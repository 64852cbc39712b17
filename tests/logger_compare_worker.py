"""Worker for test_reference_pin.py::test_logger_prints_what_the_reference_logger_prints: drives the reference utils/logger.py
(imported from the checkout in $PINN_REFERENCE_DIR, with the TF emulation for its banner) and the mirror with the same clock and calls."""
import os, sys, io, time, importlib.util, contextlib
ROOT, REF = sys.argv[1], os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")
sys.path[:0] = [ROOT + "/oracle/tf_emulation"]
def load(name, path):
    spec = importlib.util.spec_from_file_location(name, path); m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m); return m
ref = load("ref_logger", REF + "/utils/logger.py")
sys.path.insert(0, ROOT + "/pinns-tf2.0_b200/utils")
mine = load("my_logger", ROOT + "/pinns-tf2.0_b200/utils/logger.py")
hp = {"log_frequency": 10, "layers": [2, 20, 1], "tf_eps": None}
ticks = [1000.0, 1000.0, 1000.04, 1001.31, 1001.31, 1003.999, 1064.96, 1064.96, 1200.05, 4700.5, 4700.5, 4701.0]
def run(mod):
    seq = iter(ticks + [ticks[-1]] * 50)
    real = time.time
    time.time = lambda: next(seq)
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            lg = mod.Logger(hp)
            lg.set_error_fn(lambda: 0.012345)
            lg.log_train_start(object())
            lg.log_train_opt("Adam")
            lg.log_train_epoch(0, 0.45641, "")
            lg.log_train_epoch(5, 0.4, "")                 # not printed
            lg.log_train_epoch(10, 3.2e-3, "l1 = 0.5")
            lg.log_train_opt("LBFGS")
            lg.log_train_epoch(20, 1.5e-4, "", True)
            lg.log_train_epoch(30, 1.25e-5, "", True)
            lg.log_train_end(300, "done")
    finally:
        time.time = real
    return buf.getvalue().split("\n")
a, b = run(ref), run(mine)
ia = a.index("Training started"); ib = b.index("Training started")
print("\n".join(a[ia:])); print("-----"); print("\n".join(b[ib:]))
assert a[:a.index("")] == b[:b.index("")], "hyper-parameter dump differs"
assert a[ia:] == b[ib:], "log lines differ"
print("logger output identical")
