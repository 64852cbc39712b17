"""Worker for test_reference_pin.py::test_lbfgs_control_flow_equals_the_reference: drives the reference's own
utils/custom_lbfgs.lbfgs (on the TF emulation) and oracle.reference_port.lbfgs_fixed_step with the same synthetic objectives,
chosen so that every exit of the routine is taken: maxIter, maxEval, optimality at the start, optimality later, no progress
along the direction, step below tolX, f change below tolX, rejected curvature pairs, history overflow (nCorrection)."""
import contextlib
import io
import os
import sys

import numpy as np

ROOT, REF = sys.argv[1], os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")
sys.path[:0] = [ROOT + "/oracle/tf_emulation", REF + "/utils", ROOT]
import tensorflow as tf                 # noqa: E402  (emulation)
import custom_lbfgs                     # noqa: E402  (reference)
from oracle import reference_port as rp  # noqa: E402

assert custom_lbfgs.__file__.startswith(REF)


def run_reference(fn, x0, **cfgkw):
    cfg = custom_lbfgs.Struct()
    for k, v in cfgkw.items():
        setattr(cfg, k, v)
    xs, logged, said = [], [], io.StringIO()

    def opfunc(x):
        xs.append(np.asarray(x).copy())
        f, g = fn(np.asarray(x))
        return tf.convert_to_tensor(np.float64(f)), tf.convert_to_tensor(np.asarray(g, dtype=np.float64))
    state = custom_lbfgs.Struct()
    with contextlib.redirect_stdout(said):
        ret = custom_lbfgs.lbfgs(opfunc, tf.convert_to_tensor(np.asarray(x0, dtype=np.float64)), cfg, state, True,
                                 lambda it, f, is_iter: logged.append((it, float(f))))
    return ret, xs, logged, said.getvalue(), state


REASON_TEXT = {"optimality": "optimality condition below tolFun", "initial optimality": "optimality condition below tolFun",
               "no progress along direction": "Can not make progress along direction.", "step below tolX": "step size below tolX",
               "f change below tolX": "function value changing less than tolX", "max evaluations": "max nb of function evals",
               "max iterations": ""}


def compare(name, fn, x0, expect_reason, **kw):
    port = rp.lbfgs_fixed_step(lambda x: fn(x), np.asarray(x0, dtype=np.float64), max_iter=kw["maxIter"],
                               learning_rate=kw.get("learningRate", 1.0), n_correction=kw.get("nCorrection", 100),
                               tol_fun=kw.get("tolFun", 1e-5), tol_x=kw.get("tolX", 1e-19), max_eval=kw.get("maxEval"))
    ret, xs, logged, said, state = run_reference(fn, x0, verbose=True, **kw)
    assert port.stop_reason == expect_reason, (name, port.stop_reason)
    assert REASON_TEXT[expect_reason] in said, (name, said)
    assert len(xs) == len(port.x_eval) == port.n_eval, (name, len(xs), port.n_eval)
    for a, b in zip(xs, port.x_eval):
        assert np.allclose(a, b, rtol=1e-8, atol=1e-13), name      # rounding differences grow along a fixed-step run
    if expect_reason == "initial optimality":
        assert len(ret) == 2                                            # (x, f_hist) only, custom_lbfgs.py:76
        print("%-34s %-28s iterations %3d evaluations %3d" % (name, expect_reason, 0, 1))
        return
    x, f_hist, n_eval = ret
    assert n_eval == port.n_eval and np.allclose(np.asarray(x), port.x_final, rtol=1e-8, atol=1e-13), name
    assert np.allclose([float(v) for v in f_hist], port.f_hist, rtol=1e-8, atol=1e-300), name
    assert [it for it, _ in logged] == [it for it, _ in port.logged], (name, logged, port.logged)
    assert state.nIter == port.n_iter, (name, state.nIter, port.n_iter)
    if port.hist_len:
        assert len(state.old_dirs) <= kw.get("nCorrection", 100)
    print("%-34s %-28s iterations %3d evaluations %3d" % (name, expect_reason, port.n_iter, port.n_eval))


A = np.diag([1.0, 10.0, 100.0])
quad = lambda x: (0.5 * float(x @ A @ x), A @ x)
rng = np.random.default_rng(0)
B = rng.standard_normal((12, 12)); B = np.eye(12) + 0.02 * (B @ B.T)            # well conditioned: converges in a few steps
quad12 = lambda x: (0.5 * float(x @ B @ x), B @ x)
x12 = rng.standard_normal(12)
lin = lambda x: (float(np.sum(x)), np.ones_like(x))                      # y = 0: every curvature pair rejected (ys <= 1e-10)

compare("quadratic, maxIter", quad, [1.0, 1.0, 1.0], "max iterations", maxIter=4, learningRate=0.05, tolFun=1e-30)
compare("quadratic, maxEval", quad, [1.0, 1.0, 1.0], "max evaluations", maxIter=40, maxEval=3, learningRate=0.05, tolFun=1e-30)
compare("zero gradient at start", quad, [0.0, 0.0, 0.0], "initial optimality", maxIter=5)
compare("optimality after a few steps", quad12, x12, "optimality", maxIter=200, learningRate=1.0, tolFun=1e-6)
compare("history overflow (nCorrection=3)", quad12, x12, "max iterations", maxIter=15, learningRate=0.5, nCorrection=3, tolFun=1e-30)
compare("ascent direction", lambda x: (-0.5 * float(x @ x), -x), [1.0, 2.0], "max iterations", maxIter=3, learningRate=0.1, tolFun=1e-30)
compare("linear objective, no curvature", lin, [0.0, 0.0], "max iterations", maxIter=6, learningRate=0.3, tolFun=1e-30)
compare("step below tolX", quad, [1e-3, 1e-3, 1e-3], "step below tolX", maxIter=50, learningRate=1e-12, tolFun=1e-30, tolX=1e-9)
compare("f change below tolX", lambda x: (1.0, np.array([0.3, -0.2])), [0.0, 0.0], "f change below tolX", maxIter=50, learningRate=0.5,
        tolFun=1e-30, tolX=1e-7)
late = lambda x: (1.0, np.array([1.0, 0.0])) if x[0] == 0.0 else (0.5, np.array([1e-4, 0.0]))
compare("no progress along direction (it 2)", late, [0.0, 0.0], "no progress along direction", maxIter=9, learningRate=1.0,
        tolFun=1e-9, tolX=1e-5)
# The same exit at the FIRST iteration is a crash in the reference: `t` is only assigned after the direction test, and the
# state is saved unconditionally (custom_lbfgs.py:154-156 vs :233) -> UnboundLocalError.  The port (and the device L-BFGS)
# report "no progress" instead; recorded here so that the difference is a known one.
flat = lambda x: (1.0, np.array([1e-3, 0.0]))
port = rp.lbfgs_fixed_step(flat, np.zeros(2), max_iter=9, learning_rate=1.0, tol_fun=1e-9, tol_x=1e-5)
assert port.stop_reason == "no progress along direction" and port.n_iter == 1 and port.n_eval == 1
try:
    run_reference(flat, [0.0, 0.0], maxIter=9, learningRate=1.0, tolFun=1e-9, tolX=1e-5)
    raise SystemExit("the reference was expected to fail with UnboundLocalError")
except UnboundLocalError:
    print("%-34s reference raises UnboundLocalError (t unassigned); port reports 'no progress'" % "no progress at iteration 1")
print("lbfgs control flow identical")
