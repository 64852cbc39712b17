"""CPU: the HOST-side mirror (pinns-tf2.0_b200/utils/{neuralnetwork,custom_lbfgs,logger}.py + the tensorflow shim) driven end to
end without a GPU.  ``pinn_cabi.Pinn`` is replaced IN THE TEST PROCESS by tests/oracle_backend.OraclePinn (the product itself has
no CPU path), so what is under test is everything above the C ABI: PDE recognition, what is uploaded when, the epoch loops and
their logger traffic, lazy losses, the flat-parameter bridge incl. lambda_1/lambda_2, the L-BFGS wrapper's arguments and
return values, predict()/get_params() shapes.

With a checkout of the original project (PINN_REFERENCE_DIR) the classes are the reference's OWN class statements, cut out
of its scripts and executed verbatim on the mirror; the results must equal tests/golden/reference_run.npz -- what the same
class code produced on the emulated TensorFlow.  A portable variant with reference-style subclasses runs everywhere."""
import ast
import importlib.util
import io
import os
import re
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

from conftest import PKG, ROOT, load_golden, load_reference_run

REF = os.environ.get("PINN_REFERENCE_DIR", "")      # a checkout of the original project, if any
sys.path.insert(0, os.path.join(PKG, "shims"))


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.fixture()
def mirror(monkeypatch):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import pinn_cabi
    import oracle_backend
    monkeypatch.setattr(pinn_cabi, "Pinn", oracle_backend.OraclePinn)
    oracle_backend.OraclePinn.created.clear()
    import custom_lbfgs
    import logger
    import neuralnetwork
    import tensorflow as tf
    assert "shims" in tf.__file__ and neuralnetwork.__file__.startswith(PKG)
    return {"nn": neuralnetwork, "Logger": logger.Logger, "tf": tf, "lbfgs": custom_lbfgs, "backend": oracle_backend.OraclePinn}


def hp_for(layers, **kw):
    hp = {"layers": [int(v) for v in layers], "tf_epochs": 0, "tf_lr": 1e-3, "tf_b1": 0.9, "tf_eps": None, "nt_epochs": 0,
          "nt_lr": 0.8, "nt_ncorr": 50, "log_frequency": 1}
    hp.update(kw)
    return hp


def reference_class(script, name, ns):
    """The class statement of a reference script, executed verbatim on the mirror (namespace = what the script imports)."""
    src = open(os.path.join(REF, script), encoding="utf-8").read()
    try:
        tree = ast.parse(src)
    except SyntaxError:
        spec = importlib.util.spec_from_file_location("_runner", os.path.join(PKG, "run_reference_script.py"))
        runner = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(runner)
        src = runner.normalise_indentation(src)
        tree = ast.parse(src)
    node = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == name][0]
    seg = "\n" * (node.lineno - 1) + "\n".join(src.split("\n")[node.lineno - 1:node.end_lineno])
    exec(compile(seg, os.path.join(REF, script), "exec"), ns)
    return ns[name]


def logged_losses(text, tag):
    return np.array([float(m) for m in re.findall(tag + r" = +\d+ .*?loss = (\S+)", text)])


def fit_quietly(pinn, *args):
    buf = io.StringIO()
    with redirect_stdout(buf):
        pinn.fit(*args)
    return buf.getvalue()


def fmt4(values):
    return np.array([float("%.4e" % v) for v in values])


needs_ref = pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")


@needs_ref
def test_reference_burgers_inference_class_on_the_mirror(mirror):
    g, r = load_golden("burgers_inf"), load_reference_run()
    ns = {"tf": mirror["tf"], "np": np, "NeuralNetwork": mirror["nn"].NeuralNetwork}
    cls = reference_class("1d-burgers/inf_cont_burgers.py", "BurgersInformedNN", ns)

    def fresh(**kw):
        hp = hp_for(g["layers"], **kw)
        with redirect_stdout(io.StringIO()):
            lg = mirror["Logger"](hp)
        lg.set_error_fn(lambda: 0.0)
        p = cls(hp, lg, g["X_f"], g["ub"], g["lb"], float(g["nu"]))
        p._w0 = g["w"].copy()
        return p
    p = fresh()
    u_pred, f_pred = p.predict(g["X_star"])                                   # quirk Q3: f on the TRAINING points
    assert rel(u_pred, r["burgers_inf_predict"]) < 1e-12 and rel(f_pred, r["burgers_inf_residual"]) < 1e-12
    loss, grads = p.grad(g["X_u"], g["u"])
    assert abs(float(loss) - float(r["burgers_inf_loss"])) <= 1e-12 * float(r["burgers_inf_loss"])
    assert len(grads) == 18 and rel(np.concatenate([np.asarray(v).reshape(-1) for v in grads]), r["burgers_inf_grad"]) < 1e-12
    assert p.get_params(numpy=True) == float(g["nu"])
    for k, lr in enumerate(g["adam_lr"]):
        p = fresh(tf_epochs=5, tf_lr=float(lr))
        out = fit_quietly(p, g["X_u"], g["u"])
        assert rel(p.get_weights().numpy(), r["burgers_inf_adam_w_%d" % k]) < 1e-12
        assert np.array_equal(logged_losses(out, "tf_epoch"), fmt4(r["burgers_inf_adam_losses_%d" % k]))
        assert "Training finished (epoch 5)" in out
    p = fresh(nt_epochs=6)
    out = fit_quietly(p, g["X_u"], g["u"])
    assert rel(p.get_weights().numpy(), r["burgers_inf_fit_lbfgs_w"]) < 1e-12      # last EVALUATED point, not lbfgs's x
    assert np.array_equal(logged_losses(out, "nt_epoch"), fmt4(r["burgers_inf_fit_lbfgs_logged"][:, 1]))
    assert [int(v) for v in re.findall(r"nt_epoch = +(\d+)", out)] == [int(v) for v in r["burgers_inf_fit_lbfgs_logged"][:, 0]]
    call = [c for c in mirror["backend"].created[-1].calls if c[0] == "lbfgs"][0]
    assert call[1:6] == (6, 0.8, 50, np.finfo(float).eps, 1e-19)                   # maxIter, lr, nCorrection, tolFun, tolX
    # the module-level lbfgs() keeps the reference's return contract
    p = fresh()
    closure = p.get_loss_and_flat_grad(g["X_u"], g["u"])
    cfg = mirror["lbfgs"].Struct()
    cfg.learningRate, cfg.maxIter, cfg.nCorrection, cfg.tolFun = 0.8, 6, 50, np.finfo(float).eps
    x, f_hist, n_eval = mirror["lbfgs"].lbfgs(closure, p.get_weights(), cfg, mirror["lbfgs"].Struct(), True, lambda *a: None)
    assert rel(np.asarray(x), r["burgers_inf_lbfgs_x_final"]) < 1e-12 and n_eval == 6
    f0, g0 = closure(g["w"])
    assert abs(float(f0) - float(r["burgers_inf_loss"])) <= 1e-12 * float(r["burgers_inf_loss"]) and rel(np.asarray(g0), r["burgers_inf_grad"]) < 1e-12


@needs_ref
def test_reference_identification_class_on_the_mirror(mirror):
    g, r = load_golden("burgers_ide"), load_reference_run()
    ns = {"tf": mirror["tf"], "np": np, "NeuralNetwork": mirror["nn"].NeuralNetwork}
    cls = reference_class("1d-burgers/ide_cont_burgers.py", "BurgersInformedNN", ns)

    def fresh(**kw):
        hp = hp_for(g["layers"], **kw)
        with redirect_stdout(io.StringIO()):
            lg = mirror["Logger"](hp)
        lg.set_error_fn(lambda: 0.0)
        p = cls(hp, lg, g["ub"], g["lb"])
        p._w0 = g["w"][:-2].copy()                                            # lambda_1 = 0, lambda_2 = -6 come from the class
        return p
    p = fresh(tf_epochs=5)
    out = fit_quietly(p, g["X_u"], g["u"])
    w = p.get_weights().numpy()
    assert w.shape == (3023,) and rel(w, r["burgers_ide_adam_w"]) < 1e-12
    assert np.array_equal(logged_losses(out, "tf_epoch"), fmt4(r["burgers_ide_adam_losses"]))
    l1, l2 = p.get_params(numpy=True)
    assert l1 == w[-2] and abs(l2 - np.exp(w[-1])) < 1e-18 and len(p.wrap_training_variables()) == 20
    p = fresh(nt_epochs=5)
    fit_quietly(p, g["X_u"], g["u"])
    assert rel(p.get_weights().numpy(), r["burgers_ide_fit_lbfgs_w"]) < 1e-12


@needs_ref
def test_reference_schrodinger_class_on_the_mirror(mirror):
    g, r = load_golden("nls_inf"), load_reference_run()
    ns = {"tf": mirror["tf"], "np": np, "NeuralNetwork": mirror["nn"].NeuralNetwork}
    cls = reference_class("1dcomplex-schrodinger/inf_cont_schrodinger.py", "SchrodingerInformedNN", ns)
    hp = hp_for(g["layers"], tf_epochs=3, tf_lr=0.05, tf_b1=0.99, tf_eps=0.1)
    with redirect_stdout(io.StringIO()):
        lg = mirror["Logger"](hp)
    lg.set_error_fn(lambda: 0.0)
    p = cls(hp, lg, g["X_f"], g["tb"], g["ub"], g["lb"])
    p._w0 = g["w"].copy()
    u_pred, v_pred = p.predict(g["X_star"])
    assert rel(np.hstack([u_pred, v_pred]), r["nls_predict"]) < 1e-12
    out = fit_quietly(p, g["x0"], g["uv0"])                                    # (N,1) x0: quirk Q1 travels through the mirror
    assert rel(p.get_weights().numpy(), r["nls_adam_w"]) < 1e-12
    assert np.array_equal(logged_losses(out, "tf_epoch"), fmt4(r["nls_adam_losses"]))
    assert mirror["backend"].created[-1].X.shape == (50, 1)


@needs_ref
def test_reference_discrete_time_class_on_the_mirror(mirror):
    g, r = load_golden("burgers_disc"), load_reference_run()
    ns = {"tf": mirror["tf"], "np": np, "NeuralNetwork": mirror["nn"].NeuralNetwork}
    cls = reference_class("1d-burgers/inf_disc_burgers.py", "BurgersInformedNN", ns)
    hp = hp_for(g["layers"], q=int(g["q"]), tf_epochs=3, tf_eps=1e-8)
    with redirect_stdout(io.StringIO()):
        lg = mirror["Logger"](hp)
    lg.set_error_fn(lambda: 0.0)
    p = cls(hp, lg, np.array([float(g["dt"])]), g["x_1"], g["lb"], g["ub"], float(g["nu"]), g["IRK"], np.zeros(int(g["q"])))
    p._w0 = g["w"].copy()
    out = fit_quietly(p, g["x_0"], g["u_0"])
    assert rel(p.get_weights().numpy(), r["burgers_disc_adam_w"]) < 1e-12
    assert np.array_equal(logged_losses(out, "tf_epoch"), fmt4(r["burgers_disc_adam_losses"]))
    p.set_weights(g["w"])
    assert rel(np.asarray(p.predict(g["x_star"])).reshape(-1), r["burgers_disc_predict"]) < 1e-12


def test_reference_style_subclass_on_the_mirror_portable(mirror):
    """Runs everywhere (no reference checkout needed): a subclass written like the script's, compared with the oracle's golden
    Adam trajectory and L-BFGS trace."""
    tf, NeuralNetwork = mirror["tf"], mirror["nn"].NeuralNetwork
    g = load_golden("burgers_inf")

    class BurgersInformedNN(NeuralNetwork):              # 1d-burgers/inf_cont_burgers.py:48-98 (tape bodies elided)
        def __init__(self, hp, logger, X_f, ub, lb, nu):
            super().__init__(hp, logger, ub, lb)
            self.nu = nu
            self.x_f = self.tensor(X_f[:, 0:1])
            self.t_f = self.tensor(X_f[:, 1:2])

        def f_model(self):
            with tf.GradientTape(persistent=True):                               # replaced by the native path, never executed
                raise AssertionError("tape body executed")

        def get_params(self, numpy=False):
            return self.nu

    hp = hp_for(g["layers"], tf_epochs=5, nt_epochs=6, log_frequency=2)
    with redirect_stdout(io.StringIO()):
        lg = mirror["Logger"](hp)
    lg.set_error_fn(lambda: 0.5)
    p = BurgersInformedNN(hp, lg, g["X_f"], g["ub"], g["lb"], float(g["nu"]))
    p._w0 = g["w"].copy()
    out = fit_quietly(p, g["X_u"], g["u"])
    assert np.array_equal(logged_losses(out, "tf_epoch"), fmt4(g["adam_losses"][0][::2]))     # only every 2nd epoch is fetched/printed
    assert "Training finished (epoch 11)" in out and "error = 5.0000e-01" in out              # quirk Q4: the PLANNED epoch count
    backend = mirror["backend"].created[-1]
    assert [c[0] for c in backend.calls].count("adam_step") == 5 and all(c[5] is False for c in backend.calls if c[0] == "adam_step")
    assert [c for c in backend.calls if c[0] == "set_data"] == [("set_data", (100, 2), (100, 1))]      # uploaded once
    # Adam moved the weights first, so the L-BFGS part is compared through the oracle from that point
    from oracle import reference_port as rp
    pb = rp.BurgersInference(hp["layers"], g["lb"], g["ub"], float(g["nu"]), g["X_f"], g["X_u"], g["u"])
    tr = rp.lbfgs_fixed_step(lambda x: rp.loss_and_flat_grad(pb, x), g["adam_w"][0], max_iter=6, learning_rate=0.8,
                             n_correction=50, tol_fun=np.finfo(float).eps)
    assert rel(p.get_weights().numpy(), tr.x_eval[-1]) < 1e-10


@needs_ref
@pytest.mark.parametrize("script,hp_extra,expect", [
    ("1d-burgers/inf_cont_burgers.py", {"N_u": 50, "N_f": 400, "layers": [2, 20, 20, 20, 20, 20, 20, 20, 20, 1]}, "Training finished (epoch 6)"),
    ("1dcomplex-schrodinger/inf_cont_schrodinger.py", {"N_0": 20, "N_b": 20, "N_f": 200, "layers": [2, 16, 16, 2], "tf_b1": 0.99, "tf_eps": 0.1},
     "Training finished (epoch 6)"),
    ("1d-burgers/ide_cont_burgers.py", {"N_u": 60, "layers": [2, 20, 20, 20, 20, 20, 20, 20, 20, 1]}, "l2_noise"),
    ("1d-burgers/inf_disc_burgers.py", {"N_n": 40, "q": 8, "layers": [1, 12, 12, 9], "tf_eps": 1e-8}, "Training finished (epoch 6)"),
])
def test_unmodified_scripts_complete_on_the_mirror(mirror, monkeypatch, tmp_path, script, hp_extra, expect):
    """The whole unmodified script (its own hp handling, prep_data, model class, fit, predict, error function, plotting call)
    through pinns-tf2.0_b200/run_reference_script.py, with the native handle replaced by the oracle stand-in: exercises every
    host-side line a user's run touches, incl. the result artefacts."""
    import json
    spec = importlib.util.spec_from_file_location("_runner_main", os.path.join(PKG, "run_reference_script.py"))
    runner = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(runner)
    hp = {"tf_epochs": 3, "tf_lr": 0.01, "tf_b1": 0.9, "tf_eps": None, "nt_epochs": 3, "nt_lr": 0.8, "nt_ncorr": 50, "log_frequency": 1}
    hp.update(hp_extra)
    (tmp_path / "hp.json").write_text(json.dumps(hp))
    monkeypatch.setenv("PINN_RESULTS_ROOT", str(tmp_path))
    monkeypatch.setattr(sys, "argv", list(sys.argv))
    monkeypatch.setattr(sys, "path", list(sys.path))
    cwd = os.getcwd()
    for m in ("burgersutil", "schrodingerutil", "plotting"):
        sys.modules.pop(m, None)
    buf = io.StringIO()
    try:
        with redirect_stdout(buf):
            rc = runner.main(["run_reference_script.py", os.path.join(REF, script), str(tmp_path / "hp.json")])
    finally:
        os.chdir(cwd)
    out = buf.getvalue()
    runs = 2 if "ide_cont" in script else 1                     # the identification script trains twice ("clean" and "noisy")
    assert rc == 0 and expect in out and out.count("tf_epoch = ") == 3 * runs and out.count("nt_epoch = ") == 2 * runs, out[-1500:]
    res = [os.path.join(d, f) for d, _, fs in os.walk(str(tmp_path)) for f in fs]
    if "ide_cont" not in script:                                 # that script plots without save_path (plt.show() in the reference)
        assert any(f.endswith("hp.json") and "results" in f for f in res) and any(f.endswith("fields.npz") for f in res), res


def test_lazy_loss_is_current_or_an_error_never_stale(mirror):
    """tf_optimization_step returns a loss that is read back from the device only on use; reading the loss of an EARLIER step
    after a newer one was enqueued raises instead of returning the newer step's value."""
    g = load_golden("burgers_inf")
    NeuralNetwork = mirror["nn"].NeuralNetwork

    class BurgersInformedNN(NeuralNetwork):
        def __init__(self, hp, logger, X_f, ub, lb, nu):
            super().__init__(hp, logger, ub, lb)
            self.nu = nu
            self.x_f, self.t_f = self.tensor(X_f[:, 0:1]), self.tensor(X_f[:, 1:2])

    hp = hp_for(g["layers"])
    with redirect_stdout(io.StringIO()):
        p = BurgersInformedNN(hp, mirror["Logger"](hp), g["X_f"], g["ub"], g["lb"], float(g["nu"]))
    p._w0 = g["w"].copy()
    l0 = p.tf_optimization_step(g["X_u"], g["u"])
    assert abs(float(l0) - g["adam_losses"][0][0]) <= 1e-12 * g["adam_losses"][0][0]      # read before the next step: correct
    l1 = p.tf_optimization_step(g["X_u"], g["u"])
    l2 = p.tf_optimization_step(g["X_u"], g["u"])
    assert "%.6e" % l2 == "%.6e" % g["adam_losses"][0][2] and float(l0) == float(l0)       # resolved values stay valid
    with pytest.raises(RuntimeError):
        float(l1)                                                                          # never read, now stale
