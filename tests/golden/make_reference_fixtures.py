"""Execute the REFERENCE'S OWN, UNMODIFIED Python on the golden inputs and record what it computes.

    python tests/golden/make_reference_fixtures.py            # writes tests/golden/reference_run{,_nls}.npz
    python tests/golden/make_reference_fixtures.py --check    # recompute and compare with the committed file, write nothing

Needs a checkout of the original project in $PINN_REFERENCE_DIR (the tests read the committed .npz files instead).

What runs: ``utils/neuralnetwork.py``, ``utils/custom_lbfgs.py``, ``utils/logger.py`` imported as they are, and the
``*InformedNN`` class of each example script, cut out of the script by line range (the scripts train at import time) and
executed verbatim -- ``fit()``, ``grad()``, ``get_loss_and_flat_grad()``, ``lbfgs()``, ``predict()`` are the reference's.
The one substitution is the third-party dependency that cannot be installed here: ``import tensorflow`` resolves to
``oracle/tf_emulation`` (TF-2.0 eager/tape/Keras/Adam semantics on torch CPU fp64).  ``1d-burgers/ide_cont_burgers.py`` does
not parse as shipped; its indentation is repaired in memory by ``run_reference_script.normalise_indentation`` (statements
untouched) before the class is cut out.

Every number is compared with the value the restated oracle stored in tests/golden/<problem>.npz from the same inputs, so
the file pins ``oracle/reference_port.py`` (and through it ``oracle/taylor.py`` and the CUDA path) to the reference's code.
"""
import ast
import contextlib
import importlib.util
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")
TOL = 1e-13       # observed: <= 1e-16 everywhere, including the 6-iteration fixed-step L-BFGS traces
sys.path[:0] = [os.path.join(ROOT, "oracle", "tf_emulation"), os.path.join(REF, "utils")]

import tensorflow as tf                        # noqa: E402  (the emulation)
import custom_lbfgs                            # noqa: E402  (reference)
import logger as ref_logger                    # noqa: E402  (reference)
import neuralnetwork as ref_nn                 # noqa: E402  (reference)

assert "tf_emulation" in tf.__file__ and ref_nn.__file__.startswith(REF) and custom_lbfgs.__file__.startswith(REF)


def _runner():
    spec = importlib.util.spec_from_file_location("_runner", os.path.join(ROOT, "pinns-tf2.0_b200", "run_reference_script.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def reference_class(script, name, extra=None):
    """The class statement `name` of a reference script, executed verbatim in a namespace holding what the script imports."""
    src = open(os.path.join(REF, script), encoding="utf-8").read()
    try:
        tree = ast.parse(src)
    except SyntaxError:
        src = _runner().normalise_indentation(src)
        tree = ast.parse(src)
    node = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == name][0]
    seg = "\n" * (node.lineno - 1) + "\n".join(src.split("\n")[node.lineno - 1:node.end_lineno])     # keeps line numbers
    ns = {"tf": tf, "np": np, "NeuralNetwork": ref_nn.NeuralNetwork, "lbfgs": custom_lbfgs.lbfgs, "Struct": custom_lbfgs.Struct}
    ns.update(extra or {})
    exec(compile(seg, os.path.join(REF, script), "exec"), ns)
    return ns[name]


class RecordingLogger(ref_logger.Logger):
    """The reference Logger; additionally remembers what it is asked to print."""

    def __init__(self, hp):
        with contextlib.redirect_stdout(io.StringIO()):
            super().__init__(hp)
        self.tf_losses, self.nt_losses = [], []
        self.set_error_fn(lambda: 0.0)

    def log_train_epoch(self, epoch, loss, custom="", is_iter=False):
        (self.nt_losses if is_iter else self.tf_losses).append((epoch, float(loss)))
        with contextlib.redirect_stdout(io.StringIO()):
            super().log_train_epoch(epoch, loss, custom, is_iter)


def hp_for(layers, tf_epochs=0, tf_lr=1e-3, tf_b1=0.9, tf_eps=None, nt_epochs=0, nt_lr=0.8, nt_ncorr=50, **kw):
    hp = {"layers": [int(v) for v in layers], "tf_epochs": tf_epochs, "tf_lr": tf_lr, "tf_b1": tf_b1, "tf_eps": tf_eps,
          "nt_epochs": nt_epochs, "nt_lr": nt_lr, "nt_ncorr": nt_ncorr, "log_frequency": 1}
    hp.update(kw)
    return hp


def quiet_fit(model, *args):
    out, err = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(out), contextlib.redirect_stderr(err):
        model.fit(*args)


def flat_grad_of(model, grads):
    return np.concatenate([np.asarray(g).reshape(-1) for g in grads])


def lbfgs_trace(model, closure, w0, max_iter):
    """The reference's lbfgs() driven directly so that its return values are visible; the closure is the reference's own."""
    xs = []

    def opfunc(w):
        xs.append(np.asarray(w).copy())
        return closure(w)
    cfg = custom_lbfgs.Struct()
    cfg.learningRate, cfg.maxIter, cfg.nCorrection, cfg.tolFun = 0.8, max_iter, 50, 1.0 * np.finfo(float).eps
    logged = []
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        ret = custom_lbfgs.lbfgs(opfunc, tf.convert_to_tensor(w0, dtype="float64"), cfg, custom_lbfgs.Struct(), True,
                                 lambda it, f, is_iter: logged.append((it, float(f))))
    x, f_hist, n_eval = ret
    return dict(x_eval=np.array(xs), f=np.array([float(v) for v in f_hist]), x_final=np.asarray(x), n_eval=int(n_eval),
                logged=np.array(logged), model_w=np.asarray(model.get_weights()))


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def run_burgers_inf(out, dev):
    g = np.load(os.path.join(HERE, "burgers_inf.npz"))
    cls = reference_class("1d-burgers/inf_cont_burgers.py", "BurgersInformedNN")

    def fresh(**hp):
        hp = hp_for(g["layers"], **hp)
        m = cls(hp, RecordingLogger(hp), g["X_f"], g["ub"], g["lb"], float(g["nu"]))
        m.set_weights(tf.convert_to_tensor(g["w"], dtype="float64"))
        return m
    m = fresh()
    assert m.sizes_w[0] == 40 and sum(m.sizes_w) + sum(m.sizes_b) == 3021
    loss, grads = m.grad(m.tensor(g["X_u"]), m.tensor(g["u"]))
    f2, gflat = m.get_loss_and_flat_grad(m.tensor(g["X_u"]), m.tensor(g["u"]))(tf.convert_to_tensor(g["w"], dtype="float64"))
    out["burgers_inf_loss"], out["burgers_inf_grad"] = float(loss), flat_grad_of(m, grads)
    dev["burgers_inf loss"] = abs(float(loss) - float(g["loss"])) / float(g["loss"])
    dev["burgers_inf grad"] = rel(out["burgers_inf_grad"], g["grad"])
    dev["burgers_inf flat-grad closure"] = max(rel(np.asarray(gflat), g["grad"]), abs(float(f2) - float(g["loss"])) / float(g["loss"]))
    u_pred, f_pred = m.predict(g["X_star"])
    out["burgers_inf_predict"], out["burgers_inf_residual"] = u_pred, f_pred
    dev["burgers_inf predict"] = rel(u_pred, g["predict"])
    dev["burgers_inf residual (f_model)"] = rel(f_pred, g["residual"])
    for k, lr in enumerate(g["adam_lr"]):                                   # fit() with 5 Adam epochs, no L-BFGS
        m = fresh(tf_epochs=5, tf_lr=float(lr))
        quiet_fit(m, g["X_u"], g["u"])
        losses = np.array([v for _, v in m.logger.tf_losses])
        out["burgers_inf_adam_losses_%d" % k], out["burgers_inf_adam_w_%d" % k] = losses, np.asarray(m.get_weights())
        dev["burgers_inf fit(): 5 Adam epochs lr=%g, losses" % lr] = rel(losses, g["adam_losses"][k])
        dev["burgers_inf fit(): 5 Adam epochs lr=%g, weights" % lr] = rel(out["burgers_inf_adam_w_%d" % k], g["adam_w"][k])
    m = fresh(nt_epochs=6)                                                  # fit() with 6 L-BFGS iterations, no Adam
    quiet_fit(m, g["X_u"], g["u"])
    out["burgers_inf_fit_lbfgs_w"] = np.asarray(m.get_weights())
    out["burgers_inf_fit_lbfgs_logged"] = np.array(m.logger.nt_losses)
    dev["burgers_inf fit(): 6 L-BFGS its, model weights = last EVALUATED point"] = rel(out["burgers_inf_fit_lbfgs_w"], g["lbfgs_x_eval"][-1])
    dev["burgers_inf fit(): 6 L-BFGS its, logged (it, f)"] = rel(out["burgers_inf_fit_lbfgs_logged"], g["lbfgs_logged"])
    m = fresh()
    tr = lbfgs_trace(m, m.get_loss_and_flat_grad(m.tensor(g["X_u"]), m.tensor(g["u"])), g["w"], 6)
    for k in ("x_eval", "f", "x_final", "logged"):
        out["burgers_inf_lbfgs_" + k] = tr[k]
    dev["burgers_inf lbfgs(): evaluation points"] = rel(tr["x_eval"], g["lbfgs_x_eval"])
    dev["burgers_inf lbfgs(): f history"] = rel(tr["f"], g["lbfgs_f"])
    dev["burgers_inf lbfgs(): returned x (never given to the model)"] = rel(tr["x_final"], g["lbfgs_x_final"])
    assert tr["n_eval"] == int(g["lbfgs_n_eval"]), (tr["n_eval"], int(g["lbfgs_n_eval"]))
    assert rel(tr["model_w"], tr["x_eval"][-1]) == 0.0 and rel(tr["x_final"], tr["model_w"]) > 1e-6          # last step discarded


def run_burgers_ide(out, dev):
    g = np.load(os.path.join(HERE, "burgers_ide.npz"))
    cls = reference_class("1d-burgers/ide_cont_burgers.py", "BurgersInformedNN")

    def fresh(w, **hp):
        hp = hp_for(g["layers"], **hp)
        m = cls(hp, RecordingLogger(hp), g["ub"], g["lb"])
        m.set_weights(tf.convert_to_tensor(w, dtype="float64"))
        return m
    for tag, wk, lk, gk in (("", "w", "loss", "grad"), ("2", "w2", "loss2", "grad2")):
        m = fresh(g[wk])
        m.X_u = tf.convert_to_tensor(g["X_u"], dtype="float64")              # what fit() does first (ide_cont_burgers.py:116-118)
        loss, grads = m.grad(m.tensor(g["X_u"]), m.tensor(g["u"]))
        out["burgers_ide_loss" + tag], out["burgers_ide_grad" + tag] = float(loss), flat_grad_of(m, grads)
        dev["burgers_ide%s loss" % tag] = abs(float(loss) - float(g[lk])) / float(g[lk])
        dev["burgers_ide%s grad (incl. lambda_1, lambda_2)" % tag] = rel(out["burgers_ide_grad" + tag], g[gk])
        l1, l2 = m.get_params(numpy=True)
        assert l1 == g[wk][-2] and abs(l2 - np.exp(g[wk][-1])) < 1e-18
    m = fresh(g["w"], tf_epochs=5)
    quiet_fit(m, g["X_u"], g["u"])
    out["burgers_ide_adam_losses"] = np.array([v for _, v in m.logger.tf_losses])
    out["burgers_ide_adam_w"] = np.asarray(m.get_weights())
    dev["burgers_ide fit(): 5 Adam epochs, losses"] = rel(out["burgers_ide_adam_losses"], g["adam_losses"])
    dev["burgers_ide fit(): 5 Adam epochs, weights"] = rel(out["burgers_ide_adam_w"], g["adam_w"])
    m = fresh(g["w"], nt_epochs=5)
    quiet_fit(m, g["X_u"], g["u"])
    out["burgers_ide_fit_lbfgs_w"] = np.asarray(m.get_weights())
    dev["burgers_ide fit(): 5 L-BFGS its, model weights"] = rel(out["burgers_ide_fit_lbfgs_w"], g["lbfgs_x_eval"][-1])


def run_nls(out, dev):
    g = np.load(os.path.join(HERE, "nls_inf.npz"))
    cls = reference_class("1dcomplex-schrodinger/inf_cont_schrodinger.py", "SchrodingerInformedNN")

    def fresh(**hp):
        hp = hp_for(g["layers"], **hp)
        m = cls(hp, RecordingLogger(hp), g["X_f"], g["tb"], g["ub"], g["lb"])
        m.set_weights(tf.convert_to_tensor(g["w"], dtype="float64"))
        return m
    X0 = np.concatenate([g["x0"], 0 * g["x0"]], 1)
    for tag, Xin in (("q1", g["x0"]), ("x0t0", X0)):       # the script passes x0 (N,1): quirk Q1 (inf_cont_schrodinger.py:164-167)
        m = fresh()
        with contextlib.redirect_stderr(io.StringIO()):
            loss, grads = m.grad(m.tensor(Xin), m.tensor(g["uv0"]))
        out["nls_loss_" + tag], out["nls_grad_" + tag] = float(loss), flat_grad_of(m, grads)
        dev["nls %s loss" % tag] = abs(float(loss) - float(g["loss_" + tag])) / float(g["loss_" + tag])
        dev["nls %s grad" % tag] = rel(out["nls_grad_" + tag], g["grad_" + tag])
    m = fresh(tf_epochs=3, tf_lr=0.05, tf_b1=0.99, tf_eps=0.1)
    quiet_fit(m, g["x0"], g["uv0"])
    out["nls_adam_losses"], out["nls_adam_w"] = np.array([v for _, v in m.logger.tf_losses]), np.asarray(m.get_weights())
    dev["nls fit(): 3 Adam epochs (lr .05, b1 .99, eps .1), losses"] = rel(out["nls_adam_losses"], g["adam_losses"])
    dev["nls fit(): 3 Adam epochs, weights"] = rel(out["nls_adam_w"], g["adam_w"])
    m = fresh()
    u_pred, v_pred = m.predict(g["X_star"])
    out["nls_predict"] = np.hstack([u_pred, v_pred])
    dev["nls predict"] = rel(out["nls_predict"], g["predict"])
    f_u, f_v = m.f_model()
    out["nls_residual"] = np.hstack([np.asarray(f_u), np.asarray(f_v)])
    dev["nls residual (f_model)"] = rel(out["nls_residual"], g["residual"])


def run_burgers_disc(out, dev):
    g = np.load(os.path.join(HERE, "burgers_disc.npz"))
    cls = reference_class("1d-burgers/inf_disc_burgers.py", "BurgersInformedNN")
    q = int(g["q"])

    def fresh(**hp):
        hp = hp_for(g["layers"], q=q, **hp)
        m = cls(hp, RecordingLogger(hp), np.array([float(g["dt"])]), g["x_1"], g["lb"], g["ub"], float(g["nu"]),
                g["IRK"], np.zeros(q))          # IRK table float32, as np.float32(np.loadtxt(..)) in burgersutil.py:57
        m.set_weights(tf.convert_to_tensor(g["w"], dtype="float64"))
        return m
    m = fresh()
    m.dummy_x0_tf = tf.ones([g["x_0"].shape[0], m.q], dtype=m.dtype)          # what fit() does first (inf_disc_burgers.py:117-119)
    loss, grads = m.grad(m.tensor(g["x_0"]), m.tensor(g["u_0"]))
    out["burgers_disc_loss"], out["burgers_disc_grad"] = float(loss), flat_grad_of(m, grads)
    dev["burgers_disc loss"] = abs(float(loss) - float(g["loss"])) / float(g["loss"])
    dev["burgers_disc grad"] = rel(out["burgers_disc_grad"], g["grad"])
    out["burgers_disc_predict"] = np.asarray(m.predict(g["x_star"]))
    dev["burgers_disc predict"] = rel(out["burgers_disc_predict"], g["predict"])
    m = fresh(tf_epochs=3, tf_eps=1e-8)
    quiet_fit(m, g["x_0"], g["u_0"])
    out["burgers_disc_adam_losses"], out["burgers_disc_adam_w"] = np.array([v for _, v in m.logger.tf_losses]), np.asarray(m.get_weights())
    dev["burgers_disc fit(): 3 Adam epochs, losses"] = rel(out["burgers_disc_adam_losses"], g["adam_losses"])
    dev["burgers_disc fit(): 3 Adam epochs, weights"] = rel(out["burgers_disc_adam_w"], g["adam_w"])
    # The script's L-BFGS closure evaluates the loss OUTSIDE its tape (inf_disc_burgers.py:103-107): every gradient is None and
    # tf.reshape(None) raises, i.e. the shipped nt_epochs=1000 phase cannot run.  Recorded as a fact about the reference.
    m = fresh(nt_epochs=2)
    try:
        quiet_fit(m, g["x_0"], g["u_0"])
        out["burgers_disc_lbfgs_runs"] = np.array(1)
    except ValueError as exc:
        assert "None values not supported" in str(exc)
        out["burgers_disc_lbfgs_runs"] = np.array(0)


def run_burgers_ide_disc(out, dev):
    """1d-burgers/ide_disc_burgers.py:48-203.  The SCRIPT cannot run as shipped (Logger(frequency=10) :225; np.asscalar in its
    prep_data branch), the class can: its own fit() (Adam loop :163-168, L-BFGS closure :171-185 -- here the loss IS taken inside
    the tape) and predict() run here.  fit() reads the script-level `hp`, which is supplied in the class namespace."""
    g = np.load(os.path.join(HERE, "burgers_ide_disc.npz"))
    q = int(g["q"])

    def fresh(**hpkw):
        hp = hp_for(g["layers"], **hpkw)
        cls = reference_class("1d-burgers/ide_disc_burgers.py", "BurgersInformedNN", {"hp": hp})
        return cls(hp, RecordingLogger(hp), float(g["dt"]), g["lb"], g["ub"], q, g["IRK_alpha"], g["IRK_beta"])
    t64 = lambda a: tf.convert_to_tensor(a, dtype="float64")
    for tag in ("", "2"):
        m = fresh()
        m.lambda_1 = tf.Variable([0.0], dtype=m.dtype)                      # what fit() creates (:151-152) before set_weights can run
        m.lambda_2 = tf.Variable([-6.0], dtype=m.dtype)
        m.set_weights(t64(g["w" + tag]))
        m.dummy_x_0, m.dummy_x_1 = m.createDummy(t64(g["x_0"])), m.createDummy(t64(g["x_1"]))       # :155-156
        loss, grads = m.grad(t64(g["x_0"]), t64(g["u_0"]), t64(g["x_1"]), t64(g["u_1"]))
        out["burgers_ide_disc_loss" + tag], out["burgers_ide_disc_grad" + tag] = float(loss), flat_grad_of(m, grads)
        dev["burgers_ide_disc%s loss" % tag] = abs(float(loss) - float(g["loss" + tag])) / float(g["loss" + tag])
        dev["burgers_ide_disc%s grad (incl. lambda_1, lambda_2)" % tag] = rel(out["burgers_ide_disc_grad" + tag], g["grad" + tag])
    U0, U1 = m.predict(g["x_star"])
    out["burgers_ide_disc_predict_U0"], out["burgers_ide_disc_predict_U1"] = np.asarray(U0), np.asarray(U1)
    dev["burgers_ide_disc predict U_0, U_1"] = max(rel(np.asarray(U0), g["predict_U0"]), rel(np.asarray(U1), g["predict_U1"]))
    # fit() always starts from lambda = (0, -6) and the net's own initial weights, so it is compared from THAT start:
    m = fresh(tf_epochs=3, nt_epochs=4)
    m.model.layers[1].set_weights(m.model.layers[1].get_weights())           # no-op; the net keeps its seeded initial weights
    w_net0 = np.asarray(ref_nn.NeuralNetwork.get_weights(m, convert_to_tensor=False))
    quiet_fit(m, g["x_0"], g["u_0"], g["x_1"], g["u_1"])
    out["burgers_ide_disc_fit_w0"] = np.concatenate([w_net0, [0.0, -6.0]])
    out["burgers_ide_disc_fit_adam_losses"] = np.array([v for _, v in m.logger.tf_losses])
    out["burgers_ide_disc_fit_lbfgs_logged"] = np.array(m.logger.nt_losses)
    out["burgers_ide_disc_fit_w"] = np.asarray(m.get_weights())
    # the same schedule with the restated oracle from the same start
    sys.path.insert(0, ROOT)
    from oracle import reference_port as rp
    pb = rp.BurgersDiscreteIdentification([int(v) for v in g["layers"]], g["lb"], g["ub"], float(g["dt"]), g["x_0"], g["u_0"],
                                           g["x_1"], g["u_1"], g["IRK_alpha"], g["IRK_beta"])
    wa, la, _ = rp.adam_train(pb, out["burgers_ide_disc_fit_w0"], 3, lr=1e-3)
    tr = rp.lbfgs_fixed_step(lambda z: rp.loss_and_flat_grad(pb, z), wa, max_iter=4, learning_rate=0.8, n_correction=50,
                             tol_fun=np.finfo(float).eps)
    dev["burgers_ide_disc fit(): 3 Adam epochs, losses"] = rel(out["burgers_ide_disc_fit_adam_losses"], la)
    dev["burgers_ide_disc fit(): + 4 L-BFGS its, logged f"] = rel(out["burgers_ide_disc_fit_lbfgs_logged"][:, 1], np.array(tr.logged)[:, 1])
    dev["burgers_ide_disc fit(): final model weights"] = rel(out["burgers_ide_disc_fit_w"], tr.x_eval[-1])


def run_burgers_default_schedule(out, dev):
    """The reference's default training run (1d-burgers/inf_cont_burgers.py:27-43: N_u=100, N_f=10000, 100 Adam epochs at 0.03,
    200 fixed-step L-BFGS iterations at 0.8, 50 corrections) through ITS fit(), from the initial weights and data of
    tests/golden/burgers_accuracy.npz; compared with the oracle's loss curves, final weights and rel. L2 error stored there."""
    g = np.load(os.path.join(HERE, "burgers_accuracy.npz"))
    cls = reference_class("1d-burgers/inf_cont_burgers.py", "BurgersInformedNN")
    hp = hp_for([2] + [20] * 8 + [1], tf_epochs=100, tf_lr=0.03, nt_epochs=200)
    m = cls(hp, RecordingLogger(hp), g["X_f"], g["ub"], g["lb"], 0.01 / np.pi)
    m.set_weights(tf.convert_to_tensor(g["w0"], dtype="float64"))
    quiet_fit(m, g["X_u"], g["u"])
    adam = np.array([v for _, v in m.logger.tf_losses])
    lb_log = np.array([v for _, v in m.logger.nt_losses])               # f after iterations 1..199 (the last one is not logged)
    w = np.asarray(m.get_weights())
    u_pred, _ = m.predict(g["X_star"].astype(np.float64))
    err = float(np.linalg.norm(g["u_star"].astype(np.float64) - u_pred) / np.linalg.norm(g["u_star"].astype(np.float64)))
    out["schedule_adam_losses"], out["schedule_lbfgs_logged_f"], out["schedule_w"], out["schedule_error"] = adam, lb_log, w, err
    # The fixed-step L-BFGS iteration is chaotic: rounding-level differences between two fp64 implementations of the SAME
    # algorithm grow about tenfold every ten iterations (1e-16 at iteration 1, 1e-11 at 40, 1e-7 at 80, 1e-3 at 100), so only a
    # prefix can agree tightly; the end point agrees in magnitude.  The same holds between the CUDA path and the oracle.
    f_dev = np.abs(lb_log - g["oracle_lbfgs_f"][1:]) / g["oracle_lbfgs_f"][1:]
    out["schedule_lbfgs_f_deviation"] = f_dev
    dev["default schedule: 100 Adam losses"] = (rel(adam, g["oracle_adam_losses"]), 1e-13)
    dev["default schedule: L-BFGS f, iterations 1..40"] = (float(f_dev[:40].max()), 1e-9)
    dev["default schedule: L-BFGS f, iteration 199 (chaotic tail)"] = (float(f_dev[-1]), 0.25)
    dev["default schedule: final model weights (chaotic tail)"] = (rel(w, g["oracle_w"]), 0.05)
    dev["default schedule: rel. L2 error of u %.4f vs %.4f" % (err, float(g["oracle_error"]))] = \
        (abs(err - float(g["oracle_error"])) / float(g["oracle_error"]), 0.25)
    return dev


def main():
    out, dev = {}, {}
    sched = run_burgers_default_schedule(out, {})
    for k, (v, tol) in sched.items():
        print("%-70s rel. deviation from the oracle's value: %.2e (bound %.0e)" % (k, v, tol))
        assert v <= tol, k
    for fn in (run_burgers_inf, run_burgers_ide, run_nls, run_burgers_disc, run_burgers_ide_disc):
        fn(out, dev)
    width = max(len(k) for k in dev)
    for k, v in dev.items():
        print("%-*s  rel. deviation from the oracle's golden value: %.2e" % (width, k, v))
    worst = max(dev.values())
    print("worst: %.2e; discrete-time L-BFGS phase runs in the reference: %s" % (worst, bool(out["burgers_disc_lbfgs_runs"])))
    assert worst < TOL, "the restated oracle and the reference's own code disagree"
    # two files, each under 1 MB: the Schrodinger arrays (nls_*) apart from the rest
    files = {os.path.join(HERE, "reference_run.npz"): {k: v for k, v in out.items() if not k.startswith("nls_")},
             os.path.join(HERE, "reference_run_nls.npz"): {k: v for k, v in out.items() if k.startswith("nls_")}}
    if "--check" in sys.argv:
        old = {}
        for path in files:
            with np.load(path) as f:
                old.update({k: f[k] for k in f.files})
        assert sorted(old) == sorted(out), "fixture keys changed"
        for k in out:
            if k in ("schedule_adam_losses",) or not k.startswith("schedule_"):      # the chaotic tail may differ between machines
                assert rel(out[k], old[k]) < 1e-12 or np.array_equal(out[k], old[k]), k
        print("committed fixture reproduced")
    else:
        for path, part in files.items():
            np.savez_compressed(path, **{k: np.asarray(v) for k, v in part.items()})
            print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
