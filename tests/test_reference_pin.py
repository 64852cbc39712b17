"""CPU: the oracle is pinned to what the REFERENCE'S OWN Python computes.

tests/golden/reference_run.npz was produced by tests/golden/make_reference_fixtures.py: the reference's unmodified
utils/neuralnetwork.py, utils/custom_lbfgs.py, utils/logger.py and the *InformedNN classes of its scripts, executed in the
build container on the TF-2.0 API emulation of oracle/tf_emulation (TensorFlow itself cannot be installed).  Here:
  * the committed reference run equals the oracle's golden values (the ones every GPU parity test compares against);
  * where a checkout of the original project is given (PINN_REFERENCE_DIR), the run is repeated live and must reproduce the committed file;
  * the emulation's tape/Keras/Adam semantics are unit-tested against TensorFlow's documented behaviour.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden, load_reference_run

REF = os.environ.get("PINN_REFERENCE_DIR", "")      # a checkout of the original project, if any
TOL = 1e-13


def _rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _ref_run():
    return load_reference_run()


def test_reference_run_equals_oracle_golden_burgers_inference():
    r, g = _ref_run(), load_golden("burgers_inf")
    assert abs(float(r["burgers_inf_loss"]) - float(g["loss"])) <= TOL * float(g["loss"])
    assert _rel(r["burgers_inf_grad"], g["grad"]) <= TOL
    assert _rel(r["burgers_inf_predict"], g["predict"]) <= TOL and _rel(r["burgers_inf_residual"], g["residual"]) <= TOL
    for k in range(2):                                        # NeuralNetwork.fit(): 5 Adam epochs at lr 1e-3 and 0.03
        assert _rel(r["burgers_inf_adam_losses_%d" % k], g["adam_losses"][k]) <= TOL
        assert _rel(r["burgers_inf_adam_w_%d" % k], g["adam_w"][k]) <= TOL
    # custom_lbfgs.lbfgs(): evaluation points, f history, the returned x and the log lines
    assert _rel(r["burgers_inf_lbfgs_x_eval"], g["lbfgs_x_eval"]) <= TOL and _rel(r["burgers_inf_lbfgs_f"], g["lbfgs_f"]) <= TOL
    assert _rel(r["burgers_inf_lbfgs_x_final"], g["lbfgs_x_final"]) <= TOL
    assert _rel(r["burgers_inf_lbfgs_logged"], g["lbfgs_logged"]) <= TOL
    # after fit() the MODEL holds the last evaluated point, not lbfgs's returned x (quirk: last update discarded)
    assert _rel(r["burgers_inf_fit_lbfgs_w"], g["lbfgs_x_eval"][-1]) <= TOL
    assert _rel(r["burgers_inf_fit_lbfgs_w"], g["lbfgs_x_final"]) > 1e-6


def test_reference_run_equals_oracle_golden_identification():
    r, g = _ref_run(), load_golden("burgers_ide")
    for tag in ("", "2"):
        assert abs(float(r["burgers_ide_loss" + tag]) - float(g["loss" + tag])) <= TOL * float(g["loss" + tag])
        assert _rel(r["burgers_ide_grad" + tag], g["grad" + tag]) <= TOL
    assert _rel(r["burgers_ide_adam_losses"], g["adam_losses"]) <= TOL and _rel(r["burgers_ide_adam_w"], g["adam_w"]) <= TOL
    assert _rel(r["burgers_ide_fit_lbfgs_w"], g["lbfgs_x_eval"][-1]) <= TOL


def test_reference_run_equals_oracle_golden_schrodinger():
    r, g = _ref_run(), load_golden("nls_inf")
    for tag in ("q1", "x0t0"):
        assert abs(float(r["nls_loss_" + tag]) - float(g["loss_" + tag])) <= TOL * float(g["loss_" + tag])
        assert _rel(r["nls_grad_" + tag], g["grad_" + tag]) <= TOL
    assert abs(float(g["loss_q1"]) - float(g["loss_x0t0"])) > 1e-3 * float(g["loss_q1"])      # quirk Q1 is a real difference
    assert _rel(r["nls_adam_losses"], g["adam_losses"]) <= TOL and _rel(r["nls_adam_w"], g["adam_w"]) <= TOL
    assert _rel(r["nls_predict"], g["predict"]) <= TOL and _rel(r["nls_residual"], g["residual"]) <= TOL


def test_reference_run_equals_oracle_golden_discrete_time():
    r, g = _ref_run(), load_golden("burgers_disc")
    assert abs(float(r["burgers_disc_loss"]) - float(g["loss"])) <= TOL * float(g["loss"])
    assert _rel(r["burgers_disc_grad"], g["grad"]) <= TOL and _rel(r["burgers_disc_predict"], g["predict"]) <= TOL
    assert _rel(r["burgers_disc_adam_losses"], g["adam_losses"]) <= TOL and _rel(r["burgers_disc_adam_w"], g["adam_w"]) <= TOL
    # fact about the reference: its discrete-time L-BFGS closure takes the loss outside the tape, the phase cannot run
    assert int(r["burgers_disc_lbfgs_runs"]) == 0


def test_reference_run_equals_oracle_golden_discrete_time_identification():
    """ide_disc_burgers.py's class (the script around it is broken as shipped): loss, gradient incl. lambda_1/lambda_2 at two
    parameter points, both predictions.  This comparison is what exposed that the reference forms (beta - alpha) in float32."""
    r, g = _ref_run(), load_golden("burgers_ide_disc")
    for tag in ("", "2"):
        assert abs(float(r["burgers_ide_disc_loss" + tag]) - float(g["loss" + tag])) <= TOL * float(g["loss" + tag])
        assert _rel(r["burgers_ide_disc_grad" + tag], g["grad" + tag]) <= TOL
    assert _rel(r["burgers_ide_disc_predict_U0"], g["predict_U0"]) <= TOL and _rel(r["burgers_ide_disc_predict_U1"], g["predict_U1"]) <= TOL
    # its fit(): 3 Adam epochs + 4 L-BFGS iterations from the stored start, replayed here with the oracle
    sys.path.insert(0, ROOT)
    from oracle import reference_port as rp
    pb = rp.BurgersDiscreteIdentification([int(v) for v in g["layers"]], g["lb"], g["ub"], float(g["dt"]), g["x_0"], g["u_0"],
                                           g["x_1"], g["u_1"], g["IRK_alpha"], g["IRK_beta"])
    wa, la, _ = rp.adam_train(pb, r["burgers_ide_disc_fit_w0"], 3, lr=1e-3)
    tr = rp.lbfgs_fixed_step(lambda z: rp.loss_and_flat_grad(pb, z), wa, max_iter=4, learning_rate=0.8, n_correction=50,
                             tol_fun=np.finfo(float).eps)
    assert _rel(r["burgers_ide_disc_fit_adam_losses"], la) <= TOL
    assert _rel(r["burgers_ide_disc_fit_lbfgs_logged"][:, 1], np.array(tr.logged)[:, 1]) <= 1e-12
    assert _rel(r["burgers_ide_disc_fit_w"], tr.x_eval[-1]) <= 1e-12


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_reference_sources_reproduce_the_committed_run():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "golden", "make_reference_fixtures.py"), "--check"],
                       capture_output=True, text=True, timeout=900, cwd="/tmp")
    assert r.returncode == 0 and "committed fixture reproduced" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


# ---------------------------------------------------------------------------------------------------------------------------
# semantics of the emulation itself (run in a subprocess: `import tensorflow` must not leak into this test process, where the
# product's own shim of the same name may be imported by other tests)
_SEMANTICS = r'''
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import tensorflow as tf
assert "tf_emulation" in tf.__file__
c = lambda v: tf.convert_to_tensor(np.array(v, dtype=float), dtype="float64")

# 1. higher order through a persistent tape; gradient called after the context still works; x**3 -> 3x^2 -> 6x
x = c([[1.0], [2.0]])
with tf.GradientTape(persistent=True) as tape:
    tape.watch(x)
    y = x * x * x
    yx = tape.gradient(y, x)
yxx = tape.gradient(yx, x)
assert np.allclose(yx.numpy().ravel(), [3, 12]) and np.allclose(yxx.numpy().ravel(), [6, 12])

# 2. operations executed OUTSIDE the context are not recorded -> None (the inf_disc_burgers.py:103-107 situation)
with tf.GradientTape() as t2:
    t2.watch(x)
z = x * x
assert t2.gradient(z, x) is None

# 3. a value computed before the tape started is a constant for that tape, even if it depends on the source
v = tf.Variable([2.0], dtype="float64")
pre = v * v
with tf.GradientTape() as t3:
    w = pre * 3.0
assert t3.gradient(w, v) is None
with tf.GradientTape() as t3:
    w = v * v * 3.0
assert np.allclose(t3.gradient(w, v).numpy(), [12.0])          # trainable variables are watched automatically

# 4. unwatched constants give None; a non-persistent tape serves exactly one gradient call
k = c([1.0, 2.0])
with tf.GradientTape() as t4:
    s = tf.reduce_sum(k * k)
assert t4.gradient(s, k) is None
try:
    t4.gradient(s, k)
    raise SystemExit("second gradient() on a non-persistent tape must raise")
except RuntimeError:
    pass

# 5. gradients are sums over the target; list of sources -> list; nested tapes: inner result differentiable by the outer one
a, b = tf.Variable([1.0, 2.0], dtype="float64"), tf.Variable([3.0], dtype="float64")
with tf.GradientTape() as outer:
    with tf.GradientTape() as inner:
        f = tf.reduce_sum(a * a * b)
    ga = inner.gradient(f, a)                    # 2 a b, recorded by `outer`
    h = tf.reduce_sum(ga * ga)                   # 4 a^2 b^2 summed
gs = outer.gradient(h, [a, b])
assert np.allclose(gs[0].numpy(), 8 * np.array([1.0, 2.0]) * 9) and np.allclose(gs[1].numpy(), [8 * 5 * 3.0])

# 6. output_gradients / the dummy trick: per-column derivative of a matrix-valued function
d = tf.ones([2, 3], dtype="float64")
W = tf.Variable(np.arange(3.0).reshape(1, 3) + 1, dtype="float64")
with tf.GradientTape(persistent=True) as tape:
    tape.watch(x); tape.watch(d)
    U = tf.matmul(x * x, W)
    gU = tape.gradient(U, x, output_gradients=d)
    Ux = tape.gradient(gU, d)
assert np.allclose(Ux.numpy(), 2 * x.numpy() * (np.arange(3.0) + 1))

# 7. eager tensors are values: += rebinds, the original object is untouched (custom_lbfgs.py:175 relies on it)
p = c([1.0, 1.0]); q = p
p += c([1.0, 1.0])
assert np.allclose(q.numpy(), [1, 1]) and np.allclose(p.numpy(), [2, 2])
assert min(1, 1 / tf.reduce_sum(tf.abs(c([4.0])))).numpy() == 0.25 and format(tf.reduce_sum(c([1.5])), ".4e") == "1.5000e+00"
assert (np.array([1.0, 2.0]) * c([2.0, 2.0])).numpy().tolist() == [2.0, 4.0]      # numpy on the left defers to the tensor
assert (0.1 * c([1.0])).numpy()[0] == 0.1                                         # python floats stay float64

# 8. Keras pieces: layers hides the InputLayer, trainable_variables is a fresh list in (kernel, bias) order, set_weights checks
tf.keras.backend.set_floatx("float64")
tf.random.set_seed(1234)
m = tf.keras.Sequential()
m.add(tf.keras.layers.InputLayer(input_shape=(2,)))
m.add(tf.keras.layers.Lambda(lambda X: 2.0 * X - 1.0))
m.add(tf.keras.layers.Dense(5, activation=tf.nn.tanh, kernel_initializer="glorot_normal"))
m.add(tf.keras.layers.Dense(1, activation=None, kernel_initializer="glorot_normal"))
assert len(m.layers) == 3 and len(m.layers[1:]) == 2
tv = m.trainable_variables; tv.append(None)
assert len(m.trainable_variables) == 4 and [v.shape for v in m.trainable_variables] == [(2, 5), (5,), (5, 1), (1,)]
k0, b0 = m.layers[1].get_weights()
assert np.all(b0 == 0) and np.abs(k0).max() <= 2 * np.sqrt(2 / 7) / 0.87962566103423978 + 1e-12
X = np.array([[0.25, 0.5]])
assert np.allclose(m(X).numpy(), np.tanh((2 * X - 1) @ k0) @ m.layers[2].get_weights()[0])
try:
    m.layers[1].set_weights([np.zeros((3, 5)), np.zeros(5)])
    raise SystemExit("shape mismatch must raise")
except ValueError:
    pass

# 9. Adam = TF-2.0 OptimizerV2: epsilon=None -> 1e-7, epsilon OUTSIDE the bias correction
var = tf.Variable([1.0], dtype="float64")
opt = tf.keras.optimizers.Adam(learning_rate=0.1, beta_1=0.9, epsilon=None)
m_, v_, th = 0.0, 0.0, 1.0
for t in range(1, 4):
    with tf.GradientTape() as tp:
        L = tf.reduce_sum(var * var * var)
    gr = tp.gradient(L, [var])
    opt.apply_gradients(zip(gr, [var]))
    g_ = 3 * th * th
    m_ += (g_ - m_) * 0.1; v_ += (g_ * g_ - v_) * 0.001
    th -= 0.1 * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t) * m_ / (np.sqrt(v_) + 1e-7)
    assert abs(var.numpy()[0] - th) < 1e-15
print("emulation semantics ok")
'''


def test_tf_emulation_semantics():
    r = subprocess.run([sys.executable, "-c", _SEMANTICS, os.path.join(ROOT, "oracle", "tf_emulation")],
                       capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert r.returncode == 0 and "emulation semantics ok" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_reference_default_schedule_run():
    """The reference's default Burgers run (100 Adam @0.03 + 200 fixed-step L-BFGS @0.8) through its own fit(): the Adam phase
    and the first 40 L-BFGS iterations equal the oracle's to rounding; the fixed-step L-BFGS tail is chaotic (deviation grows
    ~10x per 10 iterations), so the end points agree in magnitude only -- which is also the bar of the GPU accuracy test."""
    r, a = _ref_run(), load_golden("burgers_accuracy")
    assert _rel(r["schedule_adam_losses"], a["oracle_adam_losses"]) <= TOL
    dev = r["schedule_lbfgs_f_deviation"]
    assert dev.shape == (199,) and dev[:40].max() <= 1e-9 and dev[:10].max() <= 1e-12
    assert dev[-1] > 1e-6                                              # the tail really does diverge
    assert abs(float(r["schedule_error"]) - float(a["oracle_error"])) <= 0.25 * float(a["oracle_error"])
    assert _rel(r["schedule_w"], a["oracle_w"]) <= 0.05


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_logger_prints_what_the_reference_logger_prints():
    """SURVEY 8(a) a11: with the same clock, the mirror's Logger emits the reference Logger's lines character for character
    (hyper-parameter dump, epoch lines with truncated tenths, `:.4e` losses, end line); only the version banner differs."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "logger_compare_worker.py"), ROOT],
                       capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert r.returncode == 0 and "logger output identical" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_mirror_host_attributes_equal_the_reference():
    """sizes_w / sizes_b (incl. the uniform-width assumption, quirk Q7), nt_config, tf_epochs, dtype, get_params and the
    custom_lbfgs module surface of the mirror equal those of the reference classes built from the same hp."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "surface_compare_worker.py"), ROOT],
                       capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert r.returncode == 0 and "host attributes identical" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_prep_data_equals_the_reference():
    """SURVEY 8(f)1: every array returned by the package's prep_data restatements (Burgers inference / identification /
    discrete-time inference, Schrodinger) is bit-identical to what the reference's own prep_data returns from the same seed."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "prep_data_compare_worker.py"), ROOT],
                       capture_output=True, text=True, timeout=600, cwd="/tmp")
    assert r.returncode == 0 and "prep_data identical" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_unmodified_reference_script_runs_end_to_end_on_the_emulation(tmp_path):
    """oracle/run_reference_on_emulation.py: the whole inf_cont_burgers.py (data prep, model, fit, predict, error, result
    directory) executes on the CPU with a small hp.json; its printed log has the reference Logger's shape."""
    import json
    hp = {"N_u": 50, "N_f": 500, "layers": [2, 20, 20, 20, 20, 20, 20, 20, 20, 1], "tf_epochs": 3, "tf_lr": 0.03, "tf_b1": 0.9,
          "tf_eps": None, "nt_epochs": 3, "nt_lr": 0.8, "nt_ncorr": 50, "log_frequency": 1}
    (tmp_path / "hp.json").write_text(json.dumps(hp))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "run_reference_on_emulation.py"),
                        os.path.join(REF, "1d-burgers", "inf_cont_burgers.py"), str(tmp_path / "hp.json")],
                       capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    out = r.stdout
    assert r.returncode == 0, out[-2000:] + r.stderr[-3000:]
    assert "TensorFlow version: 2.0.0-rc0 (API emulation" in out and "-- Starting Adam optimization --" in out
    assert out.count("tf_epoch = ") == 3 and out.count("nt_epoch = ") == 2      # the last L-BFGS iteration is never logged
    assert "Training finished (epoch 6)" in out and "Saving results to directory" in out


def test_gpu_tests_reference_run_keys_exist():
    """The GPU parity tests compare the CUDA results with reference_run.npz through conftest.assert_matches_reference_run;
    exercise exactly those key pairs here (with the oracle's golden values standing in for the CUDA output), so that a typo
    cannot surface only on the GPU box."""
    from conftest import assert_matches_reference_run
    g = load_golden("burgers_inf")
    assert_matches_reference_run(float(g["loss"]), g["grad"], "burgers_inf_loss", "burgers_inf_grad")
    g = load_golden("burgers_ide")
    for fk, gk in (("loss", "grad"), ("loss2", "grad2")):
        assert_matches_reference_run(float(g[fk]), g[gk], "burgers_ide_" + fk, "burgers_ide_" + gk)
    g = load_golden("nls_inf")
    for tag in ("q1", "x0t0"):
        assert_matches_reference_run(float(g["loss_" + tag]), g["grad_" + tag], "nls_loss_" + tag, "nls_grad_" + tag)
    g = load_golden("burgers_disc")
    assert_matches_reference_run(float(g["loss"]), g["grad"], "burgers_disc_loss", "burgers_disc_grad")
    with pytest.raises(AssertionError):
        assert_matches_reference_run(float(g["loss"]) * (1 + 1e-8), g["grad"], "burgers_disc_loss", "burgers_disc_grad")


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_lbfgs_control_flow_equals_the_reference():
    """Every exit of the reference's lbfgs() (maxIter, maxEval, optimality at the start / later, no progress, step below tolX,
    f change below tolX) plus rejected curvature pairs and history overflow: evaluation points, f history, returned x, logged
    iterations, evaluation and iteration counts of oracle.reference_port.lbfgs_fixed_step equal the reference's on synthetic
    objectives.  One known difference: 'no progress' at the very first iteration is an UnboundLocalError in the reference."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "lbfgs_compare_worker.py"), ROOT],
                       capture_output=True, text=True, timeout=600, cwd="/tmp")
    assert r.returncode == 0 and "lbfgs control flow identical" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    assert "reference raises UnboundLocalError" in r.stdout


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_golden_fixtures_are_reproduced_by_their_generator(tmp_path):
    """tests/golden/make_golden.py (committed with the fixtures it made) regenerates every array of the five problem fixtures
    exactly; the generator reads only the reference's data files and the oracle."""
    env = dict(os.environ, PINN_GOLDEN_OUT=str(tmp_path), PYTHONPATH=ROOT)
    for flags in ([], ["--disc"], ["--ide-disc"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "golden", "make_golden.py")] + flags, env=env,
                           capture_output=True, text=True, timeout=900, cwd="/tmp")
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    for name in ("burgers_inf", "burgers_ide", "nls_inf", "burgers_disc", "burgers_ide_disc"):
        a, b = load_golden(name), np.load(os.path.join(str(tmp_path), name + ".npz"))
        assert sorted(a.files) == sorted(b.files), name
        for k in a.files:
            assert np.array_equal(a[k], b[k]), (name, k)
