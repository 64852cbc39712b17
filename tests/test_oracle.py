"""CPU: the oracle against the committed golden vectors, and the two oracle formulations against each other."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import reference_port as rp, taylor as ty

EPS = np.finfo(float).eps


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def test_flat_layout_matches_reference_sizes():
    # utils/neuralnetwork.py:40-45 sizes_w / sizes_b for the Burgers net
    layers = [2] + [20] * 8 + [1]
    sizes_w = [int(w * layers[1]) for i, w in enumerate(layers) if i != 1]
    sizes_b = [int(w if i != 0 else layers[1]) for i, w in enumerate(layers) if i != 1]
    offs = rp.param_offsets(layers)
    o = 0
    for (wo, bo), sw, sb in zip(offs, sizes_w, sizes_b):
        assert wo == o and bo == o + sw
        o += sw + sb
    assert o == rp.num_params(layers) == 3021
    assert rp.num_params([2, 100, 100, 100, 100, 2]) == 30802


def test_burgers_inf_golden_both_oracles():
    g = load_golden("burgers_inf")
    layers = list(g["layers"])
    pb = rp.BurgersInference(layers, g["lb"], g["ub"], float(g["nu"]), g["X_f"], g["X_u"], g["u"])
    f, gr = rp.loss_and_flat_grad(pb, g["w"])
    assert abs(f - g["loss"]) <= 1e-13 * abs(g["loss"])
    assert rel(gr, g["grad"]) < 1e-12
    f2, g2, parts = ty.burgers_loss_grad(g["w"], layers, g["lb"], g["ub"], g["X_f"], g["X_u"], g["u"], nu=float(g["nu"]))
    assert abs(f2 - g["loss"]) <= 1e-13 * abs(g["loss"])
    assert rel(g2, g["grad"]) < 1e-12
    assert np.allclose(parts, g["parts"][[0, 1]] if len(g["parts"]) == 2 else g["parts"], rtol=1e-12)
    (U, Ux, Ut, Uxx), _ = ty.forward(g["w"], layers, g["lb"], g["ub"], g["X_f"][:64])
    assert rel(np.hstack([U, Ux, Ut, Uxx]), g["probes"]) < 1e-12


def test_burgers_ide_golden_both_oracles():
    g = load_golden("burgers_ide")
    layers = list(g["layers"])
    pb = rp.BurgersIdentification(layers, g["lb"], g["ub"], g["X_u"], g["u"])
    for wk, fk, gk in (("w", "loss", "grad"), ("w2", "loss2", "grad2")):
        f, gr = rp.loss_and_flat_grad(pb, g[wk])
        f2, g2, _ = ty.burgers_loss_grad(g[wk], layers, g["lb"], g["ub"], None, g["X_u"], g["u"], identification=True)
        assert abs(f - g[fk]) <= 1e-13 * abs(g[fk]) and abs(f2 - g[fk]) <= 1e-13 * abs(g[fk])
        assert rel(gr, g[gk]) < 1e-12 and rel(g2, g[gk]) < 1e-12
    assert g["grad2"].shape == (3023,)


def test_nls_golden_taylor_oracle_and_q1_quirk():
    g = load_golden("nls_inf")
    layers = list(g["layers"])
    x0 = g["x0"]
    for tag, X0 in (("q1", x0), ("x0t0", np.concatenate([x0, 0 * x0], 1))):
        f2, g2, parts = ty.schrodinger_loss_grad(g["w"], layers, g["lb"], g["ub"], g["X_f"], g["tb"], X0, g["uv0"])
        assert abs(f2 - g["loss_" + tag]) <= 1e-13 * abs(g["loss_" + tag])
        assert rel(g2, g["grad_" + tag]) < 1e-12
        assert np.allclose(parts, g["parts_" + tag], rtol=1e-12)
    # quirk Q1 changes only the initial-condition term
    assert g["parts_q1"][0] != g["parts_x0t0"][0]
    assert g["parts_q1"][1] == g["parts_x0t0"][1] and g["parts_q1"][2] == g["parts_x0t0"][2]


def test_adam_tf2_semantics_by_hand():
    # one step: m = (1-b1) g, v = (1-b2) g^2, alpha = lr sqrt(1-b2)/(1-b1) -> w -= lr*g/(|g| + eps*sqrt(1-b2)) approx
    w = np.array([1.0, -2.0]); g = np.array([0.5, -0.25])
    st = rp.adam_init(2)
    w1 = rp.adam_update(w, g, st, lr=0.1, b1=0.9, b2=0.999, eps=None)
    alpha = 0.1 * np.sqrt(1 - 0.999) / (1 - 0.9)
    exp = w - alpha * (0.1 * g) / (np.sqrt(0.001 * g * g) + 1e-7)
    assert np.allclose(w1, exp, rtol=0, atol=1e-15)
    assert st.t == 1


def test_adam_golden_trajectory():
    g = load_golden("burgers_inf")
    pb = rp.BurgersInference(list(g["layers"]), g["lb"], g["ub"], float(g["nu"]), g["X_f"], g["X_u"], g["u"])
    w, losses, _ = rp.adam_train(pb, g["w"], 5, lr=float(g["adam_lr"][0]))
    assert rel(w, g["adam_w"][0]) < 1e-12 and rel(losses, g["adam_losses"][0]) < 1e-12


def _quad(A, b):
    def f(x):
        return float(0.5 * x @ A @ x - b @ x), A @ x - b
    return f


def test_lbfgs_control_flow_quirks():
    rng = np.random.default_rng(0)
    M = rng.standard_normal((6, 6)); A = M @ M.T + 6 * np.eye(6); b = rng.standard_normal(6)
    x0 = rng.standard_normal(6)
    op = _quad(A, b)
    assert rp.lbfgs_fixed_step(op, x0, 0) is None                       # custom_lbfgs.py:43-44
    tr = rp.lbfgs_fixed_step(op, x0, max_iter=8, learning_rate=0.8, n_correction=3, tol_fun=EPS)
    f0, g0 = op(x0)
    assert tr.t[0] == min(1.0, 1.0 / np.abs(g0).sum())                 # :159-161
    assert all(t == 0.8 for t in tr.t[1:])                             # :163 fixed step, no line search
    assert np.allclose(tr.d[0], -g0)
    assert tr.n_iter == 8 and tr.n_eval == 8                           # the last update is NOT evaluated (:176-182)
    assert len(tr.x_eval) == 8 and not np.allclose(tr.x_eval[-1], tr.x_final)
    assert np.allclose(tr.x_final, tr.x_eval[-1] + tr.t[-1] * tr.d[-1])
    assert max(tr.hist_len) <= 3
    assert [it for it, _ in tr.logged] == list(range(1, 8))            # iteration maxIter breaks before the log
    # initial optimality
    xs = np.linalg.solve(A, b)
    tr2 = rp.lbfgs_fixed_step(op, xs, max_iter=5, tol_fun=1e-6)
    assert tr2.stop_reason == "initial optimality" and tr2.n_iter == 0


def test_lbfgs_golden_trace():
    g = load_golden("burgers_inf")
    pb = rp.BurgersInference(list(g["layers"]), g["lb"], g["ub"], float(g["nu"]), g["X_f"], g["X_u"], g["u"])
    tr = rp.lbfgs_fixed_step(lambda x: rp.loss_and_flat_grad(pb, x), g["w"], max_iter=6, learning_rate=0.8,
                             n_correction=50, tol_fun=EPS)
    assert tr.n_iter == int(g["lbfgs_n_iter"]) and tr.n_eval == int(g["lbfgs_n_eval"])
    assert rel(np.array(tr.f_hist), g["lbfgs_f"]) < 1e-9
    assert rel(tr.x_final, g["lbfgs_x_final"]) < 1e-9


def test_lua_struct_defaults_to_zero():
    s = rp.LuaStruct()
    s.maxIter = 3
    assert s.maxIter == 3 and s.lineSearch == 0 and (s.tolX or 1e-19) == 1e-19    # custom_lbfgs.py:242-246


def test_burgers_disc_golden_both_oracles():
    """Discrete-time IRK model (1d-burgers/inf_disc_burgers.py:61-101): nested autograd with the reference's dummy-gradient
    trick and the closed-form Taylor oracle against the committed vector (upstream q=100 Butcher table)."""
    g = load_golden("burgers_disc")
    layers = [int(v) for v in g["layers"]]
    IRK = g["IRK"].astype(np.float64)
    pb = rp.BurgersDiscreteInference(layers, g["lb"], g["ub"], float(g["nu"]), float(g["dt"]), g["x_0"], g["u_0"], g["x_1"], IRK)
    f, gr = rp.loss_and_flat_grad(pb, g["w"])
    f2, g2, parts = ty.burgers_disc_loss_grad(g["w"], layers, g["lb"], g["ub"], g["x_0"], g["u_0"], g["x_1"], float(g["nu"]),
                                              float(g["dt"]), IRK)
    for fv, gv in ((f, gr), (f2, g2)):
        assert abs(fv - g["loss"]) <= 1e-13 * abs(g["loss"]) and rel(gv, g["grad"]) < 1e-12
    assert np.allclose(parts, g["parts"], rtol=1e-12)
    assert IRK.shape == (101, 100) and abs(IRK[-1].sum() - 1.0) < 1e-5        # last row: the quadrature weights b_j


def test_burgers_ide_disc_golden_both_oracles():
    """Discrete-time identification (1d-burgers/ide_disc_burgers.py:48-203): nested-autograd restatement (dummy-gradient trick)
    and the closed-form Taylor oracle against the golden vector (q = 81 upstream table, float32 like the reference loads it)."""
    g = load_golden("burgers_ide_disc")
    layers = [int(v) for v in g["layers"]]
    assert layers == [1, 50, 50, 50, 81] and g["IRK_alpha"].dtype == np.float32 and g["IRK_alpha"].shape == (81, 81)
    pb = rp.BurgersDiscreteIdentification(layers, g["lb"], g["ub"], float(g["dt"]), g["x_0"], g["u_0"], g["x_1"], g["u_1"],
                                           g["IRK_alpha"], g["IRK_beta"])
    for tag in ("", "2"):
        f, gr = rp.loss_and_flat_grad(pb, g["w" + tag])
        f2, g2, parts = ty.burgers_ide_disc_loss_grad(g["w" + tag], layers, g["lb"], g["ub"], g["x_0"], g["u_0"], g["x_1"], g["u_1"],
                                                      float(g["dt"]), g["IRK_alpha"], g["IRK_beta"])
        for fv, gv in ((f, gr), (f2, g2)):
            assert abs(fv - float(g["loss" + tag])) <= 1e-13 * abs(float(g["loss" + tag]))
            assert np.linalg.norm(gv - g["grad" + tag]) <= 1e-12 * np.linalg.norm(g["grad" + tag])
        assert np.allclose(parts, g["parts" + tag], rtol=1e-13)
    # beta - alpha is rounded in float32 by the reference (numpy arithmetic before TensorFlow sees it): doing it in float64 is
    # a DIFFERENT function at the 1e-10 level, which the pin against the reference's own code detects
    pb64 = rp.BurgersDiscreteIdentification(layers, g["lb"], g["ub"], float(g["dt"]), g["x_0"], g["u_0"], g["x_1"], g["u_1"],
                                             g["IRK_alpha"].astype(np.float64), g["IRK_beta"].astype(np.float64))
    f64, _ = rp.loss_and_flat_grad(pb64, g["w2"])
    assert 1e-14 < abs(f64 - float(g["loss2"])) / float(g["loss2"]) < 1e-8
    U0, U1 = pb.predict(g["w2"], g["x_star"])
    assert np.allclose(U0, g["predict_U0"], rtol=0, atol=1e-13) and np.allclose(U1, g["predict_U1"], rtol=0, atol=1e-13)


LD = np.longdouble
needs_long_double = pytest.mark.skipif(np.finfo(np.longdouble).eps >= 1e-18,
                                       reason="np.longdouble is no wider than float64 on this platform")


def _golden_cases():
    """(name, function, kwargs) of the five models at the golden (initialisation) inputs."""
    b, i, n, d, e = (load_golden(k) for k in ("burgers_inf", "burgers_ide", "nls_inf", "burgers_disc", "burgers_ide_disc"))
    return [
        ("burgers_inf", ty.burgers_loss_grad, dict(w=b["w"], layers=list(b["layers"]), lb=b["lb"], ub=b["ub"], X_f=b["X_f"],
                                                    X_u=b["X_u"], u=b["u"], nu=float(b["nu"]))),
        ("burgers_ide", ty.burgers_loss_grad, dict(w=i["w"], layers=list(i["layers"]), lb=i["lb"], ub=i["ub"], X_f=None, X_u=i["X_u"],
                                                    u=i["u"], identification=True)),
        ("nls_inf", ty.schrodinger_loss_grad, dict(w=n["w"], layers=list(n["layers"]), lb=n["lb"], ub=n["ub"], X_f=n["X_f"], tb=n["tb"],
                                                    X0=n["x0"], uv0=n["uv0"])),
        ("burgers_disc", ty.burgers_disc_loss_grad, dict(w=d["w"], layers=[int(v) for v in d["layers"]], lb=d["lb"], ub=d["ub"],
                                                         x_0=d["x_0"], u_0=d["u_0"], x_1=d["x_1"], nu=float(d["nu"]), dt=float(d["dt"]),
                                                         IRK_weights=d["IRK"].astype(np.float64))),
        ("burgers_ide_disc", ty.burgers_ide_disc_loss_grad, dict(w=e["w"], layers=[int(v) for v in e["layers"]], lb=e["lb"], ub=e["ub"],
                                                                 x_0=e["x_0"], u_0=e["u_0"], x_1=e["x_1"], u_1=e["u_1"], dt=float(e["dt"]),
                                                                 IRK_alpha=e["IRK_alpha"], IRK_beta=e["IRK_beta"])),
    ]


@needs_long_double
@pytest.mark.parametrize("case", range(5))
def test_long_double_oracle_agrees_with_fp64_at_init_weights(case):
    """dtype=np.longdouble carries the same inputs through 64-bit-mantissa arithmetic: results come back in that dtype, and at
    well-conditioned initialisation weights they agree with the fp64 evaluation to a few ulps of the latter."""
    name, fn, kw = _golden_cases()[case]
    f64, g64, p64 = fn(**kw)
    fld, gld, pld = fn(**kw, dtype=LD)
    assert gld.dtype == LD and np.asarray(fld).dtype == LD and all(np.asarray(v).dtype == LD for v in pld), name
    assert np.asarray(f64).dtype == np.float64 and g64.dtype == np.float64
    assert abs(f64 - fld) <= 1e-13 * abs(fld), name
    assert np.linalg.norm(g64 - gld) <= 1e-13 * np.linalg.norm(gld), name
    for a, b in zip(p64, pld):
        assert abs(a - b) <= 1e-13 * abs(b), name


@needs_long_double
def test_fp64_oracle_loses_digits_at_trained_weights():
    """At the trained Burgers weights (100 Adam steps + 200 L-BFGS iterations, N_f = 10 000) the gradient is a sum with heavy
    cancellation: the fp64 evaluation is off the long-double one by far more than at initialisation, yet still far below the
    1e-10 tolerance of the parity tests.  Kernel tests that use a flat tolerance there are either too loose or too tight; the
    extended-precision GPU tests compare each kernel with the fp64 oracle's own error instead."""
    a = load_golden("burgers_accuracy")
    kw = dict(w=a["oracle_w"], layers=[2] + [20] * 8 + [1], lb=a["lb"], ub=a["ub"], X_f=a["X_f"], X_u=a["X_u"], u=a["u"], nu=0.01 / np.pi)
    f64, g64, _ = ty.burgers_loss_grad(**kw)
    fld, gld, _ = ty.burgers_loss_grad(**kw, dtype=LD)
    e = float(np.linalg.norm(g64 - gld) / np.linalg.norm(gld))
    assert 1e-14 < e < 1e-11, e
    assert abs(f64 - fld) <= 1e-14 * abs(fld)
