"""GPU: every fused loss/gradient kernel, and the forward kernel behind predict / derivatives / residual, against an
extended-precision (np.longdouble, 64-bit mantissa) evaluation of the Taylor oracle on the kernel's own fp64 inputs.

The bound is relative to how well-conditioned each case is.  For every checked quantity q (the loss, each loss part, each
gradient block W_l and b_l, each lambda entry; each forward stream) let R be the long-double reference, O the plain fp64 oracle
and K the kernel, e_K = |K_q - R_q| / |R_q| and e_O = |O_q - R_q| / |R_q|.  The kernel must satisfy

    e_K <= max(FACTOR * e_O, FLOOR)

i.e. be about as accurate as a plain fp64 implementation of the same maths.  A part that is zero in R must be exactly 0 in K.
At trained weights the gradient is a sum with heavy cancellation and the fp64 oracle's own error reaches ~1e-12, so a flat
tolerance is either too loose at initialisation or too tight there.

The fused loss/gradient kernels evaluate tanh with their own branch-free routine (pinn_common.cuh: tanh_fast, <= 4 ulp) where
numpy's tanh is within 1 ulp.  At trained identification weights the lambda_1 gradient is so sensitive to the rounding of the
activations that this alone moves it by ~1e-13 while numpy's evaluation is off by 6e-15.  For those kernels e_O is therefore the
larger error of two fp64 evaluations of the oracle: with numpy's tanh and with the kernels' own (pinn_cabi.device_tanh).  The
forward kernel (predict / derivatives / residual) uses the CUDA math library's tanh and is held to numpy's evaluation alone.

Regimes: trained weights, saturated tanh units (initialisation weights x 2 and x 3), non-unit asymmetric domains (a kernel that
drops the input scale 2/(ub-lb) or the offset lb must fail), and point-position edges (points on lb/ub, outside the box, duplicated).
Kernel variants: PINN_FUSED_TAIL and PINN_GENERIC_DFMA are read once per process, so each environment runs in a worker process of
its own (tests/extended_precision_worker.py) that evaluates all the cases it serves."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden, load_reference_run

pytestmark = pytest.mark.gpu

LD = np.longdouble
EPS = np.finfo(np.float64).eps
FACTOR, FLOOR = 16.0, 32 * EPS
BURGERS, NLS = [2] + [20] * 8 + [1], [2, 100, 100, 100, 100, 2]
BURGERS_INF, BURGERS_IDE, NLS_INF, BURGERS_DISC, BURGERS_IDE_DISC = 0, 1, 2, 3, 4
NU = 0.01 / np.pi

# variant -> (environment, PDEs it serves)
VARIANTS = {
    "v2_fused_tail": ({}, (BURGERS_INF, BURGERS_IDE)),
    "v2_two_launch": ({"PINN_FUSED_TAIL": "0"}, (BURGERS_INF, BURGERS_IDE)),
    "v1": ({"PINN_BURGERS_KERNEL": "v1"}, (BURGERS_INF, BURGERS_IDE)),
    "nls_specialised": ({}, (NLS_INF,)),
    "generic_dmma": ({"PINN_FORCE_GENERIC": "1"}, (BURGERS_INF, BURGERS_IDE, NLS_INF, BURGERS_DISC, BURGERS_IDE_DISC)),
    "generic_dfma": ({"PINN_FORCE_GENERIC": "1", "PINN_GENERIC_DFMA": "1"},
                     (BURGERS_INF, BURGERS_IDE, NLS_INF, BURGERS_DISC, BURGERS_IDE_DISC)),
}


# ---------------------------------------------------------------------------------------------------------------- cases
def box(rng, lb, ub, n):
    lb, ub = np.asarray(lb, float), np.asarray(ub, float)
    return lb + (ub - lb) * rng.random((n, lb.size))


def edge_set(rng, lb, ub, n_interior):
    """A ragged set with points exactly on lb / ub (normalised input +-1), outside the box by one box width (normalised +-3)
    and duplicated points, shuffled among interior points."""
    lb, ub = np.asarray(lb, float), np.asarray(ub, float)
    d = ub - lb
    xm, tm = lb + d * rng.random(2)
    pts = [[lb[0], lb[1]], [lb[0], ub[1]], [ub[0], lb[1]], [ub[0], ub[1]], [lb[0], tm], [ub[0], tm], [xm, lb[1]], [xm, ub[1]],
           [lb[0] - d[0], tm], [ub[0] + d[0], tm], [xm, lb[1] - d[1]], [xm, ub[1] + d[1]], [lb[0] - d[0], lb[1] - d[1]],
           [ub[0] + d[0], ub[1] + d[1]], [lb[0] - d[0], ub[1] + d[1]]]
    X = np.vstack([np.array(pts), box(rng, lb, ub, n_interior)])
    X = np.vstack([X, X[rng.integers(0, X.shape[0], 37)], np.array(pts)])          # duplicates of edge and interior points
    return X[rng.permutation(X.shape[0])]


def burgers_cases():
    a, r, gi, gd = load_golden("burgers_accuracy"), load_reference_run(), load_golden("burgers_inf"), load_golden("burgers_ide")
    rng = np.random.default_rng(2024)
    out = []

    def inf(name, w, lb, ub, X_f, X_u, u):
        out.append(dict(name="inf/" + name, pde=BURGERS_INF, layers=BURGERS, lb=np.asarray(lb, float), ub=np.asarray(ub, float),
                        nu=NU, X_f=X_f, X_u=X_u, u=u, w=np.asarray(w, float)))

    def ide(name, w, lb, ub, X_u, u):
        out.append(dict(name="ide/" + name, pde=BURGERS_IDE, layers=BURGERS, lb=np.asarray(lb, float), ub=np.asarray(ub, float),
                        X_u=X_u, u=u, w=np.asarray(w, float)))

    # trained weights (100 Adam steps + 200 L-BFGS iterations; the reference's default schedule), N_f = 10 000
    inf("trained_oracle_w", a["oracle_w"], a["lb"], a["ub"], a["X_f"], a["X_u"], a["u"])
    inf("trained_schedule_w", r["schedule_w"], a["lb"], a["ub"], a["X_f"], a["X_u"], a["u"])
    # identification on 2000 points of the exact solution, trained net, lambdas at the truth and far from it
    k = rng.choice(a["X_star"].shape[0], 2000, replace=False)
    for wk, wn in (("oracle_w", a["oracle_w"]), ("schedule_w", r["schedule_w"])):
        for tag, lam in (("truth", [1.0, np.log(NU)]), ("off", [0.3, -10.0])):
            ide("trained_%s_%s" % (wk, tag), np.concatenate([wn, lam]), a["lb"], a["ub"], a["X_star"][k], a["u_star"][k])
    # saturated units: initialisation weights scaled
    for s in (2.0, 3.0):
        inf("init_x%d" % s, s * gi["w"], gi["lb"], gi["ub"], gi["X_f"], gi["X_u"], gi["u"])
        ide("init_x%d" % s, np.concatenate([s * gd["w"][:-2], gd["w"][-2:]]), gd["lb"], gd["ub"], gd["X_u"], gd["u"])
    # non-unit, asymmetric domains; a ragged count
    for name, lb, ub, n in (("domain_0_2pi", [0.0, 0.0], [2 * np.pi, 5.0], 4000), ("domain_m3_8", [-3.0, 0.5], [8.0, 2.0], 4737)):
        X_f, X_u = box(rng, lb, ub, n), box(rng, lb, ub, 100)
        inf(name, gi["w"], lb, ub, X_f, X_u, np.sin(X_u[:, :1]) * np.exp(-X_u[:, 1:]))
        ide(name, np.concatenate([gi["w"], [0.7, -4.0]]), lb, ub, X_f, np.sin(X_f[:, :1]) * np.exp(-X_f[:, 1:]))
    # point-position edges, all inside one ragged set
    lb, ub = np.array([-3.0, 0.5]), np.array([8.0, 2.0])
    X_f, X_u = edge_set(rng, lb, ub, 1200), edge_set(rng, lb, ub, 60)
    inf("edges", gi["w"], lb, ub, X_f, X_u, np.cos(X_u[:, :1]))
    ide("edges", np.concatenate([gi["w"], [0.7, -4.0]]), lb, ub, X_f, np.cos(X_f[:, :1]))
    return out


def nls_cases():
    g = load_golden("nls_inf")
    rng = np.random.default_rng(2025)
    out = []
    for s in (2.0, 3.0):
        out.append(dict(name="nls/init_x%d" % s, pde=NLS_INF, layers=NLS, lb=g["lb"], ub=g["ub"], X_f=box(rng, g["lb"], g["ub"], 3000),
                        tb=g["tb"], X0=g["x0"], uv0=g["uv0"], w=s * g["w"]))
    lb, ub = np.array([-5.0, 1.0]), np.array([5.0, 3.0])
    x0 = np.linspace(-5.0, 5.0, 61)[:, None]
    out.append(dict(name="nls/domain_t_1_3", pde=NLS_INF, layers=NLS, lb=lb, ub=ub, X_f=box(rng, lb, ub, 2999),
                    tb=1.0 + 2.0 * rng.random((40, 1)), X0=np.hstack([x0, np.ones_like(x0)]),
                    uv0=np.hstack([2.0 / np.cosh(x0), 0.0 * x0]), w=g["w"]))
    return out


def disc_cases():
    d, e = load_golden("burgers_disc"), load_golden("burgers_ide_disc")
    rng = np.random.default_rng(2026)
    Ld, Le = [int(v) for v in d["layers"]], [int(v) for v in e["layers"]]
    out = []

    def disc(name, w, lb, ub, x_0, u_0, x_1):
        out.append(dict(name="disc/" + name, pde=BURGERS_DISC, layers=Ld, lb=np.asarray(lb, float), ub=np.asarray(ub, float),
                        nu=float(d["nu"]), dt=float(d["dt"]), IRK=d["IRK"].astype(np.float64), x_0=x_0, u_0=u_0, x_1=x_1, w=w))

    def ided(name, w, lb, ub, x_0, u_0, x_1, u_1):
        out.append(dict(name="ide_disc/" + name, pde=BURGERS_IDE_DISC, layers=Le, lb=np.asarray(lb, float), ub=np.asarray(ub, float),
                        dt=float(e["dt"]), IRK_alpha=e["IRK_alpha"], IRK_beta=e["IRK_beta"], x_0=x_0, u_0=u_0, x_1=x_1, u_1=u_1, w=w))

    for s in (2.0, 3.0):
        disc("init_x%d" % s, s * d["w"], d["lb"], d["ub"], d["x_0"], d["u_0"], d["x_1"])
        ided("init_x%d" % s, np.concatenate([s * e["w"][:-2], e["w"][-2:]]), e["lb"], e["ub"], e["x_0"], e["u_0"], e["x_1"], e["u_1"])
    x_0, x_1 = 4.0 * rng.random((250, 1)), 4.0 * rng.random((201, 1))
    disc("domain_0_4", d["w"], [0.0], [4.0], x_0, -np.sin(np.pi * x_0 / 2), np.array([[0.0], [4.0]]))
    ided("domain_0_4", e["w"], [0.0], [4.0], x_0[:199], -np.sin(np.pi * x_0[:199] / 2), x_1, -0.5 * np.sin(np.pi * x_1 / 2))
    return out


def oracle(c, dtype):
    """(loss, parts as the kernel reports them [3], gradient) of the Taylor oracle in `dtype`."""
    from oracle import taylor as ty
    pde = c["pde"]
    if pde == BURGERS_INF:
        f, g, (pu, pf) = ty.burgers_loss_grad(c["w"], c["layers"], c["lb"], c["ub"], c["X_f"], c["X_u"], c["u"], nu=c["nu"], dtype=dtype)
        parts = [pu, 0, pf]
    elif pde == BURGERS_IDE:
        f, g, (pu, pf) = ty.burgers_loss_grad(c["w"], c["layers"], c["lb"], c["ub"], None, c["X_u"], c["u"], identification=True,
                                              dtype=dtype)
        parts = [pu, 0, pf]
    elif pde == NLS_INF:
        f, g, parts = ty.schrodinger_loss_grad(c["w"], c["layers"], c["lb"], c["ub"], c["X_f"], c["tb"], c["X0"], c["uv0"], dtype=dtype)
    elif pde == BURGERS_DISC:
        f, g, (p0, p1) = ty.burgers_disc_loss_grad(c["w"], c["layers"], c["lb"], c["ub"], c["x_0"], c["u_0"], c["x_1"], c["nu"], c["dt"],
                                                   c["IRK"], dtype=dtype)
        parts = [p0, p1, 0]
    else:
        f, g, (p0, p1) = ty.burgers_ide_disc_loss_grad(c["w"], c["layers"], c["lb"], c["ub"], c["x_0"], c["u_0"], c["x_1"], c["u_1"],
                                                       c["dt"], c["IRK_alpha"], c["IRK_beta"], dtype=dtype)
        parts = [p0, p1, 0]
    return np.array([f], dtype), np.array(parts, dtype), np.asarray(g, dtype)


class _KernelTanhNumpy(object):
    """numpy as the oracle module sees it, except that tanh is the fused kernels' own device routine."""

    def __init__(self, device_tanh):
        self._device_tanh = device_tanh

    def __getattr__(self, name):
        return getattr(np, name)

    def tanh(self, x):
        x = np.asarray(x, np.float64)
        return self._device_tanh(x.reshape(-1)).reshape(x.shape)


def oracle_kernel_tanh(c):
    """The fp64 oracle with the fused kernels' tanh."""
    import pinn_cabi
    from oracle import taylor as ty
    pinn_cabi.load()
    ty.np = _KernelTanhNumpy(pinn_cabi.device_tanh)
    try:
        return oracle(c, np.float64)
    finally:
        ty.np = np


def blocks(c):
    """(label, slice) of every checked quantity of the flat gradient: W_l and b_l per layer, each lambda entry."""
    out, o, L = [], 0, c["layers"]
    for l in range(len(L) - 1):
        out.append(("W%d" % l, slice(o, o + L[l] * L[l + 1]))); o += L[l] * L[l + 1]
        out.append(("b%d" % l, slice(o, o + L[l + 1]))); o += L[l + 1]
    if c["pde"] in (BURGERS_IDE, BURGERS_IDE_DISC):
        out += [("lambda1", slice(o, o + 1)), ("lambda2", slice(o + 1, o + 2))]
    return out


def rel_ld(x, ref):
    """|x - ref| / |ref| evaluated in long double (x is converted exactly); None when ref is zero."""
    ref = np.asarray(ref, LD).reshape(-1)
    n = np.sqrt(np.sum(ref * ref))
    if n == 0:
        return None
    d = np.asarray(x, LD).reshape(-1) - ref
    return float(np.sqrt(np.sum(d * d)) / n)


def judge(rows, case, variant, items):
    """items: (block, K, Os, R), Os one or more fp64 oracle results.  Appends (case, variant, block, e_K, e_O, ratio, ok) to rows."""
    for block, K, Os, R in items:
        eK, eO = rel_ld(K, R), max(rel_ld(O, R) or 0.0 for O in Os)
        if eK is None:
            ok = bool(np.all(np.asarray(K) == 0))
            rows.append((case, variant, block, 0.0 if ok else np.inf, 0.0, 0.0, ok))
            continue
        rows.append((case, variant, block, eK, eO, eK / max(eO, EPS), eK <= max(FACTOR * eO, FLOOR)))


def table(rows):
    head = "%-34s %-16s %-8s %10s %10s %8s" % ("case", "variant", "block", "e_K", "e_O", "e_K/e_O")
    return "\n".join([head] + ["%-34s %-16s %-8s %10.2e %10.2e %8.2f%s" % (r[0], r[1], r[2], r[3], r[4], r[5], "" if r[6] else "  FAIL")
                               for r in rows])


# ---------------------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def cases():
    return burgers_cases() + nls_cases() + disc_cases()


@pytest.fixture(scope="module")
def references(cases):
    """name -> ((loss, parts, grad) in long double, the same in fp64, the same in fp64 with the kernels' tanh)."""
    return {c["name"]: (oracle(c, LD), oracle(c, np.float64), oracle_kernel_tanh(c)) for c in cases}


@pytest.fixture(scope="module")
def runs(cases, tmp_path_factory):
    """variant -> {name: (loss, parts, grad, [block, dyn_smem, launches])}, one worker process per kernel-selection environment."""
    d = tmp_path_factory.mktemp("extended_precision")
    src = str(d / "cases.pkl")
    with open(src, "wb") as f:
        pickle.dump(cases, f)
    out = {}
    for variant, (env, pdes) in VARIANTS.items():
        names = [c["name"] for c in cases if c["pde"] in pdes]
        dst = str(d / (variant + ".npz"))
        e = {k: v for k, v in os.environ.items() if k not in ("PINN_FUSED_TAIL", "PINN_BURGERS_KERNEL", "PINN_FORCE_GENERIC",
                                                             "PINN_GENERIC_DFMA")}
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "extended_precision_worker.py"), ROOT, src, dst] + names,
                           env=dict(e, **env), capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (variant, r.stderr[-3000:])
        with np.load(dst) as z:
            out[variant] = {n: (z[n + "/loss"], z[n + "/parts"], z[n + "/grad"], z[n + "/kernel"]) for n in names}
    return out


# ---------------------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_loss_and_gradient_as_accurate_as_fp64_oracle(variant, cases, references, runs):
    rows = []
    for c in cases:
        if c["name"] not in runs[variant]:
            continue
        (Rf, Rp, Rg), (Of, Op, Og), (Tf, Tp, Tg) = references[c["name"]]
        Kf, Kp, Kg, _ = runs[variant][c["name"]]
        items = [("loss", Kf, (Of, Tf), Rf)] + [("part%d" % i, Kp[i], (Op[i], Tp[i]), Rp[i]) for i in range(3)]
        items += [(b, Kg[s], (Og[s], Tg[s]), Rg[s]) for b, s in blocks(c)]
        judge(rows, c["name"], variant, items)
    assert rows
    worst = max(rows, key=lambda r: r[5])
    print("\n%s: largest e_K / max(e_O, eps) = %.2f (%s, %s)" % (variant, worst[5], worst[0], worst[2]))
    assert all(r[6] for r in rows), "\n" + table([r for r in rows if not r[6]] + [worst])


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_each_variant_runs_the_kernel_it_names(variant, runs):
    for name, (_, _, _, (block, smem, launches)) in runs[variant].items():
        if variant.startswith("generic"):
            assert block == 256 and smem == 0, (name, block, smem)                    # the generic kernel
        elif variant == "v1":
            assert block == 128 and smem > 100000 and launches >= 2, (name, block, smem, launches)
        else:                                                                           # v2 (256 threads) and the NLS kernel
            assert block == 256 and smem > 100000, (name, block, smem)
        if variant == "v2_fused_tail":
            assert launches == 1, (name, launches)                                      # reduction done by the last CTAs
        if variant == "v2_two_launch":
            assert launches >= 2, (name, launches)


def test_fused_tail_equals_the_tail_kernels_bit_for_bit(runs):
    """The in-kernel tail reduces the partials in the same order as the tail kernels."""
    a, b = runs["v2_fused_tail"], runs["v2_two_launch"]
    for name in a:
        assert a[name][0] == b[name][0] and np.array_equal(a[name][1], b[name][1]) and np.array_equal(a[name][2], b[name][2]), name


def test_dmma_and_dfma_forms_both_ran(runs):
    """Same maths, different summation order of the hidden-to-hidden products: results differ in the last bits."""
    a, b = runs["generic_dmma"], runs["generic_dfma"]
    for name in a:
        assert not np.array_equal(a[name][2], b[name][2]), name


def forward_ld(c, X, dtype):
    from oracle import taylor as ty
    net = c["w"][:-2] if c["pde"] in (BURGERS_IDE, BURGERS_IDE_DISC) else c["w"]
    return ty.forward(net, c["layers"], c["lb"], c["ub"], X, dtype)[0]


def residual_of(c, streams, dtype):
    U, Ux, Ut, Uxx = streams
    if c["pde"] == NLS_INF:
        u, v = U[:, 0], U[:, 1]
        h2 = u * u + v * v
        return np.stack([Ut[:, 0] + 0.5 * Uxx[:, 1] + h2 * v, Ut[:, 1] - 0.5 * Uxx[:, 0] - h2 * u], 1)
    if c["pde"] == BURGERS_IDE:
        w = np.asarray(c["w"], dtype)
        l1, kappa = w[-2], np.exp(w[-1])
    else:
        l1, kappa = 1.0, c["nu"]
    return Ut + l1 * U * Ux - kappa * Uxx


def test_predict_derivatives_residual_as_accurate_as_fp64_oracle(cases):
    """mlp_forward_generic<1> (predict) and <4> (derivatives, residual) in the saturated and non-unit-domain regimes."""
    import pinn_cabi
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from extended_precision_worker import make
    pinn_cabi.load()
    rows = []
    for c in cases:
        if not any(k in c["name"] for k in ("init_x", "domain", "edges")):
            continue
        X = c["X_u"] if c["pde"] == BURGERS_IDE else (c["x_0"] if c["pde"] in (BURGERS_DISC, BURGERS_IDE_DISC) else c["X_f"])
        p = make(c)
        p.set_weights(c["w"])
        K = p.derivatives(X)
        R, O = forward_ld(c, X, LD), forward_ld(c, X, np.float64)
        items = [(s, K[i], (O[i],), R[i]) for i, s in enumerate(("u", "u_x", "u_t", "u_xx"))]
        items.append(("predict", p.predict(X), (O[0],), R[0]))
        if c["pde"] in (BURGERS_INF, BURGERS_IDE, NLS_INF):
            items.append(("f", p.residual(), (residual_of(c, O, np.float64),), residual_of(c, R, LD)))
        p.close()
        judge(rows, c["name"], "forward", items)
    worst = max(rows, key=lambda r: r[5])
    print("\nforward: largest e_K / max(e_O, eps) = %.2f (%s, %s)" % (worst[5], worst[0], worst[2]))
    assert all(r[6] for r in rows), "\n" + table([r for r in rows if not r[6]] + [worst])
