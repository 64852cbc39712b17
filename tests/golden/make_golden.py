"""Generate the golden parity fixtures (tests/golden/*.npz).

Needs a checkout of the original project in $PINN_REFERENCE_DIR (it reads the reference's data files):
    PYTHONPATH=. python tests/golden/make_golden.py

The reference ships no golden vectors and TensorFlow 2.0 cannot be installed here (parity against TF's kernels UNPINNED), so the
vectors come from ``oracle.reference_port`` (nested reverse-mode restatement of the reference) and every
loss/gradient is cross-checked against the independent ``oracle.taylor`` before it is written.  make_reference_fixtures.py then
runs the reference's own Python (on an emulated TensorFlow) over the same inputs and must reproduce these values.
"""
import os
import sys

import numpy as np
import scipy.io

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import reference_port as rp, taylor as ty  # noqa: E402

OUT = os.environ.get("PINN_GOLDEN_OUT", os.path.dirname(os.path.abspath(__file__)))      # tests regenerate into a scratch dir
REF = os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")


def lhs(n, d, rng):
    """pyDOE ``lhs(d, n)`` classic: per-dimension stratified uniform + independent permutation."""
    cut = np.linspace(0, 1, n + 1)
    u = rng.random((n, d))
    pts = u * (cut[1:] - cut[:n])[:, None] + cut[:n][:, None]
    for j in range(d):
        pts[:, j] = pts[rng.permutation(n), j]
    return pts


def check(name, f, g, f2, g2):
    rel_f = abs(f - f2) / abs(f)
    rel_g = np.linalg.norm(g - g2) / np.linalg.norm(g)
    print(f"{name}: loss {f:.15e} cross-check rel {rel_f:.2e}, grad rel {rel_g:.2e}")
    assert rel_f < 1e-12 and rel_g < 1e-12, name


def burgers_data(rng, n_u):
    """IC/BC training points as in 1d-burgers/burgersutil.py:104-129."""
    d = scipy.io.loadmat(os.path.join(REF, "1d-burgers", "data", "burgers_shock.mat"))
    t = d["t"].flatten()[:, None]; x = d["x"].flatten()[:, None]
    Exact = np.real(d["usol"]).T
    X, T = np.meshgrid(x, t)
    X_star = np.hstack((X.flatten()[:, None], T.flatten()[:, None]))
    u_star = Exact.flatten()[:, None]
    lb, ub = X_star.min(0), X_star.max(0)
    xx = np.vstack([np.hstack((X[0:1, :].T, T[0:1, :].T)), np.hstack((X[:, 0:1], T[:, 0:1])), np.hstack((X[:, -1:], T[:, -1:]))])
    uu = np.vstack([Exact[0:1, :].T, Exact[:, 0:1], Exact[:, -1:]])
    idx = rng.choice(xx.shape[0], n_u, replace=False)
    return lb, ub, xx[idx], uu[idx], X_star, u_star


def make_burgers_inf():
    rng = np.random.default_rng(1234)
    layers = [2] + [20] * 8 + [1]
    lb, ub, X_u, u, X_star, u_star = burgers_data(rng, 100)
    n_f = 1000
    X_f = lb + (ub - lb) * lhs(n_f, 2, rng)
    nu = 0.01 / np.pi
    w0 = rp.glorot_normal_flat(layers, rng)
    # biases are zero at initialisation; perturb so that bias paths are exercised
    w = w0 + 0.02 * rng.standard_normal(w0.size)
    pb = rp.BurgersInference(layers, lb, ub, nu, X_f, X_u, u)
    f, g = rp.loss_and_flat_grad(pb, w)
    f2, g2, parts = ty.burgers_loss_grad(w, layers, lb, ub, X_f, X_u, u, nu=nu)
    check("burgers_inf", f, g, f2, g2)
    import torch
    _, (U, Ux, Ut, Uxx) = pb.residual(torch.as_tensor(w))
    probes = np.stack([a.detach().numpy()[:64, 0] for a in (U, Ux, Ut, Uxx)], 1)
    fres = (Ut + U * Ux - nu * Uxx).detach().numpy()
    wa, la, _ = rp.adam_train(pb, w, 5, lr=1e-3)
    wa2, la2, _ = rp.adam_train(pb, w, 5, lr=0.03)
    tr = rp.lbfgs_fixed_step(lambda x: rp.loss_and_flat_grad(pb, x), w, max_iter=6, learning_rate=0.8, n_correction=50,
                             tol_fun=np.finfo(float).eps)
    idxs = rng.choice(X_star.shape[0], 200, replace=False)
    np.savez_compressed(os.path.join(OUT, "burgers_inf.npz"), layers=layers, lb=lb, ub=ub, nu=nu, X_f=X_f, X_u=X_u, u=u, w=w,
                        w_init=w0, loss=f, parts=np.array(parts), grad=g, probes=probes, residual=fres,
                        adam_lr=np.array([1e-3, 0.03]), adam_losses=np.stack([la, la2]), adam_w=np.stack([wa, wa2]),
                        lbfgs_x_eval=np.array(tr.x_eval), lbfgs_f=np.array(tr.f_hist), lbfgs_t=np.array(tr.t),
                        lbfgs_x_final=tr.x_final, lbfgs_n_iter=tr.n_iter, lbfgs_n_eval=tr.n_eval,
                        lbfgs_logged=np.array(tr.logged), X_star=X_star[idxs], u_star=u_star[idxs],
                        predict=rp.predict(pb, w, X_star[idxs]))


def make_burgers_ide():
    rng = np.random.default_rng(4321)
    layers = [2] + [20] * 8 + [1]
    d = scipy.io.loadmat(os.path.join(REF, "1d-burgers", "data", "burgers_shock.mat"))
    t = d["t"].flatten()[:, None]; x = d["x"].flatten()[:, None]
    Exact = np.real(d["usol"]).T
    X, T = np.meshgrid(x, t)
    X_star = np.hstack((X.flatten()[:, None], T.flatten()[:, None]))
    u_star = Exact.flatten()[:, None]
    lb, ub = X_star.min(0), X_star.max(0)
    idx = rng.choice(X_star.shape[0], 500, replace=False)      # burgersutil.py:72-75
    X_u, u = X_star[idx], u_star[idx]
    w = rp.glorot_normal_flat(layers, rng) + 0.02 * rng.standard_normal(3021)
    w = np.concatenate([w, [0.0, -6.0]])                         # ide_cont_burgers.py:52-53
    pb = rp.BurgersIdentification(layers, lb, ub, X_u, u)
    f, g = rp.loss_and_flat_grad(pb, w)
    f2, g2, parts = ty.burgers_loss_grad(w, layers, lb, ub, None, X_u, u, identification=True)
    check("burgers_ide", f, g, f2, g2)
    w2 = w.copy(); w2[-2:] = [0.7, -4.0]
    fb, gb = rp.loss_and_flat_grad(pb, w2)
    fb2, gb2, _ = ty.burgers_loss_grad(w2, layers, lb, ub, None, X_u, u, identification=True)
    check("burgers_ide(l1=.7,l2=-4)", fb, gb, fb2, gb2)
    wa, la, _ = rp.adam_train(pb, w, 5, lr=1e-3)
    tr = rp.lbfgs_fixed_step(lambda x: rp.loss_and_flat_grad(pb, x), w, max_iter=5, learning_rate=0.8, n_correction=50,
                             tol_fun=np.finfo(float).eps)
    np.savez_compressed(os.path.join(OUT, "burgers_ide.npz"), layers=layers, lb=lb, ub=ub, X_u=X_u, u=u, w=w, loss=f,
                        parts=np.array(parts), grad=g, w2=w2, loss2=fb, grad2=gb, adam_losses=la, adam_w=wa,
                        lbfgs_x_eval=np.array(tr.x_eval), lbfgs_f=np.array(tr.f_hist), lbfgs_x_final=tr.x_final,
                        lbfgs_n_iter=tr.n_iter, lbfgs_n_eval=tr.n_eval)


def make_nls():
    rng = np.random.default_rng(777)
    layers = [2, 100, 100, 100, 100, 2]
    d = scipy.io.loadmat(os.path.join(REF, "1dcomplex-schrodinger", "data", "NLS.mat"))
    t = d["tt"].flatten()[:, None]; x = d["x"].flatten()[:, None]
    Exact = d["uu"]
    lb, ub = np.array([-5.0, 0.0]), np.array([5.0, np.pi / 2])   # schrodingerutil.py:41-42
    idx_x = rng.choice(x.shape[0], 50, replace=False)
    x0 = x[idx_x, :]
    uv0 = np.hstack([np.real(Exact)[idx_x, 0:1], np.imag(Exact)[idx_x, 0:1]])
    tb = t[rng.choice(t.shape[0], 50, replace=False), :]
    X_f = lb + (ub - lb) * lhs(400, 2, rng)
    w = rp.glorot_normal_flat(layers, rng) + 0.01 * rng.standard_normal(30802)
    out = dict(layers=layers, lb=lb, ub=ub, X_f=X_f, tb=tb, x0=x0, uv0=uv0, w=w)
    for tag, X0 in (("q1", x0), ("x0t0", np.concatenate([x0, 0 * x0], 1))):
        pb = rp.SchrodingerInference(layers, lb, ub, X_f, tb, X0, uv0)
        f, g = rp.loss_and_flat_grad(pb, w)
        f2, g2, parts = ty.schrodinger_loss_grad(w, layers, lb, ub, X_f, tb, X0, uv0)
        check("nls_" + tag, f, g, f2, g2)
        out["loss_" + tag] = f; out["grad_" + tag] = g; out["parts_" + tag] = np.array(parts)
    pb = rp.SchrodingerInference(layers, lb, ub, X_f, tb, x0, uv0)
    wa, la, _ = rp.adam_train(pb, w, 3, lr=0.05, b1=0.99, eps=0.1)   # inf_cont_schrodinger.py:33-36
    out["adam_losses"] = la; out["adam_w"] = wa
    import torch
    fu, fv, dd = pb.residual(torch.as_tensor(w))
    out["probes"] = np.stack([a.detach().numpy()[:32, 0] for a in dd], 1)    # u v u_x v_x u_t v_t u_xx v_xx
    out["residual"] = np.hstack([fu.detach().numpy(), fv.detach().numpy()])
    Xs = lb + (ub - lb) * rng.random((100, 2))
    out["X_star"] = Xs; out["predict"] = rp.predict(pb, w, Xs)
    np.savez_compressed(os.path.join(OUT, "nls_inf.npz"), **out)


if __name__ == "__main__" and "--disc" not in sys.argv and "--ide-disc" not in sys.argv:
    make_burgers_inf()
    make_burgers_ide()
    make_nls()
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, "KiB")


def make_burgers_disc():
    """Discrete-time (q-stage IRK) Burgers inference, 1d-burgers/inf_disc_burgers.py, with the upstream q=100 table."""
    sys.path.insert(0, os.path.join(ROOT, "pinns-tf2.0_b200", "1d-burgers"))
    import burgersutil
    rng = np.random.default_rng(2024)
    np.random.seed(1234)
    q = 100
    lb, ub = np.array([-1.0]), np.array([1.0])
    cwd = os.getcwd(); os.chdir(REF)
    try:
        x, t, dt, Exact_u, x_0, u_0, x_1, x_star, u_star, IRK_w, IRK_t = burgersutil.prep_data(
            os.path.join(REF, "1d-burgers", "data", "burgers_shock.mat"), N_n=250, q=q, lb=lb, ub=ub, noise=0.0, idx_t_0=10, idx_t_1=90)
    finally:
        os.chdir(cwd)
    layers = [1, 50, 50, 50, q + 1]
    w = rp.glorot_normal_flat(layers, rng) + 0.02 * rng.standard_normal(rp.num_params(layers))
    nu, dtv = 0.01 / np.pi, float(np.asarray(dt).reshape(-1)[0])
    pb = rp.BurgersDiscreteInference(layers, lb, ub, nu, dtv, x_0, u_0, x_1, IRK_w)
    f, g = rp.loss_and_flat_grad(pb, w)
    f2, g2, parts = ty.burgers_disc_loss_grad(w, layers, lb, ub, x_0, u_0, x_1, nu, dtv, IRK_w)
    check("burgers_disc", f, g, f2, g2)
    wa, la, _ = rp.adam_train(pb, w, 3, lr=1e-3, eps=1e-8)                 # inf_disc_burgers.py:38-41
    np.savez_compressed(os.path.join(OUT, "burgers_disc.npz"), layers=layers, lb=lb, ub=ub, nu=nu, dt=dtv, q=q, x_0=x_0, u_0=u_0,
                        x_1=x_1, IRK=IRK_w.astype(np.float32), w=w, loss=f, parts=np.array(parts), grad=g, adam_losses=la,
                        adam_w=wa, x_star=x_star, predict=rp.predict(pb, w, x_star)[:, -1])


if __name__ == "__main__" and "--disc" in sys.argv:
    make_burgers_disc()


def make_burgers_ide_disc():
    """Discrete-time Burgers identification, 1d-burgers/ide_disc_burgers.py, with the script's data (N_0=199, N_1=201,
    idx_t 10 -> 90, hence dt = 0.8 and the upstream q=81 table)."""
    sys.path.insert(0, os.path.join(ROOT, "pinns-tf2.0_b200", "1d-burgers"))
    import burgersutil
    rng = np.random.default_rng(81)
    np.random.seed(1234)
    lb, ub = np.array([-1.0]), np.array([1.0])
    cwd = os.getcwd(); os.chdir(REF)
    try:
        x_0, u_0, x_1, u_1, x_star, t_star, dt, q, Exact_u, alpha, beta = burgersutil.prep_data(
            os.path.join(REF, "1d-burgers", "data", "burgers_shock.mat"), N_0=199, N_1=201, lb=lb, ub=ub, noise=0.0, idx_t_0=10, idx_t_1=90)
    finally:
        os.chdir(cwd)
    layers = [1, 50, 50, 50, q]                                             # ide_disc_burgers.py:34, :222
    out = dict(layers=layers, lb=lb, ub=ub, dt=dt, q=q, x_0=x_0, u_0=u_0, x_1=x_1, u_1=u_1, IRK_alpha=alpha.astype(np.float32),
               IRK_beta=beta.astype(np.float32), x_star=x_star)
    wn = rp.glorot_normal_flat(layers, rng) + 0.02 * rng.standard_normal(rp.num_params(layers))
    pb = rp.BurgersDiscreteIdentification(layers, lb, ub, dt, x_0, u_0, x_1, u_1, alpha, beta)
    for tag, lam in (("", [0.0, -6.0]), ("2", [0.7, -4.0])):                # :151-152 initial values, then a generic point
        w = np.concatenate([wn, lam])
        f, g = rp.loss_and_flat_grad(pb, w)
        f2, g2, parts = ty.burgers_ide_disc_loss_grad(w, layers, lb, ub, x_0, u_0, x_1, u_1, dt, alpha, beta)
        check("burgers_ide_disc" + tag, f, g, f2, g2)
        out["w" + tag], out["loss" + tag], out["grad" + tag], out["parts" + tag] = w, f, g, np.array(parts)
    wa, la, _ = rp.adam_train(pb, out["w2"], 3, lr=1e-3)                    # :37-40 (tf_eps None -> 1e-7)
    out["adam_losses"], out["adam_w"] = la, wa
    tr = rp.lbfgs_fixed_step(lambda z: rp.loss_and_flat_grad(pb, z), out["w2"], max_iter=4, learning_rate=0.8, n_correction=50,
                             tol_fun=np.finfo(float).eps)
    out["lbfgs_x_eval"], out["lbfgs_f"], out["lbfgs_x_final"] = np.array(tr.x_eval), np.array(tr.f_hist), tr.x_final
    out["x_star"] = x_star[::8]                                             # 32 probe positions keep the fixture small
    U0, U1 = pb.predict(out["w2"], out["x_star"])
    out["predict_U0"], out["predict_U1"] = U0, U1
    np.savez_compressed(os.path.join(OUT, "burgers_ide_disc.npz"), **out)
    print("burgers_ide_disc.npz", os.path.getsize(os.path.join(OUT, "burgers_ide_disc.npz")) // 1024, "KiB, q =", q, "P =", out["w"].size)


if __name__ == "__main__" and "--ide-disc" in sys.argv:
    make_burgers_ide_disc()
