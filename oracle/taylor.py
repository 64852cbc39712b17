"""Independent fp64 oracle: forward Taylor-mode (streams h, h_x, h_t, h_xx) + hand-derived reverse sweep.

TEST INFRASTRUCTURE (see oracle/__init__.py).  numpy only; shares no code or derivation with
``oracle.reference_port`` (nested autograd).  The two must agree to ~1e-13 -- that agreement is what
is the independent check of the mathematics; the pin to the reference's own code is tests/golden/reference_run.npz
(parity against TensorFlow's kernels themselves remains UNPINNED: TF cannot be installed).

Maths (SURVEY.md Appendix A).  Input layer (utils/neuralnetwork.py:29-30):
    h = 2(X-lb)/(ub-lb)-1,  h_x = [2/(ub0-lb0), 0],  h_t = [0, 2/(ub1-lb1)],  h_xx = 0
tanh layer, z = hW+b, a = tanh z, s = 1-a^2:
    z_x = h_x W, z_t = h_t W, z_xx = h_xx W;  a_x = s z_x, a_t = s z_t, a_xx = s z_xx - 2 a s z_x^2
linear head: same contraction, no activation.
Reverse through a tanh layer given adjoints (A, A_x, A_t, A_xx) of (a, a_x, a_t, a_xx):
    Z_x = s A_x - 4 a s z_x A_xx;  Z_t = s A_t;  Z_xx = s A_xx
    Z   = s [A - 2a z_x A_x - 2a z_t A_t + A_xx(-2a z_xx - 2 z_x^2 (1-3a^2))]
    dW += h^T Z + h_x^T Z_x + h_t^T Z_t + h_xx^T Z_xx;  db += sum Z;  input adjoints = (Z, Z_x, Z_t, Z_xx) W^T

``dtype`` (default float64) is the arithmetic type.  With ``dtype=np.longdouble`` the same fp64 inputs (weights, points, nu, dt,
lb/ub, IRK tables) go through 64-bit-mantissa arithmetic, which gives the exact function of what a kernel receives to ~1e-19:
the reference of tests/test_gpu_extended_precision.py.  Losses come back as ``dtype`` scalars.  The float64 path is unchanged.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np


def _shapes(layers):
    return [(int(layers[i]), int(layers[i + 1])) for i in range(len(layers) - 1)]


def _unpack(w, layers):
    Ws, bs, o = [], [], 0
    for fi, fo in _shapes(layers):
        Ws.append(w[o:o + fi * fo].reshape(fi, fo)); o += fi * fo
        bs.append(w[o:o + fo]); o += fo
    return Ws, bs


def forward(w, layers, lb, ub, X, dtype=np.float64):
    """X: (N,2) -> outputs (u, u_x, u_t, u_xx), each (N, n_out), and the per-layer stash."""
    X = np.asarray(X, dtype=dtype)
    lb, ub = np.asarray(lb, dtype).reshape(-1), np.asarray(ub, dtype).reshape(-1)
    Ws, bs = _unpack(np.asarray(w, dtype=dtype), layers)
    N = X.shape[0]
    if int(layers[0]) == 1:        # discrete-time models: 1-D input x (1d-burgers/inf_disc_burgers.py:34), no t stream
        sc = 2.0 / (ub[:1] - lb[:1])
        h = sc * (X[:, :1] - lb[:1]) - 1.0
        hx = np.full((N, 1), sc[0], dtype); ht = np.zeros((N, 1), dtype); hxx = np.zeros((N, 1), dtype)
    else:
        if X.shape[1] == 1:        # quirk Q1: (N,1) input broadcast by the Lambda to (x, t:=x)
            X = np.concatenate([X, X], axis=1)
        sc = 2.0 / (ub - lb)
        h = sc * (X - lb) - 1.0
        hx = np.zeros((N, 2), dtype); hx[:, 0] = sc[0]
        ht = np.zeros((N, 2), dtype); ht[:, 1] = sc[1]
        hxx = np.zeros((N, 2), dtype)
    stash = []
    L = len(Ws)
    for l in range(L - 1):
        W, b = Ws[l], bs[l]
        z, zx, zt, zxx = h @ W + b, hx @ W, ht @ W, hxx @ W
        a = np.tanh(z)
        s = 1.0 - a * a
        stash.append((h, hx, ht, hxx, a, s, zx, zt, zxx))
        h, hx, ht, hxx = a, s * zx, s * zt, s * zxx - 2.0 * a * s * zx * zx
    W, b = Ws[-1], bs[-1]
    out = (h @ W + b, hx @ W, ht @ W, hxx @ W)
    stash.append((h, hx, ht, hxx))
    return out, stash


def backward(w, layers, stash, seeds, dtype=np.float64):
    """seeds: adjoints of (u, u_x, u_t, u_xx), each (N, n_out).  Returns the flat parameter gradient."""
    Ws, _ = _unpack(np.asarray(w, dtype=dtype), layers)
    L = len(Ws)
    g = []
    h, hx, ht, hxx = stash[-1]
    Z, Zx, Zt, Zxx = seeds
    gW = h.T @ Z + hx.T @ Zx + ht.T @ Zt + hxx.T @ Zxx
    gb = Z.sum(0)
    g.append((gW, gb))
    A, Ax, At, Axx = Z @ Ws[-1].T, Zx @ Ws[-1].T, Zt @ Ws[-1].T, Zxx @ Ws[-1].T
    for l in range(L - 2, -1, -1):
        h, hx, ht, hxx, a, s, zx, zt, zxx = stash[l]
        Zx = s * Ax - 4.0 * a * s * zx * Axx
        Zt = s * At
        Zxx = s * Axx
        Z = s * (A - 2.0 * a * zx * Ax - 2.0 * a * zt * At + Axx * (-2.0 * a * zxx - 2.0 * zx * zx * (1.0 - 3.0 * a * a)))
        gW = h.T @ Z + hx.T @ Zx + ht.T @ Zt + hxx.T @ Zxx
        gb = Z.sum(0)
        g.append((gW, gb))
        if l > 0:
            WT = Ws[l].T
            A, Ax, At, Axx = Z @ WT, Zx @ WT, Zt @ WT, Zxx @ WT
    flat = []
    for gW, gb in reversed(g):
        flat.append(gW.reshape(-1)); flat.append(gb)
    return np.concatenate(flat)


def burgers_loss_grad(w, layers, lb, ub, X_f, X_u, u, nu=None, identification=False, n_f_global=None,
                      data_weight=1.0, dtype=np.float64) -> Tuple[float, np.ndarray, Tuple[float, float]]:
    """Burgers inference (1d-burgers/inf_cont_burgers.py:59-90) or identification
    (1d-burgers/ide_cont_burgers.py:56-91; w = [net, l1, l2], residual on X_u)."""
    w = np.asarray(w, dtype=dtype)
    if identification:
        wn, l1, kappa = w[:-2], w[-2], np.exp(w[-1])
        X_f = X_u
    else:
        wn, l1, kappa = w, 1.0, nu
    nf = n_f_global or X_f.shape[0]
    (U, Ux, Ut, Uxx), st = forward(wn, layers, lb, ub, X_f, dtype)
    f = Ut + l1 * U * Ux - kappa * Uxx
    c = 2.0 * f / nf
    g = backward(wn, layers, st, (c * l1 * Ux, c * l1 * U, c, -c * kappa), dtype)
    mse_f = dtype(np.sum(f * f) / nf)
    (Ud, _, _, _), std = forward(wn, layers, lb, ub, X_u, dtype)
    r = Ud - u
    nu_ = X_u.shape[0]
    zero = np.zeros_like(r)
    g = g + backward(wn, layers, std, (data_weight * 2.0 * r / nu_, zero, zero, zero), dtype)
    mse_u = data_weight * dtype(np.sum(r * r) / nu_)
    if identification:
        g = np.concatenate([g, [np.sum(c * U * Ux), np.sum(-c * kappa * Uxx)]])
    return mse_u + mse_f, g, (mse_u, mse_f)


def schrodinger_loss_grad(w, layers, lb, ub, X_f, tb, X0, uv0, n_f_global=None, aux_weight=1.0, dtype=np.float64):
    """1dcomplex-schrodinger/inf_cont_schrodinger.py:60-129."""
    w = np.asarray(w, dtype=dtype)
    lb, ub = np.asarray(lb, dtype), np.asarray(ub, dtype)
    nf = n_f_global or X_f.shape[0]
    (H, Hx, Ht, Hxx), st = forward(w, layers, lb, ub, X_f, dtype)
    u, v = H[:, 0], H[:, 1]
    h2 = u * u + v * v
    fu = Ht[:, 0] + 0.5 * Hxx[:, 1] + h2 * v
    fv = Ht[:, 1] - 0.5 * Hxx[:, 0] - h2 * u
    cu, cv = 2.0 * fu / nf, 2.0 * fv / nf
    S = np.stack([cu * 2 * u * v - cv * (3 * u * u + v * v), cu * (u * u + 3 * v * v) - cv * 2 * u * v], 1)
    St = np.stack([cu, cv], 1)
    Sxx = np.stack([-0.5 * cv, 0.5 * cu], 1)
    g = backward(w, layers, st, (S, np.zeros_like(S), St, Sxx), dtype)
    mse_f = dtype((np.sum(fu * fu) + np.sum(fv * fv)) / nf)
    # initial condition
    (H0, _, _, _), st0 = forward(w, layers, lb, ub, X0, dtype)
    r0 = H0 - uv0
    n0 = r0.shape[0]
    z = np.zeros_like(r0)
    g = g + backward(w, layers, st0, (aux_weight * 2.0 * r0 / n0, z, z, z), dtype)
    mse_0 = aux_weight * dtype(np.sum(r0 * r0) / n0)
    # periodic boundary
    tb = np.asarray(tb, dtype)
    Xl = np.concatenate([0 * tb + lb[0], tb], 1)
    Xu = np.concatenate([0 * tb + ub[0], tb], 1)
    (Hl, Hxl, _, _), stl = forward(w, layers, lb, ub, Xl, dtype)
    (Hu, Hxu, _, _), stu = forward(w, layers, lb, ub, Xu, dtype)
    nb = tb.shape[0]
    d, dx = Hl - Hu, Hxl - Hxu
    zb = np.zeros_like(d)
    k = aux_weight * 2.0 / nb
    g = g + backward(w, layers, stl, (k * d, k * dx, zb, zb), dtype) + backward(w, layers, stu, (-k * d, -k * dx, zb, zb), dtype)
    mse_b = aux_weight * dtype((np.sum(d * d) + np.sum(dx * dx)) / nb)
    return mse_0 + mse_b + mse_f, g, (mse_0, mse_b, mse_f)


def burgers_disc_loss_grad(w, layers, lb, ub, x_0, u_0, x_1, nu, dt, IRK_weights, dtype=np.float64):
    """Discrete-time (implicit Runge-Kutta, q stages) Burgers inference, 1d-burgers/inf_disc_burgers.py:49-127:
    net [1, ..., q+1]; U_1 = net(x) (N, q+1); U = U_1[:, :q]; N = U U_x - nu U_xx;
    U_0 = U_1 + dt N IRK^T  (IRK: (q+1, q));  loss = sum((U_0 - u_0)^2) + sum(net(x_1)^2)   (sums, not means, :98-101)."""
    w = np.asarray(w, dtype=dtype)
    IRK = np.asarray(IRK_weights, dtype=dtype)
    q = IRK.shape[1]
    (U1, U1x, _, U1xx), st = forward(w, layers, lb, ub, x_0, dtype)
    U, Ux, Uxx = U1[:, :q], U1x[:, :q], U1xx[:, :q]
    Nn = U * Ux - nu * Uxx
    U0 = U1 + dt * Nn @ IRK.T
    R = 2.0 * (U0 - u_0)                                  # u_0 (N,1) broadcasts over the q+1 stages
    Nbar = dt * R @ IRK                                   # (N, q)
    S = R.copy(); S[:, :q] += Nbar * Ux
    Sx = np.zeros_like(R); Sx[:, :q] = Nbar * U
    Sxx = np.zeros_like(R); Sxx[:, :q] = -nu * Nbar
    g = backward(w, layers, st, (S, Sx, np.zeros_like(R), Sxx), dtype)
    loss0 = dtype(np.sum((U0 - u_0) ** 2))
    (B1, _, _, _), stb = forward(w, layers, lb, ub, x_1, dtype)
    zb = np.zeros_like(B1)
    g = g + backward(w, layers, stb, (2.0 * B1, zb, zb, zb), dtype)
    loss1 = dtype(np.sum(B1 ** 2))
    return loss0 + loss1, g, (loss0, loss1)


def burgers_ide_disc_loss_grad(w, layers, lb, ub, x_0, u_0, x_1, u_1, dt, IRK_alpha, IRK_beta, dtype=np.float64):
    """Discrete-time Burgers identification, 1d-burgers/ide_disc_burgers.py:81-115: w = [net, l1, l2], net [1, ..., q];
    U_0 = U + dt N alpha^T on x_0, U_1 = U - dt N (beta - alpha)^T on x_1 with N = l1 U U_x - e^{l2} U_xx;
    loss = sum((U_0 - u_0)^2) + sum((U_1 - u_1)^2).  Both snapshots are the same computation with stage matrices
    M_0 = alpha and M_1 = -(beta - alpha) (beta broadcast over rows): pred = U + dt N M^T."""
    w = np.asarray(w, dtype=dtype)
    wn, l1, kappa = w[:-2], w[-2], np.exp(w[-1])
    A = np.asarray(IRK_alpha, dtype=dtype)
    # beta - alpha is formed by numpy in the tables' own dtype (float32 in the reference, ide_disc_burgers.py:107) and only then promoted
    M1 = -np.asarray(np.asarray(IRK_beta).reshape(1, -1) - np.asarray(IRK_alpha), dtype=dtype)
    g = np.zeros(wn.size, dtype)
    dl1 = dl2 = 0.0
    parts = []
    for x, u, M in ((x_0, u_0, A), (x_1, u_1, M1)):
        (U, Ux, _, Uxx), st = forward(wn, layers, lb, ub, x, dtype)
        Nn = l1 * U * Ux - kappa * Uxx
        R = 2.0 * (U + dt * Nn @ M.T - u)                   # u (N,1) broadcasts over the q stages
        Nbar = dt * R @ M
        g = g + backward(wn, layers, st, (R + Nbar * l1 * Ux, Nbar * l1 * U, np.zeros_like(R), -kappa * Nbar), dtype)
        dl1 += dtype(np.sum(Nbar * U * Ux))
        dl2 += dtype(np.sum(Nbar * (-kappa) * Uxx))
        parts.append(dtype(np.sum((0.5 * R) ** 2)))
    return parts[0] + parts[1], np.concatenate([g, [dl1, dl2]]), tuple(parts)
