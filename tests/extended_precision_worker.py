"""Worker for tests/test_gpu_extended_precision.py: evaluates loss, loss parts and gradient of every case it is given on the GPU,
under the kernel-selection environment variables of its own process (PINN_FUSED_TAIL and PINN_GENERIC_DFMA are read once per
process), and writes the results to an .npz.

    python extended_precision_worker.py <root> <cases.pkl> <out.npz> <case name> ...
"""
import os
import pickle
import sys

import numpy as np

ROOT = sys.argv[1]
sys.path[:0] = [ROOT, os.path.join(ROOT, "pinns-tf2.0_b200", "utils")]
import pinn_cabi  # noqa: E402


def make(c):
    """A handle holding the case's problem definition (the same calls as the Python surface makes)."""
    pde = c["pde"]
    p = pinn_cabi.Pinn(pde, c["layers"], c["lb"], c["ub"])
    if pde == pinn_cabi.BURGERS_INF:
        p.set_pde_params([c["nu"]]); p.set_collocation(c["X_f"][:, 0], c["X_f"][:, 1]); p.set_data(c["X_u"], c["u"])
    elif pde == pinn_cabi.BURGERS_IDE:
        p.set_data(c["X_u"], c["u"])
    elif pde == pinn_cabi.NLS_INF:
        p.set_collocation(c["X_f"][:, 0], c["X_f"][:, 1]); p.set_boundary(c["tb"]); p.set_data(c["X0"], c["uv0"])
    elif pde == pinn_cabi.BURGERS_DISC:
        p.set_pde_params([c["nu"], c["dt"]]); p.set_irk(c["IRK"]); p.set_boundary(c["x_1"]); p.set_data(c["x_0"], c["u_0"])
    else:
        p.set_pde_params([c["dt"]]); p.set_irk(pinn_cabi.irk_ide_disc(c["IRK_alpha"], c["IRK_beta"]))
        p.set_snapshot(0, c["x_0"], c["u_0"]); p.set_snapshot(1, c["x_1"], c["u_1"])
    return p


def main():
    pinn_cabi.load()
    with open(sys.argv[2], "rb") as f:
        cases = {c["name"]: c for c in pickle.load(f)}
    out = {}
    for name in sys.argv[4:]:
        c = cases[name]
        p = make(c)
        n0 = p.launch_count()
        loss, grad, parts = p.loss_grad(w=c["w"])
        info = p.kernel_info()
        out[name + "/loss"] = np.float64(loss)
        out[name + "/parts"] = parts
        out[name + "/grad"] = grad
        out[name + "/kernel"] = np.array([info["block"], info["dyn_smem"], p.launch_count() - n0])
        p.close()
    np.savez(sys.argv[3], **out)


if __name__ == "__main__":
    main()
