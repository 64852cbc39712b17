"""Fixture for the end-of-training accuracy check (BASELINE metric, second half: rel. L2 error of u against the
reference solution burgers_shock.mat): the full evaluation grid and the default training sets of
1d-burgers/inf_cont_burgers.py (N_u=100, N_f=10000, np.random.seed(1234)), produced by OUR prep_data restatement.
Also runs the reference's default schedule with the CPU oracle and stores its loss curve / final error.
    PYTHONPATH=. python tests/golden/make_accuracy_fixture.py"""
import os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "pinns-tf2.0_b200", "1d-burgers")); sys.path.insert(0, os.path.join(ROOT, "pinns-tf2.0_b200", "utils")); sys.path.insert(0, os.path.join(ROOT, "pinns-tf2.0_b200", "shims"))
import burgersutil
from oracle import reference_port as rp
from neuralnetwork import _glorot_normal
REF = os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")
np.random.seed(1234)
x, t, X, T, Exact_u, X_star, u_star, X_u, u, X_f, ub, lb = burgersutil.prep_data(
    os.path.join(REF, "1d-burgers", "data", "burgers_shock.mat"), 100, 10000, noise=0.0)
layers = [2] + [20] * 8 + [1]
w0 = _glorot_normal(layers, np.random.default_rng(1234))
nu = 0.01 / np.pi
pb = rp.BurgersInference(layers, lb, ub, nu, X_f, X_u, u)
t0 = time.time()
w, losses, _ = rp.adam_train(pb, w0, 100, lr=0.03)                      # inf_cont_burgers.py:35-38
tr = rp.lbfgs_fixed_step(lambda z: rp.loss_and_flat_grad(pb, z), w, max_iter=200, learning_rate=0.8, n_correction=50,
                         tol_fun=np.finfo(float).eps)                   # :40-42
w_model = tr.x_eval[-1]
err = np.linalg.norm(u_star - rp.predict(pb, w_model, X_star)) / np.linalg.norm(u_star)
print("oracle schedule: %.1f s, adam loss %.4e -> %.4e, lbfgs f %.4e -> %.4e (%d its, %s), rel L2 error %.4e"
      % (time.time() - t0, losses[0], losses[-1], tr.f_hist[0], tr.f_hist[-1], tr.n_iter, tr.stop_reason, err))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "burgers_accuracy.npz"), X_star=X_star.astype(np.float32),
                    u_star=u_star.astype(np.float32), X_u=X_u, u=u, X_f=X_f, lb=lb, ub=ub, w0=w0, oracle_adam_losses=losses,
                    oracle_lbfgs_f=np.array(tr.f_hist), oracle_error=err, oracle_w=w_model)
print(os.path.getsize(os.path.join(ROOT, "tests", "golden", "burgers_accuracy.npz")) // 1024, "KiB")
