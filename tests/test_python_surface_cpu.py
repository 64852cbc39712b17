"""CPU: the host-side mirror of the reference's Python surface (SURVEY 8(b)) up to the GPU boundary:
module/symbol names, Struct semantics, hp parsing, flat sizes, PDE recognition, data preparation, and -- when the
reference checkout is given (PINN_REFERENCE_DIR) -- the UNMODIFIED inf_cont_burgers.py loading on our modules
through run_reference_script.py until it needs the GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import PKG, ROOT, load_golden

REF = os.environ.get("PINN_REFERENCE_DIR", "")      # a checkout of the original project, if any
HP = {"N_u": 100, "N_f": 1000, "layers": [2] + [20] * 8 + [1], "tf_epochs": 3, "tf_lr": 0.03, "tf_b1": 0.9, "tf_eps": None,
      "nt_epochs": 4, "nt_lr": 0.8, "nt_ncorr": 50, "log_frequency": 10}


def test_module_surface_matches_reference_names():
    import custom_lbfgs, logger, neuralnetwork
    for name in ("lbfgs", "dot", "Struct", "reset_time", "record_time", "last_time", "final_loss", "times"):
        assert hasattr(custom_lbfgs, name)
    for name in ("get_epoch_duration", "get_elapsed", "get_error_u", "set_error_fn", "log_train_start", "log_train_epoch",
                 "log_train_opt", "log_train_end"):
        assert hasattr(logger.Logger, name)
    for name in ("loss", "grad", "wrap_training_variables", "get_params", "get_weights", "set_weights", "get_loss_and_flat_grad",
                 "tf_optimization", "tf_optimization_step", "nt_optimization", "nt_optimization_steps", "fit", "predict", "summary",
                 "tensor"):
        assert hasattr(neuralnetwork.NeuralNetwork, name)


def test_struct_and_lbfgs_contract():
    from custom_lbfgs import Struct, lbfgs
    s = Struct()
    s.maxIter = 0
    assert s.anything == 0 and s.maxIter == 0
    assert lbfgs(lambda x: (0.0, x), np.zeros(3), s, Struct(), True, None) is None      # custom_lbfgs.py:43-44
    s.maxIter = 5
    import pinn_cabi
    import torch
    if not torch.cuda.is_available():
        # a foreign closure runs on the stand-alone DEVICE optimiser: without a GPU that fails loudly (no host fallback)
        with pytest.raises(pinn_cabi.PinnError, match="no CPU fallback"):
            lbfgs(lambda x: (0.0, x), np.zeros(3), s, Struct(), True, None)
    else:
        # with one it runs there: a zero gradient at the start is optimal at once, (x, f_hist) only (custom_lbfgs.py:73-76)
        state = Struct()
        ret = lbfgs(lambda x: (0.0, x), np.zeros(3), s, state, True, None)
        assert len(ret) == 2 and state.stop_reason == "initial optimality"
        assert np.array_equal(np.asarray(ret[0]), np.zeros(3))


def test_network_construction_and_pde_recognition(capsys):
    from logger import Logger
    from neuralnetwork import NeuralNetwork
    import pinn_cabi

    class BurgersInformedNN(NeuralNetwork):      # constructor of 1d-burgers/inf_cont_burgers.py:48-56
        def __init__(self, hp, logger, X_f, ub, lb, nu):
            super().__init__(hp, logger, ub, lb)
            self.nu = nu
            self.x_f = self.tensor(X_f[:, 0:1]); self.t_f = self.tensor(X_f[:, 1:2])

        def loss(self, u, u_pred):               # would be TensorFlow tape code in the reference
            raise AssertionError("tape body must have been replaced by the fused-kernel loss")

    net = BurgersInformedNN(HP, Logger(HP), np.zeros((10, 2)), np.array([1.0, 1.0]), np.array([-1.0, 0.0]), 0.01 / np.pi)
    assert net.sizes_w == [40] + [400] * 7 + [20] and net.sizes_b == [20] * 8 + [1]      # neuralnetwork.py:40-45
    assert net.nt_config.maxIter == 4 and net.nt_config.tolFun == np.finfo(float).eps and net.nt_config.lineSearch == 0
    assert net.tf_eps == 1e-7 and net.dtype == "float64"
    assert net._pde_id() == pinn_cabi.BURGERS_INF
    assert BurgersInformedNN.loss is not BurgersInformedNN._script_loss
    assert net._w0.shape == (3021,) and np.all(net._w0[40:60] == 0)                       # glorot weights, zero biases
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(pinn_cabi.PinnError, match="no CUDA device"):
            net.fit(np.zeros((5, 2)), np.zeros((5, 1)))


@pytest.fixture()
def burgers_shock_mat(tmp_path):
    """The reference's 1d-burgers/data/burgers_shock.mat (x: 256, t: 100, usol: 256 x 100), rebuilt from the evaluation grid
    prep_data made of it, which tests/golden/burgers_accuracy.npz stores (in float32)."""
    import scipy.io
    g = load_golden("burgers_accuracy")
    X_star, u_star = g["X_star"].astype(np.float64), g["u_star"].astype(np.float64)
    x, t = X_star[:256, 0], X_star[::256, 1]
    X, T = np.meshgrid(x, t)
    assert np.array_equal(X_star, np.hstack((X.flatten()[:, None], T.flatten()[:, None])))
    path = str(tmp_path / "burgers_shock.mat")
    scipy.io.savemat(path, {"x": x[:, None], "t": t[:, None], "usol": u_star.reshape(100, 256).T})
    return path


def test_prep_data_shapes_against_reference_files(burgers_shock_mat):
    sys.path.insert(0, os.path.join(PKG, "1d-burgers"))
    import burgersutil
    np.random.seed(1234)
    out = burgersutil.prep_data(burgers_shock_mat, 100, 1000, noise=0.0)
    x, t, X, T, Exact_u, X_star, u_star, X_u, u, X_f, ub, lb = out
    assert X_star.shape == (25600, 2) and X_u.shape == (100, 2) and u.shape == (100, 1) and X_f.shape == (1000, 2)
    assert np.allclose(lb, [-1, 0]) and np.allclose(ub, [1, 0.99])
    # Latin hypercube: exactly one sample per stratum in each dimension
    for j in range(2):
        strata = np.floor((X_f[:, j] - lb[j]) / (ub[j] - lb[j]) * 1000).astype(int)
        assert sorted(np.clip(strata, 0, 999)) == list(range(1000))
    # every training point is an initial/boundary point (burgersutil.py:104-118)
    assert np.all((X_u[:, 1] == 0) | (np.abs(X_u[:, 0]) == 1))
    ide = burgersutil.prep_data(burgers_shock_mat, 2000, noise=0.01)
    assert ide[7].shape == (2000, 2) and len(ide) == 11


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_unmodified_reference_script_runs_up_to_the_gpu_boundary():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    r = subprocess.run([sys.executable, os.path.join(PKG, "run_reference_script.py"),
                        os.path.join(REF, "1d-burgers", "inf_cont_burgers.py")], capture_output=True, text=True, timeout=300)
    out = r.stdout + r.stderr
    assert "Hyperparameters" in out and "Training started" in out      # data prep, Logger, class creation all worked
    assert "no CUDA device" in out and r.returncode != 0                # and it stops exactly at the GPU boundary


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
def test_indentation_normaliser_repairs_ide_cont_and_leaves_good_scripts_alone():
    import ast
    sys.path.insert(0, PKG)
    import run_reference_script as r
    src = open(os.path.join(REF, "1d-burgers", "ide_cont_burgers.py"), encoding="utf-8").read()
    with pytest.raises(SyntaxError):
        ast.parse(src)                                                   # does not parse as shipped (SURVEY 0.4)
    tree = ast.parse(r.normalise_indentation(src))
    cls = [n for n in tree.body if isinstance(n, ast.ClassDef)][0]
    methods = {m.name: m for m in cls.body if isinstance(m, ast.FunctionDef)}
    assert list(methods) == ["__init__", "f_model", "loss", "wrap_training_variables", "get_weights", "set_weights",
                             "get_params", "fit", "predict"]
    assert len(methods["__init__"].body) == 3                            # super().__init__, lambda_1, lambda_2
    with_body = [b for b in methods["f_model"].body if isinstance(b, ast.With)][0].body
    assert len(with_body) == 5                                           # watch, watch, stack, model, u_x (like inf_cont)
    for f in ("1d-burgers/inf_cont_burgers.py", "1dcomplex-schrodinger/inf_cont_schrodinger.py"):
        s0 = open(os.path.join(REF, f), encoding="utf-8").read()
        assert ast.dump(ast.parse(r.normalise_indentation(s0))) == ast.dump(ast.parse(s0))


@pytest.mark.skipif(not os.path.isdir(REF), reason="needs a checkout of the original PINNs-TF2.0 project (set PINN_REFERENCE_DIR)")
@pytest.mark.parametrize("script", ["1d-burgers/ide_cont_burgers.py", "1dcomplex-schrodinger/inf_cont_schrodinger.py",
                                    "1d-burgers/inf_disc_burgers.py"])
def test_other_reference_scripts_reach_the_gpu_boundary(script):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, os.path.join(PKG, "run_reference_script.py"), os.path.join(REF, script)],
                       capture_output=True, text=True, timeout=300)
    out = r.stdout + r.stderr
    assert "Training started" in out and "no CUDA device" in out and r.returncode != 0


def test_result_artefacts_hp_json_and_fields(tmp_path, monkeypatch, burgers_shock_mat):
    """SURVEY 8(f)3: the plot_* helpers leave <save_path>/results/<timestamp>-<script>/{hp.json, fields.npz} behind, with or
    without matplotlib (reference: utils/plotting.py:8-16, burgersutil.py:132-203)."""
    import json
    import importlib
    monkeypatch.setenv("PINN_RESULTS_ROOT", str(tmp_path))
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.setattr(sys, "argv", ["inf_cont_burgers.py"])
    sys.path.insert(0, os.path.join(PKG, "utils"))
    sys.path.insert(0, os.path.join(PKG, "1d-burgers"))
    burgersutil = importlib.import_module("burgersutil")
    np.random.seed(0)
    x, t, X, T, Exact_u, X_star, u_star, X_u, u_tr, X_f, ub, lb = burgersutil.prep_data(burgers_shock_mat, 50, 500)
    hp = {"N_u": 50, "layers": [2, 20, 1], "tf_eps": None, "np_value": np.float64(0.5)}
    out = burgersutil.plot_inf_cont_results(X_star, u_star.flatten() * 1.01, X_u, u_tr, Exact_u, X, T, x, t,
                                            save_path="1d-burgers", save_hp=hp)
    assert out.startswith(os.path.join(str(tmp_path), "1d-burgers", "results")) and out.endswith("-inf_cont_burgers")
    assert json.load(open(os.path.join(out, "hp.json"))) == {"N_u": 50, "layers": [2, 20, 1], "tf_eps": None, "np_value": 0.5}
    f = np.load(os.path.join(out, "fields.npz"))
    assert f["U_pred"].shape == Exact_u.shape == (100, 256)
    assert abs(float(f["rel_l2_error"]) - 0.01) < 1e-12
    assert burgersutil.plot_ide_cont_results(X_star, u_star, X_u, u_tr, Exact_u, X, T, x, t, 1.0, 1.0, 0.003, 0.003) is None
    # non-zero ranks of a multi-process job write nothing
    monkeypatch.setenv("RANK", "1")
    assert burgersutil.plot_inf_cont_results(X_star, u_star.flatten(), X_u, u_tr, Exact_u, X, T, x, t,
                                             save_path="1d-burgers", save_hp=hp) is None
