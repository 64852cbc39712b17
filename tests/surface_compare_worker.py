"""Worker for test_reference_pin.py::test_mirror_host_attributes_equal_the_reference: builds the reference NeuralNetwork (from
$PINN_REFERENCE_DIR, on the TF emulation) and the mirror for the same hp and compares every host-side attribute the scripts read."""
import contextlib
import importlib.util
import io
import os
import sys

import numpy as np

ROOT, REF = sys.argv[1], os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")


def load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def side(paths, nn_path):
    for k in ("custom_lbfgs", "logger", "neuralnetwork", "tensorflow", "pinn_cabi"):
        sys.modules.pop(k, None)
    old = list(sys.path)
    sys.path[:0] = paths
    try:
        nn = load("nn_" + str(len(paths)) + str(abs(hash(nn_path))), nn_path)
        import custom_lbfgs
        import logger
        return nn, custom_lbfgs, logger
    finally:
        sys.path[:] = old


ref = side([ROOT + "/oracle/tf_emulation", REF + "/utils"], REF + "/utils/neuralnetwork.py")
mine = side([ROOT + "/pinns-tf2.0_b200/shims", ROOT + "/pinns-tf2.0_b200/utils"], ROOT + "/pinns-tf2.0_b200/utils/neuralnetwork.py")
assert ref[1].__file__.startswith(REF) and mine[1].__file__.startswith(ROOT)

lb, ub = np.array([-1.0, 0.0]), np.array([1.0, 0.99])
for layers in ([2] + [20] * 8 + [1], [2, 100, 100, 100, 100, 2], [2, 16, 1], [1, 50, 50, 50, 101], [2, 8, 12, 1]):
    hp = {"layers": layers, "tf_epochs": 7, "tf_lr": 0.03, "tf_b1": 0.9, "tf_eps": None, "nt_epochs": 11, "nt_lr": 0.8,
          "nt_ncorr": 50, "log_frequency": 10}
    objs = []
    for nn, lb_mod, lg_mod in (ref, mine):
        with contextlib.redirect_stdout(io.StringIO()):
            objs.append(nn.NeuralNetwork(dict(hp), lg_mod.Logger(hp), ub[:layers[0]], lb[:layers[0]]))
    r, m = objs
    assert r.sizes_w == m.sizes_w and r.sizes_b == m.sizes_b, (layers, r.sizes_w, m.sizes_w)      # incl. quirk Q7 for [2,8,12,1]
    assert r.tf_epochs == m.tf_epochs and r.dtype == m.dtype
    for k in ("learningRate", "maxIter", "nCorrection", "tolFun", "maxEval", "tolX", "lineSearch", "verbose"):
        assert getattr(r.nt_config, k) == getattr(m.nt_config, k), k                                # Struct: missing keys are 0
    assert r.get_params() == m.get_params() == []
# Struct / dot / module globals of custom_lbfgs
rs, ms = ref[1].Struct(), mine[1].Struct()
assert rs.anything == ms.anything == 0
for k in ("lbfgs", "Struct", "dot", "reset_time", "record_time", "last_time", "final_loss", "times"):
    assert hasattr(ref[1], k) and hasattr(mine[1], k), k
cfg = mine[1].Struct(); cfg.maxIter = 0
assert ref[1].lbfgs(None, None, cfg, None, True, None) is None and mine[1].lbfgs(None, None, cfg, None, True, None) is None
print("host attributes identical")
