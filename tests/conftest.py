import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "pinns-tf2.0_b200")
for p in (ROOT, os.path.join(PKG, "utils")):
    if p not in sys.path:
        sys.path.insert(0, p)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def _cuda_device_present():
    try:
        import ctypes
        n = ctypes.c_int(0)
        rt = ctypes.CDLL("libcudart.so")
        return rt.cudaGetDeviceCount(ctypes.byref(n)) == 0 and n.value > 0
    except Exception:
        try:
            import torch
            return torch.cuda.is_available()
        except Exception:
            return False


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a box without a GPU skips the gpu-marked tests instead of failing in pinn_create (the oracle
    stand-in plugin of tests/test_gpu_testcode_dryrun.py runs them on the CPU on purpose and opts out)."""
    if os.environ.get("PINN_GPU_TESTS_ON_ORACLE") == "1" or config.pluginmanager.hasplugin("oracle_backend_plugin"):
        return
    if _cuda_device_present():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device (B200); there is no CPU fallback")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def load_reference_run():
    """What the reference's OWN Python computed on the golden inputs (tests/golden/make_reference_fixtures.py), kept in two
    files so that each stays under 1 MB: the Schrodinger arrays (nls_*) in reference_run_nls.npz, the rest in reference_run.npz."""
    run = {}
    for name in ("reference_run", "reference_run_nls"):
        with np.load(os.path.join(GOLDEN, name + ".npz")) as f:
            run.update({k: f[k] for k in f.files})
    return run


def assert_matches_reference_run(loss, grad, loss_key, grad_key, tol=1e-10):
    """The CUDA result against the numbers produced by the reference's own code (not only against the restated oracle)."""
    r = load_reference_run()
    ref_loss, ref_grad = float(r[loss_key]), np.asarray(r[grad_key], dtype=np.float64)
    assert abs(float(loss) - ref_loss) <= tol * abs(ref_loss), (loss_key, float(loss), ref_loss)
    grad = np.asarray(grad, dtype=np.float64)
    assert grad.shape == ref_grad.shape, (grad_key, grad.shape, ref_grad.shape)
    assert np.linalg.norm(grad - ref_grad) <= tol * np.linalg.norm(ref_grad), grad_key


@pytest.fixture(scope="session")
def lib_built():
    """Build libpinn_b200.so if it is stale/missing (nvcc cross-compiles without a GPU)."""
    sys.path.insert(0, PKG)
    import build as pinn_build
    return pinn_build.build()
