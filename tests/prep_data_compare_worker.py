"""Worker for test_reference_pin.py::test_prep_data_equals_the_reference: runs the reference's own prep_data functions
(1d-burgers/burgersutil.py, 1dcomplex-schrodinger/schrodingerutil.py imported from $PINN_REFERENCE_DIR; matplotlib is stubbed --
it is only imported there, never used by prep_data -- and pyDOE.lhs is the stand-in of pinns-tf2.0_b200/shims) and the
restatements of this package from the same numpy seed; every returned array must be bit-identical."""
import importlib.util
import os
import sys
import types

import numpy as np

ROOT, REF = sys.argv[1], os.environ.get("PINN_REFERENCE_DIR") or sys.exit("set PINN_REFERENCE_DIR to a checkout of the original PINNs-TF2.0 project")


class _Anything(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything(self.__name__ + "." + name)

    def __call__(self, *a, **k):
        return _Anything(self.__name__ + "()")

    def update(self, *a, **k):
        return None


for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.gridspec", "mpl_toolkits", "mpl_toolkits.mplot3d", "mpl_toolkits.axes_grid1"):
    sys.modules[name] = _Anything(name)


def load(name, path, paths):
    for k in ("plotting", "burgersutil", "schrodingerutil", "tensorflow"):
        sys.modules.pop(k, None)
    old = list(sys.path)
    sys.path[:0] = paths
    try:
        spec = importlib.util.spec_from_file_location(name, path)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m
    finally:
        sys.path[:] = [p for p in old]


os.chdir(REF)                      # the reference modules resolve ./PINNs/Utilities and sys.path.append("utils") relative to the cwd
shims = os.path.join(ROOT, "pinns-tf2.0_b200", "shims")
ref_b = load("ref_burgersutil", REF + "/1d-burgers/burgersutil.py", [ROOT + "/oracle/tf_emulation", shims, REF + "/utils"])
ref_s = load("ref_schrodingerutil", REF + "/1dcomplex-schrodinger/schrodingerutil.py", [ROOT + "/oracle/tf_emulation", shims, REF + "/utils"])
my_b = load("my_burgersutil", ROOT + "/pinns-tf2.0_b200/1d-burgers/burgersutil.py", [shims, ROOT + "/pinns-tf2.0_b200/utils"])
my_s = load("my_schrodingerutil", ROOT + "/pinns-tf2.0_b200/1dcomplex-schrodinger/schrodingerutil.py", [shims, ROOT + "/pinns-tf2.0_b200/utils"])
assert ref_b.prep_data.__code__.co_filename.startswith(REF) and my_b.prep_data.__code__.co_filename.startswith(ROOT)


def same(name, a, b):
    assert len(a) == len(b), (name, len(a), len(b))
    for i, (u, v) in enumerate(zip(a, b)):
        u, v = np.asarray(u), np.asarray(v)
        assert u.shape == v.shape and u.dtype == v.dtype and np.array_equal(u, v), (name, i, u.shape, v.shape, u.dtype, v.dtype)
    print("%-38s %2d outputs bit-identical" % (name, len(a)))


burgers = os.path.join(REF, "1d-burgers", "data", "burgers_shock.mat")
nls = os.path.join(REF, "1dcomplex-schrodinger", "data", "NLS.mat")
cases = [
    ("burgers inference (N_u=100, N_f=10000)", lambda m: m.prep_data(burgers, 100, 10000, noise=0.0)),          # inf_cont_burgers.py:104-106
    ("burgers identification (N_u=2000)", lambda m: m.prep_data(burgers, 2000, noise=0.0)),                     # ide_cont_burgers.py:176-177
    ("burgers identification, noise=0.01", lambda m: m.prep_data(burgers, 2000, noise=0.01)),                   # noise is ignored there
    ("burgers discrete inference (q=500)", lambda m: m.prep_data(burgers, N_n=250, q=500, lb=np.array([-1.0]), ub=np.array([1.0]),
                                                               noise=0.0, idx_t_0=10, idx_t_1=90)),             # inf_disc_burgers.py:135-139
    ("burgers discrete inference, noise", lambda m: m.prep_data(burgers, N_n=250, q=100, lb=np.array([-1.0]), ub=np.array([1.0]),
                                                              noise=0.05, idx_t_0=10, idx_t_1=90)),
]
# discrete-time identification (ide_disc_burgers.py:216-218).  The reference branch calls np.asscalar, which numpy >= 1.23 no longer
# has; it is supplied for the reference call only (np.asscalar(a) was a.item()).
if not hasattr(np, "asscalar"):
    np.asscalar = lambda a: a.item()
cases.append(("burgers discrete identification", lambda m: m.prep_data(burgers, N_0=199, N_1=201, lb=np.array([-1.0]), ub=np.array([1.0]),
                                                                        noise=0.0, idx_t_0=10, idx_t_1=90)))
cases.append(("burgers discrete identification, noise", lambda m: m.prep_data(burgers, N_0=199, N_1=201, lb=np.array([-1.0]),
                                                                               ub=np.array([1.0]), noise=0.01, idx_t_0=10, idx_t_1=90)))
for name, fn in cases:
    np.random.seed(1234); a = fn(ref_b)
    np.random.seed(1234); b = fn(my_b)
    same(name, a, b)
np.random.seed(1234); a = ref_s.prep_data(nls, 50, 50, 20000, 0.0)                                              # inf_cont_schrodinger.py:144-147
np.random.seed(1234); b = my_s.prep_data(nls, 50, 50, 20000, 0.0)
same("schrodinger (N_0=50, N_b=50, N_f=20000)", a, b)
print("prep_data identical")
