"""CPU: bench.py's host logic end to end against a FAKE backend (no GPU, no oracle timing): argument handling, the timed
loops, the e2e modes, extras and the JSON contract (one line, required keys).  The fake only counts calls and returns
plausible numbers; nothing here measures anything."""
import ctypes as C
import io
import json
import os
import sys
from contextlib import redirect_stdout

import numpy as np

from conftest import ROOT


class FakePinn(object):
    instances = []

    def __init__(self, pde, layers, lb, ub, device=0, rank=0, world=1, nccl_uid=None):
        self.pde, self.layers, self.launches, self.events, self.steps = pde, list(layers), 0, {}, 0
        self.P = sum(a * b + b for a, b in zip(layers[:-1], layers[1:])) + (2 if pde == 1 else 0)
        FakePinn.instances.append(self)

    def _noop(self, *a, **k):
        return None

    set_pde_params = set_data = set_collocation = set_collocation_ptr = set_collocation_mapped = _noop
    set_boundary = set_irk = sync = flush_l2 = close = _noop

    def set_weights(self, w):
        self.steps = 0

    def adam_step(self, lr, b1=0.9, b2=0.999, eps=1e-7, sync=True):
        self.launches += 2
        self.steps += 1
        return 0.5 if sync else None

    def adam_steps(self, n, lr, b1=0.9, b2=0.999, eps=1e-7):
        self.launches += 2 * n
        self.steps += n

    def last_loss(self):
        return 1.0 / self.steps

    def event_record(self, idx):
        self.events[idx] = True

    def event_elapsed_ms(self, i, j):
        assert i in self.events and j in self.events
        return 0.46

    def launch_count(self):
        return self.launches

    def time_kernel_ms(self, iters):
        return 0.445 * iters

    def kernel_info(self):
        return {"grid": 148, "block": 256, "dyn_smem": 196376, "regs": 252, "local_bytes": 0, "sms": 148}

    def lbfgs(self, max_iter, **k):
        return {"n_iter": max_iter, "n_eval": max_iter, "reason": 1, "reason_str": "max iterations", "x_final": np.ones(self.P),
                "f_hist": [0.5] * max_iter}

    def loss_grad(self, w=None, want_grad=True):
        return 0.25, np.ones(self.P), np.zeros(3)

    def get_weights(self):
        return np.full(self.P, float(self.steps))         # Adam steps since set_weights

    adam_reset = _noop


def _fake_backend(monkeypatch):
    sys.path.insert(0, ROOT)
    import torch
    import pinn_cabi
    import bench
    monkeypatch.setattr(pinn_cabi, "Pinn", FakePinn)
    monkeypatch.setattr(pinn_cabi, "host_alloc", lambda n: (np.zeros(n), C.c_void_p(0)))
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(bench, "time_reference_port", lambda n_f, steps, warmup, seed=1234, budget_s=0: (0.4, 8, 0.1, n_f))
    monkeypatch.setattr(bench, "_port_baseline", lambda kind, data, w, steps, warmup, n, what, **kw: {"value": 1e5, "unit": "points/s", "cores": 8,
                                                                                                  "kind": "port", "sample": what})
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    return bench


def test_bench_gpu_arm_control_flow_with_fake_backend(monkeypatch):
    bench = _fake_backend(monkeypatch)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "4", "--warmup", "1"])
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    lines = [l for l in buf.getvalue().strip().split("\n") if l]
    assert len(lines) == 1                                   # exactly one JSON line on stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline", "extras"):
        assert key in d, key
    assert d["warmup"] == 3 and d["steps"] == 4              # warm-up is raised to the minimum of 3
    assert d["dtype"] == "f64" and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["gpu_launches"] == 2 * 4 and abs(d["ms_per_step"] - 0.46) < 1e-9
    assert d["config"]["workload"] == bench.workload_string(100000)        # the string both arms print
    c5 = d["cfg5"]
    assert c5["n_f_global"] == 2000000 and c5["n_gpus"] == 1 and c5["adam_ms_per_step"] > 0 and c5["lbfgs_ms_per_iteration"] > 0
    assert abs(d["value"] - 100000 / 0.46e-3) / d["value"] < 1e-9
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "copy_mode", "mapped_mode"}
    assert d["e2e"]["h2d_bytes_per_step"] == 1600000 and d["e2e"]["d2h_bytes_per_step"] == 8
    r = d["roofline"]
    assert r["bound"] == "tensor" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and r["traffic"] > 1e6
    assert set(d["extras"]) == {"burgers_lbfgs", "burgers_cfg1_10k", "burgers_identification", "schrodinger", "burgers_8x40_generic",
                                "burgers_discrete_time"}
    assert all("error" not in v for v in d["extras"].values()), d["extras"]
    for k in ("burgers_cfg1_10k", "burgers_identification", "schrodinger"):
        assert d["extras"][k]["cpu_baseline"]["kind"] == "port"
    assert d["extras"]["schrodinger"]["roofline"]["bound"] == "tensor"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 8


def test_bench_dump_outputs_are_those_of_the_last_timed_step(monkeypatch, tmp_path):
    """--dump-outputs writes the loss and the weights as they stand after the last timed step (3 warm-up + 5 timed Adam steps),
    not after the untimed steps that follow."""
    bench = _fake_backend(monkeypatch)
    out = tmp_path / "out"
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "5", "--warmup", "3", "--no-extras", "--no-cpu-baseline",
                                      "--dump-outputs", str(out)])
    with redirect_stdout(io.StringIO()):
        bench.main()
    assert sorted(os.listdir(out)) == ["loss.npy", "weights.npy"]
    loss, w = np.load(out / "loss.npy"), np.load(out / "weights.npy")
    assert loss.dtype == w.dtype == np.float64 and loss.tolist() == [1.0 / 8] and w.shape == (3021,) and np.all(w == 8.0)


def _launch_two(extra_args, tmp_path):
    import subprocess
    port = 29600 + os.getpid() % 300
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "bench_fake_worker.py")] + extra_args,
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = []
    for p in procs:
        try:
            o, e = p.communicate(timeout=240)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        assert p.returncode == 0, e[-2000:]
        outs.append(o)
    return outs


def test_bench_two_ranks_gloo(tmp_path):
    """Both ranks run the same number of steps (the keep-alive count is broadcast), exit 0, and only rank 0 prints."""
    outs = _launch_two([], tmp_path)
    assert outs[1].strip() == ""
    lines = [l for l in outs[0].strip().split("\n") if l]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["n_gpus"] == 2 and "cpu_baseline" not in d and "extras" not in d
    assert abs(d["value"] - 200000 / 0.46e-3) / d["value"] < 1e-9          # whole-job aggregate over both shards
    assert "ncclAllReduce" in d["config"]["parallelism"]
    pc = d["parity_check"]                                                  # sharded vs whole-set evaluation ran before the timing
    assert pc["ok"] and pc["world"] == 2 and pc["points"] == 200000 and pc["lbfgs_iters_equal"] and pc["weights_bitwise_identical_across_ranks"]
    assert d["cfg5"]["n_gpus"] == 2 and d["cfg5"]["n_f_global"] == 2000000


def test_reference_arm_under_two_ranks_only_rank0_works(tmp_path, monkeypatch):
    """--impl reference under a 2-rank launch: rank 0 alone runs and prints, the other rank exits 0 without work."""
    outs = _launch_two(["--impl", "reference", "--steps", "1", "--warmup", "1", "--n-f", "2000"], tmp_path)
    assert outs[1].strip() == ""
    d = json.loads(outs[0].strip().split("\n")[-1])
    assert d["impl"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["cpu_baseline"]["value"] == d["value"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"]["workload"] == bench.workload_string(2000)           # same string as the GPU arm prints for this --n-f
