#!/usr/bin/env python
"""Benchmark of the PINN training hot path (BASELINE.json metric: collocation-points/sec per training step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (config.workload, identical on both arms): BASELINE.json configs[1] -- 1D Burgers, [2,20x8,1] tanh MLP,
N_f = 100 000 collocation points per GPU (+ N_u = 100 data points), one Adam training step = fused loss/gradient
evaluation + on-device Adam update.  A "step" is one pass of that hot path.  N > 1 (torchrun): collocation points are
sharded, weak scaling (100 000 per GPU), one exchange of [gradient | loss] (3024 doubles) per step.

value    : whole-job collocation points / second, inputs resident in HBM, each step timed with CUDA events on the
           launching stream (L2 flushed between timed iterations), max over ranks.
e2e      : the same metric through the public API with HOST buffers: every step hands over that step's collocation batch in
           pinned host memory and reads the loss back (pinn_adam_step(&loss)).
roofline : fused kernel alone (CUDA events); algorithmic FLOPs = 24*S per collocation point + 6*S per data point
           (S = 2860 weight entries; SURVEY 8(d)) against the MEASURED FP64 pipe peak of this pool's B200
           (profiles/microbench/fp64_peak_r01.jsonl: DMMA.8x8x4 37.0 TFLOP/s, which is also the HGX B200 datasheet figure;
           MEASURED_PEAKS.json has no FP64 entry).  The path is FP64-pipe-bound (4 300 FLOP per HBM byte); the HBM fraction is
           reported beside it.
cpu_baseline / --impl reference: the restated reference (oracle/reference_port.py: nested reverse-mode autograd, torch CPU
           fp64, TF-2.0 Adam semantics) timed on this box's host cores (fixed thread count, printed with nproc).
parity_check (N > 1): before anything is timed, loss/gradient, 3 Adam steps and 4 L-BFGS iterations on the SHARDED handles are
           compared with a world = 1 handle holding the whole point set on rank 0; the run fails when they differ by > 1e-10.
cfg5     : BASELINE configs[4] -- N_f = 2 000 000 GLOBAL points strong-scaled over the N GPUs of this run (N = 1: all on one
           GPU), Adam ms/step and L-BFGS ms/iteration.
extras (N = 1): the other SURVEY section-8 configurations (cfg 1: N_f = 10 000; cfg 4: identification N = 2000; Schrodinger;
           discrete time), each with its own cpu_baseline.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pinns-tf2.0_b200")
for p in (ROOT, PKG, os.path.join(PKG, "utils")):
    if p not in sys.path:
        sys.path.insert(0, p)

LAYERS = [2] + [20] * 8 + [1]
S_WEIGHTS = 2 * 20 + 7 * 400 + 20            # 2860
FLOP_PER_COLLOC = 24 * S_WEIGHTS             # 68 640 (forward 8S, input adjoint 8S, weight gradient 8S)
FLOP_PER_DATA = 6 * S_WEIGHTS                # one stream
N_F_PER_GPU = 100_000
N_F_CFG5 = 2_000_000
N_U = 100
LB, UB = np.array([-1.0, 0.0]), np.array([1.0, 0.99])
NU = 0.01 / np.pi
ADAM_LR = 1e-3
FP64_PEAK_TFLOPS_DATASHEET = 37.0            # HGX B200 FP64 / FP64 tensor (dense), per GPU
CPU_THREADS = 16                             # reference arm: fixed (round-1 calibration: 8-16 threads are fastest for torch's
                                             # small-tensor ops on this pool's 128-CPU hosts; more threads are slower)
PARITY_TOL = 1e-10
NLS_LAYERS = [2, 100, 100, 100, 100, 2]
NLS_LB, NLS_UB = np.array([-5.0, 0.0]), np.array([5.0, np.pi / 2])
NLS_S = 2 * 100 + 3 * 100 * 100 + 100 * 2    # 30 400


def workload_string(n_f):
    return ("1d-burgers inf_cont [2,20x8,1] tanh, N_f=%d collocation points per GPU, N_u=100, Adam lr 1e-3, fp64 "
            "(BASELINE configs[1])" % n_f)


def fp64_peak():
    path = os.path.join(ROOT, "profiles", "microbench", "fp64_peak_r01.jsonl")
    best = None
    try:
        for line in open(path):
            d = json.loads(line)
            if "dmma_tflops" in d:
                best = max(best or 0.0, d["dmma_tflops"])
    except Exception:
        pass
    return (best, "measured (profiles/microbench/fp64_peak_r01.jsonl, DMMA.8x8x4); datasheet %.1f" % FP64_PEAK_TFLOPS_DATASHEET) \
        if best else (FP64_PEAK_TFLOPS_DATASHEET, "datasheet fallback")


def _ncu_summary(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from a committed `ncu --set full` summary under profiles/."""
    for rnd in ("r02", "r01"):
        path = os.path.join(ROOT, "profiles", "ncu_%s_%s_summary.csv" % (name, rnd))
        try:
            tot = 0.0
            for line in open(path):
                f = line.strip().split(",")
                if len(f) == 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(f[1], None)
                    if mult is None:
                        return None, None
                    tot += float(f[2]) * mult
            if tot:
                return tot, os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


def ncu_traffic_bytes():
    return _ncu_summary("burgers_v2")[0]


def hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback"


def synthetic_problem(seed, n_f):
    rng = np.random.default_rng(seed)
    X_f = LB + (UB - LB) * rng.random((n_f, 2))
    X_u = LB + (UB - LB) * rng.random((N_U, 2))
    u = rng.uniform(-1, 1, (N_U, 1))
    return X_f, X_u, u


def init_weights(layers=None):
    from neuralnetwork import _glorot_normal
    return _glorot_normal(layers or LAYERS, np.random.default_rng(1234))


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self._stop, self._th = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([v.strip() for v in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=10)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU (reference) arm
def cpu_threads():
    """Thread count of the CPU arm: fixed per box (min(16, CPUs available)), so that repeated runs are comparable.
    torchrun exports OMP_NUM_THREADS=1, which would cripple this arm, hence the explicit set_num_threads."""
    try:
        ncpu = len(os.sched_getaffinity(0))
    except Exception:
        ncpu = os.cpu_count() or 1
    return max(1, min(CPU_THREADS, ncpu)), ncpu


def time_port_steps(problem, w, steps, warmup, lr=ADAM_LR, b1=0.9, b2=0.999, eps=None):
    """Mean seconds per (loss + flat gradient + Adam update) of the restated reference on the host cores."""
    from oracle import reference_port as rp
    st = rp.adam_init(w.size)
    ts, f = [], None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        f, g = rp.loss_and_flat_grad(problem, w)
        w = rp.adam_update(w, g, st, lr, b1, b2, eps)
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    return float(np.mean(ts)), f


def time_reference_port(n_f, steps, warmup, seed=1234, budget_s=110.0):
    """The restated reference on the host cores: loss + flat gradient (nested reverse mode) + Adam update.
    Bounded sample: the whole (warmup + steps) run stays within ~budget_s whatever --steps the caller passes; throughput in
    points/s is nearly size-independent at these sizes (1.5e5 - 4e5 pts/s from N_f = 1e4 to 1e5)."""
    import torch
    from oracle import reference_port as rp
    threads, ncpu = cpu_threads()
    torch.set_num_threads(threads)
    Xc, Xuc, uc = synthetic_problem(seed + 1, 5000)
    pbc = rp.BurgersInference(LAYERS, LB, UB, NU, Xc, Xuc, uc)
    wc = init_weights()
    rp.loss_and_flat_grad(pbc, wc)
    t0 = time.perf_counter()
    rp.loss_and_flat_grad(pbc, wc)
    est_step = (time.perf_counter() - t0) * n_f / 5000.0
    if est_step * (steps + warmup) > budget_s:
        n_f = max(2000, int(n_f * budget_s / (est_step * (steps + warmup))))
    X_f, X_u, u = synthetic_problem(seed, n_f)
    pb = rp.BurgersInference(LAYERS, LB, UB, NU, X_f, X_u, u)
    sec, f = time_port_steps(pb, init_weights(), steps, warmup)
    return sec, threads, f, n_f


def _port_baseline(kind, data, w, steps, warmup, n_pts, what, **adam):
    """cpu_baseline of one of the extra configurations: the restated reference problem `kind` built from `data`, timed like
    the headline arm (same fixed thread count)."""
    import torch
    from oracle import reference_port as rp
    threads, ncpu = cpu_threads()
    torch.set_num_threads(threads)
    problem = {"burgers_inf": lambda: rp.BurgersInference(LAYERS, LB, UB, NU, *data),
               "burgers_ide": lambda: rp.BurgersIdentification(LAYERS, LB, UB, *data),
               "nls_inf": lambda: rp.SchrodingerInference(NLS_LAYERS, NLS_LB, NLS_UB, *data)}[kind]()
    sec, _ = time_port_steps(problem, w, steps, warmup, **adam)
    return {"value": n_pts / sec, "unit": "points/s", "ms_per_step": sec * 1e3, "cores": threads, "nproc": ncpu, "kind": "port",
            "sample": "%d Adam steps after %d warm-up, %s (oracle/reference_port.py)" % (steps, warmup, what)}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    n_f = args.n_f
    sec, cores, _, n_used = time_reference_port(n_f, args.steps, args.warmup)
    _, ncpu = cpu_threads()
    val = n_used / sec
    line = {
        "impl": "reference", "metric": "collocation-points/sec per training step (1D Burgers 8x20 tanh, Adam step)",
        "value": val, "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_string(n_f)},
        "cpu_baseline": {"value": val, "unit": "points/s", "cores": cores, "nproc": ncpu, "kind": "port",
                         "sample": f"{args.steps} Adam steps on a bounded sample of N_f={n_used} points after {args.warmup} warm-up, "
                                   "oracle/reference_port.py (TF-free restatement of the reference's nested-tape step; "
                                   "TensorFlow 2.0 is not installable here)"},
        "e2e": {"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU helpers
def timed_adam_steps(p, steps, flush, lr=ADAM_LR, b1=0.9, b2=0.999, eps=1e-7, ev0=0):
    """Per-step device times (ms): CUDA events on the launching stream around each asynchronous step."""
    for i in range(steps):
        if flush:
            p.flush_l2()
        p.event_record(ev0 + 2 * i)
        p.adam_step(lr, b1, b2, eps, sync=False)
        p.event_record(ev0 + 2 * i + 1)
    p.sync()
    return [p.event_elapsed_ms(ev0 + 2 * i, ev0 + 2 * i + 1) for i in range(steps)]


def timed_adam_batch(p, steps, lr=ADAM_LR, b1=0.9, b2=0.999, eps=1e-7, ev0=0):
    """Device time (ms) per step of `steps` Adam steps enqueued by ONE native call (pinn_adam_steps): no per-step binding cost, which
    for the small configurations is comparable to the step itself."""
    p.event_record(ev0)
    p.adam_steps(steps, lr, b1, b2, eps)
    p.event_record(ev0 + 1)
    p.sync()
    return p.event_elapsed_ms(ev0, ev0 + 1) / steps


def timed_lbfgs(p, iters, ev0=0):
    """Device time (ms) per L-BFGS iteration: events around one pinn_lbfgs call that enqueues all iterations blind."""
    eps = float(np.finfo(float).eps)
    p.lbfgs(2, learning_rate=0.8, n_correction=50, tol_fun=eps)       # allocates the history buffers
    p.sync()
    p.event_record(ev0)
    r = p.lbfgs(iters, learning_rate=0.8, n_correction=50, tol_fun=eps, sync_every=iters)
    p.event_record(ev0 + 1)
    p.sync()
    return p.event_elapsed_ms(ev0, ev0 + 1) / max(1, r["n_iter"]), r["n_iter"]


def max_over_ranks(dist, v):
    if dist is None:
        return float(v)
    import torch
    tt = torch.tensor([float(v)], dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return float(tt.item())


def parity_check(pinn_cabi, dist, p, rank, local_rank, world, n_f, X_u, u):
    """Sharded (world ranks) against whole-set (one GPU, rank 0) evaluation of the SAME points the bench times: loss and
    gradient, 3 Adam steps, 4 L-BFGS iterations.  Every rank executes the same number of exchanges."""
    eps = float(np.finfo(float).eps)
    w0 = init_weights()
    p.set_weights(w0); p.adam_reset()
    lN, gN, _ = p.loss_grad()
    aN = [p.adam_step(ADAM_LR) for _ in range(3)]
    wN = p.get_weights()
    p.set_weights(w0); p.adam_reset()
    rN = p.lbfgs(4, learning_rate=0.8, n_correction=50, tol_fun=eps, sync_every=2, want_x_final=True)
    p.set_weights(w0); p.adam_reset()
    p.sync()
    dist.barrier()                       # the other ranks wait HERE (on the host), not inside an exchange kernel
    out = [None]
    if rank == 0:
        whole = np.concatenate([synthetic_problem(1234 + r, n_f)[0] for r in range(world)], 0)
        s = pinn_cabi.Pinn(pinn_cabi.BURGERS_INF, LAYERS, LB, UB, device=local_rank)
        s.set_pde_params([NU]); s.set_data(X_u, u); s.set_collocation(whole[:, 0], whole[:, 1]); s.set_weights(w0)
        l1, g1, _ = s.loss_grad()
        a1 = [s.adam_step(ADAM_LR) for _ in range(3)]
        w1 = s.get_weights()
        s.set_weights(w0); s.adam_reset()
        r1 = s.lbfgs(4, learning_rate=0.8, n_correction=50, tol_fun=eps, sync_every=2, want_x_final=True)
        s.close()
        res = {"rel_loss": abs(lN - l1) / abs(l1), "rel_grad": rel(gN, g1), "rel_adam_losses": rel(aN, a1),
               "rel_adam_weights": rel(wN, w1), "lbfgs_iters_equal": bool(rN["n_iter"] == r1["n_iter"] and rN["n_eval"] == r1["n_eval"]),
               "rel_lbfgs_x": rel(rN["x_final"], r1["x_final"]), "rel_lbfgs_f_hist": rel(rN["f_hist"], r1["f_hist"]),
               "tolerance": PARITY_TOL, "points": int(whole.shape[0]), "world": world,
               "what": "sharded handles (this run's collocation shards) vs one world=1 handle holding all points on rank 0"}
        res["ok"] = bool(res["lbfgs_iters_equal"] and all(res[k] <= PARITY_TOL for k in
                                                         ("rel_loss", "rel_grad", "rel_adam_losses", "rel_adam_weights",
                                                          "rel_lbfgs_x", "rel_lbfgs_f_hist")))
        out = [res]
    dist.broadcast_object_list(out, src=0)
    # replicated state really is replicated: every rank holds bit-identical weights after the sharded Adam steps
    import torch
    wt = torch.from_numpy(np.ascontiguousarray(wN))
    ws = [torch.empty_like(wt) for _ in range(world)]
    dist.all_gather(ws, wt)
    out[0]["weights_bitwise_identical_across_ranks"] = bool(all(torch.equal(ws[0], x) for x in ws))
    out[0]["ok"] = bool(out[0]["ok"] and out[0]["weights_bitwise_identical_across_ranks"])
    return out[0]


def cfg5_block(p, dist, rank, world, steps=20, iters=20):
    """BASELINE configs[4]: N_f = 2 000 000 global points, strong-scaled over the ranks of this run."""
    n5 = N_F_CFG5 // world
    rng = np.random.default_rng(5000 + rank)
    X = LB + (UB - LB) * rng.random((n5, 2))
    p.set_collocation(X[:, 0], X[:, 1], n_global=n5 * world)
    p.set_weights(init_weights()); p.adam_reset()
    for _ in range(3):
        p.adam_step(ADAM_LR, sync=False)
    p.sync()
    if dist is not None:
        dist.barrier()
    ms = timed_adam_steps(p, steps, flush=True)
    adam_ms = max_over_ranks(dist, float(np.mean(ms)))
    lb_ms, n_it = timed_lbfgs(p, iters)
    lb_ms = max_over_ranks(dist, lb_ms)
    return {"config": "BASELINE configs[4]: Burgers inf_cont, N_f=%d GLOBAL points strong-scaled over %d GPU(s) (%d per GPU), N_u=100; "
                      "Adam lr 1e-3, then L-BFGS lr 0.8 / 50 corrections" % (n5 * world, world, n5),
            "n_f_global": n5 * world, "n_gpus": world, "adam_ms_per_step": adam_ms, "adam_points_per_s": n5 * world / (adam_ms * 1e-3),
            "adam_steps_timed": steps, "lbfgs_ms_per_iteration": lb_ms, "lbfgs_points_per_s": n5 * world / (lb_ms * 1e-3),
            "lbfgs_iterations_timed": n_it, "timing": "CUDA events on the launching stream, L2 flushed between Adam steps, max over ranks"}


def measure_extras(pinn_cabi, n_f, with_cpu=True):
    """Other SURVEY section-8 configurations, measured briefly on the same box (not the headline metric), each with the
    restated reference timed on the host cores beside it."""
    out = {}
    peak = fp64_peak()[0]
    eps = float(np.finfo(float).eps)
    # ---- BASELINE configs[1] L-BFGS phase at the headline size
    try:
        X_f, X_u, u = synthetic_problem(4321, n_f)
        p = pinn_cabi.Pinn(pinn_cabi.BURGERS_INF, LAYERS, LB, UB)
        p.set_pde_params([NU]); p.set_data(X_u, u); p.set_collocation(X_f[:, 0], X_f[:, 1]); p.set_weights(init_weights())
        for _ in range(20):
            p.adam_step(ADAM_LR, sync=False)
        ms, n_it = timed_lbfgs(p, 60)
        out["burgers_lbfgs"] = {"config": "BASELINE configs[1] L-BFGS phase: N_f=%d, lr 0.8, 50 corrections, all iterations enqueued blind" % n_f,
                                "ms_per_iteration": ms, "points_per_s": n_f / (ms * 1e-3), "iterations": n_it}
        p.close()
    except Exception as e:  # pragma: no cover
        out["burgers_lbfgs"] = {"error": str(e)}
    # ---- BASELINE configs[0] size (the north_star target is quoted at N_f = 10 000): Adam and L-BFGS
    try:
        n1 = 10000
        X_f, X_u, u = synthetic_problem(1234, n1)
        p = pinn_cabi.Pinn(pinn_cabi.BURGERS_INF, LAYERS, LB, UB)
        p.set_pde_params([NU]); p.set_data(X_u, u); p.set_collocation(X_f[:, 0], X_f[:, 1]); p.set_weights(init_weights())
        for _ in range(20):
            p.adam_step(ADAM_LR, sync=False)
        p.sync()
        ms = float(np.mean(timed_adam_steps(p, 200, flush=False)))
        ms_b = timed_adam_batch(p, 400)
        k_ms = p.time_kernel_ms(50) / 50
        lb_ms, n_it = timed_lbfgs(p, 100)
        d = {"config": "BASELINE configs[0] size on 1xB200: N_f=10000, N_u=100, Adam lr 1e-3; L-BFGS lr 0.8 / 50 corrections",
             "adam_ms_per_step": ms, "adam_points_per_s": n1 / (ms * 1e-3), "adam_ms_per_step_batched": ms_b,
             "batched": "400 steps enqueued by one pinn_adam_steps call, one event pair", "kernel_ms": k_ms,
             "roofline_frac_fp64": (n1 * FLOP_PER_COLLOC + N_U * FLOP_PER_DATA) / (k_ms * 1e-3) / 1e12 / peak,
             "lbfgs_ms_per_iteration": lb_ms, "lbfgs_points_per_s": n1 / (lb_ms * 1e-3), "lbfgs_iterations": n_it,
             "timing": "CUDA events, 200 back-to-back asynchronous steps (inputs 160 KB: L2-resident by nature)"}
        p.close()
        if with_cpu:
            d["cpu_baseline"] = _port_baseline("burgers_inf", (X_f, X_u, u), init_weights(), 8, 2, n1, "N_f=10000 (the whole configuration)")
            d["speedup_vs_cpu_baseline"] = d["adam_points_per_s"] / d["cpu_baseline"]["value"]
        out["burgers_cfg1_10k"] = d
    except Exception as e:  # pragma: no cover
        out["burgers_cfg1_10k"] = {"error": str(e)}
    # ---- BASELINE configs[3]: identification
    try:
        rng = np.random.default_rng(7)
        X_u = LB + (UB - LB) * rng.random((2000, 2)); u = rng.uniform(-1, 1, (2000, 1))
        w_ide = np.concatenate([init_weights(), [0.0, -6.0]])
        p = pinn_cabi.Pinn(pinn_cabi.BURGERS_IDE, LAYERS, LB, UB)
        p.set_data(X_u, u); p.set_weights(w_ide)
        for _ in range(20):
            p.adam_step(ADAM_LR, sync=False)
        p.sync()
        ms = float(np.mean(timed_adam_steps(p, 200, flush=False)))
        ms_b = timed_adam_batch(p, 400)
        lb_ms, n_it = timed_lbfgs(p, 100)
        d = {"config": "BASELINE configs[3]: N=2000 data=collocation points, lambda_1, lambda_2 trainable; Adam lr 1e-3, L-BFGS lr 0.8",
             "ms_per_step": ms, "points_per_s": 2000 / (ms * 1e-3), "ms_per_step_batched": ms_b,
             "batched": "400 steps enqueued by one pinn_adam_steps call, one event pair",
             "lbfgs_ms_per_iteration": lb_ms, "lbfgs_iterations": n_it}
        p.close()
        if with_cpu:
            d["cpu_baseline"] = _port_baseline("burgers_ide", (X_u, u), w_ide, 10, 2, 2000, "N=2000 (the whole configuration)")
            d["speedup_vs_cpu_baseline"] = d["points_per_s"] / d["cpu_baseline"]["value"]
        out["burgers_identification"] = d
    except Exception as e:  # pragma: no cover
        out["burgers_identification"] = {"error": str(e)}
    # ---- BASELINE configs[2]: Schrodinger
    try:
        rng = np.random.default_rng(9)
        n_nls = 20000
        X_f = NLS_LB + (NLS_UB - NLS_LB) * rng.random((n_nls, 2)); tb = rng.uniform(0, NLS_UB[1], (50, 1)); x0 = rng.uniform(-5, 5, (50, 1))
        uv0 = np.stack([2 / np.cosh(x0[:, 0]), 0 * x0[:, 0]], 1)
        w_nls = init_weights(NLS_LAYERS)
        p = pinn_cabi.Pinn(pinn_cabi.NLS_INF, NLS_LAYERS, NLS_LB, NLS_UB)
        p.set_collocation(X_f[:, 0], X_f[:, 1]); p.set_boundary(tb); p.set_data(x0, uv0)
        p.set_weights(w_nls)
        for _ in range(3):
            p.adam_step(0.05, 0.99, 0.999, 0.1, sync=False)
        p.sync()
        ms = float(np.mean(timed_adam_steps(p, 30, flush=True, lr=0.05, b1=0.99, b2=0.999, eps=0.1)))
        p.time_kernel_ms(2)
        k_ms = p.time_kernel_ms(10) / 10
        flops = (n_nls + 150) * 24.0 * NLS_S
        traffic, traffic_src = _ncu_summary("nls")
        alg_bytes = 16.0 * (n_nls + 150) + 2 * 8.0 * 30802
        d = {"config": "BASELINE configs[2]: [2,100x4,2], N_f=20000, N_0=N_b=50, Adam lr .05 b1 .99 eps .1",
             "ms_per_step": ms, "points_per_s": n_nls / (ms * 1e-3), "kernel_ms": k_ms,
             "roofline": {"bound": "tensor", "pipe": "fp64 (DMMA.8x8x4)", "achieved": flops / (k_ms * 1e-3) / 1e12, "peak": peak,
                          "unit": "TFLOP/s", "frac": flops / (k_ms * 1e-3) / 1e12 / peak, "kernel": "pinn::nls::fused_loss_grad",
                          "algorithmic_flop_per_point": 24 * NLS_S, "traffic": traffic, "traffic_source": traffic_src,
                          "algorithmic_bytes": alg_bytes},
             "roofline_frac_fp64": flops / (k_ms * 1e-3) / 1e12 / peak}
        p.close()
        if with_cpu:
            d["cpu_baseline"] = _port_baseline("nls_inf", (X_f[:5000], tb, x0, uv0), w_nls, 4, 1, 5000,
                                               "bounded sample: N_f=5000 of the 20000 points", lr=0.05, b1=0.99, eps=0.1)
            d["speedup_vs_cpu_baseline"] = d["points_per_s"] / d["cpu_baseline"]["value"]
        out["schrodinger"] = d
    except Exception as e:  # pragma: no cover
        out["schrodinger"] = {"error": str(e)}
    # ---- a net the specialised DMMA kernels do not cover: upstream's 8 x 40 table (Burgers_systematic.py:187-202) on the
    # generic fused kernel (any width; hidden-to-hidden layers on DMMA.8x8x4 with operands from global memory)
    try:
        L40 = [2] + [40] * 8 + [1]
        n40 = 20000
        S40 = 2 * 40 + 7 * 1600 + 40
        X_f, X_u, u = synthetic_problem(40, n40)
        p = pinn_cabi.Pinn(pinn_cabi.BURGERS_INF, L40, LB, UB)
        p.set_pde_params([NU]); p.set_data(X_u, u); p.set_collocation(X_f[:, 0], X_f[:, 1]); p.set_weights(init_weights(L40))
        for _ in range(3):
            p.adam_step(ADAM_LR, sync=False)
        p.sync()
        ms = float(np.mean(timed_adam_steps(p, 10, flush=False)))
        k_ms = p.time_kernel_ms(5) / 5
        out["burgers_8x40_generic"] = {"config": "[2,40x8,1] tanh (upstream's systematic table), N_f=%d, generic fused kernel (any layer list; hidden layers on DMMA.8x8x4)" % n40,
                                       "ms_per_step": ms, "points_per_s": n40 / (ms * 1e-3), "kernel_ms": k_ms,
                                       "roofline_frac_fp64": (n40 * 24.0 * S40 + N_U * 6.0 * S40) / (k_ms * 1e-3) / 1e12 / peak}
        p.close()
    except Exception as e:  # pragma: no cover
        out["burgers_8x40_generic"] = {"error": str(e)}
    # ---- discrete time (SURVEY 8(f)2)
    try:
        q = 500
        L = [1, 50, 50, 50, q + 1]
        rng = np.random.default_rng(11)
        x0 = rng.uniform(-1, 1, (250, 1)); u0 = -np.sin(np.pi * x0)
        p = pinn_cabi.Pinn(pinn_cabi.BURGERS_DISC, L, [-1.0], [1.0])
        p.set_pde_params([NU, 0.8]); p.set_irk(rng.standard_normal((q + 1, q)) / q); p.set_boundary(np.array([-1.0, 1.0]))
        p.set_data(x0, u0); p.set_weights(init_weights(L))
        for _ in range(5):
            p.adam_step(1e-3, eps=1e-8, sync=False)
        p.sync()
        ms = float(np.mean(timed_adam_steps(p, 50, flush=False, lr=1e-3, eps=1e-8)))
        out["burgers_discrete_time"] = {"config": "1d-burgers/inf_disc_burgers.py: [1,50,50,50,501], N=250 + 2 boundary points, q=500 "
                                                  "(synthetic stage matrix)", "ms_per_step": ms, "points_per_s": 250 / (ms * 1e-3)}
        p.close()
    except Exception as e:  # pragma: no cover
        out["burgers_discrete_time"] = {"error": str(e)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-f", type=int, default=N_F_PER_GPU, help="collocation points per GPU (default: BASELINE configs[1])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cfg5", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (loss.npy, weights.npy, float64) to DIR, so that two builds "
                         "can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 implementation")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 10
        args.warmup = args.warmup if args.warmup is not None else 3
        run_reference_arm(args, rank, world)
        return
    args.steps = args.steps if args.steps is not None else 200      # no flags: a longer timed region than the driver's K
    args.warmup = args.warmup if args.warmup is not None else 20
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import pinn_cabi
    dist = None
    uid = None
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's version banner (printed at VERSION and WARN level) and any other
        # NCCL debug output go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # Control plane (uid exchange, barriers, max over ranks) on gloo: the ONLY NCCL communicator in this process is
        # the library's data-path one.  Two NCCL communicators with kernels in flight at the same time can deadlock
        # (observed at 4 ranks when torch's NCCL barrier overlapped the library's allreduce).
        dist.init_process_group("gloo")
        box = [pinn_cabi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]

    handle = []

    def barrier():
        for hh in handle:
            hh.sync()                      # drain the library's stream (incl. its exchange kernels) first
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    n_f = args.n_f
    n_f_global = n_f * world
    X_f, X_u, u = synthetic_problem(1234 + rank, n_f)
    _, X_u, u = synthetic_problem(1234, 1)     # data term identical on all ranks
    p = pinn_cabi.Pinn(pinn_cabi.BURGERS_INF, LAYERS, LB, UB, device=local_rank, rank=rank, world=world, nccl_uid=uid)
    handle.append(p)
    import sharding
    used_p2p = sharding.connect_p2p(dist, p, world) if dist is not None else False
    fused_tail = os.environ.get("PINN_FUSED_TAIL", "1") != "0"
    exchange = "none" if world == 1 else (
        ("inside the fused kernel: its last CTAs reduce the partials, push over NVLink into every peer's memory, sum in rank order and "
         "apply Adam (fused_tail / exchange_block; one launch per step)" if fused_tail else
         "fused reduce + NVLink all-to-all push + Adam kernel (reduce_exchange, P2P stores into peer memory)")
        if used_p2p else "reduce_partials + ncclAllReduce + adam_update")
    p.set_pde_params([NU])
    p.set_data(X_u, u, weight=1.0 if rank == 0 else 0.0)
    # pinned host copies of this rank's collocation batch (e2e leg uploads them every step)
    hx, hx_ptr = pinn_cabi.host_alloc(n_f)
    ht, ht_ptr = pinn_cabi.host_alloc(n_f)
    hx[:] = X_f[:, 0]; ht[:] = X_f[:, 1]
    import ctypes as C
    dp = C.POINTER(C.c_double)
    p.set_collocation_ptr(C.cast(hx_ptr, dp), C.cast(ht_ptr, dp), n_f, n_f_global)
    p.set_weights(init_weights())

    # ---------------- multi-GPU parity BEFORE anything is timed: sharded vs whole-set evaluation of the timed points
    parity = None
    if dist is not None:
        parity = parity_check(pinn_cabi, dist, p, rank, local_rank, world, n_f, X_u, u)
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"error": "multi-GPU parity check failed", "parity_check": parity}), flush=True)
            barrier()
            os._exit(3)

    # ---------------- device-resident steps, CUDA events per step, L2 flushed between timed iterations
    for _ in range(args.warmup):
        p.adam_step(ADAM_LR, sync=False)
    barrier()
    l0 = p.launch_count()
    with ClockSampler(local_rank) as clocks:
        t_wall0 = time.perf_counter()
        ms_steps = timed_adam_steps(p, args.steps, flush=True)
        barrier()
        launches = p.launch_count() - l0          # kernels of this library launched inside the timed region
        wall = time.perf_counter() - t_wall0
        # read back before the untimed steps below move the weights on
        dumped = {"loss": np.array([p.last_loss()]), "weights": p.get_weights()} if args.dump_outputs else None
        # keep the sampler alive for at least ~1.5 s of load so that it sees clocks under load; the same (fixed) number of
        # extra steps on every rank -- ranks MUST execute the same number of exchanges
        extra = int(max(0.0, 1.5 - wall) / max(wall / args.steps, 1e-5)) + 1
        if dist is not None:
            te = torch.tensor([extra], dtype=torch.int64)
            dist.broadcast(te, src=0)
            extra = int(te.item())
        long_ms = timed_adam_steps(p, min(extra, 2000), flush=False, ev0=2 * args.steps)
        for _ in range(max(0, extra - 2000)):
            p.adam_step(ADAM_LR, sync=False)
        p.sync()
        barrier()
    ms_step = max_over_ranks(dist, float(np.mean(ms_steps)))
    launches_per_step = launches / args.steps
    value = n_f_global / (ms_step * 1e-3)

    # ---------------- fused kernel alone (roofline)
    barrier()
    p.time_kernel_ms(3)
    k_iters = 50
    ms_kernel = min(p.time_kernel_ms(k_iters) / k_iters for _ in range(3))
    flops = n_f * FLOP_PER_COLLOC + (N_U * FLOP_PER_DATA if rank == 0 else 0)
    peak, peak_src = fp64_peak()
    hbm, hbm_src = hbm_peak()
    achieved = flops / (ms_kernel * 1e-3) / 1e12
    alg_bytes = 16.0 * n_f + 8.0 * 3021 + 8.0 * 3024
    traffic, traffic_src = _ncu_summary("burgers_v2")
    roofline = {"bound": "tensor", "pipe": "fp64 (DMMA.8x8x4 + DFMA share one pipe)", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic,
                "traffic_unit": "bytes per launch (dram read+write, ncu --set full, %s)" % traffic_src,
                "algorithmic_bytes": alg_bytes, "algorithmic_flop_per_launch": flops,
                "kernel": "pinn::burgers2::fused_loss_grad", "kernel_ms": ms_kernel,
                "hbm": {"achieved": alg_bytes / (ms_kernel * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                        "frac": alg_bytes / (ms_kernel * 1e-3) / 1e9 / hbm, "peak_source": hbm_src,
                        "note": "algorithmic bytes 16 B/point + weights in + gradient out; the path is FP64-bound"}}

    # ---------------- end to end through the public API with HOST buffers: every step hands the library that step's
    # collocation batch in pinned host memory and reads the loss back.  Two ways to get the batch across PCIe:
    #   copy  : pinn_set_collocation  -> explicit H2D copy (2 x 0.8 MB) + sync, then the step
    #   mapped: pinn_set_collocation_mapped -> zero-copy, the fused kernel reads the pinned batch itself over PCIe
    #           (prefetched one tile ahead), so the transfer overlaps the arithmetic.  Same bytes cross the bus per step.
    def e2e_loop(mapped):
        setter = p.set_collocation_mapped if mapped else p.set_collocation_ptr
        barrier()
        for _ in range(3):
            setter(C.cast(hx_ptr, dp), C.cast(ht_ptr, dp), n_f, n_f_global)
            p.adam_step(ADAM_LR, sync=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            setter(C.cast(hx_ptr, dp), C.cast(ht_ptr, dp), n_f, n_f_global)
            lv = p.adam_step(ADAM_LR, sync=True)
        barrier()
        sec = max_over_ranks(dist, (time.perf_counter() - t0) / args.steps)
        return sec, lv

    e2e_copy_s, loss = e2e_loop(False)
    e2e_map_s, loss = e2e_loop(True)
    p.set_collocation_ptr(C.cast(hx_ptr, dp), C.cast(ht_ptr, dp), n_f, n_f_global)     # back to the device-resident batch
    e2e_s = min(e2e_copy_s, e2e_map_s)
    e2e = {"value": n_f_global / e2e_s, "unit": "points/s", "h2d_bytes_per_step": 16 * n_f, "d2h_bytes_per_step": 8,
           "ms_per_step": e2e_s * 1e3, "timing": "wall clock around the API calls, barrier+synchronize both sides",
           "mode": "mapped (zero-copy: kernel reads the pinned batch over PCIe)" if e2e_map_s <= e2e_copy_s else "copy",
           "copy_mode": {"value": n_f_global / e2e_copy_s, "ms_per_step": e2e_copy_s * 1e3},
           "mapped_mode": {"value": n_f_global / e2e_map_s, "ms_per_step": e2e_map_s * 1e3}}
    kernel_info = p.kernel_info()

    # ---------------- BASELINE configs[4]: 2 000 000 global points over the GPUs of this run (replaces p's collocation set)
    cfg5 = None
    if not args.no_cfg5:
        barrier()
        try:
            cfg5 = cfg5_block(p, dist, rank, world)
        except Exception as e:  # pragma: no cover
            cfg5 = {"error": str(e)}
        barrier()

    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        extras = measure_extras(pinn_cabi, n_f, with_cpu=not args.no_cpu_baseline)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sec, cores, _, n_used = time_reference_port(n_f, 10, 3, budget_s=40.0)
        cpu = {"value": n_used / sec, "unit": "points/s", "cores": cores, "nproc": cpu_threads()[1], "kind": "port",
               "sample": f"10 Adam steps of N_f={n_used} after 3 warm-up, oracle/reference_port.py (nested reverse-mode, torch CPU fp64)"}

    if rank == 0:
        line = {
            "metric": "collocation-points/sec per training step (1D Burgers 8x20 tanh, Adam step)",
            "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "ms_per_step_median": float(np.median(ms_steps)), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(n_f), "global_points": n_f_global,
                       "l2": "flushed (256 MB memset) between timed iterations; inputs are 1.6 MB, the path is compute-bound",
                       "parallelism": "dp%d (collocation shards; per step one exchange of 3024 doubles = 24 KB per rank pair: %s)" % (world, exchange)},
            "clocks": clocks.summary(),
            "e2e": e2e, "gpu_launches": launches, "launches_per_step": launches_per_step,
            "roofline": roofline, "kernel_info": kernel_info, "final_loss": loss,
            "long_run": {"steps": len(long_ms), "ms_per_step": float(np.mean(long_ms)), "ms_per_step_median": float(np.median(long_ms)),
                         "note": "back-to-back asynchronous steps without L2 flush, timed per step with CUDA events (this rank)"},
        }
        if world > 1:
            line["nvlink_bytes_per_step"] = {"per_rank_sent": (world - 1) * 3024 * 8 if used_p2p else None,
                                             "note": "push exchange: every rank stores its 3024-double vector into each peer's buffer"
                                             if used_p2p else "NCCL allreduce (ring/tree chosen by NCCL)"}
        if parity is not None:
            line["parity_check"] = parity
        if cfg5 is not None:
            line["cfg5"] = cfg5
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if extras is not None:
            line["extras"] = extras
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr.astype(np.float64))
        print(json.dumps(line), flush=True)
    if dist is not None:
        barrier()
        p.close()
        dist.barrier()
        dist.destroy_process_group()
        sys.stdout.flush()
        os._exit(0)          # no lingering helper threads: the next launch on this box must find the GPUs and ports free


if __name__ == "__main__":
    # stdout carries exactly ONE JSON line.  C libraries loaded into this process write to file descriptor 1 on their own (NCCL
    # prints its version banner there whatever NCCL_DEBUG_FILE says), so descriptor 1 is pointed at stderr for the whole run
    # and Python's sys.stdout keeps the real one.
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_real_stdout, "w", buffering=1)
    main()
    sys.stdout.flush()
