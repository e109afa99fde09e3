#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 differentiable-A* engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[1]: NeuralAstar inference (CNN encoder + differentiable A*),
mazes_032_moore_c8 32x32, batch 100 per GPU.  A "step" is one `planner(map_designs, start_maps, goal_maps)` forward
over one batch.  Inputs are the reference's test split (100 maps, start positions drawn with seed 1234) and the
reference's shipped checkpoint, both committed as small fixtures under tests/golden/ (tests/golden/make_golden.py).

The K timed steps run through `neural_astar.utils.inference.PipelinedPlanner` (public API): one CUDA-graph launch
per step in which the search kernel of batch k overlaps the encoder convolutions of batch k+1.  `value` = device
resident inputs (rotated through a ring larger than L2); `e2e` = the same loop with every step's inputs copied from
pinned host memory and its results copied back (copies inside the graph).  Both are timed with CUDA events around
the WHOLE K-step loop (pipeline fill and drain included), barrier + synchronize on both sides, max over ranks.
Step k reads the 100 maps rolled by k % 112 positions, so the inputs of every step depend on k alone; `--dump-outputs DIR`
saves what the last step returned (histories, paths) for output-for-output comparison of two builds.

Prints ONE JSON line (rank 0) with the contract keys plus `roofline`, `cpu_baseline`, `e2e`, `clocks`,
`gpu_launches`, and `configs` (BASELINE.json configs[2..4]: training step, WarCraft-shaped 12x12, 256x256).
`--impl reference` times the reference's own PyTorch CPU implementation of the path when it was staged under
oracle/_ref (oracle/stage_ref.py), else the C restatement (oracle/astar_oracle.c, LITERAL form) + torch-CPU encoder.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "neural-astar_b200")
REF_STAGE = os.path.join(ROOT, "oracle", "_ref")

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "maps/sec, NeuralAstar inference (encoder + differentiable A*), 32x32 Moore mazes, b=100 per GPU"
UNIT = "maps/s"
BATCH = 100
H = W = 32
N_CELLS = H * W
ALGO_BYTES_PER_MAP = 28 * N_CELLS  # SURVEY.md 8(d): read cost+start+goal+obstacles, write histories(f32)+paths(i64)
WORKLOAD = "NeuralAstar inference, mazes_032_moore_c8 32x32, batch=100 (BASELINE.json configs[1])"
DATA = "mazes_032_moore_c8 test split (100 maps, seed-1234 starts) + shipped checkpoint, committed fixtures"
RING_N = 112   # 112 x 1.2 MB of inputs = 138 MB > 126 MB L2: a step's inputs are never L2-resident


def shared_config(world: int) -> dict:
    """`config` of the JSON line — identical in both arms (ours / --impl reference) so the two lines are comparable."""
    return {"workload": WORKLOAD, "batch_per_gpu": BATCH, "grid": "32x32", "g_ratio": 0.5, "T_max": W * W,
            "parallelism": f"dp{world} (independent map shards, no data-path collective; the reference arm runs on rank 0's "
                           f"host cores only)",
            "l2": f"GPU arm: inputs rotate through a ring of {RING_N} device-resident batches (138 MB > 126 MB L2), or come "
                  f"from pinned host memory every step (e2e); not applicable to the CPU reference arm",
            "timing": "GPU arm: CUDA events around the whole K-step loop (pipeline fill + drain inside), barrier + "
                      "synchronize both sides, max over ranks; reference arm: host wall clock"}


def _paths(ours: bool):
    for p in ((ROOT, PKG, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")) if ours
              else (ROOT, REF_STAGE, os.path.join(ROOT, "tests"))):
        if p not in sys.path:
            sys.path.insert(0, p)


def load_problem(name="mazes032_vanilla_test"):
    from golden_util import Golden

    g = Golden(name)
    return g.obst.astype(np.float32), g.start.astype(np.float32), g.goal.astype(np.float32), g


def load_planner(device):
    """NeuralAstar with the reference's shipped weights — from OUR package, or from the staged reference when the
    process runs `--impl reference` (sys.path decides which `neural_astar` is imported; never both)."""
    from neural_astar.planner import NeuralAstar

    planner = NeuralAstar(encoder_input="m+", encoder_arch="CNN", encoder_depth=4)
    state = np.load(os.path.join(ROOT, "tests", "golden", "mazes032_ckpt_planner_state.npz"))
    msg = planner.load_state_dict({k: torch.from_numpy(state[k]) for k in state.files})
    assert not msg.missing_keys and not msg.unexpected_keys, msg
    return planner.to(device).eval()


def dump_outputs(dirname, arrays):
    """Write each array as <dirname>/<name>.npy (float32), so that two builds run with the same arguments can be
    compared output for output."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


# ------------------------------------------------------------------------------------------------ clocks
_SAMPLER_SRC = r"""
import json, sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
samples, reasons = [], set()
mx = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
print("ready", flush=True)
import select
while True:
    if select.select([sys.stdin], [], [], 0)[0]:
        break
    try:
        samples.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        for bit, nm in names.items():
            if r & bit:
                reasons.add(nm)
    except Exception:
        pass
    time.sleep(0.002)
print(json.dumps({"samples": samples, "reasons": sorted(reasons), "max": mx}), flush=True)
"""


class ClockSampler:
    """SM clocks / throttle reasons sampled through NVML every 2 ms by a SEPARATE PROCESS while the timed regions
    run (a polling thread inside this interpreter would compete for the GIL with the launching thread)."""

    def __init__(self, index: int):
        self.index, self.proc, self.result = index, None, None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, str(self.index)], stdin=subprocess.PIPE,
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            if self.proc.stdout.readline().strip() != "ready":
                self.proc = None
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            try:
                out, _ = self.proc.communicate("stop\n", timeout=10)
                self.result = json.loads(out.strip().splitlines()[-1])
            except Exception:
                self.result = None

    def summary(self):
        r = self.result
        if not r or not r.get("samples"):
            return {"sm_mhz": None, "sm_max_mhz": (r or {}).get("max"), "reasons": (r or {}).get("reasons", []), "samples": 0}
        return {"sm_mhz": float(np.median(r["samples"])), "sm_max_mhz": r["max"], "reasons": r["reasons"],
                "samples": len(r["samples"]), "sampler": "NVML, separate process, 2 ms period, over all timed legs"}


def pin_to_gpu_numa(index: int):
    """Run this rank on the CPU cores NVML reports as local to its GPU (SCALE_r01: GPU0-3 -> CPUs 0-31,64-95)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_traffic():
    """DRAM bytes per launch of the search kernel from the committed ncu summary, if any."""
    path = os.path.join(ROOT, "profiles", "latest_kernel_summary.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------ reference arm
class _SweepTimeout(Exception):
    pass


def _bounded(fn, limit_s):
    """Wall time of fn(), or inf when it is still running after limit_s seconds (SIGALRM raises inside the Python-level
    loop of the reference, which executes thousands of small ops per call)."""
    import signal

    def on_alarm(signum, frame):
        raise _SweepTimeout()

    old = signal.signal(signal.SIGALRM, on_alarm)
    signal.setitimer(signal.ITIMER_REAL, limit_s)
    try:
        t0 = time.perf_counter()
        fn()
        return time.perf_counter() - t0
    except _SweepTimeout:
        return float("inf")
    finally:
        signal.setitimer(signal.ITIMER_REAL, 0.0)
        signal.signal(signal.SIGALRM, old)


def _pick_threads(fn, set_threads):
    """The host's best thread count.  The reference's loop is thousands of tiny ops, each an OpenMP fork-join: past a
    few dozen threads (and across sockets) it collapses — measured on the B200 host: 16 threads fastest, 128 unpinned
    threads took minutes per batch.  Counts are tried in ascending order on the CPUs this process may use; every trial
    after the first is cut off at 4x the best time so far, and the sweep stops at the first count that is slower."""
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({min(avail, c) for c in (8, 16, 32, 64, avail)})
    best, best_t, tried = cands[0], float("inf"), []
    for c in cands:
        set_threads(c)
        limit = 300.0 if best_t == float("inf") else 4.0 * best_t + 1.0
        warm = _bounded(fn, limit)
        dt = _bounded(fn, limit) if warm != float("inf") else float("inf")
        tried.append(c)
        if dt < best_t:
            best, best_t = c, dt
        else:
            break
    set_threads(best)
    return best, tried, best_t


def bench_reference(args):
    """The reference's CPU implementation of the path on this box's host cores, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    pinned = pin_to_gpu_numa(0)   # one socket's cores, like the GPU arm's rank 0 (cross-socket OpenMP teams are far slower)
    staged = os.path.isdir(os.path.join(REF_STAGE, "neural_astar", "planner")) and not args.port
    _paths(ours=False)
    maps, start, goal, _ = load_problem()
    if staged:
        # the reference's own modules (staged by oracle/stage_ref.py at build time): NeuralAstar.forward =
        # encoder + the PyTorch DifferentiableAstar loop (differentiable_astar.py:150-267), unmodified
        import neural_astar

        assert os.path.realpath(neural_astar.__file__).startswith(os.path.realpath(REF_STAGE)), neural_astar.__file__
        planner = load_planner(torch.device("cpu"))
        tm, ts, tg = (torch.from_numpy(x) for x in (maps, start, goal))

        def run(m=BATCH):
            with torch.no_grad():
                return planner(tm[:m], ts[:m], tg[:m])

        threads, cands, t_full = _pick_threads(run, torch.set_num_threads)
        kind = "reference"
        what = "the reference's own PyTorch NeuralAstar.forward (staged, unmodified: encoder + DifferentiableAstar loop)"
    else:
        # fallback when nothing was staged: C restatement of the loop (LITERAL form) + torch-CPU encoder of our package
        _paths(ours=True)
        from oracle import oracle

        oracle.build()
        planner = load_planner(torch.device("cpu"))

        class _Out:
            pass

        def run(m=BATCH):
            with torch.no_grad():
                cost = planner.encode(*(torch.from_numpy(x[:m]) for x in (maps, start, goal))).numpy()
            return oracle.forward(cost, start[:m], goal[:m], maps[:m], g_ratio=0.5, mode="literal")

        def set_threads(c):
            torch.set_num_threads(c)
            oracle.set_threads(c)

        threads, cands, t_full = _pick_threads(run, set_threads)
        kind = "port"
        what = "torch-CPU encoder + oracle LITERAL loop (oracle/astar_oracle.c, OpenMP over maps)"
    # bound the whole run (warm-up + K timed steps) to a few minutes: when K full batches would take longer, every
    # step processes the first m maps of the batch instead (maps/s stays the unit; the sample is stated)
    budget_s = float(args.budget)
    m = BATCH
    total = args.steps + args.warmup
    if t_full * total > budget_s:
        m = int(max(10, min(BATCH, BATCH * budget_s / (t_full * total))))
    out = None
    for _ in range(args.warmup):
        out = run(m)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = run(m)
    dt = time.perf_counter() - t0
    value = m * args.steps / dt
    hist_sum = float(out.histories.sum())
    sample = (f"each step = the first {m} of the b={BATCH} maps through {what}; {threads} threads = fastest of {cands} "
              f"(ascending sweep, stopped at the first slower count) on {len(os.sched_getaffinity(0))} of "
              f"{os.cpu_count()} logical CPUs" + (" (GPU 0's NUMA node)" if pinned else ""))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": DATA,
        "config": shared_config(args.gpus),
        "expansions_per_s": hist_sum * args.steps / dt,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def run_cpu_baseline(budget_s=20.0):
    """cpu_baseline of our own line (rank 0, N=1): the reference arm in a SUBPROCESS (its `neural_astar` package is
    the staged reference, which must not meet ours in one interpreter), bounded to ~`budget_s` seconds."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "5", "--warmup", "1",
           "--budget", str(budget_s)]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env).stdout
        line = json.loads([ln for ln in out.splitlines() if ln.startswith("{")][-1])
        return line["cpu_baseline"]
    except Exception as e:  # pragma: no cover
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": f"reference arm failed: {e!r}"}


# ------------------------------------------------------------------------------------------------ ours
class Timer:
    def __init__(self, dist, dev):
        self.dist, self.dev = dist, dev

    def barrier(self, all_ranks=True):
        if self.dist is not None and all_ranks:
            self.dist.barrier()
        torch.cuda.synchronize()

    def loop(self, body, all_ranks=True):
        """Device time of `body()` as a whole (events on the launching stream), barrier + sync on both sides."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier(all_ranks)
        a.record()
        out = body()
        b.record()
        self.barrier(all_ranks)
        return a.elapsed_time(b), out

    def per_step(self, fn, steps, flush):
        """Sum of per-step event pairs with the L2 flushed (outside the pairs) between steps: rank-local."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        out = None
        for a, b in evs:
            flush.zero_()
            a.record()
            out = fn()
            b.record()
        torch.cuda.synchronize()
        ts = [a.elapsed_time(b) for a, b in evs]
        return ts, out


def config_c3(dev, peak):
    """BASELINE.json configs[2]: NeuralAstar training step (scripts/train.py semantics: Tmax=0.25, B=100, RMSprop
    1e-3, L1 loss) on the reference's first training batch (tests/golden/train_curve_mazes032.npz)."""
    from types import SimpleNamespace

    from neural_astar import _native
    from neural_astar.planner import NeuralAstar
    from neural_astar.utils.training import PlannerModule

    z = np.load(os.path.join(ROOT, "tests", "golden", "train_curve_mazes032.npz"))
    B, Hh, Ww = (int(v) for v in z["shape"])
    N = Hh * Ww

    def bits(k):
        return np.unpackbits(z[k], axis=1)[:, :N].reshape(B, 1, Hh, Ww).astype(np.float32)

    def onehot(k):
        x = np.zeros((B, N), np.float32)
        x[np.arange(B), z[k]] = 1
        return x.reshape(B, 1, Hh, Ww)

    batch = [torch.from_numpy(x).to(dev) for x in (bits("obst_bits"), onehot("start_idx"), onehot("goal_idx"), bits("opt_bits"))]
    torch.manual_seed(1234)
    planner = NeuralAstar(encoder_input="m+", encoder_arch="CNN", encoder_depth=4, Tmax=0.25)
    module = PlannerModule(planner, SimpleNamespace(params=SimpleNamespace(lr=1e-3))).to(dev).train()
    opt = module.configure_optimizers()

    def step():
        opt.zero_grad(set_to_none=True)
        loss = module.training_step(batch, 0)
        loss.backward()
        opt.step()
        return loss

    for _ in range(5):
        step()
    torch.cuda.synchronize()
    K = 20
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(K):
        step()
    b.record()
    torch.cuda.synchronize()
    ms_eager = a.elapsed_time(b) / K
    # the same step as ONE CUDA-graph launch (neural_astar.utils.training.GraphedTrainStep)
    from neural_astar.utils.training import GraphedTrainStep

    gstep = GraphedTrainStep(module, batch)
    for _ in range(3):
        gstep(batch)
    torch.cuda.synchronize()
    a.record()
    for _ in range(K):
        gstep(batch)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / K
    # the two search kernels alone: forward (T = 256 cap) and closed-form backward, on the current cost maps
    with torch.no_grad():
        cost = planner.encode(*batch[:3]).contiguous()
    T = int(0.25 * Ww * Ww)
    fw = lambda: _native.forward(cost, batch[1], batch[2], batch[0], 0.5, T)  # noqa: E731
    hist, _, ts, ns, _ = fw()
    Tb = _native.batch_steps(ts, ns, T)
    gh = torch.sign(hist - batch[3]) / hist.numel()
    bw = lambda: _native.backward(cost, batch[1], batch[2], batch[0], gh, Tb, ts, 0.5)  # noqa: E731

    def t_of(fn):
        for _ in range(3):
            fn()
        x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x.record()
        for _ in range(10):
            fn()
        y.record()
        torch.cuda.synchronize()
        return x.elapsed_time(y) / 10 * 1e3

    fwd_us, bwd_us = t_of(fw), t_of(bw)
    algo = 36 * N * B    # SURVEY 8(d): 28*N forward + read grad_histories + write grad_cost
    ach = algo / ((fwd_us + bwd_us) * 1e-6) / 1e9
    # the same pair on 64x64 maps (the reference's all_064 set: tests/golden/all064_vanilla.npz, 12 maps x8), training
    # cap T = 0.25*64*64: forward and event-based backward on the warp64 engine
    g64 = load_problem("all064_vanilla")[3]
    rep = 8
    o64, s64, g64t = (torch.from_numpy(np.tile(x, (rep, 1, 1, 1))).to(dev) for x in (g64.obst, g64.start, g64.goal))
    gen = torch.Generator().manual_seed(7)
    c64 = (o64.cpu() * (0.3 + 0.7 * torch.rand(o64.shape, generator=gen))).to(dev)
    T64 = int(0.25 * 64 * 64)
    fw64 = lambda: _native.forward(c64, s64, g64t, o64, 0.5, T64)  # noqa: E731
    h64, _, ts64, ns64, _ = fw64()
    Tb64 = _native.batch_steps(ts64, ns64, T64)
    gh64 = torch.randn(h64.shape, generator=gen).to(dev) / h64.numel()
    bw64 = lambda: _native.backward(c64, s64, g64t, o64, gh64, Tb64, ts64, 0.5)  # noqa: E731
    f64_us, b64_us = t_of(fw64), t_of(bw64)
    return {"workload": "NeuralAstar training step (Tmax=0.25 -> T=256, b=100, RMSprop, L1), mazes_032 first train batch",
            "train_steps_per_s": 1e3 / ms, "maps_per_s": B * 1e3 / ms, "ms_per_step": ms, "ms_per_step_eager": ms_eager,
            "api": "neural_astar.utils.training.GraphedTrainStep (forward + L1 loss + backward + RMSprop as one CUDA graph); "
                   "ms_per_step_eager = the same step issued op by op from Python",
            "search_fwd_us": fwd_us, "search_bwd_us": bwd_us,
            "grid64": {"workload": "search kernels alone, all_064 maps (12 distinct x8 = 96), learned-like costs, T = 1024 cap",
                       "fwd_us": f64_us, "bwd_us": b64_us, "bwd_over_fwd": b64_us / f64_us,
                       "engines": "forward and backward: warp64 (engine 4), event-based closed form"},
            "roofline": {"bound": "hbm", "kernel": "astar_warp32_kernel<0,0,0> + <0,1,0>", "achieved": ach, "peak": peak,
                         "unit": "GB/s", "frac": ach / peak, "algorithmic_bytes_per_launch": algo}}


def config_c4(dev, peak):
    """BASELINE.json configs[3]: WarCraft-shaped inference, b=512, 96x96 RGB -> 12x12 costs (data not shipped:
    synthetic RGB as SURVEY.md 8(d) C4 prescribes), CNNDownSize depth 3, const 10, learn_obstacles."""
    from neural_astar import _native
    from neural_astar.planner import NeuralAstar
    from neural_astar.utils.inference import GraphedPlanner

    B = 512
    g = torch.Generator().manual_seed(1234)
    maps = torch.rand(B, 3, 96, 96, generator=g).to(dev)
    start = torch.zeros(B, 1, 12, 12, device=dev); start[:, :, 0, 0] = 1
    goal = torch.zeros(B, 1, 12, 12, device=dev); goal[:, :, 11, 11] = 1
    torch.manual_seed(1234)
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):      # the constructor prints a learn_obstacles warning (like the reference)
        na = NeuralAstar(encoder_input="rgb+", encoder_arch="CNNDownSize", encoder_depth=3, learn_obstacles=True, const=10.0)
    na = na.to(dev).eval()
    fast = GraphedPlanner(na, maps, start, goal)
    for _ in range(3):
        fast.replay()
    K = 20
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(K):
        out = fast.replay()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / K
    with torch.no_grad():
        cost = na.encode(maps, start, goal)
        ones = torch.ones_like(start)
        for _ in range(3):
            _native.forward(cost, start, goal, ones, 0.5, 144)
        x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x.record()
        for _ in range(10):
            _native.forward(cost, start, goal, ones, 0.5, 144)
        y.record()
        torch.cuda.synchronize()
    kus = x.elapsed_time(y) / 10 * 1e3
    algo = 28 * 144 * B
    ach = algo / (kus * 1e-6) / 1e9
    return {"workload": "NeuralAstar inference, synthetic 96x96 RGB -> 12x12 (CNNDownSize d3, const 10, learn_obstacles), b=512",
            "maps_per_s": B * 1e3 / ms, "ms_per_step": ms, "expansions_per_map": float(out.histories.sum()) / B,
            "search_kernel_us": kus, "api": "GraphedPlanner replay (encoder + search in one CUDA graph)",
            "roofline": {"bound": "hbm", "kernel": "astar_warp32_kernel<0,0,0>", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "algorithmic_bytes_per_launch": algo}}


def config_c5(dev, peak, rank, timer, dist, world):
    """BASELINE.json configs[4]: synthetic 256x256 Moore grids, 1024 DISTINCT maps per GPU (seed 1234 + rank),
    VanillaAstar semantics; sharded over the ranks with no data-path collective."""
    from c5_data import c5_maps
    from neural_astar import _native

    Hh = Ww = 256
    per_gpu = 1024
    t0 = time.time()
    obst, start, goal = c5_maps(per_gpu, Hh, Ww, 1234 + rank)
    gen_s = time.time() - t0
    o, s, g = (torch.from_numpy(x).to(dev) for x in (obst, start, goal))
    fn = lambda: _native.forward(o, s, g, o, 0.5, Ww * Ww)  # noqa: E731
    for _ in range(3):
        out = fn()
    # (1) one launch at a time: the launch lasts as long as its longest map (latency figure, roofline denominator).
    # Every call allocates its 0.8 GB of outputs; the loops below keep at most two result sets alive, exactly like the
    # warm-up above, so the caching allocator serves them from its pool (a fresh 0.8 GB cudaMalloc inside the timed
    # region costs tens of ms and used to make this figure jump between runs).  Median of three timed loops.
    reps = 3

    def serial(n):
        last = None
        for _ in range(n):
            last = fn()
        return last

    trials = []
    for _ in range(3):
        t_ms, out = timer.loop(lambda: serial(reps))
        trials.append(t_ms / reps)
    ms_serial = sorted(trials)[1]
    # (2) throughput: consecutive batches on 4 streams.  Engine 5 runs persistent CTAs that leave as their work queue
    # drains, so the next batch's CTAs move onto the SMs the current batch has already vacated while its last, longest
    # maps are still being searched on a few SMs.  Every launch does its full work and completes inside the timed region.
    n_streams, reps_t = 4, 16
    from neural_astar.planner import VanillaAstar
    from neural_astar.utils.inference import OverlappedPlanner

    over = OverlappedPlanner(VanillaAstar().to(dev).eval(), n_streams=n_streams, device=dev)

    def overlapped(n):
        last = None
        for _ in range(n):
            last = over.submit(o, s, g)
        over.wait_all()
        return last.result()

    overlapped(2 * n_streams)
    trials_t = []
    for _ in range(3):
        t_ms, out_t = timer.loop(lambda: overlapped(reps_t))
        trials_t.append(t_ms / reps_t)
    ms = sorted(trials_t)[1]
    assert torch.equal(out_t.histories, out[0]) and torch.equal(out_t.paths, out[1])   # same results as the serial launch
    ns = out[3].float()
    stats = torch.tensor([ms, float(ns.sum()), float(ns.max()), float((out[2] >= 0).sum()), ms_serial], device=dev,
                         dtype=torch.float64)
    if dist is not None:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, exp_total, exp_max, solved, ms_serial = float(mx[0]), float(sm[1]), float(mx[2]), float(sm[3]), float(mx[4])
    else:
        ms, exp_total, exp_max, solved, ms_serial = (float(v) for v in stats)
    maps_total = per_gpu * world
    algo = 24 * Hh * Ww * per_gpu     # cost aliases obstacles: 24*N bytes per map (SURVEY 8(d))
    traffic = None                    # DRAM bytes per launch from the committed ncu capture (296 maps), scaled to this batch
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_bin16_v3.json")))
        traffic = prof["dram_bytes_per_launch"] / 296.0 * per_gpu
    except Exception:
        pass
    ach = algo / (ms_serial * 1e-3) / 1e9
    return {"workload": f"VanillaAstar, synthetic 256x256 Moore grids (p_obst 0.2, Chebyshev(start,goal) >= 128), "
                        f"{per_gpu} distinct maps per GPU x {world} GPU(s), seed 1234+rank",
            "maps_per_s": maps_total / (ms * 1e-3), "maps_per_s_per_gpu": per_gpu / (ms * 1e-3), "ms_per_batch": ms,
            "throughput_mode": f"utils.inference.OverlappedPlanner(VanillaAstar): {reps_t} batches round-robin on {n_streams} streams, max over ranks (tails of one batch "
                               "overlap the next batches); `serial` = one launch at a time",
            "ms_per_batch_trials": trials_t,
            "serial": {"ms_per_launch": ms_serial, "ms_per_launch_trials": trials, "maps_per_s": maps_total / (ms_serial * 1e-3),
                       "us_per_step_longest_map": ms_serial * 1e3 / max(exp_max, 1.0)},
            "expansions_per_s": exp_total / (ms * 1e-3), "mean_expansions_per_map": exp_total / maps_total,
            "max_expansions_per_map": exp_max, "solved": solved,
            "engine": "5 (binary-cost, CTA per map, nastar_bin16.cuh)" if _native.lib().nastar_b200_bin16_supported(Hh, Ww)
                      and os.environ.get("NASTAR_B200_BIN16", "1") != "0" else "3 (generic, HBM workspace)",
            "map_generation_s_per_rank": gen_s,
            "roofline": {"bound": "hbm", "kernel": "astar_bin16_kernel<8>", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "algorithmic_bytes_per_launch": algo, "traffic": traffic, "per_gpu": True,
                         "note": "one launch alone (serial.ms_per_launch) is latency-bound: it lasts as long as its longest "
                                 "map (one dependent step chain per map); see serial.us_per_step_longest_map"}}


def bench_ours(args):
    _paths(ours=True)
    from neural_astar import _native
    from neural_astar.planner import encoder as _enc
    from neural_astar.utils.inference import PipelinedPlanner

    _native.lib()  # fail loudly when the CUDA engine is not built
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    pinned_cpus = pin_to_gpu_numa(local_rank)
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        dist = None
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    timer = Timer(dist, dev)
    K, Wm = args.steps, max(args.warmup, 3)

    maps_np, start_np, goal_np, golden = load_problem()
    planner = load_planner(dev)
    maps, start, goal = (torch.from_numpy(x).to(dev) for x in (maps_np, start_np, goal_np))
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # ---- the two timed legs: pipelined planner, device-resident ring / pinned host buffers -----------------------
    ring_n = RING_N
    ring = torch.stack([torch.stack([t.roll(i, 0) for t in (maps, start, goal)]) for i in range(ring_n)])
    pipe_dev = PipelinedPlanner(planner, maps, start, goal)
    pipe_host = PipelinedPlanner(planner, maps, start, goal, host=True)
    pipe_dev.prepare()
    pipe_host.prepare()
    step_evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]

    def loop_dev(n, evs=None):
        for k in range(n):
            pipe_dev.submit_stacked(ring[k % ring_n])
            if evs is not None:
                evs[k + 1].record()
        return pipe_dev.drain()

    def loop_host(n):
        for _ in range(n):
            pipe_host.submit()
        return pipe_host.drain()

    loop_dev(Wm)
    loop_host(Wm)
    torch.cuda.synchronize()

    with ClockSampler(local_rank) as clk:
        l0 = pipe_dev.native_launches

        def body():
            step_evs[0].record()
            return loop_dev(K, step_evs)

        total_ms, out = timer.loop(body)
        # the last step's results live in graph-owned buffers that later replays overwrite: copy them now
        dumped = ({"histories": out.histories.cpu().numpy(), "paths": out.paths.to(torch.float32).cpu().numpy()}
                  if args.dump_outputs else None)
        launches = pipe_dev.native_launches - l0
        step_ms = [step_evs[i].elapsed_time(step_evs[i + 1]) for i in range(K)]
        e2e_ms, _ = timer.loop(lambda: loop_host(K))
        torch.cuda.synchronize()
        expansions = float(out.histories.sum())     # last batch (a rotation of the same 100 maps)
        # search kernel alone (roofline denominator): finished cost maps, same stream; like the timed loop above the
        # inputs rotate through rings larger than L2 (maps/start/goal ring 138 MB + cost ring 46 MB), so every launch
        # reads its planes from HBM while the kernel's instructions stay cached as they are in the real pipeline
        # (flushing L2 with a 512 MB memset also evicts the kernel's code, which a one-warp-per-SM launch then
        # re-fetches line by line: measured 411 us instead of ~65 us)
        with torch.no_grad():
            cost = planner.encode(maps, start, goal)
        cost_ring = torch.stack([cost.roll(i, 0) for i in range(ring_n)])
        kern_evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for i in range(3):
            _native.forward(cost_ring[i], ring[i][1], ring[i][2], ring[i][0], 0.5, W * W)
        torch.cuda.synchronize()
        for i, (ea, eb) in enumerate(kern_evs):
            sl = (i + 3) % ring_n
            ea.record()
            _native.forward(cost_ring[sl], ring[sl][1], ring[sl][2], ring[sl][0], 0.5, W * W)
            eb.record()
        torch.cuda.synchronize()
        kern_ms = float(sum(ea.elapsed_time(eb) for ea, eb in kern_evs))
        # the same kernel with the SMs filled: the 1000 distinct maps of mazes_032 (train+valid+test) x100 =
        # 100 000 maps, 2.87 GB of algorithmic traffic (larger than L2)
        sat = None
        if rank == 0 and not args.no_saturated:
            o1k, s1k, g1k, _ = load_problem("inputs_mazes032_all1000")
            o1k, s1k, g1k = (torch.from_numpy(x).to(dev) for x in (o1k, s1k, g1k))
            with torch.no_grad():
                c1k = torch.cat([planner.encode(o1k[i:i + 200], s1k[i:i + 200], g1k[i:i + 200]) for i in range(0, 1000, 200)])
            rep = 100
            big = [x.repeat(rep, 1, 1, 1) for x in (c1k, s1k, g1k, o1k)]
            sat_fn = lambda: _native.forward(*big, 0.5, W * W)  # noqa: E731
            for _ in range(3):   # warm-up: the 1.2 GB of outputs must come from the caching allocator, not cudaMalloc
                sat_out = sat_fn()
            del sat_out
            sat_ts, sat_out = timer.per_step(sat_fn, 5, flush)
            sat_s = float(np.mean(sat_ts)) * 1e-3
            nb = 1000 * rep
            sat = {"batch": nb, "distinct_maps": 1000, "kernel_ms": sat_s * 1e3, "maps_per_s": nb / sat_s,
                   "expansions_per_s": float(sat_out[0].sum()) / sat_s,
                   "achieved": ALGO_BYTES_PER_MAP * nb / sat_s / 1e9, "unit": "GB/s"}
            del big, sat_out
        peak, peak_src = peak_hbm()
        configs = {}
        if not args.no_configs:
            if rank == 0 and world == 1:
                configs["c3"] = config_c3(dev, peak)
                configs["c4"] = config_c4(dev, peak)
            c5 = config_c5(dev, peak, rank, timer, dist, world)
            if rank == 0:
                configs["c5"] = c5

    # parity spot-check against the committed reference output for these inputs (learned costs differ in the last
    # ulp between cuDNN and the CPU encoder, so compare the vanilla search exactly)
    van = _native.forward(maps, start, goal, maps, 0.5, W * W)
    assert np.array_equal(van[0].cpu().numpy() != 0, golden.bits("hist_bits") != 0), "search parity lost"

    if dist is not None:
        t = torch.tensor([total_ms, e2e_ms, kern_ms, max(step_ms)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms, kern_ms, step_max = (float(x) for x in t)
        e = torch.tensor([expansions, float(launches)], device=dev, dtype=torch.float64)
        dist.all_reduce(e, op=dist.ReduceOp.SUM)
        expansions, launches = float(e[0]), int(e[1])
    else:
        step_max = max(step_ms)
    if rank == 0:
        maps_total = BATCH * world * K
        value = maps_total / (total_ms * 1e-3)
        kern_s = kern_ms * 1e-3 / K
        achieved = ALGO_BYTES_PER_MAP * BATCH / kern_s / 1e9
        h2d = int(sum(x.numel() * x.element_size() for x in pipe_host.host_inputs[0]))
        d2h = int(sum(x.numel() * x.element_size() for x in pipe_host.host_outputs[0]))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": total_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 search (bit-exact masks) / " + ("tf32" if _enc.ALLOW_TF32 else "fp32")
                     + " encoder 3x3 convs (cuDNN tensor cores, torch's default), fp32 head",
            "data": DATA,
            "config": shared_config(world),
            "api": "neural_astar.utils.inference.PipelinedPlanner (one CUDA-graph launch per step: search of batch k || "
                   "encoder of batch k+1)",
            "rank_cpu_affinity": pinned_cpus,
            "ms_per_step_median": float(np.median(step_ms)), "ms_per_step_max": step_max,
            "expansions_per_s": expansions * K / (total_ms * 1e-3),
            "search_kernel_us": kern_s * 1e6,
            "e2e": {"value": maps_total / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / K,
                    "api": "PipelinedPlanner(host=True), three stages per step graph: pinned H2D(batch k) || encoder(k-1) || "
                           "search(k-2) + D2H of histories+paths; K submits + drain inside the timed region"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "nastar::astar_warp32_kernel<0,0,0>",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src, "traffic": ncu_traffic(),
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_MAP * BATCH,
                         "timing": "CUDA events around each launch, inputs rotated through rings larger than L2 (184 MB)",
                         "note": "b=100 occupies 100 of 148 SMs with one warp each: latency-bound by the longest map's "
                                 "dependent steps; `saturated` is the same kernel at b=100000 (1000 distinct maps x100)"},
            "clocks": clk.summary(),
        }
        if sat is not None:
            sat["peak"] = peak
            sat["frac"] = sat["achieved"] / peak
            line["roofline"]["saturated"] = sat
        if configs:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = run_cpu_baseline()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-saturated", action="store_true", help="skip the b=100000 kernel-only measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs block (training / WarCraft / 256x256)")
    ap.add_argument("--port", action="store_true", help="--impl reference: use the C restatement even if the reference is staged")
    ap.add_argument("--budget", type=float, default=150.0, help="--impl reference: seconds for warm-up + timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the histories and paths of the last timed step as DIR/histories.npy and DIR/paths.npy "
                         "(float32, [100,1,32,32] each; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_ours(args)


if __name__ == "__main__":
    main()
