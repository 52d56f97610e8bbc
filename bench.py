#!/usr/bin/env python
"""Benchmark of the DDPG / TD3 update hot path (BASELINE.json metric:
"DDPG update-steps/sec @ batch 4096, 1/2/4/8xB200; embed-gather HBM GB/s").

  python bench.py --gpus N --steps K --warmup W            # this framework (CUDA path), DDPG (BASELINE configs[1])
  python bench.py --algo td3 ...                           # the same line for TD3 (BASELINE configs[2])
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's losses and weights
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores
                                                           # (numpy port in oracle/; /root/reference is Python
                                                           # and does not exist on the GPU box)

One "step" = one update (ddpg_update / td3_update) over one synthetic ML-20M-shaped minibatch:
26,744 items x 128-d table, frame_size 10, 4096 sample rows per GPU, policy step every 10th
step, Adam(lr=1e-5), dropout active (perf mode: on-device Philox).  Prints ONE JSON line.

Timing protocol: both CUDA-graph variants of the step (policy / non-policy) are primed before any timed
region whatever --warmup is; W untimed warm-up steps; then R repeats (R >= 3) of EXACTLY K steps, each
repeat bracketed by barrier + synchronize, every step timed on the device with CUDA events (L2 flushed by
a 256 MB write between steps, outside the events), max over ranks; `value` is the median repeat and
`spread` gives min / max.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ITEMS, DIM, FRAME, HIDDEN = 26744, 128, 10, 256
S_DIM = DIM * FRAME + FRAME
ROWS_PER_GPU = 4096
STRONG_ROWS = 8192                    # BASELINE configs[3]: 8192 rows sharded over the GPUs (strong scaling)
POLICY_STEP = 10
# SURVEY.md 8d: algorithmic work per sample row
GATHER_BYTES_PER_ROW = 16604
GATHER_READ_BYTES_PER_ROW = 5764
FLOP = {"ddpg": (5276160, 6526976), "td3": (7980544, 9231360)}      # (non-policy step, policy step)
L1_FWD_FLOP_PER_ROW = 2 * S_DIM * HIDDEN           # the dominant kernel: layer-1 forward GEMM


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            p = json.load(fh)
        return dict(hbm=float(p["hbm_gbs"]), bf16=float(p["bf16_tflops"]),
                    bf16_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    except Exception:
        return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()          # exact PID, never by pattern
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.strip().split(",") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
            sm = [float(r[0]) for r in rows]
            out["samples"] = len(sm)
            if sm:
                busy = [x for x in sm if x > 0.5 * max(sm)] or sm
                out["sm_mhz"] = float(np.median(busy))
                out["sm_max_mhz"] = float(rows[0][1])
                out["power_w_max"] = max(float(r[2]) for r in rows)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for i, nm in enumerate(names):
                    if any(r[3 + i].strip().lower().startswith("active") for r in rows):
                        out["reasons"].append(nm)
        except Exception:
            pass
        return out


def synth_step_inputs(seed, n_rows, n_steps):
    """Per-step minibatches: items ~ U{0..n_items-1}, ratings ~ U{-4..5}, one pseudo-user."""
    rng = np.random.default_rng(seed)
    items = rng.integers(0, N_ITEMS, size=(n_steps, n_rows, FRAME + 1), dtype=np.int64)
    ratings = rng.integers(-4, 6, size=(n_steps, n_rows, FRAME + 1)).astype(np.float32)
    done = np.zeros((n_rows,), dtype=np.float32)
    done[-1] = 1.0
    return items, ratings, done


def workload_name(algo, n_rows=ROWS_PER_GPU, per_gpu=True):
    cfg = "configs[1]" if algo == "ddpg" else "configs[2]"
    return "%s batch %d rows%s, 128-d embeddings, 26744 items, frame 10 (BASELINE %s)" % (
        algo.upper(), n_rows, "/GPU" if per_gpu else "", cfg)


# =============================================================================== reference arm
class _OracleStepper:
    """Reference algorithm (gather + ddpg_update / td3_update) on the host: numpy port in oracle/."""

    def __init__(self, n_rows, algo="ddpg"):
        from oracle import recnn_oracle as O
        from oracle import cases as C
        self.O, self.C, self.n, self.algo = O, C, n_rows, algo
        rng = np.random.default_rng(0)
        self.rng = rng
        self.table = rng.standard_normal((N_ITEMS, DIM), dtype=np.float32)
        self.nets = {"policy_net": O.make_actor(rng, S_DIM, DIM, HIDDEN, 6e-1)}
        self.nets["target_policy_net"] = O.copy_net(self.nets["policy_net"])
        self.opts = {"policy_optimizer": O.make_optimizer("adam", lr=1e-5)}
        for sfx in ([""] if algo == "ddpg" else ["1", "2"]):
            self.nets["value_net" + sfx] = O.make_critic(rng, S_DIM, DIM, HIDDEN, 54e-2)
            self.nets["target_value_net" + sfx] = O.copy_net(self.nets["value_net" + sfx])
            self.opts["value_optimizer" + sfx] = O.make_optimizer("adam", lr=1e-5)
        self.sizes = np.asarray([n_rows + FRAME], dtype=np.int64)
        self.items, self.ratings, _ = synth_step_inputs(1, n_rows, 4)
        self.step = 0

    def run(self):
        """One step; returns its wall time (the dropout / noise draws are not timed: RNGs differ per implementation)."""
        O = self.O
        masks = O.synth_masks(self.rng, 6 if self.algo == "ddpg" else 8, self.n, HIDDEN)
        noise = None
        if self.algo == "td3":
            noise = (self.rng.standard_normal((self.n, DIM)) * self.C.TD3_PARAMS["noise_std"]).astype(np.float32)
        i = self.step % 4
        t0 = time.perf_counter()
        batch = O.frame_gather(self.table, self.items[i], self.ratings[i], self.sizes, FRAME)
        if self.algo == "ddpg":
            O.ddpg_update(batch, dict(self.C.DDPG_PARAMS), self.nets, self.opts, masks, self.step, learn=True)
        else:
            O.td3_update(batch, dict(self.C.TD3_PARAMS), self.nets, self.opts, masks, noise, self.step, learn=True)
        dt = time.perf_counter() - t0
        self.step += 1
        return dt


def pick_blas_threads(stepper):
    """One BLAS thread per hardware thread is far from OpenBLAS's best on a 100+ core box for GEMMs of this
    size; give the CPU arm the thread count that maximises ITS step rate (2 steps at each candidate)."""
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return None, os.cpu_count() or 1
    ncpu = os.cpu_count() or 1
    best, best_t = ncpu, None
    for n in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):
        with threadpool_limits(limits=n):
            stepper.run()
            t = min(stepper.run(), stepper.run())
        if best_t is None or t < best_t:
            best, best_t = n, t
    return threadpool_limits, best


def cpu_sample(n_rows, algo, seconds_budget, min_steps=10, max_steps=60):
    """Oracle port on the host cores, bounded: steps until ~budget seconds are used."""
    stepper = _OracleStepper(n_rows, algo)
    limiter, threads = pick_blas_threads(stepper)
    ctx = limiter(limits=threads) if limiter is not None else None
    if ctx is not None:
        ctx.__enter__()
    try:
        timed, t_total = 0, 0.0
        t_start = time.perf_counter()
        while True:
            t_total += stepper.run()
            timed += 1
            if (timed >= min_steps and time.perf_counter() - t_start > seconds_budget) or timed >= max_steps:
                break
    finally:
        if ctx is not None:
            ctx.__exit__(None, None, None)
    return {"value": timed / t_total, "unit": "steps/s", "cores": threads, "host_cpus": os.cpu_count() or 1,
            "kind": "port",
            "sample": "%d %s steps at %d rows (gather + update, numpy/OpenBLAS fp32, best-of thread count)"
                      % (timed, algo.upper(), n_rows)}


def run_reference(args):
    """`--impl reference`: the reference algorithm on the host CPU (numpy port in oracle/; /root/reference is
    Python and is not on the GPU box).  Rank 0 only.  Whatever --gpus is, one unit of work is ONE 4096-row
    minibatch through the update step -- the same unit the CUDA arm's `value` counts -- so the ratio of the two
    arms is like for like at every N."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_rows = ROWS_PER_GPU
    stepper = _OracleStepper(n_rows, args.algo)
    limiter, threads = pick_blas_threads(stepper)
    ctx = limiter(limits=threads) if limiter is not None else None
    if ctx is not None:
        ctx.__enter__()
    try:
        for _ in range(args.warmup):
            stepper.run()
        t_total = sum(stepper.run() for _ in range(args.steps))
    finally:
        if ctx is not None:
            ctx.__exit__(None, None, None)
    value = args.steps / t_total
    line = {
        "impl": "reference", "metric": "%s_update_steps_per_sec" % args.algo, "value": value, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.algo), "rows_per_gpu": n_rows, "rows_per_step": n_rows,
                   "unit_def": "4096-row minibatches through the update step per second (one host, all the BLAS "
                               "threads that help; the same unit the CUDA arm counts over its N GPUs)",
                   "optimizer": "adam lr=1e-5", "policy_step": POLICY_STEP},
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "host_cpus": os.cpu_count() or 1,
                         "kind": "port",
                         "sample": "%d full steps at %d rows (gather + %s_update, numpy/OpenBLAS fp32, best-of thread count)"
                                   % (args.steps, n_rows, args.algo)},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# =============================================================================== native arm
class Bench:
    """One agent (DDPG or TD3) + synthetic per-step inputs on this rank's GPU."""

    def __init__(self, algo, n_rows, dev, rank, world, data_parallel, n_distinct=16, seed=1234, flush=None):
        import torch
        import recnn_b200
        self.torch, self.algo, self.n_rows, self.dev, self.rank, self.world = torch, algo, n_rows, dev, rank, world
        torch.manual_seed(seed)                       # same weights on every rank
        rng = np.random.default_rng(0)
        self.table = torch.from_numpy(rng.standard_normal((N_ITEMS, DIM), dtype=np.float32)).to(dev)
        actor = recnn_b200.nn.Actor(S_DIM, DIM, HIDDEN, 6e-1)
        if algo == "ddpg":
            agent = recnn_b200.nn.DDPG(actor, recnn_b200.nn.Critic(S_DIM, DIM, HIDDEN, 54e-2)).to(dev)
        else:
            agent = recnn_b200.nn.TD3(actor, recnn_b200.nn.Critic(S_DIM, DIM, HIDDEN, 54e-2),
                                      recnn_b200.nn.Critic(S_DIM, DIM, HIDDEN, 54e-2)).to(dev)
        for k in list(agent.optimizers):
            net = k.replace("optimizer", "net")
            agent.optimizers[k] = recnn_b200.optim.Adam(agent.nets[net].parameters(), lr=1e-5)
        if data_parallel and world > 1:
            recnn_b200.dist.enable_data_parallel(agent)
        self.agent = agent
        self.n_distinct = n_distinct
        items_np, ratings_np, done_np = synth_step_inputs(100 + rank, n_rows, n_distinct)
        self.items_h = [torch.from_numpy(items_np[i]).pin_memory() for i in range(n_distinct)]
        self.ratings_h = [torch.from_numpy(ratings_np[i]).pin_memory() for i in range(n_distinct)]
        self.done_h = torch.from_numpy(done_np).pin_memory()
        self.items_d = [t.to(dev) for t in self.items_h]
        self.ratings_d = [t.to(dev) for t in self.ratings_h]
        self.done_d = self.done_h.to(dev)
        self.flush = flush if flush is not None else torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def engine(self):
        from recnn_b200 import _lib
        from recnn_b200.nn.update._engine import get_engine
        return get_engine(_lib.ALGO_DDPG if self.algo == "ddpg" else _lib.ALGO_TD3, self.agent.nets, self.dev)

    def batch(self, i, host):
        return {"items": self.items_h[i] if host else self.items_d[i],
                "ratings": self.ratings_h[i] if host else self.ratings_d[i],
                "done": self.done_h if host else self.done_d, "table": self.table}

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def prime(self, host):
        """Both variants of the step (policy / non-policy) seen twice: direct launch, then graph capture --
        so no capture can land inside a timed region whatever --warmup is."""
        for s in (0, 0, 1, 1):
            self.agent._step = s
            self.agent.update(self.batch(0, host), learn=True)
        self.agent._step = 0

    def run(self, host_inputs, steps, warmup, repeats, flush_l2=True, batch_fn=None):
        """-> dict(ms = [per-repeat device ms of `steps` steps, max over ranks], kernels per repeat, last loss)."""
        torch = self.torch
        self.prime(host_inputs)
        agent = self.agent
        agent._step = 0
        it = 0
        loss = None

        def one(timed_events=None):
            nonlocal it, loss
            if flush_l2:
                self.flush.zero_()
            b = batch_fn() if batch_fn is not None else self.batch(it % self.n_distinct, host_inputs)
            if timed_events is not None:
                timed_events[0].record()
            loss = agent.update(b, learn=True)          # H2D (if host) + fused step + D2H of the losses
            agent.step()
            if timed_events is not None:
                timed_events[1].record()
            it += 1

        for _ in range(warmup):
            one()
        rep_ms, kernels = [], 0
        wall = 0.0
        for _ in range(repeats):
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            self.barrier()
            k0 = self.engine().kernels
            t0 = time.perf_counter()
            for s in range(steps):
                one(ev[s])
            self.barrier()
            wall += time.perf_counter() - t0
            kernels = self.engine().kernels - k0
            ms = sum(a.elapsed_time(b) for a, b in ev)
            t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
            if self.world > 1:
                import torch.distributed as dist
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            rep_ms.append(float(t.item()))
        return {"ms": rep_ms, "kernels": int(kernels), "loss": loss, "wall_s": wall}


def timed_outputs(agent, loss):
    """What a caller of the timed path holds after its last step: the dict update() returned and every net's
    weights (updated in place), as host float64 / float32 arrays keyed by output file name."""
    out = {"loss.%s" % k: np.asarray(v, dtype=np.float64) for k, v in loss.items()}
    for net, module in sorted(agent.nets.items()):
        for k, p in module.state_dict().items():
            out["%s.%s" % (net, k)] = p.detach().float().cpu().numpy()
    return out


def summarize(rep_ms, steps, world):
    """steps/s per repeat -> median (whole job: x world 4096-row minibatches), min, max."""
    v = sorted(steps / (m / 1e3) * world for m in rep_ms)
    med = float(np.median(v))
    return med, {"repeats": len(v), "min": v[0], "max": v[-1], "rel": (v[-1] - v[0]) / med if med else None}


def dp_check(dev, rank, world):
    """N > 1 only (the driver's GPU test box has one GPU): three parity-mode DDPG steps (SGD, replayed dropout
    masks) on a small canonical-shape case, rows sharded over the ranks with the peer-memory all-reduce, checked
    (1) replicas bit-identical after the steps and (2) equal to the SAME steps run unsharded on one GPU
    (losses 1e-5 relative; every weight within 2e-3 of the largest weight change + 1e-5 relative).  Raises on failure."""
    import torch
    import torch.distributed as dist
    import recnn_b200
    from recnn_b200.nn.arena import param_arena
    S, A, H, n, n_items, steps = S_DIM, DIM, HIDDEN, 64 * world, 2000, 3
    g = torch.Generator().manual_seed(4242)
    table = torch.randn(n_items, DIM, generator=g)
    items = torch.randint(0, n_items, (n, FRAME + 1), generator=g)
    ratings = torch.randint(-4, 6, (n, FRAME + 1), generator=g).float()
    done = torch.zeros(n)
    done[n // 3] = 1.0
    done[-1] = 1.0
    masks = [[(torch.rand(n, H, generator=g) < 0.5).to(torch.uint8) for _ in range(6)] for _ in range(steps)]

    def make():
        torch.manual_seed(99)
        agent = recnn_b200.nn.DDPG(recnn_b200.nn.Actor(S, A, H, 6e-1), recnn_b200.nn.Critic(S, A, H, 54e-2)).to(dev)
        for k in list(agent.optimizers):
            agent.optimizers[k] = recnn_b200.optim.SGD(agent.nets[k.replace("optimizer", "net")].parameters(), lr=1e-3)
        return agent

    def run(agent, lo, hi, n_global):
        losses = []
        tab = table.to(dev)
        init = {k: param_arena(m).clone() for k, m in agent.nets.items()}
        for s in range(steps):
            agent._step = s * POLICY_STEP          # every step is a policy step: actor all-reduce + Polyak covered
            b = {"items": items[lo:hi], "ratings": ratings[lo:hi], "done": done[lo:hi], "table": tab,
                 "dropout_masks": [m[lo:hi].contiguous() for m in masks[s]], "n_rows_global": n_global}
            losses.append(agent.update(b, learn=True))
        return losses, init

    dp = make()
    recnn_b200.dist.enable_data_parallel(dp)
    lo, hi = recnn_b200.dist.shard_rows(n, rank, world)
    dp_losses, _ = run(dp, lo, hi, n)
    torch.cuda.synchronize(dev)
    # (1) replicas bit-identical
    for name in sorted(dp.nets):
        a = param_arena(dp.nets[name])
        ref = a.clone()
        dist.broadcast(ref, src=0)
        if not torch.equal(a, ref):
            raise AssertionError("dp_check: replica %d of %s differs from rank 0 after %d steps" % (rank, name, steps))
    # (2) equal to the unsharded run (every rank runs it: cheap, and keeps the ranks in lock step)
    single = make()
    s_losses, init = run(single, 0, n, n)
    worst = 0.0
    for a, b in zip(dp_losses, s_losses):
        for k in ("value", "policy"):
            err = abs(a[k] - b[k]) / (abs(b[k]) + 0.1)
            worst = max(worst, err)
            if err > 1e-5:
                raise AssertionError("dp_check: %s loss %r (sharded) vs %r (one GPU)" % (k, a[k], b[k]))
    wdiff = 0.0
    for name in sorted(dp.nets):
        a, b = param_arena(dp.nets[name]), param_arena(single.nets[name])
        change = (b - init[name]).abs().max().item()
        d = (a - b).abs().max().item()
        tol = 2e-3 * change + 1e-5 * b.abs().max().item()
        wdiff = max(wdiff, d / (change + 1e-30))
        if d > tol:
            raise AssertionError("dp_check: %s differs from the one-GPU run by %.3e (largest change %.3e)" % (name, d, change))
    return {"status": "ok", "ranks": world, "rows": n, "steps": steps, "replicas_bit_identical": True,
            "max_loss_rel_err_vs_one_gpu": worst, "max_weight_diff_over_largest_change": wdiff,
            "transport": "peer" if getattr(dp.nets["policy_net"], "_recnn_dp", (0, 0, None))[2] is not None else "nccl"}


def run_native(args):
    import torch
    import torch.distributed as dist
    import recnn_b200
    from recnn_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "WARN"      # NCCL would print its banner on stdout, which carries the ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    algo = args.algo
    steps, warmup = args.steps, max(args.warmup, 3)
    repeats = args.repeats if args.repeats > 0 else (5 if steps <= 100 else 3)

    check = dp_check(dev, rank, world) if world > 1 else None

    main = Bench(algo, ROWS_PER_GPU, dev, rank, world, data_parallel=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    r_dev = main.run(False, steps, warmup, repeats)
    clocks = sampler.stop() if rank == 0 else {}
    dump = timed_outputs(main.agent, r_dev["loss"]) if (args.dump_outputs and rank == 0) else None
    r_e2e = main.run(True, steps, 3, repeats)
    r_warm = main.run(False, steps, 3, 1, flush_l2=False)
    value, spread = summarize(r_dev["ms"], steps, world)
    e2e_value, e2e_spread = summarize(r_e2e["ms"], steps, world)
    warm_value, _ = summarize(r_warm["ms"], steps, world)
    ms_per_step = float(np.median(r_dev["ms"])) / steps

    # strong scaling (BASELINE configs[3]): 8192 global rows sharded over the GPUs, optimizer updates/s
    strong = None
    if STRONG_ROWS % world == 0:
        sb = Bench("ddpg", STRONG_ROWS // world, dev, rank, world, data_parallel=True, flush=main.flush)
        k = min(steps, 50)
        r = sb.run(False, k, 3, 3)
        sv, ss = summarize(r["ms"], k, 1)
        strong = {"workload": "DDPG batch %d rows sharded over %d GPU(s) (BASELINE configs[3])" % (STRONG_ROWS, world),
                  "global_rows": STRONG_ROWS, "rows_per_gpu": STRONG_ROWS // world, "updates_per_sec": sv,
                  "ms_per_step": 1e3 / sv, "spread": ss, "steps": k}
        del sb

    line = None
    if rank == 0:
        L = _lib.lib()
        st = torch.cuda.current_stream(dev).cuda_stream
        flush = main.flush
        n_rows = ROWS_PER_GPU
        agent, table = main.agent, main.table

        def time_kernel(fn, iters=20):
            for _ in range(3):
                fn()
            ts = []
            for _ in range(iters):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize(dev)
                ts.append(a.elapsed_time(b))
            return float(np.mean(ts))

        def graph_time(fns, reps=10):
            """Average DEVICE time of one launch: the launches `fns` (each on its own operands, together larger than
            the 126 MB L2, so no launch finds its streamed operand cached) are captured into one CUDA graph and the
            graph is replayed `reps` times between two events.  Unlike an event pair around a single host launch this
            contains no host-side launch preparation (tensor-map encoding) and is not limited by the ~2 us event
            resolution; it does contain the inter-kernel gaps, as the step's own graph does."""
            for f in fns:
                f()
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for f in fns:
                    f()
            g.replay()
            torch.cuda.synchronize(dev)
            ts = []
            for _ in range(reps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                g.replay()
                b.record()
                torch.cuda.synchronize(dev)
                ts.append(a.elapsed_time(b) / len(fns))
            return float(np.median(ts)), float(min(ts)), float(max(ts))

        # (1) the materialising gather kernel  (HBM bound)
        items_d, ratings_d = main.items_d, main.ratings_d
        g_state = torch.empty(n_rows, S_DIM, device=dev)
        g_next = torch.empty(n_rows, S_DIM, device=dev)
        g_act = torch.empty(n_rows, DIM, device=dev)
        g_rew = torch.empty(n_rows, device=dev)
        gather_single_ms = time_kernel(lambda: _lib.check(L.recnn_frame_gather(
            table.data_ptr(), N_ITEMS, DIM, items_d[0].data_ptr(), ratings_d[0].data_ptr(), n_rows, FRAME,
            g_state.data_ptr(), g_next.data_ptr(), g_act.data_ptr(), g_rew.data_ptr(), None, st)))
        # four launches with their own ids and outputs (4 x 44 MB written > L2) in one graph: average device time
        g_outs = [(torch.empty(n_rows, S_DIM, device=dev), torch.empty(n_rows, S_DIM, device=dev),
                   torch.empty(n_rows, DIM, device=dev), torch.empty(n_rows, device=dev)) for _ in range(4)]

        def gather_launch(i):
            o = g_outs[i]
            return lambda: _lib.check(L.recnn_frame_gather(
                table.data_ptr(), N_ITEMS, DIM, items_d[i].data_ptr(), ratings_d[i].data_ptr(), n_rows, FRAME,
                o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), None,
                torch.cuda.current_stream(dev).cuda_stream))

        gather_ms, gather_ms_min, gather_ms_max = graph_time([gather_launch(i) for i in range(4)])
        del g_outs
        gather_gbs = n_rows * GATHER_BYTES_PER_ROW / (gather_ms * 1e-3) / 1e9
        # the same kernel on a batch whose output does not fit in L2 (16x the rows): its HBM-bound regime
        big = 16 * n_rows
        gb_items = torch.randint(0, N_ITEMS, (big, FRAME + 1), device=dev, dtype=torch.int64)
        gb_ratings = torch.rand(big, FRAME + 1, device=dev)
        gb_state = torch.empty(big, S_DIM, device=dev)
        gb_next = torch.empty(big, S_DIM, device=dev)
        gb_act = torch.empty(big, DIM, device=dev)
        gb_rew = torch.empty(big, device=dev)
        gather_big_ms = time_kernel(lambda: _lib.check(L.recnn_frame_gather(
            table.data_ptr(), N_ITEMS, DIM, gb_items.data_ptr(), gb_ratings.data_ptr(), big, FRAME,
            gb_state.data_ptr(), gb_next.data_ptr(), gb_act.data_ptr(), gb_rew.data_ptr(), None, st)), iters=10)
        gather_big_gbs = big * GATHER_BYTES_PER_ROW / (gather_big_ms * 1e-3) / 1e9
        del gb_state, gb_next, gb_act, gb_rew, gb_items, gb_ratings
        # (2) the dominant kernel of the step: layer-1 forward GEMM [4096,1290] x [1290,256]
        #     (same tcgen05 3xTF32 kernel and operand pitches as inside the step; plain-store epilogue).
        #     Eight launches on eight different state images (8 x 21 MB > L2) in one graph: average device time.
        ld_s = (S_DIM + 3) // 4 * 4
        x_imgs = [torch.randn(n_rows, ld_s, device=dev) for _ in range(8)]
        w1 = agent.nets["policy_net"].linear1.weight            # strided view into the arena, pitch 1292
        h1s = [torch.empty(n_rows, HIDDEN, device=dev) for _ in range(8)]

        def l1_launch(i, tile):      # the stream is looked up at call time: graph capture runs on its own stream
            return lambda: _lib.check(L.recnn_gemm_tf32x3(
                n_rows, HIDDEN, S_DIM, x_imgs[i].data_ptr(), ld_s, 0, w1.data_ptr(), w1.stride(0), 0,
                h1s[i].data_ptr(), HIDDEN, tile, torch.cuda.current_stream(dev).cuda_stream))

        l1 = {}
        for tile in (64, 128):
            med, lo, hi = graph_time([l1_launch(i, tile) for i in range(8)])
            l1[tile] = {"ms": med, "ms_min": lo, "ms_max": hi,
                        "tf32_tflops": 3.0 * n_rows * L1_FWD_FLOP_PER_ROW / (med * 1e-3) / 1e12}
        l1_single_ms = time_kernel(l1_launch(0, 64))                # round-1 method (one host launch between events)
        best_tile = min(l1, key=lambda t: l1[t]["ms"])
        l1_ms = l1[best_tile]["ms"]
        l1_tflops = n_rows * L1_FWD_FLOP_PER_ROW / (l1_ms * 1e-3) / 1e12
        del x_imgs, h1s
        tf32_peak = peaks["bf16"] / 2.0           # dense TF32 = half the dense bf16 rate
        rows_global = n_rows * world
        updates_per_sec = value / world

        def flop_per_step(a, rows):
            return rows * (FLOP[a][1] + (POLICY_STEP - 1) * FLOP[a][0]) / POLICY_STEP

        feed_info = bench_device_feed(main, time_kernel, steps) if (world == 1 and algo == "ddpg") else None
        # (3) the other algorithm (BASELINE configs[2] next to configs[1]) on one GPU, shorter run
        other = None
        if world == 1 and not args.no_other_algo:
            oa = "td3" if algo == "ddpg" else "ddpg"
            ob = Bench(oa, n_rows, dev, rank, 1, data_parallel=False, flush=flush)
            k = min(steps, 100)
            ro = ob.run(False, k, 3, 3)
            ro_e2e = ob.run(True, k, 3, 3)
            ov, osp = summarize(ro["ms"], k, 1)
            oe, _ = summarize(ro_e2e["ms"], k, 1)
            other = {"workload": workload_name(oa), "steps_per_sec": ov, "ms_per_step": 1e3 / ov, "spread": osp,
                     "e2e_steps_per_sec": oe, "steps": k, "gpu_launches": ro["kernels"],
                     "update_tflops": flop_per_step(oa, n_rows) * ov / 1e12,
                     "step_tensor_frac": 3.0 * flop_per_step(oa, n_rows) * ov / 1e12 / tf32_peak}
            if not args.no_cpu_baseline:
                other["cpu_baseline"] = cpu_sample(n_rows, oa, 8.0, min_steps=6, max_steps=30)
            del ob
        reinforce = bench_reinforce(dev, not args.no_cpu_baseline) if (world == 1 and not args.no_other_algo) else None
        cpu = cpu_sample(n_rows, algo, 15.0) if (world == 1 and not args.no_cpu_baseline) else None
        cpu256 = cpu_sample(256, "ddpg", 4.0, min_steps=20, max_steps=400) if (world == 1 and not args.no_cpu_baseline) else None
        comm = getattr(agent.nets["policy_net"], "_recnn_dp", (0, 0, None))[2]
        line = {
            "metric": "%s_update_steps_per_sec" % algo, "value": value, "unit": "steps/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(algo),
                       "rows_per_gpu": n_rows, "global_rows": rows_global, "parallelism": "dp%d" % world,
                       "unit_def": "4096-row minibatches through the update step per second, whole job "
                                   "(each data-parallel step consumes n_gpus of them; optimizer updates/s = value / n_gpus)",
                       "grad_allreduce": ("none" if world == 1 else
                                          "in-graph NVLink peer-memory kernels (recnn_comm_*)" if comm is not None
                                          else "NCCL between the step's phases"),
                       "optimizer": "adam lr=1e-5 (fused)", "policy_step": POLICY_STEP,
                       "dropout": "on (device Philox)", "l2": "flushed between timed steps (256 MB write)",
                       "timing": "both graph variants primed before the timed region; %d repeats of %d steps, median" % (repeats, steps),
                       "inputs": "items/ratings/done resident in HBM; frames gathered on device inside the step",
                       "matmul": "tcgen05 3xTF32 (error-compensated, fp32-grade) with fp32 CUDA-core fallbacks for the 256->1 head"},
            "spread": spread,
            "optimizer_updates_per_sec": updates_per_sec,
            "rows_per_sec": updates_per_sec * rows_global,
            "update_tflops": flop_per_step(algo, rows_global) * updates_per_sec / 1e12,
            # SURVEY 8d: (algorithmic FLOPs x 3 TF32 passes) / (t_step x TF32 peak x GPUs): the whole step, not one kernel
            "step_tensor_frac": 3.0 * flop_per_step(algo, rows_global) * updates_per_sec / 1e12 / (tf32_peak * world),
            "value_warm_l2": warm_value,
            "wall_s": r_dev["wall_s"],
            "e2e": {"value": e2e_value, "unit": "steps/s", "spread": e2e_spread,
                    "h2d_bytes_per_step": int(n_rows * ((FRAME + 1) * 12 + 4)), "d2h_bytes_per_step": 32,
                    "what": "%s_update(batch of pinned host items/ratings/done) -> dict of python floats" % algo},
            "gpu_launches": int(r_dev["kernels"]),
            "roofline": {"bound": "tensor", "kernel": "layer-1 forward GEMM [4096x1290]x[1290x256] (tc_gemm_kernel, tcgen05 kind::tf32, 3 MMA passes/product)",
                         "achieved": 3.0 * l1_tflops, "algorithmic_fp32": l1_tflops, "peak": tf32_peak, "unit": "TFLOP/s",
                         "frac": 3.0 * l1_tflops / tf32_peak,
                         "traffic": 22518784, "traffic_source": "dram__bytes_read+write per launch, profiles/r2k/r2k_tc_gemm_raw.csv (ncu --set full)", "peak_source": "%s bf16 %.0f TF/s / 2 (TF32 kind)" % (peaks["source"], peaks["bf16"]),
                         "ms": l1_ms, "tile_n": best_tile, "per_tile": {str(k): v for k, v in l1.items()},
                         "timing": "8 launches on 8 distinct state images (8 x 21 MB > L2) captured in one CUDA graph, "
                                   "replayed 10x between CUDA events, L2 flushed between replays; median per launch",
                         "ms_single_launch_between_events": l1_single_ms},
            "roofline_gather": {"bound": "hbm", "kernel": "frame_gather_kernel", "achieved": gather_gbs,
                                "peak": peaks["hbm"], "unit": "GB/s", "frac": gather_gbs / peaks["hbm"],
                                "traffic": 12184064, "traffic_source": "dram__bytes_read+write per launch, profiles/r2k/r2k_gather_raw.csv: the 44 MB of "
                                "output is absorbed by the 126 MB L2 inside the kernel, so DRAM traffic << algorithmic bytes", "peak_source": peaks["source"], "ms": gather_ms, "ms_min": gather_ms_min, "ms_max": gather_ms_max,
                                "ms_single_launch_between_events": gather_single_ms,
                                "timing": "4 launches (own ids / outputs, 4 x 44 MB > L2) in one CUDA graph, replayed 10x between events; median per launch",
                                "bytes_per_launch": n_rows * GATHER_BYTES_PER_ROW,
                                "at_16x_rows": {"rows": big, "ms": gather_big_ms, "algorithmic_gbs": gather_big_gbs,
                                                "traffic": 710117376, "traffic_source": "profiles/r2k/r2k_gather_big_raw.csv (58.2 MB read + 651.9 MB written)",
                                                "dram_gbs_est": (big * 10840 + N_ITEMS * DIM * 4) / (gather_big_ms * 1e-3) / 1e9,
                                                "dram_frac_est": (big * 10840 + N_ITEMS * DIM * 4) / (gather_big_ms * 1e-3) / 1e9 / peaks["hbm"],
                                                "note": "same kernel, 16x the rows: the 710 MB of output no longer fits in L2 and goes to HBM, "
                                                        "the 13.7 MB table is still served by L2, so DRAM traffic ~ output + table once"}},
            "clocks": clocks,
            "last_loss": r_dev["loss"],
        }
        if strong is not None:
            line["strong"] = strong
        if check is not None:
            line["dp_check"] = check
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if cpu256 is not None:
            cpu256["what"] = "BASELINE configs[0]: DDPG batch 256 on the CPU path"
            line["cpu_baseline_n256"] = cpu256
        if other is not None:
            line["td3" if algo == "ddpg" else "ddpg"] = other
        if reinforce is not None:
            line["reinforce"] = reinforce
        if feed_info is not None:
            line["feed"] = feed_info
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if line is not None:
        print(json.dumps(line))


def bench_reinforce(dev, with_cpu):
    """SURVEY 8f-2 at the shapes of the reference's Top-K notebook (DiscreteActor 1290 -> 2048 -> 5000 items,
    Critic(1290, 5000, 2048), K = 10, policy_step = 10) with 128 rows per env step: recnn.nn.Reinforce.update() calls
    per second, policy updates included (every 10th call back-propagates through the 10 saved batches)."""
    import torch
    import recnn_b200
    from recnn_b200.nn import ChooseREINFORCE
    S, H, I, N = FRAME * DIM + FRAME, 2048, 5000, 128
    torch.manual_seed(7)
    agent = recnn_b200.nn.Reinforce(recnn_b200.nn.DiscreteActor(S, I, H), recnn_b200.nn.Critic(S, I, H, 54e-2)).to(dev)
    policy = agent.nets["policy_net"]
    bw = torch.randn(I, S, device=dev) * 0.02

    def select(state, action, K, writer, step, **kw):
        beta = lambda s, action=None: torch.softmax(s @ bw.T, dim=1)       # noqa: E731  (the notebook's Beta net, frozen)
        return policy._select_action_with_TopK_correction(state, beta, action, K=K, writer=writer, step=step)

    policy.select_action = select
    agent.params["reinforce"] = ChooseREINFORCE(ChooseREINFORCE.reinforce_with_TopK_correction)
    agent.optimizers = {"policy_optimizer": recnn_b200.optim.Adam(policy.parameters(), lr=1e-5),
                        "value_optimizer": recnn_b200.optim.Adam(agent.nets["value_net"].parameters(), lr=1e-5)}
    g = torch.Generator(device="cpu").manual_seed(3)
    batches = []
    for _ in range(4):
        a = torch.randint(0, I, (N,), generator=g)
        batches.append({"state": torch.randn(N, S, generator=g).to(dev), "next_state": torch.randn(N, S, generator=g).to(dev),
                        "action": torch.nn.functional.one_hot(a, I).float().to(dev),
                        "reward": (torch.randint(1, 6, (N,), generator=g).float() - 3).to(dev),
                        "done": torch.zeros(N).to(dev)})
    lib = recnn_b200._lib.lib()

    def run(k):
        for i in range(k):
            agent.update(batches[i % 4])
            agent.step()
        torch.cuda.synchronize(dev)

    run(21)                                   # two policy updates: every shape seen
    k = 100
    k0 = lib.recnn_b200_launch_count()
    t0 = time.perf_counter()
    run(k)
    dt = time.perf_counter() - t0
    out = {"workload": "REINFORCE Top-K off-policy correction, DiscreteActor 1290-2048-%d, Critic(1290,%d,2048), %d rows/step, "
                       "K=10, policy_step=10" % (I, I, N),
           "updates_per_sec": k / dt, "ms_per_update": 1e3 * dt / k, "steps": k,
           "gpu_launches": int(lib.recnn_b200_launch_count() - k0), "timing": "wall clock around %d Reinforce.update() calls "
           "(host-driven: sampling, critic step, every 10th call the policy backward over 1280 saved rows), synchronised" % k,
           "reference_incidental": "9.48 it/s at batch_size=10 users in the notebook's own log (unknown GPU, DataLoader included)"}
    if with_cpu:
        out["cpu_baseline"] = cpu_reinforce_sample(S, H, I, N)
    return out


def cpu_reinforce_sample(S, H, I, N):
    """The float64 oracle of the POLICY update (forward + closed-form backward over 10 x N saved rows) on the host:
    the part of a policy step that dominates; a bounded sample (3 updates)."""
    from oracle import reinforce_oracle as RO
    rng = np.random.default_rng(0)
    p = RO.make_discrete_actor(rng, S, I, H)
    rows = 10 * N
    state = rng.normal(0, 1, (rows, S)).astype(np.float32)
    act = rng.integers(0, I, rows)
    blp = np.log(rng.uniform(1e-4, 5e-4, rows)).astype(np.float32)
    ret = rng.normal(0, 1, rows).astype(np.float32)
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        RO.reinforce_policy_grad(p, state, act, blp, ret, RO.TOPK, 10)
    dt = (time.perf_counter() - t0) / reps
    return {"value": 1.0 / dt, "unit": "policy updates/s (policy half only, 1280 saved rows)", "kind": "port",
            "cores": int(os.environ.get("OMP_NUM_THREADS", os.cpu_count() or 1)), "sample": "%d policy updates, float64 numpy" % reps}


FEED_BYTES_PER_ROW = (FRAME + 1) * 12 * 2 + 4          # read ids+ratings, write ids+ratings, write done


def bench_device_feed(main, time_kernel, steps):
    """SURVEY.md 8f rank 1: minibatches cut on the device out of resident user histories
    (recnn_b200.data.DeviceFrameFeed) instead of a DataLoader worker + H2D.  Synthetic "rolling users":
    2048 users x 138 interactions (128 windows each, 262,144 windows).  Reports the window-gather kernel
    alone and the update step fed by ``feed.sample(4096)`` (no host->device traffic at all)."""
    import torch
    from recnn_b200.data.feed import HistoryCSR, DeviceFrameFeed
    dev = main.dev
    rng = np.random.default_rng(7)
    n_users, length = 2048, 138
    items = rng.integers(0, N_ITEMS, size=(n_users, length), dtype=np.int64)
    rates = rng.integers(-4, 6, size=(n_users, length)).astype(np.float64)
    feed = DeviceFrameFeed(HistoryCSR(np.arange(n_users), list(items), list(rates), FRAME), main.table, dev)
    n_rows = ROWS_PER_GPU
    w = torch.randint(0, feed.csr.n_windows, (n_rows,), device=dev)
    ids_ms = time_kernel(lambda: feed.windows(w))
    users32 = list(range(0, 32 * 8, 8))                    # 32 users x 128 windows = 4096 rows
    users_ms = time_kernel(lambda: feed.batch(users32))
    k = min(steps, 100)
    r = main.run(False, k, 3, 3, batch_fn=lambda: feed.sample(n_rows))   # randint + window gather + fused step + loss read-back
    v, sp = summarize(r["ms"], k, 1)
    return {"what": "update step fed by DeviceFrameFeed.sample(4096): windows cut on the device from resident "
                    "histories (2048 users x 138 interactions), no host->device copies",
            "steps_per_sec": v, "ms_per_step": 1e3 / v, "spread": sp, "h2d_bytes_per_step": 0,
            "window_gather_ids_ms": ids_ms, "window_gather_users_ms": users_ms,
            "window_gather_bytes_per_launch": n_rows * FEED_BYTES_PER_ROW,
            "note": "window_gather_*_ms include the output allocation and (users form) a 520-byte plan upload; "
                    "1.1 MB per launch: latency-bound, not bandwidth-bound"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=0, help="repeats of the K timed steps (default: 5 if K <= 100 else 3)")
    ap.add_argument("--algo", default="ddpg", choices=["ddpg", "td3"])
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline legs (A/B runs)")
    ap.add_argument("--no-other-algo", action="store_true", help="skip the sub-object of the other algorithm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (losses) and left in the nets (weights, ~7 MB for "
                         "DDPG, ~10 MB for TD3) as DIR/<name>.npy; the inputs are seeded, so runs with the same "
                         "arguments can be compared output for output")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl native")
        args.warmup = min(args.warmup, 3)
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
