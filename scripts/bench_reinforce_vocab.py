#!/usr/bin/env python
"""Time of one REINFORCE policy-gradient call (Top-K corrected loss, DiscreteActor 1290 -> 256 -> I) against the size of
the item vocabulary, up to BASELINE configs[4] (2^20 items, 16,384 rows x policy_step 10 = 163,840 saved rows).

  python scripts/bench_reinforce_vocab.py [--repeats 3] [--quick]

Prints one JSON line per point.  Each (rows, items) point runs the path the policy update picks for it
(recnn_b200.nn.update.reinforce._policy_grad_plan); at 5,000 items both the materialised and the streamed C entries are
timed, which places the size threshold between the two with a measurement.  Timing: CUDA events around each call, one
untimed warm-up call, median / min / max of the repeats.  Algorithmic FLOP per call (fp32 multiply-adds x 2):
  streamed      8 R H I + 4 R S H   (logits twice, dW2, dh; dW1 and layer 1)
  materialised  6 R H I + 4 R S H
`tensor_frac` = 3 x FLOP / time / TF32 peak (three TF32 passes per fp32 product), the peak read as bench.py reads it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import recnn_b200                                                     # noqa: E402
from recnn_b200 import _lib                                           # noqa: E402
from recnn_b200.nn.arena import param_arena, grad_arena               # noqa: E402
from recnn_b200.nn.update.reinforce import _policy_grad_plan          # noqa: E402
from bench import load_peaks                                          # noqa: E402

S, H, K = 1290, 256, 10


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception:
        pass
    return info


def run_point(policy, R, items, chunk, repeats, peak_tf32, info):
    L = _lib.lib()
    d = policy.dims
    g = torch.Generator(device="cuda").manual_seed(R + items)
    state = torch.randn(R, S, device="cuda", generator=g)
    action = torch.randint(0, items, (R,), device="cuda", generator=g)
    beta = torch.log(torch.rand(R, device="cuda", generator=g) * 4e-6 + 1e-7)
    ret = torch.randn(R, device="cuda", generator=g)
    floats = L.recnn_reinforce_streamed_scratch_floats(d, R, chunk) if chunk else L.recnn_discrete_scratch_floats(d, R, 1)
    scratch = torch.empty(floats, device="cuda")
    out = torch.zeros(2, device="cuda")
    flat, grads = param_arena(policy), grad_arena(policy)
    args = (d, flat.data_ptr(), grads.data_ptr(), state.data_ptr(), action.data_ptr(), beta.data_ptr(), ret.data_ptr(),
            R, _lib.REINFORCE_TOPK, K)
    st = _lib.stream_ptr(0)

    def call():
        if chunk:
            _lib.check(L.recnn_reinforce_policy_grad_streamed(*args, chunk, out.data_ptr(), scratch.data_ptr(), st))
        else:
            _lib.check(L.recnn_reinforce_policy_grad(*args, out.data_ptr(), scratch.data_ptr(), st))

    call()                                                              # warm-up (module load, tensor maps)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    assert np.isfinite(float(out[0])) and int(out.view(torch.int32)[1]) == 0
    flop = (8 if chunk else 6) * R * H * items + 4 * R * S * H
    med = float(np.median(ms))
    line = {"path": "streamed" if chunk else "materialised", "rows": R, "items": items, "hidden": H, "state_dim": S,
            "method": "topk", "item_chunk": chunk, "ms": med, "ms_min": min(ms), "ms_max": max(ms), "repeats": repeats,
            "flop": flop, "tflops": flop / (med * 1e-3) / 1e12,
            "tensor_frac": 3.0 * flop / (med * 1e-3) / 1e12 / peak_tf32, "tf32_peak_tflops": peak_tf32,
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9,
            "scratch_gb": floats * 4 / 1e9, **info}
    print(json.dumps(line), flush=True)
    del scratch, state


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a check of the script, not a measurement)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this script measures the GPU"
    repeats = max(3, a.repeats)
    peaks = load_peaks()
    peak_tf32 = peaks["bf16"] / 2.0
    info = dict(gpu_info(), peak_source=peaks["source"])
    item_sizes = [5000, 262144, 1 << 20] if not a.quick else [5000, 40000]
    row_sizes = [16384, 163840] if not a.quick else [1024, 8192]
    for items in item_sizes:
        torch.manual_seed(items)
        policy = recnn_b200.nn.DiscreteActor(S, items, H).cuda()
        for R in row_sizes:
            plan = _policy_grad_plan(R, items)
            # both entries at 5,000 items; the streamed one with the chunk the plan picks for R rows once it streams
            paths = [0, _policy_grad_plan(R, 1 << 40)] if items == 5000 else [plan]
            for chunk in paths:
                run_point(policy, R, items, chunk, repeats, peak_tf32, info)
        del policy
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
