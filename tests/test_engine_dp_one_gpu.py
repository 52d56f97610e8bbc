"""Data parallel with NCCL-style all-reduces between the step's phases, on a single GPU: two spawned ranks share
cuda:0 and exchange through gloo (RECNN_B200_COMM=nccl, so no peer-memory communicator is built).  This runs the
engine's host-side exchange -- the three-call fused schedule, the phase-by-phase schedule of external optimizers
and value_update's critic step -- on machines with one GPU; test_gpu_parity.py::test_data_parallel_equals_reference
covers the real multi-GPU transports."""
import os
import socket

import numpy as np
import pytest
import torch

import recnn_b200
from oracle import cases as C
from oracle import recnn_oracle as O
from tests._golden import load_golden, compare_with_golden
from tests._cuda import run_cuda_case, build_nets, build_optimizers

pytestmark = pytest.mark.gpu
WORLD = 2
VALUE_STEPS = 3


def _value_batches(spec, inp, lo, hi):
    ref = O.frame_gather(inp["table"], inp["items"], inp["ratings"], inp["sizes"], spec["frame"])
    for step in range(VALUE_STEPS):
        batch = {k: torch.from_numpy(np.ascontiguousarray(v[lo:hi])) for k, v in ref.items()}
        batch["dropout_masks"] = [torch.from_numpy(np.ascontiguousarray(m[lo:hi])) for m in inp["masks"][step]]
        yield step, batch


def _value_losses(shard):
    """value_update losses of VALUE_STEPS critic steps (built-in Adam) on this rank's rows of the canonical batch."""
    spec = C.CASES["canon"]
    inp = C.make_inputs(spec, "ddpg")
    dev = torch.device("cuda:0")
    nets = build_nets(spec, inp, dev)
    opts = build_optimizers("adam", nets, "ddpg")
    if shard is not None:
        recnn_b200.dist.enable_data_parallel(nets)
    lo, hi = (0, spec["n_rows"]) if shard is None else recnn_b200.dist.shard_rows(spec["n_rows"], *shard)
    return np.asarray([float(recnn_b200.nn.update.value_update(b, dict(C.DDPG_PARAMS), nets, opts, dev, {},
                                                               learn=True, step=step))
                       for step, b in _value_batches(spec, inp, lo, hi)])


def _worker(rank, port, what, algo, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["RECNN_B200_COMM"] = "nccl"
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        if what == "value_update":
            got = {"value_loss": _value_losses((rank, WORLD))}
        else:
            gold = load_golden("%s_canon_adam.npz" % algo)
            got = run_cuda_case("canon", algo, "adam", golden=gold, form="frames", device="cuda:0",
                                shard=(rank, WORLD), external=(what == "external"))
            nets = got.pop("_nets")
            got["_peer_comm"] = np.asarray(nets["policy_net"].__dict__["_recnn_dp"][2] is not None)
        q.put((rank, got))
    finally:
        dist.destroy_process_group()


def _run_ranks(what, algo="ddpg"):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, port, what, algo, q)) for r in range(WORLD)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in range(WORLD))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def _assert_replicas_identical(res):
    for k in res[0]:
        if k.startswith("final."):
            assert np.array_equal(res[0][k], res[1][k]), "replicas diverged: %s" % k


@pytest.mark.parametrize("algo", ["ddpg", "td3"])
def test_builtin_optimizers_split_into_three_graphed_calls(algo):
    """Built-in Adam under NCCL-style data parallel: the fused step cut into three calls (one CUDA graph each
    after the first sighting) with the gradient and loss all-reduces between the replays."""
    res = _run_ranks("builtin", algo)
    gold = load_golden("%s_canon_adam.npz" % algo)
    for rank in range(WORLD):
        assert not bool(res[rank].pop("_peer_comm"))
        compare_with_golden(res[rank], gold, check_grads=False)
    _assert_replicas_identical(res)


@pytest.mark.parametrize("algo", ["ddpg", "td3"])
def test_external_optimizers_all_reduce_between_phases(algo):
    """torch.optim.Adam under NCCL-style data parallel: phase by phase, gradients all-reduced before each
    Python step(); the same golden bar as the single-process split-phase path."""
    res = _run_ranks("external", algo)
    gold = load_golden("%s_canon_adam.npz" % algo)
    for rank in range(WORLD):
        assert not bool(res[rank].pop("_peer_comm"))
        compare_with_golden(res[rank], gold)
    _assert_replicas_identical(res)


def test_value_update_returns_the_global_loss():
    """value_update at world 2 returns the loss of the whole batch (the ranks' partial sums all-reduced), not
    this rank's share of it.  Two shard sums are not bit-identical to one sum over all rows: 1e-6 relative."""
    res = _run_ranks("value_update")
    want = _value_losses(None)
    assert np.array_equal(res[0]["value_loss"], res[1]["value_loss"])
    np.testing.assert_allclose(res[0]["value_loss"], want, rtol=1e-6, atol=0)
