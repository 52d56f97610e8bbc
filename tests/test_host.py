"""CPU-side checks: the C-ABI library loads and exports every symbol the header
declares, the ctypes mirrors match the C structs, and the host logic (arenas,
optimizer binding, collate, import aliases) behaves.  No kernel is launched."""
import copy
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

import recnn_b200
from recnn_b200 import _lib
from recnn_b200.nn.arena import param_arena, grad_arena
from oracle import recnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "recnn_b200.h")).read()
    declared = set(re.findall(r"RECNN_API\s+[\w\s\*]+?\b(recnn_\w+)\s*\(", header))
    assert len(declared) >= 15
    L = _lib.lib()                       # builds the library if missing; also verifies struct size / offsets
    handle = ctypes.CDLL(_lib.lib_path())
    for name in declared:
        assert hasattr(handle, name), name
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert L.recnn_b200_abi_version() == 3
    assert L.recnn_sizeof_step_args() == ctypes.sizeof(_lib.StepArgs)


def test_param_counts_match_reference_shapes():
    L = _lib.lib()
    d = _lib.Dims(1290, 128, 256, 0)
    # 429,184 / 429,313 parameters (SURVEY.md 8) + 16-byte row padding of linear1.weight (1290 -> 1292,
    # 1418 -> 1420) and of the critic's 1-element linear3.bias
    assert L.recnn_actor_param_count(d) == 429184 + 256 * 2
    assert L.recnn_critic_param_count(d) == 429313 + 256 * 2 + 3
    a = recnn_b200.nn.Actor(1290, 128, 256)
    c = recnn_b200.nn.Critic(1290, 128, 256)
    assert sum(p.numel() for p in a.parameters()) == 429184 and sum(p.numel() for p in c.parameters()) == 429313
    from recnn_b200.nn.arena import net_layout
    offs, lds, count = net_layout(c)
    assert lds == [1420, 256, 256] and count == 429313 + 515 and offs[0] == 0 and offs[1] == 256 * 1420
    assert L.recnn_step_workspace_bytes(d, 4096, 0) > 0


def test_error_reporting_without_gpu():
    L = _lib.lib()
    assert L.recnn_polyak_update(None, None, 10, 0.5, None) == -1
    assert b"non-null" in L.recnn_b200_last_error()
    with pytest.raises(_lib.RecnnError):
        _lib.check(-1)


def test_state_dict_layout_matches_reference():
    a = recnn_b200.nn.Actor(1290, 128, 256, 6e-1)
    c = recnn_b200.nn.Critic(1290, 128, 256, 54e-2)
    assert list(a.state_dict()) == ["linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias",
                                    "linear3.weight", "linear3.bias"]
    assert a.linear1.weight.shape == (256, 1290) and a.linear3.weight.shape == (128, 256)
    assert c.linear1.weight.shape == (256, 1418) and c.linear3.weight.shape == (1, 256)
    assert a.linear3.weight.abs().max() <= 6e-1 and c.linear3.bias.abs().max() <= 54e-2
    assert isinstance(a.drop_layer, torch.nn.Dropout) and a.drop_layer.p == 0.5


def test_arena_aliasing_survives_copies_and_moves():
    a = recnn_b200.nn.Actor(170, 16, 32)
    before = [p.detach().clone() for p in a.parameters()]
    flat = param_arena(a)
    assert flat.numel() >= sum(p.numel() for p in a.parameters())
    assert a.linear1.weight.stride() == (172, 1) and a.linear1.weight.shape == (32, 170)   # 170 -> pitch 172
    for p, q in zip(a.parameters(), before):
        assert torch.equal(p, q)
    flat.mul_(2.0)                                           # writes through to the parameters
    assert torch.equal(a.linear2.bias, before[3] * 2)
    assert param_arena(a) is flat                            # still valid -> reused
    b = copy.deepcopy(a)
    fb = param_arena(b)
    assert fb.data_ptr() != flat.data_ptr() and torch.equal(fb, flat)
    a.load_state_dict({k: v * 0 + 1 for k, v in a.state_dict().items()})
    assert param_arena(a).sum().item() == sum(p.numel() for p in a.parameters())          # pads stay 0
    assert all(torch.equal(p, torch.ones_like(p)) for p in a.parameters())
    g = grad_arena(a)
    assert a.linear1.weight.grad.data_ptr() == g.data_ptr()
    torch.optim.SGD(a.parameters(), lr=0.1).zero_grad(set_to_none=True)
    assert a.linear1.weight.grad is None
    assert grad_arena(a) is g and a.linear1.weight.grad is not None


def test_builtin_optimizer_binding():
    a = recnn_b200.nn.Actor(170, 16, 32)
    c = recnn_b200.nn.Critic(170, 16, 32)
    opt = recnn_b200.optim.Adam(a.parameters(), lr=1e-5, weight_decay=1e-2)
    opt.bind(a)
    with pytest.raises(ValueError):
        opt.bind(c)
    co = opt.c_optim()
    assert co.kind == _lib.OPT_ADAM and co.lr == 1e-5 and co.weight_decay == 1e-2 and co.beta2 == 0.999
    opt.param_groups[0]["lr"] = 3e-4
    assert opt.c_optim().lr == 3e-4
    assert "param_groups" in opt.state_dict()


def test_collate_matches_oracle():
    rng = np.random.default_rng(0)
    users = [{"items": rng.integers(0, 50, size=n, dtype=np.int64), "rates": rng.integers(-4, 6, size=n).astype(np.float64),
              "sizes": n, "users": i} for i, n in enumerate((14, 11, 25))]
    table = torch.zeros(50, 8)
    got = recnn_b200.data.prepare_batch_static_size(users, table, frame_size=10, embed_batch=recnn_b200.data.batch_frames)
    want = O.collate_users(users, 10)
    assert np.array_equal(got["items"].numpy(), want["items"])
    assert got["ratings"].dtype == torch.float32 and np.array_equal(got["ratings"].numpy(), want["ratings"])
    assert np.array_equal(got["sizes"].numpy(), want["sizes"]) and np.array_equal(got["users"].numpy(), want["users"])
    assert got["table"] is None           # CPU table is never handed to the device path


def test_no_cpu_fallback():
    table = torch.zeros(50, 8)
    batch = {"items": torch.zeros(4, 11, dtype=torch.int64), "ratings": torch.zeros(4, 11),
             "sizes": torch.tensor([14]), "users": torch.tensor([0])}
    with pytest.raises(_lib.RecnnError):
        recnn_b200.data.batch_tensor_embeddings(batch, table, 10)
    a = recnn_b200.nn.Actor(170, 16, 32)
    with pytest.raises(_lib.RecnnError):
        a(torch.zeros(2, 170))
    nets = {"policy_net": a, "target_policy_net": copy.deepcopy(a),
            "value_net": recnn_b200.nn.Critic(170, 16, 32), "target_value_net": recnn_b200.nn.Critic(170, 16, 32)}
    with pytest.raises(_lib.RecnnError):
        recnn_b200.nn.ddpg_update({}, {}, nets, {}, torch.device("cpu"), {}, learn=True, step=0)


def test_reference_import_names_resolve():
    mod = recnn_b200.install_as_recnn()
    import recnn
    assert recnn is mod
    from recnn.nn import Actor, Critic, ddpg_update, td3_update, DDPG, TD3          # noqa: F401
    from recnn.nn.update import value_update, temporal_difference                  # noqa: F401
    from recnn.utils import soft_update, DummyWriter                               # noqa: F401
    from recnn.data import get_base_batch, batch_tensor_embeddings                 # noqa: F401
    r, d, t = torch.ones(3, 1), torch.tensor([[0.], [1.], [0.]]), torch.full((3, 1), 2.0)
    assert torch.equal(temporal_difference(r, d, 0.5, t), torch.tensor([[2.], [1.], [2.]]))
    for k in [k for k in sys.modules if k == "recnn" or k.startswith("recnn.")]:
        del sys.modules[k]


def test_algo_wrappers_keep_reference_wiring():
    ddpg = recnn_b200.nn.DDPG(recnn_b200.nn.Actor(170, 16, 32), recnn_b200.nn.Critic(170, 16, 32))
    assert ddpg.params == {"gamma": 0.99, "min_value": -10, "max_value": 10, "policy_step": 10, "soft_tau": 0.001}
    assert set(ddpg.nets) == {"value_net", "target_value_net", "policy_net", "target_policy_net"}
    for name, net in ddpg.nets.items():
        assert net.training == ("target" not in name)
    for p, q in zip(ddpg.nets["policy_net"].parameters(), ddpg.nets["target_policy_net"].parameters()):
        assert torch.equal(p, q) and p.data_ptr() != q.data_ptr()
    td3 = recnn_b200.nn.TD3(recnn_b200.nn.Actor(170, 16, 32), recnn_b200.nn.Critic(170, 16, 32),
                            recnn_b200.nn.Critic(170, 16, 32))
    assert td3.params["policy_update"] == 10 and td3.params["noise_clip"] == 3
    assert ddpg._step == 0
    ddpg.step()
    assert ddpg._step == 1


def test_frame_env_feed_matches_oracle_collate():
    """FrameEnv (in-memory constructor) -> DataLoader -> collate -> frame-form batch."""
    rng = np.random.default_rng(3)
    table = torch.from_numpy(rng.standard_normal((40, 8), dtype=np.float32))
    user_dict = {u: {"items": rng.integers(0, 40, size=n, dtype=np.int64),
                     "ratings": rng.integers(-4, 6, size=n).astype(np.float64)}
                 for u, n in enumerate((14, 30, 11, 12, 9, 25))}          # user 4 is too short for frame 10
    env = recnn_b200.data.FrameEnv.from_user_dict(table, user_dict, frame_size=10, batch_size=3, num_workers=0,
                                                  test_size=0.0, embed_batch=recnn_b200.data.batch_frames)
    assert len(env.base.train_user_dataset) == 5
    seen = 0
    for batch in env.train_dataloader:
        users = batch["users"].tolist()
        want = O.collate_users([{"items": user_dict[u]["items"], "rates": user_dict[u]["ratings"],
                                 "sizes": len(user_dict[u]["items"]), "users": u} for u in users], 10)
        assert np.array_equal(batch["items"].numpy(), want["items"])
        assert np.array_equal(batch["ratings"].numpy(), want["ratings"])
        assert batch["items"].shape[0] == sum(len(user_dict[u]["items"]) - 10 for u in users)
        seen += len(users)
    assert seen == 5
    from recnn_b200.data.env import DataPath
    p = DataPath("/tmp/", "r.csv", "e.pkl", "c.pkl", use_cache=False)
    assert p.ratings == "/tmp/r.csv" and p.cache == "/tmp/c.pkl"
