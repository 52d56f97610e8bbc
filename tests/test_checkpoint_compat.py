"""Checkpoint compatibility with the reference (SURVEY 8f rank 4): state_dicts written by the reference's own
Actor / Critic (oracle/make_ckpt_golden.py, torch.save as readme.md:152 / streamlit_demo.py:151-160 use it) load
into recnn_b200's nets and reproduce the reference's forward outputs; state_dicts written here load back."""
import os

import numpy as np
import pytest
import torch

import recnn_b200

CKPT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_checkpoint.pt")


def _load():
    return torch.load(CKPT, map_location="cpu", weights_only=True)


def test_reference_state_dict_loads_with_identical_keys_and_values():
    ck = _load()
    S, A, H = ck["dims"]
    actor, critic = recnn_b200.nn.Actor(S, A, H), recnn_b200.nn.Critic(S, A, H)
    assert list(actor.state_dict().keys()) == list(ck["actor"].keys())
    assert list(critic.state_dict().keys()) == list(ck["critic"].keys())
    actor.load_state_dict(ck["actor"], strict=True)
    critic.load_state_dict(ck["critic"], strict=True)
    for k, v in ck["actor"].items():
        assert torch.equal(actor.state_dict()[k], v) and actor.state_dict()[k].dtype == v.dtype
    for k, v in ck["critic"].items():
        assert torch.equal(critic.state_dict()[k], v)


def test_saved_state_dict_round_trips_through_torch_save(tmp_path):
    ck = _load()
    S, A, H = ck["dims"]
    actor = recnn_b200.nn.Actor(S, A, H)
    actor.load_state_dict(ck["actor"])
    path = tmp_path / "ddpg_policy.model"
    torch.save(actor.state_dict(), path)                       # what the reference publishes
    back = torch.load(path, map_location="cpu", weights_only=True)
    for k, v in ck["actor"].items():
        assert torch.equal(back[k], v) and back[k].is_contiguous() and tuple(back[k].shape) == tuple(v.shape)


def test_saved_state_dict_loads_into_the_reference_classes(tmp_path):
    """The fixture's state_dicts were written by the reference's own Actor / Critic, so they record what its
    load_state_dict(strict=True) accepts: these keys in this order, these shapes and dtypes.  A file saved by
    recnn_b200 must match that layout, and after loading the fixture it must carry the very weights on which the
    reference computed ck["out"]."""
    ck = _load()
    S, A, H = ck["dims"]
    for kind, cls in (("actor", recnn_b200.nn.Actor), ("critic", recnn_b200.nn.Critic)):
        ref = ck[kind]
        for loaded in (False, True):
            ours = cls(S, A, H)
            if loaded:
                ours.load_state_dict(ref)
            path = tmp_path / ("%s_%d.model" % (kind, loaded))
            torch.save(ours.state_dict(), path)
            back = torch.load(path, map_location="cpu", weights_only=True)
            assert list(back.keys()) == list(ref.keys()), kind
            for k, v in ref.items():
                assert tuple(back[k].shape) == tuple(v.shape) and back[k].dtype == v.dtype, (kind, k)
                assert not loaded or torch.equal(back[k], v), (kind, k)


@pytest.mark.gpu
def test_loaded_checkpoint_reproduces_the_reference_forward():
    ck = _load()
    S, A, H = ck["dims"]
    actor = recnn_b200.nn.Actor(S, A, H)
    critic = recnn_b200.nn.Critic(S, A, H)
    actor.load_state_dict(ck["actor"])
    critic.load_state_dict(ck["critic"])
    actor, critic = actor.cuda().eval(), critic.cuda().eval()
    got = actor(ck["state"]).cpu().numpy()
    np.testing.assert_allclose(got, ck["out"]["actor"].numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(actor(ck["state"], tanh=True).cpu().numpy(), ck["out"]["actor_tanh"].numpy(),
                               rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(critic(ck["state"], ck["action"]).cpu().numpy(), ck["out"]["critic"].numpy(),
                               rtol=1e-5, atol=1e-6)
