"""Item-streamed REINFORCE policy gradient (recnn_reinforce_policy_grad_streamed) on the GPU: against the float64 oracle,
against the materialised entry, bit-for-bit repeatable, and through the public API at a million items, where the
materialised logits would not fit.  Tolerances as tests/test_reinforce_gpu.py: loss 2e-4 relative, every gradient within
3e-4 of the tensor's largest entry."""
from __future__ import annotations

import numpy as np
import pytest
import torch

import recnn_b200
from recnn_b200 import _lib
from recnn_b200.nn.arena import param_arena, grad_arena
from oracle import reinforce_oracle as RO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
K = 10
GRADS = ("w1", "b1", "w2", "b2")
METHODS = ["basic_reinforce", "reinforce_with_correction", "reinforce_with_TopK_correction"]
MIB = 1 << 20


def make_policy(p, S, H, I):
    m = recnn_b200.nn.DiscreteActor(S, I, H)
    with torch.no_grad():
        m.linear1.weight.copy_(torch.from_numpy(p["w1"]))
        m.linear1.bias.copy_(torch.from_numpy(p["b1"]))
        m.linear2.weight.copy_(torch.from_numpy(p["w2"]))
        m.linear2.bias.copy_(torch.from_numpy(p["b2"]))
    return m.to(DEV)


def grads_of(m):
    return {"w1": m.linear1.weight.grad, "b1": m.linear1.bias.grad, "w2": m.linear2.weight.grad, "b2": m.linear2.bias.grad}


def make_case(seed, S, H, I, R):
    rng = np.random.default_rng(seed)
    p = RO.make_discrete_actor(rng, S, I, H)
    return {"p": p, "state": rng.normal(0, 1, (R, S)).astype(np.float32), "action": rng.integers(0, I, R),
            "beta": np.log(rng.uniform(1e-4, 5e-4, R)).astype(np.float32),
            "ret": rng.normal(0, 1, R).astype(np.float32)}


def device_call(m, c, method, chunk):
    """One call of the streamed (chunk > 0) or materialised (chunk == 0) C entry; (loss, oob flag, {name: grad copy})."""
    L = _lib.lib()
    d = m.dims
    n = c["state"].shape[0]
    st = torch.from_numpy(c["state"]).to(DEV)
    act = torch.as_tensor(c["action"], dtype=torch.int64).to(DEV)
    beta = torch.from_numpy(c["beta"]).to(DEV) if method != RO.BASIC else None
    ret = torch.from_numpy(c["ret"]).to(DEV)
    floats = L.recnn_reinforce_streamed_scratch_floats(d, n, chunk) if chunk else L.recnn_discrete_scratch_floats(d, n, 1)
    scratch = torch.empty(floats, device=DEV)
    out = torch.zeros(2, device=DEV)
    flat, grads = param_arena(m), grad_arena(m)
    grads.fill_(float("nan"))                     # every gradient element must be written
    args = (d, flat.data_ptr(), grads.data_ptr(), st.data_ptr(), act.data_ptr(), _lib.ptr(beta), ret.data_ptr(), n,
            method, K)
    if chunk:
        _lib.check(L.recnn_reinforce_policy_grad_streamed(*args, chunk, out.data_ptr(), scratch.data_ptr(),
                                                          _lib.stream_ptr(DEV)))
    else:
        _lib.check(L.recnn_reinforce_policy_grad(*args, out.data_ptr(), scratch.data_ptr(), _lib.stream_ptr(DEV)))
    torch.cuda.synchronize()
    return float(out[0]), int(out.view(torch.int32)[1]), {k: v.detach().clone() for k, v in grads_of(m).items()}


def oracle(c, method):
    return RO.reinforce_policy_grad(c["p"], c["state"], c["action"], None if method == RO.BASIC else c["beta"], c["ret"],
                                    method, K)


def assert_close(loss, grads, want_loss, want, keys=GRADS, loss_terms_abs=0.0):
    """loss_terms_abs: sum of |row loss term|.  The rows' terms cancel (the returns are normalised to zero mean), so over
    tens of thousands of rows the fp32 sum of the terms is only as exact as a few ulp of this magnitude."""
    assert loss == pytest.approx(want_loss, rel=2e-4, abs=max(1e-4 * (1 + abs(want_loss)), 4e-7 * loss_terms_abs))
    for k in keys:
        w = want[k].cpu().numpy() if torch.is_tensor(want[k]) else want[k]
        scale = np.abs(w).max()
        assert scale > 0, k
        err = np.abs(grads[k].double().cpu().numpy() - w).max()
        assert err <= 3e-4 * scale, (k, err, scale)


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("S,H,I,R,chunk", [(13, 16, 37, 40, 8), (13, 16, 37, 40, 37), (52, 64, 300, 96, 128),
                                           (1290, 256, 5000, 1280, 1024), (1290, 2048, 5000, 1280, 1024)])
def test_streamed_matches_oracle(method, S, H, I, R, chunk):
    """Chunks 8 (ragged 37 = 4 x 8 + 5) and 37 at the tiny shape run the CUDA-core fallbacks of the GEMMs; 128 of 300
    leaves a ragged 44-wide chunk; 1024 of 5000 a ragged 904-wide one on the tensor cores."""
    mid = RO.METHODS[method]
    c = make_case(S + I + chunk, S, H, I, R)
    m = make_policy(c["p"], S, H, I)
    loss, oob, grads = device_call(m, c, mid, chunk)
    assert oob == 0
    want_loss, want, _ = oracle(c, mid)
    assert_close(loss, grads, want_loss, want)


def test_streamed_against_materialised():
    S, H, I, R = 1290, 2048, 5000, 1280
    c = make_case(7, S, H, I, R)
    m = make_policy(c["p"], S, H, I)
    want_loss, want, _ = oracle(c, RO.TOPK)
    l_s, _, g_s = device_call(m, c, RO.TOPK, 1024)
    l_m, _, g_m = device_call(m, c, RO.TOPK, 0)
    assert_close(l_s, g_s, want_loss, want)
    assert_close(l_m, g_m, want_loss, want)
    assert_close(l_s, g_s, l_m, {k: v.double() for k, v in g_m.items()})


def test_streamed_is_deterministic():
    S, H, I, R = 1290, 256, 5000, 1280
    c = make_case(8, S, H, I, R)
    m = make_policy(c["p"], S, H, I)
    l1, _, g1 = device_call(m, c, RO.TOPK, 1024)
    l2, _, g2 = device_call(m, c, RO.TOPK, 1024)
    assert l1 == l2
    for k in GRADS:
        assert torch.equal(g1[k], g2[k]), k
    want_loss, want, _ = oracle(c, RO.TOPK)
    for chunk in (512, 5000):
        l3, _, g3 = device_call(m, c, RO.TOPK, chunk)
        assert_close(l3, g3, want_loss, want)
        assert_close(l3, g3, l1, {k: v.double() for k, v in g1.items()})


# ---------------------------------------------------------------------------------------------------- million items
def reference_blocks(m, state, action, beta, ret, method, block=128, need_w2=True):
    """float64 policy gradient of DiscreteActor m computed on the GPU in blocks of rows (never more than [block, items]
    at a time).  Returns (loss, {name: grad}, sum of |row loss term|)."""
    w1 = m.linear1.weight.detach().double()
    b1 = m.linear1.bias.detach().double()
    w2 = m.linear2.weight.detach().double()
    b2 = m.linear2.bias.detach().double()
    H, I = w1.shape[0], w2.shape[0]
    out = {"w1": torch.zeros_like(w1), "b1": torch.zeros_like(b1), "b2": torch.zeros_like(b2)}
    if need_w2:
        out["w2"] = torch.zeros_like(w2)
    loss = terms_abs = 0.0
    for r0 in range(0, state.shape[0], block):
        x = state[r0:r0 + block].double()
        a = action[r0:r0 + block]
        h = torch.relu(x @ w1.T + b1)
        z = h @ w2.T + b2
        probs = torch.softmax(z, dim=1)
        del z
        rows = torch.arange(x.shape[0], device=x.device)
        pa = probs[rows, a].cpu().numpy()
        Lr, g, _ = RO.row_terms(pa, None if beta is None else beta[r0:r0 + block].cpu().numpy(),
                                ret[r0:r0 + block].cpu().numpy(), method, K)
        loss += float(Lr.sum())
        terms_abs += float(np.abs(Lr).sum())
        g = torch.from_numpy(g).to(x.device)
        dz = probs.mul_(-g[:, None])
        dz[rows, a] += g
        if need_w2:
            out["w2"] += dz.T @ h
        out["b2"] += dz.sum(0)
        dh = (dz @ w2) * (h > 0)
        del dz, probs
        out["w1"] += dh.T @ x
        out["b1"] += dh.sum(0)
    return loss, out, terms_abs


def saved_rows(m, rng, T, N, S, I):
    """T env steps of N rows each, saved as DiscreteActor._select_action_with_TopK_correction saves them."""
    for _ in range(T):
        m._saved.append({"state": torch.from_numpy(rng.normal(0, 1, (N, S)).astype(np.float32)).to(DEV),
                         "action": torch.from_numpy(rng.integers(0, I, N)).to(DEV),
                         "beta_log_prob": torch.from_numpy(np.log(rng.uniform(1e-7, 5e-6, N)).astype(np.float32)).to(DEV),
                         "K": K})
        m.rewards.append(torch.tensor(float(rng.normal()), device=DEV))


def flatten_saved(m):
    state = torch.cat([r["state"] for r in m._saved])
    action = torch.cat([r["action"] for r in m._saved])
    beta = torch.cat([r["beta_log_prob"] for r in m._saved])
    rewards = [float(r) for r in m.rewards]
    N = m._saved[0]["state"].shape[0]
    ret = torch.from_numpy(np.repeat(RO.normalised_returns(rewards), N))
    return state, action, beta, ret


def test_million_items_through_the_public_api():
    S, H, I, T, N = 1290, 256, 1 << 20, 4, 1024
    from recnn_b200.nn.update.reinforce import _policy_grad_plan
    assert _policy_grad_plan(T * N, I) > 0
    torch.manual_seed(0)
    m = recnn_b200.nn.DiscreteActor(S, I, H).to(DEV)
    saved_rows(m, np.random.default_rng(1), T, N, S, I)
    want_loss, want, terms_abs = reference_blocks(m, *flatten_saved(m), RO.TOPK)
    chooser = recnn_b200.nn.ChooseREINFORCE(recnn_b200.nn.ChooseREINFORCE.reinforce_with_TopK_correction)
    loss = chooser(m, None, learn=False)
    assert_close(float(loss), grads_of(m), want_loss, want, loss_terms_abs=terms_abs)
    assert len(m._saved) == 0


def test_bounded_memory_at_a_million_items():
    """65,536 saved rows x 2^20 items: the materialised logits would be 275 GB."""
    S, H, I, T, N = 1290, 256, 1 << 20, 8, 8192
    R = T * N
    torch.manual_seed(1)
    m = recnn_b200.nn.DiscreteActor(S, I, H).to(DEV)
    opt = recnn_b200.optim.Adam(m.parameters(), lr=1e-3)
    saved_rows(m, np.random.default_rng(2), T, N, S, I)
    want_loss, want, terms_abs = reference_blocks(m, *flatten_saved(m), RO.TOPK, block=256, need_w2=False)
    w0 = m.linear2.weight.detach().clone()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    chooser = recnn_b200.nn.ChooseREINFORCE(recnn_b200.nn.ChooseREINFORCE.reinforce_with_TopK_correction)
    loss = chooser(m, opt, learn=True)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - before
    # what the update may add: the gradient arena and Adam's two moments (created on first use, 3 x 1 GB here), the
    # streamed entry's scratch (state image, hidden activations, dh, one [R, chunk] logits chunk: 1.5 GB) and the
    # concatenated saved states (0.34 GB), plus 512 MiB for the small tensors and the allocator's rounding
    from recnn_b200.nn.update.reinforce import _policy_grad_plan
    arena = param_arena(m).numel() * 4
    scratch = _lib.lib().recnn_reinforce_streamed_scratch_floats(m.dims, R, _policy_grad_plan(R, I)) * 4
    assert scratch < 2 * 1024 * MIB
    bound = 3 * arena + scratch + R * S * 4 + 512 * MIB
    assert grown < bound, (grown / MIB, bound / MIB)
    assert_close(float(loss), grads_of(m), want_loss, want, keys=("w1", "b1", "b2"), loss_terms_abs=terms_abs)
    assert opt.steps_taken() == 1
    assert not torch.equal(w0, m.linear2.weight.detach())
    assert R * I * 4 > 180e9


def test_reinforce_agent_at_a_million_items():
    """recnn.nn.Reinforce with a 2^20-wide DiscreteActor and Critic: 64 rows per env step, the policy update on step 10
    takes the streamed path; losses finite, policy and targets move only then."""
    S, H, I, N = 52, 64, 1 << 20, 64
    torch.manual_seed(3)
    rng = np.random.default_rng(4)
    agent = recnn_b200.nn.Reinforce(recnn_b200.nn.DiscreteActor(S, I, H), recnn_b200.nn.Critic(S, I, H, 54e-2))
    agent = agent.to(torch.device(DEV))
    policy = agent.nets["policy_net"]
    bw = torch.from_numpy(rng.normal(0, 0.3, (I, S)).astype(np.float32)).to(DEV)

    def select_action_corr(state, action, K, writer, step, **kwargs):
        beta = lambda s, action=None: torch.softmax(s @ bw.T, dim=1)       # noqa: E731
        return policy._select_action_with_TopK_correction(state, beta, action, K=K, writer=writer, step=step)

    policy.select_action = select_action_corr
    agent.params["reinforce"] = recnn_b200.nn.ChooseREINFORCE(recnn_b200.nn.ChooseREINFORCE.reinforce_with_TopK_correction)
    agent.params["K"] = 10
    agent.optimizers["policy_optimizer"] = recnn_b200.optim.Adam(policy.parameters(), lr=1e-3)
    agent.optimizers["value_optimizer"] = recnn_b200.optim.Adam(agent.nets["value_net"].parameters(), lr=1e-3)
    w0 = policy.linear2.weight.detach().clone()
    t0 = agent.nets["target_policy_net"].linear2.weight.detach().clone()
    out = []
    for i in range(11):
        a = torch.from_numpy(rng.integers(0, I, N)).to(DEV)
        batch = {"state": torch.from_numpy(rng.normal(0, 1, (N, S)).astype(np.float32)).to(DEV),
                 "action": torch.nn.functional.one_hot(a, I).float(),
                 "reward": torch.from_numpy(rng.integers(-2, 3, N).astype(np.float32)).to(DEV),
                 "next_state": torch.from_numpy(rng.normal(0, 1, (N, S)).astype(np.float32)).to(DEV),
                 "done": torch.from_numpy((rng.random(N) < 0.1).astype(np.float32)).to(DEV)}
        if i == 10:
            from recnn_b200.nn.update.reinforce import _policy_grad_plan
            assert _policy_grad_plan(len(policy._saved) * N + N, I) > 0
        out.append(agent.update(batch))
        agent.step()
        if i == 9:
            assert torch.equal(w0, policy.linear2.weight.detach())
            assert torch.equal(t0, agent.nets["target_policy_net"].linear2.weight.detach())
    assert [o is not None for o in out] == [i == 10 for i in range(11)]
    o = out[10]
    assert set(o) == {"value", "policy", "step"} and np.isfinite(o["value"]) and np.isfinite(o["policy"])
    assert not torch.equal(w0, policy.linear2.weight.detach())
    assert not torch.equal(t0, agent.nets["target_policy_net"].linear2.weight.detach())
    assert len(policy._saved) == 0


# ---------------------------------------------------------------------------------------------------- errors
def test_out_of_range_action_on_the_streamed_path():
    S, H, I, R = 52, 64, 300, 96
    c = make_case(5, S, H, I, R)
    m = make_policy(c["p"], S, H, I)
    bad = dict(c, action=c["action"].copy())
    bad["action"][7] = I
    bad["action"][11] = -1
    l_bad, oob, g_bad = device_call(m, bad, RO.TOPK, 128)
    assert oob == 1
    keep = np.setdiff1d(np.arange(R), [7, 11])             # the flagged rows contribute nothing
    rest = {k: (v[keep] if k != "p" else v) for k, v in c.items()}
    want_loss, want, _ = oracle(rest, RO.TOPK)
    assert_close(l_bad, g_bad, want_loss, want)
    # through the public API, at a size that selects the streamed path
    from recnn_b200.nn.update.reinforce import _policy_grad_plan
    big = recnn_b200.nn.DiscreteActor(8, 1 << 20, 8).to(DEV)
    rows = 300
    assert _policy_grad_plan(rows, 1 << 20) > 0
    act = torch.zeros(rows, dtype=torch.int64, device=DEV)
    act[5] = 1 << 20
    for r in (1.0, 2.0):
        big._saved.append({"state": torch.zeros(rows // 2, 8, device=DEV), "action": act[:rows // 2] if r == 1.0 else
                           act[rows // 2:], "beta_log_prob": None})
        big.rewards.append(torch.tensor(r))
    with pytest.raises(IndexError):
        recnn_b200.nn.ChooseREINFORCE()(big, None, learn=False)


def test_item_chunk_must_be_positive():
    c = make_case(6, 13, 16, 37, 8)
    m = make_policy(c["p"], 13, 16, 37)
    for chunk in (0, -1):
        L = _lib.lib()
        out = torch.zeros(2, device=DEV)
        scratch = torch.empty(L.recnn_reinforce_streamed_scratch_floats(m.dims, 8, 8), device=DEV)
        st = torch.from_numpy(c["state"]).to(DEV)
        act = torch.as_tensor(c["action"], dtype=torch.int64).to(DEV)
        ret = torch.from_numpy(c["ret"]).to(DEV)
        with pytest.raises(_lib.RecnnError):
            _lib.check(L.recnn_reinforce_policy_grad_streamed(
                m.dims, param_arena(m).data_ptr(), grad_arena(m).data_ptr(), st.data_ptr(), act.data_ptr(), None,
                ret.data_ptr(), 8, RO.BASIC, 1, chunk, out.data_ptr(), scratch.data_ptr(), _lib.stream_ptr(DEV)))
