"""Drop-in for recnn.nn.update.reinforce (recnn/nn/update/reinforce.py:10-129): ChooseREINFORCE and reinforce_update.

The policy loss and its gradient are ONE device call (recnn_reinforce_policy_grad: recomputed forward, closed-form
d loss / d logits, three tensor-core GEMMs; past 1 GiB of logits its item-streamed form, which never holds more than one
chunk of them) over the rows ``DiscreteActor`` saved since the last policy update; the
optimizer step is the fused arena kernel (recnn_b200.optim) or any torch optimizer stepping the aliased ``.grad``
views.  The critic half is the DDPG critic step (value_update) fed with the target policy's probabilities.
"""
from __future__ import annotations

import gc

import torch

from ... import _lib
from ... import utils
from ...utils.misc import DummyWriter
from ..arena import param_arena, grad_arena
from .misc import value_update


_MAX_LOGIT_FLOATS = 1 << 28          # 1 GiB of fp32 logits


def _policy_grad_plan(rows, items):
    """Item chunk width of the policy gradient over ``rows`` saved rows and ``items`` outputs; 0 = materialise.

    Up to 1 GiB of logits the materialised entry (one logits GEMM, 3/4 of the streamed FLOPs) is used; beyond, the
    item-streamed entry with the widest multiple of 128 whose [rows, chunk] logits stay within 1 GiB (at least 128)."""
    if rows * items <= _MAX_LOGIT_FLOATS:
        return 0
    return max(128, _MAX_LOGIT_FLOATS // rows // 128 * 128)


def _policy_loss(policy, returns, method):
    """Loss (0-dim tensor) of ``method`` over policy._saved; the gradient of every parameter lands in the policy's
    gradient arena (= ``p.grad`` of its parameters), overwriting what was there (zero_grad + backward)."""
    saved = policy._saved
    if not saved:
        raise RuntimeError("no saved actions: select_action was not called since the last policy update")
    if len(returns) != len(saved):
        raise ValueError("%d returns for %d saved env steps" % (len(returns), len(saved)))
    flat = param_arena(policy)
    dev = flat.device
    if dev.type != "cuda":
        raise _lib.RecnnError("recnn_b200 nets run on CUDA only (policy is on %s)" % dev)
    grads = grad_arena(policy)
    state = torch.cat([r["state"] for r in saved], 0).contiguous()
    action = torch.cat([r["action"] for r in saved], 0).contiguous()
    beta_lp = None
    if method != _lib.REINFORCE_BASIC:
        if any(r["beta_log_prob"] is None for r in saved):
            raise RuntimeError("the corrected REINFORCE losses need select_action to be one of the *_with_correction "
                               "variants (no behaviour-policy log-probs were saved)")
        beta_lp = torch.cat([r["beta_log_prob"] for r in saved], 0).contiguous()
    rows = torch.tensor([r["state"].shape[0] for r in saved])
    ret_rows = torch.repeat_interleave(torch.as_tensor(returns, dtype=torch.float32).cpu(), rows).to(dev, non_blocking=True)
    n = state.shape[0]
    d = policy.dims
    L = _lib.lib()
    chunk = _policy_grad_plan(n, d.num_items)
    floats = L.recnn_reinforce_streamed_scratch_floats(d, n, chunk) if chunk else L.recnn_discrete_scratch_floats(d, n, 1)
    scratch = torch.empty(floats, device=dev, dtype=torch.float32)
    out = torch.zeros(2, device=dev, dtype=torch.float32)
    ks = {r.get("K") for r in saved if r.get("K") is not None}
    if len(ks) > 1:
        raise ValueError("select_action was called with different K since the last policy update: %s" % sorted(ks))
    K = ks.pop() if ks else 1
    args = (d, flat.data_ptr(), grads.data_ptr(), state.data_ptr(), action.data_ptr(), _lib.ptr(beta_lp),
            ret_rows.data_ptr(), n, method, K)
    with torch.cuda.device(dev):
        if chunk:
            _lib.check(L.recnn_reinforce_policy_grad_streamed(*args, chunk, out.data_ptr(), scratch.data_ptr(),
                                                              _lib.stream_ptr(dev)))
        else:
            _lib.check(L.recnn_reinforce_policy_grad(*args, out.data_ptr(), scratch.data_ptr(), _lib.stream_ptr(dev)))
    if int(out.view(torch.int32)[1].item()) != 0:
        raise IndexError("saved action index out of range for the policy's output layer")
    return out[0].clone()


class ChooseREINFORCE:
    def __init__(self, method=None):
        if method is None:
            method = ChooseREINFORCE.basic_reinforce
        self.method = method

    @staticmethod
    def basic_reinforce(policy, returns, *args, **kwargs):
        """sum over saved steps and rows of -log pi(a) R   (reinforce.py:16-22)"""
        return _policy_loss(policy, returns, _lib.REINFORCE_BASIC)

    @staticmethod
    def reinforce_with_correction(policy, returns, *args, **kwargs):
        """... of (pi(a)/beta(a)) (-log pi(a)) R   (reinforce.py:24-33)"""
        return _policy_loss(policy, returns, _lib.REINFORCE_CORRECTED)

    @staticmethod
    def reinforce_with_TopK_correction(policy, returns, *args, **kwargs):
        """... of lambda_K (pi(a)/beta(a)) (-log pi(a)) R, lambda_K = K (1 - pi(a))^(K-1)   (reinforce.py:35-44)"""
        return _policy_loss(policy, returns, _lib.REINFORCE_TOPK)

    _BUILT_IN = ("basic_reinforce", "reinforce_with_correction", "reinforce_with_TopK_correction")

    def __call__(self, policy, optimizer, learn=True):
        if getattr(self.method, "__name__", None) not in self._BUILT_IN or \
                getattr(ChooseREINFORCE, self.method.__name__) is not self.method:
            raise TypeError("recnn_b200 computes the REINFORCE gradient in closed form for the three built-in methods; "
                            "a custom method would need the autograd graph the reference keeps in saved_log_probs")
        # discounted returns over the saved env steps, normalised (reinforce.py:44-52; the discount is the literal 0.99)
        R = 0
        returns = []
        rewards = [r.detach().float().cpu() if torch.is_tensor(r) else torch.tensor(float(r)) for r in policy.rewards]
        for r in rewards[::-1]:
            R = r + 0.99 * R
            returns.insert(0, R)
        returns = torch.tensor(returns)
        returns = (returns - returns.mean()) / (returns.std() + 0.0001)

        policy_loss = self.method(policy, returns)

        if learn:
            # zero_grad + backward happened inside the method (the gradient arena was overwritten)
            from ... import optim as _optim
            if isinstance(optimizer, _optim._ArenaOptimizer) and optimizer._module is not policy:
                optimizer.bind(policy)
            optimizer.step()

        policy.gc()
        gc.collect()
        return policy_loss


def reinforce_update(batch, params, nets, optimizer, device=torch.device("cpu"), debug=None,
                     writer=DummyWriter(), learn=True, step=-1):
    """Same signature, side effects and return value as the reference (reinforce.py:68-129): returns the losses dict
    on policy steps (step % policy_step == 0 and step > 0) and None otherwise."""
    # Due to its mechanics, reinforce doesn't support testing (reinforce.py:80-81)
    learn = True
    policy = nets["policy_net"]
    dev = policy.linear1.weight.device
    if dev.type != "cuda":
        raise _lib.RecnnError("recnn_b200 update functions run on CUDA only (policy net is on %s); there is no CPU path" % dev)
    state = batch["state"].to(dev)
    action = batch["action"].to(dev)

    predicted_probs = policy.select_action(state=state, action=action, K=params["K"], learn=learn, writer=writer, step=step)
    if not isinstance(writer, DummyWriter):
        writer.add_histogram("predicted_probs_std", predicted_probs.std(), step)
        writer.add_histogram("predicted_probs_mean", predicted_probs.mean(), step)
        mx = predicted_probs.max(dim=1).values
        writer.add_histogram("predicted_probs_max_mean", mx.mean(), step)
        writer.add_histogram("predicted_probs_max_std", mx.std(), step)
    reward = nets["value_net"](state, predicted_probs).detach()
    policy.rewards.append(reward.mean())

    value_loss = value_update(batch, params, nets, optimizer, writer=writer, device=dev, debug=debug, learn=True, step=step)

    if step % params["policy_step"] == 0 and step > 0:
        policy_loss = params["reinforce"](policy, optimizer["policy_optimizer"])
        utils.soft_update(nets["value_net"], nets["target_value_net"], soft_tau=params["soft_tau"])
        utils.soft_update(nets["policy_net"], nets["target_policy_net"], soft_tau=params["soft_tau"])
        losses = {"value": value_loss.item(), "policy": policy_loss.item(), "step": step}
        utils.write_losses(writer, losses, kind="train" if learn else "test")
        return losses
