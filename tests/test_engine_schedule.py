"""The update's phase schedule (recnn_b200/nn/update/_engine.py: schedule) on the CPU: which phase masks go to the
C side and which host work runs between them, pinned for every path, plus the ordering invariants over all inputs."""
import itertools

import pytest

from recnn_b200 import _lib as P
from recnn_b200.nn.update._engine import (schedule, ALLREDUCE_VALUE_GRADS as AR_V, ALLREDUCE_POLICY_GRADS as AR_P,
                                          ALLREDUCE_LOSSES as AR_L, STEP_VALUE_OPTIMIZERS as STEP_V,
                                          STEP_POLICY_OPTIMIZER as STEP_P)

# run_step's phase order (recnn_b200/csrc/step.cu)
ORDER = (P.PH_GATHER, P.PH_VALUE_GRAD, P.PH_VALUE_OPT, P.PH_POLICY_LOSS, P.PH_POLICY_GRAD, P.PH_POLICY_OPT,
         P.PH_SOFT_UPDATE, P.PH_FINISH)
HEAD = P.PH_GATHER | P.PH_VALUE_GRAD
SPLIT = (P.PH_GATHER | P.PH_VALUE_GRAD, P.PH_VALUE_OPT | P.PH_POLICY_LOSS | P.PH_POLICY_GRAD,
         P.PH_POLICY_OPT | P.PH_SOFT_UPDATE | P.PH_FINISH)


def sched(value_only=False, learn=True, do_policy=False, value_builtin=True, policy_builtin=True, debug=None,
          world=1, peer_comm=False):
    return schedule(value_only, learn, do_policy, value_builtin, policy_builtin, (not learn) if debug is None else debug,
                    world, peer_comm)


def all_inputs():
    """Every combination a caller can produce: do_policy only on learning steps, value-only calls never take a
    policy step, debug outputs exactly when learn=False, and a peer communicator only with several ranks."""
    for value_only, learn, do_policy, vb, pb, world, peer in itertools.product(
            (False, True), (False, True), (False, True), (False, True), (False, True), (1, 2, 8), (False, True)):
        if (do_policy and (not learn or value_only)) or (peer and world == 1):
            continue
        yield dict(value_only=value_only, learn=learn, do_policy=do_policy, value_builtin=vb, policy_builtin=pb,
                   world=world, peer_comm=peer)


# ----------------------------------------------------------------------------- each path, pinned
@pytest.mark.parametrize("do_policy", [False, True])
@pytest.mark.parametrize("world,peer", [(1, False), (2, True), (8, True)])
def test_fused_one_gpu_or_peer_comm_is_one_call(do_policy, world, peer):
    s = sched(do_policy=do_policy, world=world, peer_comm=peer)
    assert s.segments == ((P.PH_ALL, ()),)
    assert s.capturable


def test_fused_nccl_is_three_calls_cut_where_gradients_are_complete():
    s = sched(world=2)
    assert s.segments == ((SPLIT[0], (AR_V,)), (SPLIT[1], (AR_L,)), (SPLIT[2], ()))
    assert s.capturable
    s = sched(world=2, do_policy=True)
    assert s.segments == ((SPLIT[0], (AR_V,)), (SPLIT[1], (AR_P, AR_L)), (SPLIT[2], ()))
    assert s.capturable


def test_external_optimizers_run_phase_by_phase():
    s = sched(do_policy=True, value_builtin=False, policy_builtin=False)
    assert s.segments == ((HEAD, (STEP_V,)), (P.PH_POLICY_LOSS, ()), (P.PH_POLICY_GRAD, ()),
                          (P.PH_POLICY_OPT, (STEP_P,)), (P.PH_SOFT_UPDATE, ()), (P.PH_FINISH, ()))
    assert not s.capturable
    s = sched(do_policy=False, value_builtin=False, policy_builtin=False)
    assert s.segments == ((HEAD, (STEP_V,)), (P.PH_POLICY_LOSS, ()), (P.PH_FINISH, ()))
    assert not s.capturable


@pytest.mark.parametrize("peer", [False, True])
def test_external_optimizers_data_parallel_all_reduce_with_nccl(peer):
    s = sched(do_policy=True, value_builtin=False, policy_builtin=False, world=2, peer_comm=peer)
    assert s.segments == ((HEAD, (AR_V, STEP_V)), (P.PH_POLICY_LOSS, ()), (P.PH_POLICY_GRAD, (AR_P,)),
                          (P.PH_POLICY_OPT, (STEP_P,)), (P.PH_SOFT_UPDATE, (AR_L,)), (P.PH_FINISH, ()))
    s = sched(do_policy=False, value_builtin=False, policy_builtin=False, world=2, peer_comm=peer)
    assert s.segments == ((HEAD, (AR_V, STEP_V)), (P.PH_POLICY_LOSS, (AR_L,)), (P.PH_FINISH, ()))


def test_mixed_optimizers_step_each_once():
    """Built-in policy optimizer with an external value optimizer and vice versa: the built-in one is the C
    side's optimizer phase, the external one is stepped in Python, never both."""
    s = sched(do_policy=True, value_builtin=False, policy_builtin=True)
    assert s.segments == ((HEAD, (STEP_V,)), (P.PH_POLICY_LOSS, ()), (P.PH_POLICY_GRAD, ()),
                          (P.PH_POLICY_OPT, ()), (P.PH_SOFT_UPDATE, ()), (P.PH_FINISH, ()))
    s = sched(do_policy=True, value_builtin=True, policy_builtin=False)
    assert s.segments == ((HEAD, ()), (P.PH_VALUE_OPT, ()), (P.PH_POLICY_LOSS, ()), (P.PH_POLICY_GRAD, ()),
                          (P.PH_POLICY_OPT, (STEP_P,)), (P.PH_SOFT_UPDATE, ()), (P.PH_FINISH, ()))
    assert not s.capturable


@pytest.mark.parametrize("world", [1, 2])
def test_learn_false_trains_nothing(world):
    s = sched(learn=False, value_builtin=False, policy_builtin=False, world=world)
    losses = (AR_L,) if world > 1 else ()
    assert s.segments == ((HEAD, ()), (P.PH_POLICY_LOSS, losses), (P.PH_FINISH, ()))
    assert not s.capturable


def test_value_only():
    assert sched(value_only=True).segments == ((HEAD, ()), (P.PH_VALUE_OPT, ()), (P.PH_FINISH, ()))
    assert sched(value_only=True, value_builtin=False).segments == ((HEAD, (STEP_V,)), (P.PH_FINISH, ()))
    assert sched(value_only=True, learn=False, value_builtin=False).segments == ((HEAD, ()), (P.PH_FINISH, ()))
    # several ranks: the critic gradient before its optimizer, the loss before FINISH reads it back
    assert sched(value_only=True, world=2).segments == ((HEAD, (AR_V,)), (P.PH_VALUE_OPT, (AR_L,)), (P.PH_FINISH, ()))
    assert sched(value_only=True, value_builtin=False, world=2).segments == ((HEAD, (AR_V, STEP_V, AR_L)),
                                                                             (P.PH_FINISH, ()))
    assert sched(value_only=True, learn=False, world=2).segments == ((HEAD, (AR_L,)), (P.PH_FINISH, ()))
    assert not any(sched(value_only=True, value_builtin=vb, world=w).capturable for vb in (False, True) for w in (1, 2))


def test_debug_outputs_are_never_captured():
    assert not sched(learn=True, debug=True).capturable


# ----------------------------------------------------------------------------- invariants over all inputs
def _events(s):
    """The schedule as one flat sequence: ('phase', bit) for every phase bit of a call, in run_step's order
    within the call, then ('host', action) for each host action after it."""
    ev = []
    for phases, actions in s.segments:
        ev += [("phase", b) for b in ORDER if phases & b]
        ev += [("host", act) for act in actions]
    return ev


@pytest.mark.parametrize("inp", list(all_inputs()), ids=lambda d: "-".join("%s=%s" % kv for kv in d.items()))
def test_invariants(inp):
    s = sched(**inp)
    ev = _events(s)
    bits = [b for kind, b in ev if kind == "phase"]
    # every phase bit at most once, in run_step's order; GATHER first, FINISH last
    assert len(bits) == len(set(bits))
    assert bits == sorted(bits, key=ORDER.index)
    assert bits[0] == P.PH_GATHER and bits[-1] == P.PH_FINISH
    assert ev[-1] == ("phase", P.PH_FINISH)
    for phases, _ in s.segments:
        assert phases and phases & ~P.PH_ALL == 0
    acts = [a for kind, a in ev if kind == "host"]
    assert len(acts) == len(set(acts))

    def at(e):
        return ev.index(e)

    def maybe(phase):
        return at(("phase", phase)) if ("phase", phase) in ev else len(ev)

    # a gradient all-reduce after the phase that completes the gradient, before its optimizer phase / step()
    if AR_V in acts:
        assert at(("phase", P.PH_VALUE_GRAD)) < at(("host", AR_V)) < maybe(P.PH_VALUE_OPT)
        if STEP_V in acts:
            assert at(("host", AR_V)) < at(("host", STEP_V))
    if AR_P in acts:
        assert at(("phase", P.PH_POLICY_GRAD)) < at(("host", AR_P)) < at(("phase", P.PH_POLICY_OPT))
        if STEP_P in acts:
            assert at(("host", AR_P)) < at(("host", STEP_P))
    # an external optimizer steps after the C side finished (and, for the policy, clipped) its gradient
    if STEP_V in acts:
        assert at(("phase", P.PH_VALUE_GRAD)) < at(("host", STEP_V)) < maybe(P.PH_POLICY_LOSS)
    if STEP_P in acts:
        assert at(("phase", P.PH_POLICY_OPT)) < at(("host", STEP_P)) < at(("phase", P.PH_SOFT_UPDATE))

    learn, dp = inp["learn"], inp["world"] > 1
    # the exchange: in the kernels through the peer communicator when fused, otherwise NCCL between the calls
    if dp and not (inp["peer_comm"] and s.capturable):
        assert at(("host", AR_L)) < at(("phase", P.PH_FINISH))
        assert (AR_V in acts) == learn
        assert (AR_P in acts) == inp["do_policy"]
    else:
        assert not {AR_V, AR_P, AR_L} & set(acts)
    # each optimizer stepped exactly once: by the C side (its phase) or in Python, never both
    if learn:
        assert (STEP_V in acts) == (not inp["value_builtin"])
        assert (("phase", P.PH_VALUE_OPT) in ev) == inp["value_builtin"]
        if inp["do_policy"]:
            assert ("phase", P.PH_POLICY_OPT) in ev
            assert (STEP_P in acts) == (not inp["policy_builtin"])
        else:
            assert STEP_P not in acts
    else:
        assert not {STEP_V, STEP_P} & set(acts)
        assert ("phase", P.PH_VALUE_OPT) not in ev
    if inp["value_only"]:
        assert not {P.PH_POLICY_LOSS, P.PH_POLICY_GRAD, P.PH_POLICY_OPT, P.PH_SOFT_UPDATE} & set(bits)
    # graphs only for a learning step with every optimizer on the device, and never with Python work inside
    assert s.capturable == (learn and not inp["value_only"] and inp["value_builtin"] and inp["policy_builtin"])
    if s.capturable:
        assert not {STEP_V, STEP_P} & set(acts)
    # one GPU with built-in optimizers: no host work at all
    if inp["world"] == 1 and inp["value_builtin"] and inp["policy_builtin"]:
        assert acts == []
