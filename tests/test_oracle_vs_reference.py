"""Differential test: the numpy oracle against vectors recorded from the UNMODIFIED reference on seeds and shapes
that are NOT in the screened golden fixtures (oracle/cases.py UNSCREENED_CASES, tests/golden/vs_reference.npz
written by ``python -m oracle.make_golden vs_reference``)."""
import numpy as np
import pytest

from oracle import cases as C
from oracle import recnn_oracle as O
from tests._golden import compare_with_golden, load_golden, run_oracle_case


def _recorded(name, algo, opt):
    """The reference's run of one case in the key layout of oracle/make_golden.py:run_update_case."""
    gold = load_golden("vs_reference.npz")
    pre = "%s.%s.%s." % (name, algo, opt)
    out = {k[len(pre):]: v for k, v in gold.items() if k.startswith(pre)}
    if "samples" in out:
        split = np.split(out.pop("samples"), np.cumsum(out.pop("sample_sizes"))[:-1])
        out.update(zip(out.pop("sample_keys").tolist(), split))
    if algo == "td3" and name + ".noise" in gold:
        out.update(("noise.%d" % s, x) for s, x in enumerate(gold[name + ".noise"]))
    return out


@pytest.mark.parametrize("opt", ["adam", "sgd"])
@pytest.mark.parametrize("algo", ["ddpg", "td3"])
@pytest.mark.parametrize("name", list(C.UNSCREENED_CASES))
def test_oracle_tracks_the_live_reference(name, algo, opt):
    live = _recorded(name, algo, opt)
    if float(live["gate_margin"]) <= C.GATE_GUARD:
        pytest.skip("unscreened seed with an ambiguous ReLU gate (margin %.2g): torch/MKL and numpy may gate "
                    "differently; the screened golden seeds cover this algorithm" % float(live["gate_margin"]))
    got = run_oracle_case(C.UNSCREENED_CASES[name], algo, opt, golden=live if algo == "td3" else None)
    got = {k: v[:C.UNSCREENED_SAMPLES] if k.endswith(".sample") else v for k, v in got.items()}
    compare_with_golden(got, live, check_grads=(algo == "ddpg"))


def test_reference_gather_equals_oracle_on_random_users():
    ref = load_golden("vs_reference.npz")
    table, users, frame = C.random_gather_users()
    col = O.collate_users(users, frame)
    out = O.frame_gather(table, col["items"], col["ratings"], col["sizes"], frame)
    for k in ("state", "next_state", "action", "reward", "done"):
        assert np.array_equal(out[k].view(np.uint32), ref["gather." + k].view(np.uint32)), k
