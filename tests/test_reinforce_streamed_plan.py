"""Host-side pieces of the item-streamed REINFORCE policy gradient: which path the policy update takes for a given
size, and how the streamed entry's scratch scales.  No GPU needed."""
from __future__ import annotations

import pytest

from recnn_b200 import _lib
from recnn_b200.nn.update.reinforce import _policy_grad_plan

LIMIT = 1 << 28                          # floats of materialised logits (1 GiB)


def test_plan_threshold():
    assert _policy_grad_plan(1 << 14, 1 << 14) == 0                # exactly 2^28 floats: materialised
    assert _policy_grad_plan(1 << 14, (1 << 14) + 1) > 0          # one item more: streamed
    assert _policy_grad_plan(1, LIMIT) == 0


@pytest.mark.parametrize("rows,items", [(640, 1 << 20), (704, 1 << 20), (4096, 1 << 20), (65536, 1 << 20),
                                        (163840, 1 << 20), (163840, 5000), (1 << 14, (1 << 14) + 1), (300000, 1000)])
def test_plan_chunks_are_the_widest_multiple_of_128_within_the_limit(rows, items):
    c = _policy_grad_plan(rows, items)
    assert c >= 128 and c % 128 == 0
    if rows * 128 <= LIMIT:
        assert rows * c <= LIMIT < rows * (c + 128)
    else:
        assert c == 128                                           # the floor, even past the limit


def test_plan_known_shapes():
    assert _policy_grad_plan(163840, 1 << 20) == 1536
    assert _policy_grad_plan(65536, 1 << 20) == 4096
    assert _policy_grad_plan(4096, 1 << 20) == 65536
    assert _policy_grad_plan(10 ** 6, 1 << 20) == 256
    assert _policy_grad_plan(3 * 10 ** 6, 1 << 20) == 128


@pytest.mark.parametrize("rows,items", [(1280, 5000),                    # bench.py's reinforce leg
                                        (128, 5000), (100, 5000), (96, 5000), (10, 5000),   # GPU test shapes
                                        (60, 37), (60, 300), (20, 20)])
def test_existing_shapes_stay_materialised(rows, items):
    assert _policy_grad_plan(rows, items) == 0


def _floats(rows, items, chunk, S=1290, H=256):
    return _lib.lib().recnn_reinforce_streamed_scratch_floats(_lib.DiscreteDims(S, H, items, 0), rows, chunk)


@pytest.mark.parametrize("rows", [640, 4096, 65536])
def test_streamed_scratch_does_not_grow_with_items(rows):
    base = _floats(rows, 1 << 20, 1024)
    assert base > 0
    for items in (1 << 16, (1 << 20) + 77, 1 << 24, (1 << 31) - 1):
        assert _floats(rows, items, 1024) == base
    # far below the materialised entry's scratch at a million items
    assert base < _lib.lib().recnn_discrete_scratch_floats(_lib.DiscreteDims(1290, 256, 1 << 20, 0), rows, 1) / 100


@pytest.mark.parametrize("rows", [4096, 65536])
def test_streamed_scratch_grows_linearly_with_the_chunk(rows):
    H = 256
    chunks = [1024, 2048, 4096, 8192, 16384]
    f = [_floats(rows, 1 << 20, c, H=H) for c in chunks]
    for (c0, f0), (c1, f1) in zip(zip(chunks, f), zip(chunks[1:], f[1:])):
        # one [rows, chunk] logits buffer, plus the split-K partials of one chunk's dW2 [chunk, H + 1], which grow by
        # less than one partial per added column
        extra = (f1 - f0) - rows * (c1 - c0)
        assert 0 <= extra <= (H + 1) * (c1 - c0), (c0, c1, extra)


def test_streamed_scratch_rejects_bad_arguments():
    assert _floats(64, 1000, 0) == 0
    assert _floats(64, 1000, -5) == 0
    assert _floats(0, 1000, 128) == 0
