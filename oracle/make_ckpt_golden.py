"""Generate tests/golden/ref_checkpoint.pt by running the UNMODIFIED reference (build container only).

    python -m oracle.make_ckpt_golden

What is pinned (SURVEY.md 8f rank 4, checkpoint compatibility): the reference publishes trained policies as
``torch.save(policy_net.state_dict())`` files (readme.md:152, loaded by examples/streamlit_demo.py:151-160 with
``recnn.nn.models.Actor(1290, 128, 256).load_state_dict(torch.load(...))``).  The published files themselves are not
available offline, so the fixture is the same artefact made here: state_dicts of the reference's own Actor / Critic
(constructed by the reference, reduced dims to keep the fixture small), saved with torch.save exactly as the
reference does, plus eval-mode inputs and the REFERENCE's forward outputs on them.
tests/test_checkpoint_compat.py loads the file into recnn_b200.nn.Actor / Critic (CUDA forward must reproduce the
stored outputs) and checks that a state_dict saved by recnn_b200 has the layout of the reference classes' own
(same keys in the same order, shapes, dtypes), so that they load it with strict=True.
"""
from __future__ import annotations

import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.ref_import import import_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_checkpoint.pt")
S, A, H, N = 44, 8, 32, 19          # state = frame 4 x dim 10 + 4, hidden 32


def main():
    recnn = import_reference()
    torch.manual_seed(20260923)
    actor = recnn.nn.models.Actor(S, A, H, 6e-1).eval()
    critic = recnn.nn.models.Critic(S, A, H, 54e-2).eval()
    state = torch.randn(N, S)
    action = torch.randn(N, A)
    with torch.no_grad():
        out = {"actor": actor(state), "actor_tanh": actor(state, tanh=True), "critic": critic(state, action)}
    torch.save({"dims": (S, A, H), "actor": actor.state_dict(), "critic": critic.state_dict(),
                "state": state, "action": action, "out": out}, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
