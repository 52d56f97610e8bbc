"""Generate tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python -m oracle.make_golden

What is pinned (SURVEY.md 8c -- the reference ships no golden vectors, so they
are produced here by differential execution of its own functions):

* gather.npz  -- recnn.data.utils.prepare_batch_static_size + batch_tensor_embeddings
                 on three synthetic users (full inputs and outputs, bit-exact).
* collate.npz -- recnn.data.utils.prepare_batch_static_size up to (not including) the embedding
                 gather: the [N, F+1] item-id / rating windows, sizes and users it hands to
                 ``embed_batch`` (captured by passing an identity ``embed_batch``), plus ``done``
                 from batch_tensor_embeddings, for (i) all 14 synthetic users in storage order and
                 (ii) a shuffled 6-user minibatch.  Ragged lengths incl. the minimum F+1, float64
                 ratings that are not fp32-representable (pins the ``.float()`` rounding).
* ingest.npz  -- recnn.data.dataset_functions.prepare_dataset + utils.make_items_tensor + sort_users_itemwise on a
                 synthetic ratings table (24 users, sparse movie ids, unsorted timestamps): surviving users and
                 their order, per-user time-ordered item rows / mapped ratings.
* ddpg_<case>.npz / td3_<case>.npz -- recnn.nn.update.ddpg_update / td3_update,
                 12 consecutive steps (policy steps 0 and 10 included), torch.optim
                 Adam(lr=1e-5) and SGD(lr=1e-3) passed through the reference's
                 ``optimizer`` dict, dropout made reproducible by assigning a
                 mask-replaying module to ``net.drop_layer`` (an attribute of the
                 reference's nets; no reference source is modified), TD3 noise
                 made reproducible by seeding torch's CPU generator right before
                 each call and storing the identical draw.
  Stored: input checksums, per-step losses, digests (sampled values + sums) of
  every parameter of every net after steps {1, 2, 11, 12}, critic .grad after
  step index 1 (a non-policy step: pure value-loss gradient) and actor .grad
  after step index 0 (post "clip": sign-flipped, L1-normalised).
* vs_reference.npz -- the same update cases on the unscreened seeds and shapes of
                 C.UNSCREENED_CASES, and the gather on C.random_gather_users(),
                 reduced to what tests/test_oracle_vs_reference.py compares.
"""
from __future__ import annotations

import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import cases as C            # noqa: E402
from oracle import recnn_oracle as O     # noqa: E402
from oracle.ref_import import import_reference  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
SNAP_AFTER = (1, 2, 11, 12)     # number of completed steps


class ReplayDropout(torch.nn.Module):
    """Stands in for nn.Dropout(p=0.5): train mode multiplies by the next
    supplied mask * 2 (== x * mask / (1-p), bit-identical to torch's dropout
    for p=.5 since *2 is exact); eval mode is the identity."""

    def __init__(self):
        super().__init__()
        self.queue = []

    def feed(self, masks):
        self.queue = [torch.from_numpy(np.asarray(m, dtype=np.float32)) for m in masks]

    def forward(self, x):
        if not self.training:
            return x
        return x * (self.queue.pop(0) * 2.0)


def _load(module, p):
    with torch.no_grad():
        module.linear1.weight.copy_(torch.from_numpy(p["w1"]))
        module.linear1.bias.copy_(torch.from_numpy(p["b1"]))
        module.linear2.weight.copy_(torch.from_numpy(p["w2"]))
        module.linear2.bias.copy_(torch.from_numpy(p["b2"]))
        module.linear3.weight.copy_(torch.from_numpy(p["w3"]))
        module.linear3.bias.copy_(torch.from_numpy(p["b3"]))
    return module


def _dump(module):
    ps = [q.detach().numpy().copy() for q in module.parameters()]
    return dict(zip(O.PARAM_ORDER, ps))


def _dump_grad(module):
    ps = [q.grad.detach().numpy().copy() for q in module.parameters()]
    return dict(zip(O.PARAM_ORDER, ps))


def build_ref_nets(recnn, spec, inp, algo):
    s_dim, a_dim, h = C.dims(spec)
    nets = {}
    for name, p in inp["nets"].items():
        if "policy" in name:
            m = recnn.nn.Actor(s_dim, a_dim, h, spec["actor_init_w"])
        else:
            m = recnn.nn.Critic(s_dim, a_dim, h, spec["critic_init_w"])
        _load(m, p)
        m.drop_layer = ReplayDropout()
        if "target" in name:
            m.eval()                      # algo.py:76-77
        else:
            m.train()
        nets[name] = m
    return nets


def make_optimizers(kind, nets, algo):
    def mk(net):
        if kind == "adam":
            return torch.optim.Adam(net.parameters(), lr=1e-5)
        return torch.optim.SGD(net.parameters(), lr=1e-3)
    if algo == "ddpg":
        return {"policy_optimizer": mk(nets["policy_net"]), "value_optimizer": mk(nets["value_net"])}
    return {"policy_optimizer": mk(nets["policy_net"]),
            "value_optimizer1": mk(nets["value_net1"]),
            "value_optimizer2": mk(nets["value_net2"])}


def ref_batch(recnn, inp, spec):
    batch = {"items": torch.from_numpy(inp["items"]), "ratings": torch.from_numpy(inp["ratings"]),
             "sizes": torch.from_numpy(inp["sizes"]), "users": torch.arange(len(inp["sizes"]))}
    return recnn.data.utils.batch_tensor_embeddings(
        batch, torch.from_numpy(inp["table"]), spec["frame"])


def run_update_case(recnn, case, algo, opt_kind):
    spec = C.CASES[case] if isinstance(case, str) else case      # a case name or a spec dict
    inp = C.make_inputs(spec, algo)
    nets = build_ref_nets(recnn, spec, inp, algo)
    opts = make_optimizers(opt_kind, nets, algo)
    batch = ref_batch(recnn, inp, spec)
    params = dict(C.DDPG_PARAMS if algo == "ddpg" else C.TD3_PARAMS)
    out = {"input_checksums": C.input_checksums(inp)}
    loss_keys = ("value", "policy") if algo == "ddpg" else ("value1", "value2", "policy")
    losses = {k: [] for k in loss_keys}
    writer = recnn.utils.misc.DummyWriter()
    for step in range(spec["steps"]):
        masks = inp["masks"][step]
        if algo == "ddpg":
            # drop_layer call order: value(2) -> policy(2) -> value(2)  (misc.py:37, ddpg.py:78-79)
            nets["value_net"].drop_layer.feed(masks[0:2] + masks[4:6])
            nets["policy_net"].drop_layer.feed(masks[2:4])
            loss = recnn.nn.update.ddpg_update(batch, params, nets, opts, torch.device("cpu"),
                                               {}, writer, learn=True, step=step)
        else:
            nets["value_net1"].drop_layer.feed(masks[0:2] + masks[6:8])   # td3.py:88,117
            nets["value_net2"].drop_layer.feed(masks[2:4])                # td3.py:89
            nets["policy_net"].drop_layer.feed(masks[4:6])                # td3.py:116
            # the noise draw is the first consumer of the CPU generator (td3.py:74)
            torch.manual_seed(9000 + step)
            probe = torch.normal(torch.zeros(spec["n_rows"], spec["dim"]), params["noise_std"])
            torch.manual_seed(9000 + step)
            out["noise.%d" % step] = probe.numpy().copy()
            loss = recnn.nn.update.td3_update(batch, params, nets, opts, torch.device("cpu"),
                                              {}, writer, learn=True, step=step)
        for m in nets.values():
            assert not m.drop_layer.queue, "mask queue not drained"
        for k in loss_keys:
            losses[k].append(loss[k])
        assert loss["step"] == step
        done_steps = step + 1
        if done_steps in SNAP_AFTER:
            for name, m in nets.items():
                for k, v in C.net_digest(_dump(m)).items():
                    out["after%d.%s.%s" % (done_steps, name, k)] = v
        if step == 0:
            for k, v in C.net_digest(_dump_grad(nets["policy_net"])).items():
                out["grad_step0.policy_net.%s" % k] = v
        if step == 1:
            crit = "value_net" if algo == "ddpg" else "value_net1"
            for k, v in C.net_digest(_dump_grad(nets[crit])).items():
                out["grad_step1.%s.%s" % (crit, k)] = v
    for k in loss_keys:
        out["loss." + k] = np.asarray(losses[k], dtype=np.float64)
    # initial-weight digests so tests can form deltas
    for name, p in inp["nets"].items():
        for k, v in C.net_digest(p).items():
            out["init.%s.%s" % (name, k)] = v
    # gate margin of this case (numpy oracle on the same inputs; see oracle/cases.py GATE_GUARD)
    from tests._golden import run_oracle_case
    O.reset_gate_margin()
    run_oracle_case(case, algo, opt_kind, golden=out if algo == "td3" else None)
    out["gate_margin"] = np.float64(O.GATE_MARGIN["min"])
    if case == "tiny":           # small enough to store every final tensor verbatim
        for name, m in nets.items():
            for k, v in _dump(m).items():
                out["final.%s.%s" % (name, k)] = v
    return out


def run_vs_reference_cases(recnn):
    """vs_reference.npz: the update cases of C.UNSCREENED_CASES (keys '<case>.<algo>.<opt>.*') and the gather on
    C.random_gather_users() ('gather.*'), both run by the reference.  Only what tests/test_oracle_vs_reference.py
    compares is kept: losses, input checksums, the gate margin, TD3's noise draws ('<case>.noise' [steps, rows,
    dim], the same for both optimizers) and the first C.UNSCREENED_SAMPLES entries of each weight sample (and of
    DDPG's gradient samples), concatenated in the order of 'sample_keys' with lengths 'sample_sizes'.  A case with
    an ambiguous ReLU gate, which the test skips, keeps its gate margin only."""
    out = {}
    for name, spec in C.UNSCREENED_CASES.items():
        for algo in ("ddpg", "td3"):
            for opt_kind in ("adam", "sgd"):
                got = run_update_case(recnn, spec, algo, opt_kind)
                pre = "%s.%s.%s." % (name, algo, opt_kind)
                out[pre + "gate_margin"] = got["gate_margin"]
                if float(got["gate_margin"]) <= C.GATE_GUARD:
                    continue
                for k in ["input_checksums"] + [k for k in got if k.startswith("loss.")]:
                    out[pre + k] = got[k]
                if algo == "td3":
                    out[name + ".noise"] = np.stack([got["noise.%d" % s] for s in range(spec["steps"])])
                keys = sorted(k for k in got if k.endswith(".sample") and (algo == "ddpg" or not k.startswith("grad_")))
                samples = [got[k][:C.UNSCREENED_SAMPLES] for k in keys]
                out[pre + "sample_keys"] = np.asarray(keys)
                out[pre + "sample_sizes"] = np.asarray([s.size for s in samples], dtype=np.int64)
                out[pre + "samples"] = np.concatenate(samples)
    table, users, frame = C.random_gather_users()
    ref = recnn.data.utils.prepare_batch_static_size(copy.deepcopy(users), torch.from_numpy(table), frame_size=frame)
    for k in ("state", "next_state", "action", "reward", "done"):
        out["gather." + k] = ref[k].numpy()
    return out


def run_gather_case(recnn):
    rng = np.random.default_rng(2024)
    frame = 10
    table = rng.standard_normal((300, 128), dtype=np.float32)
    users = []
    for uid, length in ((7, 14), (3, 11), (11, 20)):
        users.append({"items": rng.integers(0, 300, size=length, dtype=np.int64),
                      "rates": rng.integers(-4, 6, size=length).astype(np.float64),
                      "sizes": length, "users": uid})
    got = recnn.data.utils.prepare_batch_static_size(
        copy.deepcopy(users), torch.from_numpy(table), frame_size=frame)
    out = {"table": table, "frame_size": np.int64(frame)}
    for i, u in enumerate(users):
        out["user%d.items" % i] = u["items"]
        out["user%d.rates" % i] = u["rates"]
        out["user%d.id" % i] = np.int64(u["users"])
    for k in ("state", "next_state", "action", "reward", "done"):
        out["out." + k] = got[k].numpy()
    out["out.sizes"] = got["meta"]["sizes"].numpy()
    out["out.users"] = got["meta"]["users"].numpy()
    return out


COLLATE_LENGTHS = (11, 12, 30, 11, 57, 13, 100, 25, 11, 19, 64, 33, 12, 47)
COLLATE_MINIBATCH = (9, 0, 13, 4, 3, 6)      # positions in storage order, as a shuffling DataLoader would pick


def collate_case_users(frame=10, n_items=500):
    """Synthetic user histories of the collate fixture (shared with the tests through the stored arrays)."""
    rng = np.random.default_rng(77)
    users = []
    for pos, length in enumerate(COLLATE_LENGTHS):
        rates = 2.0 * (rng.integers(1, 11, size=length) / 2.0 - 2.5)          # ML-20M half stars -> 2(r-2.5)
        rates = rates + (rng.random(length) < 0.3) * rng.standard_normal(length) * 0.1   # some non-representable
        users.append({"items": rng.integers(0, n_items, size=length, dtype=np.int64),
                      "rates": rates.astype(np.float64), "sizes": length, "users": 1000 + 7 * pos})
    return users


def run_collate_case(recnn):
    frame = 10
    users = collate_case_users(frame)
    table = np.random.default_rng(78).standard_normal((500, 4), dtype=np.float32)
    ident = lambda batch, item_embeddings_tensor, frame_size: batch      # noqa: E731  (captures embed_batch's input)
    out = {"frame_size": np.int64(frame), "n_users": np.int64(len(users)),
           "minibatch": np.asarray(COLLATE_MINIBATCH, dtype=np.int64)}
    for i, u in enumerate(users):
        out["user%d.items" % i] = u["items"]
        out["user%d.rates" % i] = u["rates"]
        out["user%d.id" % i] = np.int64(u["users"])
    for tag, sel in (("all", list(range(len(users)))), ("mini", list(COLLATE_MINIBATCH))):
        picked = [copy.deepcopy(users[i]) for i in sel]
        got = recnn.data.utils.prepare_batch_static_size(copy.deepcopy(picked), torch.from_numpy(table),
                                                         frame_size=frame, embed_batch=ident)
        emb = recnn.data.utils.prepare_batch_static_size(copy.deepcopy(picked), torch.from_numpy(table),
                                                         frame_size=frame)
        out[tag + ".items"] = got["items"].numpy()
        out[tag + ".ratings"] = got["ratings"].numpy()
        out[tag + ".sizes"] = got["sizes"].numpy()
        out[tag + ".users"] = got["users"].numpy()
        out[tag + ".done"] = emb["done"].numpy()
        assert out[tag + ".ratings"].dtype == np.float32 and out[tag + ".items"].dtype == np.int64
    return out


def ingest_case_frames(n_users=24, n_items=60, dim=6, seed=5):
    """A small ML-20M-shaped ratings table (userId, movieId, rating, timestamp) and {movieId: embedding}:
    sparse non-contiguous movie ids, half-star ratings, unique timestamps (so the time order is unambiguous),
    users with 3..40 interactions (some at or below frame_size, which the ingest must drop)."""
    import pandas as pd
    rng = np.random.default_rng(seed)
    movie_ids = np.sort(rng.choice(np.arange(1, 5000), size=n_items, replace=False))
    emb = {int(m): torch.from_numpy(rng.standard_normal(dim).astype(np.float32)) for m in movie_ids}
    rows = []
    t = 1_000_000
    for u in range(n_users):
        uid = 10 + 13 * u
        n = int(rng.integers(3, 41))
        for _ in range(n):
            t += int(rng.integers(1, 1000))
            rows.append((uid, int(rng.choice(movie_ids)), float(rng.integers(1, 11)) / 2.0, t))
    order = rng.permutation(len(rows))                       # the CSV is not time-sorted
    df = pd.DataFrame([rows[i] for i in order], columns=["userId", "movieId", "rating", "timestamp"])
    return df, emb


def run_ingest_case(recnn):
    """recnn.data.dataset_functions.prepare_dataset (the ingest behind Env.process_env, recnn/data/env.py:133-176)
    on the synthetic table: which users survive, in which order, and their time-ordered item-row / rating arrays."""
    frame = 10
    df, emb = ingest_case_frames()
    table, key_to_id, id_to_key = recnn.data.utils.make_items_tensor(emb)
    base = recnn.data.env.EnvBase()
    base.embeddings, base.key_to_id, base.id_to_key = table, key_to_id, id_to_key
    dset = recnn.data.dataset_functions
    args = dset.DataFuncArgsMut(df=df.copy(), base=base, users=None, user_dict=None)
    dset.prepare_dataset(args, dset.DataFuncKwargs(frame_size=frame))
    out = {"frame_size": np.int64(frame), "table": table.numpy(), "users": np.asarray(list(args.users), dtype=np.int64),
           "keys": np.asarray(sorted(emb), dtype=np.int64), "all_users": np.asarray(sorted(args.user_dict), dtype=np.int64)}
    for col in ("userId", "movieId", "rating", "timestamp"):                # the input table itself
        out["csv." + col] = df[col].to_numpy()
    out["emb"] = np.stack([emb[k].numpy() for k in sorted(emb)])
    for u in args.user_dict:
        out["u%d.items" % u] = np.asarray(args.user_dict[u]["items"])
        out["u%d.ratings" % u] = np.asarray(args.user_dict[u]["ratings"])
    sorted_users = recnn.data.utils.sort_users_itemwise(args.user_dict, list(args.users))
    out["sorted_users"] = np.asarray(list(sorted_users), dtype=np.int64)
    return out


def main():
    torch.set_num_threads(max(1, min(8, os.cpu_count() or 1)))
    recnn = import_reference()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    only = set(sys.argv[1:])
    if not only or "ingest" in only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "ingest.npz"), **run_ingest_case(recnn))
        print("wrote ingest.npz")
    if not only or "collate" in only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "collate.npz"), **run_collate_case(recnn))
        print("wrote collate.npz")
    if not only or "vs_reference" in only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "vs_reference.npz"), **run_vs_reference_cases(recnn))
        print("wrote vs_reference.npz")
    if only and "gather" not in only and "update" not in only:
        return
    if not only or "gather" in only:
        np.savez_compressed(os.path.join(GOLDEN_DIR, "gather.npz"), **run_gather_case(recnn))
        print("wrote gather.npz")
    if only and "update" not in only:
        return
    for case in C.CASES:
        for algo in ("ddpg", "td3"):
            for opt_kind in ("adam", "sgd"):
                out = run_update_case(recnn, case, algo, opt_kind)
                name = "%s_%s_%s.npz" % (algo, case, opt_kind)
                np.savez_compressed(os.path.join(GOLDEN_DIR, name), **out)
                print("wrote", name, {k: [round(x, 6) for x in v[:3]] for k, v in
                                      ((kk, out[kk]) for kk in out if kk.startswith("loss."))})


if __name__ == "__main__":
    main()
