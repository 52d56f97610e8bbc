"""Host-side driver of the fused device step (one instance per set of nets).

Responsibilities (all plumbing; the arithmetic is in recnn_b200/csrc):
  * validate / (re)build the flat parameter, gradient and optimizer arenas;
  * stage the batch into fixed device buffers (one async copy per tensor) so the
    step is replayable as a CUDA graph;
  * run the phase schedule of the update (``schedule``): which phase masks go to the C
    side, and which all-reduces / external ``optimizer.step()`` calls run between them;
  * read the 3-4 loss scalars back (the only synchronisation of a step -- the
    reference API returns Python floats, recnn/nn/update/ddpg.py:102).
"""
from __future__ import annotations

import os
import warnings
from typing import NamedTuple

import torch

from ... import _lib
from ... import optim as _optim
from ..arena import param_arena, grad_arena

_USE_GRAPHS = os.environ.get("RECNN_B200_GRAPHS", "1") != "0"
_MAX_GRAPH_KEYS = 16            # bound of the graph cache (first sightings included)
MASK_KEY = "dropout_masks"      # optional batch entries for bit-reproducible runs
NOISE_KEY = "noise"

DDPG_NETS = ("value_net", "target_value_net", "policy_net", "target_policy_net")
TD3_NETS = ("value_net1", "target_value_net1", "value_net2", "target_value_net2", "policy_net",
            "target_policy_net")

# Host actions that run between two C calls of a step, on the step's stream.
ALLREDUCE_VALUE_GRADS = "allreduce_value_grads"
ALLREDUCE_POLICY_GRADS = "allreduce_policy_grads"
ALLREDUCE_LOSSES = "allreduce_losses"
STEP_VALUE_OPTIMIZERS = "step_value_optimizers"
STEP_POLICY_OPTIMIZER = "step_policy_optimizer"


class Schedule(NamedTuple):
    segments: tuple     # ((phase mask, (host action, ...)), ...): C calls in order, each followed by its host actions
    capturable: bool    # may run as one CUDA graph per segment (the host actions stay between the replays)


def schedule(value_only, learn, do_policy, value_builtin, policy_builtin, debug, world, peer_comm) -> Schedule:
    """The C calls of one update and the host work between them (the same for DDPG and TD3: the host actions
    on the value gradients / optimizers cover both of TD3's critics).

    A learning step whose optimizers are all built in runs fused: one call with every phase, its gradient
    exchange inside the kernels when there is one GPU or a peer communicator; with NCCL it is cut into three
    calls where the critic and then the actor gradients are complete.  Only these fused steps are captured
    into CUDA graphs.  Anything else -- an external optimizer, learn=False (debug outputs), the critic-only
    ``value_only`` step -- runs phase by phase with direct launches: a built-in optimizer is the C side's
    optimizer phase, an external one is stepped in Python, and with several ranks the gradients and the loss
    scalars go through NCCL between the calls."""
    P = _lib
    if learn and not value_only and not debug and value_builtin and policy_builtin:
        if world == 1 or peer_comm:
            return Schedule(((P.PH_ALL, ()),), True)
        grads = (ALLREDUCE_POLICY_GRADS,) if do_policy else ()
        return Schedule(((P.PH_GATHER | P.PH_VALUE_GRAD, (ALLREDUCE_VALUE_GRADS,)),
                         (P.PH_VALUE_OPT | P.PH_POLICY_LOSS | P.PH_POLICY_GRAD, grads + (ALLREDUCE_LOSSES,)),
                         (P.PH_POLICY_OPT | P.PH_SOFT_UPDATE | P.PH_FINISH, ())), True)
    dp = world > 1
    segs = []

    def call(phases):
        segs.append((phases, []))

    def then(action):
        segs[-1][1].append(action)

    call(P.PH_GATHER | P.PH_VALUE_GRAD)
    if learn:
        if dp:
            then(ALLREDUCE_VALUE_GRADS)
        if value_builtin:
            call(P.PH_VALUE_OPT)
        else:
            then(STEP_VALUE_OPTIMIZERS)
    if not value_only:
        call(P.PH_POLICY_LOSS)
        if do_policy:
            call(P.PH_POLICY_GRAD)
            if dp:
                then(ALLREDUCE_POLICY_GRADS)
            # clip coefficient (+ the fused optimizer when the policy optimizer is built in; for an
            # external one the C side only scales the gradient in place)
            call(P.PH_POLICY_OPT)
            if not policy_builtin:
                then(STEP_POLICY_OPTIMIZER)
            call(P.PH_SOFT_UPDATE)
    if dp:
        then(ALLREDUCE_LOSSES)
    call(P.PH_FINISH)                    # ++rng_step, losses -> pinned host
    return Schedule(tuple((ph, tuple(acts)) for ph, acts in segs), False)


class StepEngine:
    def __init__(self, algo, nets, device):
        self.algo = algo
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.RecnnError("recnn_b200 update functions run on CUDA only (device=%s); there is no CPU path"
                                  % self.device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.names = DDPG_NETS if algo == _lib.ALGO_DDPG else TD3_NETS
        for k in self.names:
            if k not in nets:
                raise KeyError(k)
        self.policy = nets["policy_net"]
        pol = self.policy            # any module with linear1/2/3 works (also the reference's own classes)
        crit = nets[self.names[0]]
        # REINFORCE (recnn/nn/update/reinforce.py:92-102): the policy is a two-layer DiscreteActor whose probabilities
        # are the critic's "action"; only the critic half of the step runs here, fed with the target policy's output
        self.discrete = not hasattr(pol, "linear3")
        if self.discrete:
            if algo != _lib.ALGO_DDPG:
                raise ValueError("a DiscreteActor policy only goes with the DDPG-style critic step (value_update)")
            self.dims = _lib.Dims(pol.linear1.in_features, pol.linear2.out_features, crit.linear1.out_features, 0)
        else:
            self.dims = _lib.Dims(pol.linear1.in_features, pol.linear3.out_features, pol.linear1.out_features, 0)
        if (crit.linear1.in_features != self.dims.state_dim + self.dims.action_dim
                or crit.linear1.out_features != self.dims.hidden or crit.linear3.out_features != 1):
            raise ValueError("critic shape does not match the actor (expects input state_dim+action_dim, same hidden, 1 output)")
        self.n_rows = -1
        self.form = None
        self.graphs = {}             # bytes(StepArgs) -> None once run directly, then [(CUDAGraph, kernels)] per segment
        self._fast = {}              # (value_only, do_policy, form, n) -> (tokens, StepArgs, Schedule, graphs)
        self.group = None            # torch.distributed process group for data parallel
        self.world = 1
        self.comm = None             # recnn_b200.dist.PeerComm: in-kernel all-reduce over NVLink peer memory
        self.seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFFFFFF
        # value(1), value2, policy, ||actor grad||_1, error bits (int32), 3 spare  (include/recnn_b200.h: losses)
        self.losses = torch.zeros(8, dtype=torch.float32, device=self.device)
        self.losses_host = torch.zeros(8, dtype=torch.float32).pin_memory()
        self._flags_host = self.losses_host.view(torch.int32)
        self.rng_step = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.buf = {}
        self._probes = {}            # net name -> (module, first parameter, last parameter): see _tokens
        self._params_seen, self._params_version = None, 0
        self.kernels = 0             # kernels of this library launched by this engine (graph replays included)

    def set_data_parallel(self, group, world, comm):
        """Exchange gradients and losses over ``group`` (``world`` ranks), in the step's kernels through the
        peer communicator ``comm`` or, when it is None, with NCCL between the step's phases."""
        self.group, self.world, self.comm = group, world, comm
        self._invalidate()

    # ------------------------------------------------------------------ staging
    def _invalidate(self):
        """Drop everything that baked device addresses or the schedule in: the graph cache (first sightings
        included) and the fast-path table.  Called whenever a staging buffer or the workspace is (re)allocated,
        the batch shape changes, or data parallelism is (re)configured -- a stale graph would run against freed
        memory."""
        self.graphs.clear()
        self._fast.clear()

    def _buffer(self, name, shape, dtype):
        b = self.buf.get(name)
        if b is None or tuple(b.shape) != tuple(shape) or b.dtype != dtype:
            b = torch.empty(shape, dtype=dtype, device=self.device)
            self.buf[name] = b
            self._invalidate()
        return b

    def _stage(self, name, src, dtype, shape=None):
        if not torch.is_tensor(src):
            src = torch.as_tensor(src)
        if src.requires_grad:
            src = src.detach()
        if shape is not None and tuple(src.shape) != tuple(shape):
            src = src.reshape(shape)
        dst = self.buf.get(name)
        if dst is None or dst.shape != src.shape or dst.dtype != dtype:
            dst = self._buffer(name, src.shape, dtype)
        dst.copy_(src, non_blocking=True)
        return dst

    def _stage_batch(self, batch):
        d = self.dims
        if "items" in batch and batch.get("table") is not None:
            form = "frames"
            items = batch["items"]
            n = int(items.shape[0])
            table = batch["table"]
            if table.device != self.device or table.dtype != torch.float32 or not table.is_contiguous():
                raise _lib.RecnnError("batch['table'] must be a contiguous fp32 tensor on %s" % self.device)
            frame = int(items.shape[1]) - 1
            emb = int(table.shape[1])
            if frame * emb + frame != d.state_dim or emb != d.action_dim:
                raise ValueError("frame batch (frame=%d, dim=%d) does not match the nets (state_dim=%d, action_dim=%d)"
                                 % (frame, emb, d.state_dim, d.action_dim))
            st = dict(form=form, n=n, table=table, frame=frame, emb=emb,
                      items=self._stage("items", items, torch.int64),
                      ratings=self._stage("ratings", batch["ratings"], torch.float32))
            if batch.get("done") is not None:
                st["done"] = self._stage("done", batch["done"], torch.float32, (n,))
            else:
                sizes = self._stage("sizes", batch["sizes"], torch.int64)
                done = self._buffer("done", (n,), torch.float32)
                _lib.check(_lib.lib().recnn_done_from_sizes(sizes.data_ptr(), sizes.numel(), frame, done.data_ptr(),
                                                            n, _lib.stream_ptr(self.device)))
                st["done"] = done
            st["reward"] = (self._stage("reward", batch["reward"], torch.float32, (n,))
                            if batch.get("reward") is not None else None)
        else:
            form = "dense"
            n = int(batch["state"].shape[0])
            st = dict(form=form, n=n,
                      state=self._stage("state", batch["state"], torch.float32),
                      next_state=self._stage("next_state", batch["next_state"], torch.float32),
                      action=self._stage("action", batch["action"], torch.float32),
                      reward=self._stage("reward", batch["reward"], torch.float32, (n,)),
                      done=self._stage("done", batch["done"], torch.float32, (n,)))
            if st["state"].shape[1] != d.state_dim or st["action"].shape[1] != d.action_dim:
                raise ValueError("batch shapes do not match the nets")
        n_masks = 6 if self.algo == _lib.ALGO_DDPG else 8
        masks = batch.get(MASK_KEY)
        if masks is not None:
            if len(masks) != n_masks:
                raise ValueError("%s needs %d masks" % (MASK_KEY, n_masks))
            st["masks"] = [self._stage("mask%d" % i, m, torch.uint8, (n, d.hidden)) for i, m in enumerate(masks)]
        else:
            st["masks"] = None
        noise = batch.get(NOISE_KEY) if self.algo == _lib.ALGO_TD3 else None
        st["noise"] = self._stage("noise", noise, torch.float32, (n, d.action_dim)) if noise is not None else None
        # data parallel: the loss means and gradient scales use the GLOBAL row count.  Equal shards are
        # assumed (n * world) unless the caller says otherwise (uneven shards, e.g. dist.shard_rows of a batch
        # that does not divide by the world size, must pass batch["n_rows_global"]).
        st["n_global"] = int(batch["n_rows_global"]) if batch.get("n_rows_global") is not None else n * self.world
        if st["n_global"] < n:
            raise ValueError("batch['n_rows_global'] (%d) is smaller than this rank's row count (%d)" % (st["n_global"], n))
        if n != self.n_rows or form != self.form:
            self.n_rows, self.form = n, form
            self._invalidate()
        return st

    # ------------------------------------------------------------------ arenas / args
    def _c_net(self, module, opt, with_grads):
        flat = param_arena(module)
        if flat.device != self.device:
            raise _lib.RecnnError("net is on %s but the update runs on %s (call Algo.to(device) / net.cuda())"
                                  % (flat.device, self.device))
        if not with_grads:
            return _lib.Net(flat.data_ptr(), None, None, None, None, None)
        if isinstance(opt, _optim._ArenaOptimizer):
            if opt._module is not module:
                opt.bind(module)
            return opt.c_net(module)
        g = grad_arena(module)
        return _lib.Net(flat.data_ptr(), g.data_ptr(), None, None, None, None)

    @staticmethod
    def _c_optim(opt):
        if isinstance(opt, _optim._ArenaOptimizer):
            return opt.c_optim()
        return _lib.Optim(_lib.OPT_EXTERNAL, 0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0)

    def _build_args(self, st, nets, optimizer, params, learn, do_policy):
        a = _lib.StepArgs()
        a.algo = self.algo
        a.learn = int(bool(learn))
        a.do_policy_step = int(bool(do_policy))
        a.dims = self.dims
        a.n_rows = st["n"]
        a.n_rows_global = st["n_global"]
        if st["form"] == "frames":
            a.table = st["table"].data_ptr()
            a.n_items = int(st["table"].shape[0])
            a.frame = st["frame"]
            a.emb_dim = st["emb"]
            a.items = st["items"].data_ptr()
            a.ratings = st["ratings"].data_ptr()
        else:
            a.state = st["state"].data_ptr()
            a.next_state = st["next_state"].data_ptr()
            a.action = st["action"].data_ptr()
        a.reward = _lib.ptr(st["reward"])
        a.done = st["done"].data_ptr()
        td3 = self.algo == _lib.ALGO_TD3
        pol_opt = optimizer.get("policy_optimizer") if learn else None
        if self.discrete:
            pol_opt = None           # the step never touches the DiscreteActor: next_action_in replaces its forward
            a.next_action_in = st["next_action"].data_ptr()
        else:
            a.policy = self._c_net(nets["policy_net"], pol_opt, learn)
            a.target_policy = self._c_net(nets["target_policy_net"], None, False)
        a.policy_optim = self._c_optim(pol_opt)
        val_opts = []
        for i in range(2 if td3 else 1):
            sfx = str(i + 1) if td3 else ""
            vo = optimizer.get("value_optimizer" + sfx) if learn else None
            val_opts.append(vo)
            a.value[i] = self._c_net(nets["value_net" + sfx], vo, learn)
            a.target_value[i] = self._c_net(nets["target_value_net" + sfx], None, False)
        kinds = {type(v) for v in val_opts}
        a.value_optim = self._c_optim(val_opts[0])
        if td3 and isinstance(val_opts[0], _optim._ArenaOptimizer):
            o0, o1 = val_opts[0].c_optim(), (val_opts[1].c_optim() if isinstance(val_opts[1], _optim._ArenaOptimizer) else None)
            same = o1 is not None and all(getattr(o0, f) == getattr(o1, f) for f, _ in _lib.Optim._fields_)
            if len(kinds) != 1 or not same:
                raise ValueError("the two TD3 value optimizers must be the same built-in optimizer with equal hyper-parameters")
        a.gamma = float(params["gamma"])
        if not td3:
            a.min_value = float(params["min_value"])
            a.max_value = float(params["max_value"])
        else:
            a.noise_std = float(params["noise_std"])
            a.noise_clip = float(params["noise_clip"])
        a.soft_tau = float(params["soft_tau"])
        online = [nets[k] for k in self.names if not k.startswith("target") and not (self.discrete and k == "policy_net")]
        if len({bool(m.training) for m in online}) != 1:
            raise ValueError("the online nets must all be in the same mode (train() / eval()): dropout is applied "
                             "to every online net or to none; the target nets always run in eval mode")
        a.dropout = int(bool(online[-1].training))
        if st["masks"] is not None:
            for i, m in enumerate(st["masks"]):
                a.masks[i] = m.data_ptr()
        a.noise = _lib.ptr(st["noise"])
        a.seed = self.seed
        a.rng_step = self.rng_step.data_ptr()
        a.losses = self.losses.data_ptr()
        a.losses_host = self.losses_host.data_ptr()
        nbytes = _lib.lib().recnn_step_workspace_bytes(self.dims, st["n"], self.algo)
        ws = self.buf.get("workspace")
        if ws is None or ws.numel() < nbytes:
            ws = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            self.buf["workspace"] = ws
            self._invalidate()
        a.workspace = ws.data_ptr()
        a.workspace_bytes = ws.numel()
        return a, pol_opt, val_opts

    def _launch(self, a, phases):
        """One C call of the step on the current stream; returns the number of kernels it launched."""
        a.phases = phases
        L = _lib.lib()
        fn = L.recnn_ddpg_step if self.algo == _lib.ALGO_DDPG else L.recnn_td3_step
        before = L.recnn_b200_launch_count()
        _lib.check(fn(a, _lib.stream_ptr(self.device)))
        return L.recnn_b200_launch_count() - before

    def _allreduce(self, t):
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def _host_action(self, action, nets, pol_opt, val_opts):
        value_nets = [nets[k] for k in self.names if k.startswith("value_net")]
        if action == ALLREDUCE_VALUE_GRADS:
            for vn in value_nets:
                self._allreduce(grad_arena(vn))
        elif action == ALLREDUCE_POLICY_GRADS:
            self._allreduce(grad_arena(nets["policy_net"]))
        elif action == ALLREDUCE_LOSSES:
            self._allreduce(self.losses[:3])
        elif action == STEP_VALUE_OPTIMIZERS:
            for vn, vo in zip(value_nets, val_opts):
                grad_arena(vn)          # re-attach p.grad views if zero_grad(set_to_none) dropped them
                vo.step()
        else:
            assert action == STEP_POLICY_OPTIMIZER, action
            grad_arena(nets["policy_net"])
            pol_opt.step()

    def _graphs(self, a, sched):
        """The CUDA graphs of a capturable schedule with these arguments: None the first time they are seen
        (direct launches, which also warm lazy module loading) or when capture fails, captured the second time.
        Keyed by the arguments' bytes, i.e. every pointer and scalar the graphs bake in."""
        a.phases = 0
        key = bytes(a)
        if key not in self.graphs:
            if len(self.graphs) >= _MAX_GRAPH_KEYS:     # e.g. hyper-parameters that change every step
                self._invalidate()
            self.graphs[key] = None
            return None
        graphs = self.graphs[key]
        if graphs is None:
            try:
                torch.cuda.synchronize(self.device)
                graphs = []
                for phases, _ in sched.segments:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        n = self._launch(a, phases)
                    graphs.append((g, n))
            except Exception as exc:      # capture unsupported in this context: stay on direct launches
                warnings.warn("recnn_b200: CUDA graph capture failed (%s); using direct launches" % exc)
                globals()["_USE_GRAPHS"] = False
                return None
            self.graphs[key] = graphs
        return graphs

    def _run(self, a, sched, nets, pol_opt=None, val_opts=None, graphs=None):
        """Every segment of the schedule -- a graph replay or a direct C call -- followed by its host actions.
        Returns the graphs used (None: direct launches)."""
        if graphs is None and sched.capturable and _USE_GRAPHS:
            graphs = self._graphs(a, sched)
        for i, (phases, actions) in enumerate(sched.segments):
            if graphs is not None:
                g, n = graphs[i]
                g.replay()
            else:
                n = self._launch(a, phases)
            self.kernels += n
            for act in actions:
                self._host_action(act, nets, pol_opt, val_opts)
        return graphs

    def _read_losses(self):
        """After the stream synchronisation of a step: the loss scalars, or the step's error."""
        bits = int(self._flags_host[4])
        if bits & 1:
            raise IndexError("batch['items'] holds an item id outside [0, n_items) (the update was applied with the "
                             "offending rows reading table row 0)")
        if bits & 2:
            raise _lib.RecnnError("data parallel: the ranks disagree on the global row count; pass "
                                  "batch['n_rows_global'] when the shards are uneven")
        return self.losses_host[:4].tolist()

    def _tokens(self, nets, optimizer, params, st):
        """Cheap fingerprint of everything a cached StepArgs / CUDA graph depends on: storage addresses of the nets
        (first and last parameter, gradient), optimizer hyper-parameters and state arenas, the algorithm's scalars
        and the staged batch buffers.  This runs on every step between the batch copies and the graph launch, i.e.
        while the GPU idles, so it avoids nn.Module attribute lookups (the Parameter objects are cached per net) and
        compares the params dict with one C-level dict comparison."""
        tok = []
        probes = self._probes
        for name in self.names:
            m = nets[name]
            pr = probes.get(name)
            if pr is None or pr[0] is not m:
                pr = probes[name] = (m, m.linear1.weight, m.linear3.bias if hasattr(m, "linear3") else m.linear2.bias)
            w, b = pr[1], pr[2]
            g = w.grad
            tok.append((w.data_ptr(), b.data_ptr(), 0 if g is None else g.data_ptr(), m.training))
        for k in optimizer:
            o = optimizer[k]
            if isinstance(o, _optim._ArenaOptimizer):
                g = o.param_groups[0]
                tok.append((k, id(o), g["lr"], g.get("betas"), g.get("eps"), g["weight_decay"], g.get("momentum"),
                            g.get("alpha"), g.get("k"), g.get("N_sma_threshhold"),
                            0 if o._m is None else o._m.data_ptr(), 0 if o._t is None else o._t.data_ptr()))
            else:
                tok.append((k, id(o)))
        if self._params_seen is None or self._params_seen != params:
            self._params_seen = dict(params)
            self._params_version += 1
        tok.append(self._params_version)
        for k in ("table", "items", "ratings", "state", "next_state", "action", "reward", "done", "noise"):
            t = st.get(k)
            tok.append(0 if t is None else t.data_ptr())
        if st["masks"] is not None:
            tok.append(tuple(m.data_ptr() for m in st["masks"]))
        ws = self.buf.get("workspace")
        tok.append((0 if ws is None else ws.data_ptr(), st["n_global"], self.world,
                    0 if self.comm is None else self.comm.ptr))
        return tok

    # ------------------------------------------------------------------ the step
    def step(self, batch, params, nets, optimizer, learn, step, debug, policy_every_key):
        """One DDPG / TD3 update (recnn/nn/update/ddpg.py, td3.py)."""
        do_policy = bool(learn and step % params[policy_every_key] == 0)
        with torch.cuda.device(self.device):
            return self._update(batch, params, nets, optimizer, learn, do_policy, debug, False)

    def value_only(self, batch, params, nets, optimizer, learn, debug):
        """recnn/nn/update/misc.py:10-55 on its own: critic step without the policy half."""
        with torch.cuda.device(self.device):
            return self._update(batch, params, nets, optimizer, learn, False, debug, True)

    def _update(self, batch, params, nets, optimizer, learn, do_policy, debug, value_only):
        st = self._stage_batch(batch)
        if value_only and self.discrete:
            # next_action = target_policy_net(next_state)   (misc.py:28 with a DiscreteActor: probabilities)
            st["next_action"] = self._stage("next_action", nets["target_policy_net"](st["next_state"]), torch.float32)
        # ---- fast path: same variant as a previous step -> replay its graphs
        vkey = (value_only, do_policy, st["form"], st["n"])
        ent = self._fast.get(vkey) if learn and _USE_GRAPHS else None
        if ent is not None and ent[0] == self._tokens(nets, optimizer, params, st):
            self._run(ent[1], ent[2], nets, graphs=ent[3])
            torch.cuda.current_stream(self.device).synchronize()
            return self._read_losses()
        a, pol_opt, val_opts = self._build_args(st, nets, optimizer, params, learn, do_policy)
        want_debug = None
        if not learn:
            n, A = st["n"], self.dims.action_dim
            want_debug = {k: torch.empty(n, A, device=self.device)
                          for k in (("next_action",) if value_only else ("next_action", "gen_action"))}
            a.next_action_out = _lib.ptr(want_debug.get("next_action"))
            a.gen_action_out = _lib.ptr(want_debug.get("gen_action"))
        sched = schedule(value_only, learn, do_policy, isinstance(val_opts[0], _optim._ArenaOptimizer),
                         isinstance(pol_opt, _optim._ArenaOptimizer), want_debug is not None, self.world,
                         self.comm is not None)
        if sched.capturable and self.comm is not None:
            a.comm = self.comm.ptr        # the fused step all-reduces in its kernels
        graphs = self._run(a, sched, nets, pol_opt, val_opts)
        if graphs is not None:
            # arenas may have been (re)built by _build_args: fingerprint after the fact
            self._fast[vkey] = (self._tokens(nets, optimizer, params, st), a, sched, graphs)
        torch.cuda.current_stream(self.device).synchronize()
        vals = self._read_losses()
        for k, t in (want_debug or {}).items():
            debug[k] = t                  # debug=None fails like the reference (misc.py:47)
        return vals


def get_engine(algo, nets, device) -> StepEngine:
    """Engines are cached on the policy net (they own graphs and staging buffers)."""
    policy = nets["policy_net"]
    cache = policy.__dict__.setdefault("_recnn_engines", {})
    dev = torch.device(device)
    key = (algo, dev.type, dev.index)
    eng = cache.get(key)
    if eng is None:
        eng = StepEngine(algo, nets, dev)
        dp = policy.__dict__.get("_recnn_dp")
        if dp is not None:
            eng.set_data_parallel(*dp)
        cache[key] = eng
    return eng
