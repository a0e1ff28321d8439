"""Generic (any-model) round executor of the device engine.

Same plan semantics as the fused ``fed_round_small`` kernel (W-pool / time-weighted / index-list batch selection with
the same counter-based RNG, per-pair optimizer state that persists across rounds, per-cluster weighted aggregation,
train/test evaluation with optional ensembles) but built from separate native kernels so it works for every
architecture and for algorithms that must look at raw client updates before aggregating (CFL):

* local step: LSTM federations → ``sim/lstm_exec.py`` (all pairs per launch on the persistent LSTM kernels); stackable conv
  nets → ``sim/stacked.py`` (all pairs in one channel-stacked network on the grouped implicit-GEMM kernels); everything else
  per pair: bank-bound ``nn.Module`` forward/backward (TcLinear → tcgen05 GEMM, TcConv2d → implicit-GEMM convolution),
  gradients land in a flat scratch row, ``ops.adam_amsgrad_rows_`` / ``ops.sgd_rows_`` update the client row;
* aggregation: ``ops.cluster_aggregate_`` over the ``[C, M, P]`` client arena (K1);
* evaluation: clients are grouped by the model they are scored with → one batched forward per (model, split), per-client
  sums by masked reduction on device, ONE host copy per block of rounds.

The per-(client, model) local step is launch-bound for every architecture in the zoo at federated batch sizes (a CNN
step is ~60 small kernels), so on CUDA it is captured ONCE into a CUDA graph over static buffers (``_GraphedStep``:
parameters, optimizer moments, gradient row, batch) and replayed for every pair and step; gradients accumulate directly
into a flat row because each parameter's ``.grad`` is a view of it (no per-tensor gather).  ``FDB_NO_GRAPHS=1`` or a
failed capture falls back to eager execution of the same ops.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

from .. import ops
from ..ops.reference import batch_hash, mix32


def _pair_sampler(st: Dict, c: int, m: int, t: int, nb: torch.Tensor, B: int):
    """(n_cm, sampler(h1) -> index tensor into the flattened [T1*S] sample axis of client c)."""
    from ..ops.reference import _pair_plan
    return _pair_plan(st, c, m, t, nb, B)


def run_rounds_generic(sim, rounds: int) -> Dict[str, torch.Tensor]:
    a, bank, data = sim.args, sim.bank, sim.data
    dev = sim.device
    plan = sim.current_plan()
    t, C, M, P = sim.t, sim.C, sim.M, bank.P
    T1, S = data.steps, data.X.shape[2]
    B, E = a.batch_size, a.epochs
    W = plan["W"]
    nsamp_h = sim.data_host.nsamp
    nb = (nsamp_h.to(torch.int64) + B - 1) // B
    st = {"W": W.cpu(), "nsamp": nsamp_h, "X": sim.data_host.X, "sample_mode": plan.get("sample_mode", "pool"),
          "n_mode": plan.get("n_mode", "batches"), "train_index": _cpu(plan.get("train_index")),
          "train_count": _cpu(plan.get("train_count"))}
    use_adam = plan.get("optimizer", "sgd" if a.client_optimizer == "sgd" else "adam") != "sgd"
    lr = float(plan.get("lr", a.lr))
    seed = int(a.dummy_arg) * 7919 + 13 + 1000003 * t
    feat_mask = plan.get("feat_mask")
    ens_mode = int(plan.get("ens_mode", 0) or 0)
    metrics = torch.zeros(rounds, C, 4, dtype=torch.float32, device=dev)
    cl = sim.clients
    Xc_all = data.X.reshape(T1, C, S, *data.X.shape[3:])
    for r in range(rounds):
        rnd = sim.round_in_step + r
        Wt = st["W"][t]
        active = (st["train_count"] > 0).any(dim=1) if st["sample_mode"] == "index" else (Wt != 0).any(dim=1)
        cl.n.zero_()
        world, rank = _world_rank(sim)
        from . import lstm_exec, stacked
        lstm_b = lstm_exec.applicable(sim, feat_mask)    # LSTM federations: all pairs advance in the same few launches
        stack_b = not lstm_b and stacked.applicable(sim, feat_mask)   # conv nets: all pairs in one channel-stacked network
        batched = lstm_b or stack_b
        bpairs, n_host = [], np.zeros((C, M), dtype=np.float32)
        slots = [] if batched else _stream_slots(sim)    # K side streams: independent (client, model) pairs replay concurrently
        pair_i = 0
        # worker slot s trains client sampled[s] in arena row s (slot == client under full participation)
        sampled = sim.participants(rnd)
        for s, c in enumerate(sampled):
            if world > 1 and c % world != rank:   # clients are sharded over the ranks (one process per GPU)
                continue
            xy = _lazy_client_xy(Xc_all, data, c, T1, S)
            for m in range(M):
                if not bool(active[m]):
                    continue
                n_cm, sampler = _pair_sampler(st, c, m, t, nb, B)
                if n_cm <= 0:
                    continue
                if batched:
                    bpairs.append((s, c, m, sampler))
                    n_host[s, m] = n_cm
                    continue
                if slots:
                    with torch.cuda.stream(slots[pair_i % len(slots)]):
                        cl.params[s, m].copy_(bank.theta[m])
                        _local_steps(sim, c, m, xy, sampler, seed, rnd, E, use_adam, lr, a.wd, feat_mask, pair_i % len(slots), s=s)
                else:
                    cl.params[s, m].copy_(bank.theta[m])
                    _local_steps(sim, c, m, xy, sampler, seed, rnd, E, use_adam, lr, a.wd, feat_mask, s=s)
                pair_i += 1
                cl.n[s, m] = n_cm
        _join_slots(sim, slots)
        if batched:
            if lstm_b:
                lstm_exec.train_pairs(sim, bpairs, seed, rnd, E, use_adam, lr, a.wd)
            elif not stacked.train_pairs(sim, bpairs, seed, rnd, E, use_adam, lr, a.wd):
                for (s, c, m, sampler) in bpairs:         # unequal batch sizes: the per-pair path
                    cl.params[s, m].copy_(bank.theta[m])
                    _local_steps(sim, c, m, _lazy_client_xy(Xc_all, data, c, T1, S), sampler, seed, rnd, E, use_adam, lr, a.wd, feat_mask,
                                 s=s)
            cl.n.copy_(torch.from_numpy(n_host), non_blocking=True)
        # the raw-update hooks address W columns by client id: they get the slot → client list under partial participation
        uploaded = None if sim.participants_table is None else sampled
        # raw-update hooks (CFL family) may veto the aggregation of this round
        skip = False
        wants_raw = (hasattr(sim.algo, "state") and "cfl" in getattr(sim.algo, "arg", "")) or \
            (hasattr(sim.algo, "on_client_updates") and not sim.algo.split_done and rnd == sim.algo.split_round)
        if world > 1 and wants_raw:
            # every rank trained only its own clients, but the split decision (norms, cosine bipartition, slot allocation)
            # must be taken on ALL updates and identically everywhere: complete the arena first (cold path, NCCL)
            import torch.distributed as dist
            others = [c for c in range(C) if c % world != rank]
            if others:
                cl.params[others] = 0
                cl.n[others] = 0
            dist.all_reduce(cl.params)
            dist.all_reduce(cl.n)
        if hasattr(sim.algo, "state") and "cfl" in getattr(sim.algo, "arg", ""):
            skip = sim.algo.state.cluster_cfl(t, rnd + 1, bank, cl.params, cl.n, clients=uploaded)
            if skip:
                plan["W"] = sim.algo.state.weights_tensor(t)
                st["W"] = plan["W"].cpu()
        if hasattr(sim.algo, "on_client_updates") and not sim.algo.split_done and rnd == sim.algo.split_round:
            sim.algo.on_client_updates(t, cl.params, cl.n, clients=uploaded)
        if not skip:
            if world > 1:
                _peer_aggregate(sim, world, rank)
            else:
                ops.cluster_aggregate_(bank.theta, cl.params, cl.n)
        if plan.get("recluster_hard"):
            acc = sim.evaluator.acc_matrix(list(range(M)), t)
            best = np.argmax(acc, axis=0)
            st["W"][t].zero_()
            st["W"][t][torch.from_numpy(best), torch.arange(C)] = 1.0
            st.pop("_np", None)   # the host numpy mirror of W used by the pair planner is stale
            plan["W"] = st["W"].clone()
            sim.algo.absorb_weights(t, st["W"])
        _evaluate(sim, plan, st, r, metrics, ens_mode)
    if _world_rank(sim)[0] > 1:   # cold path: every rank evaluated only its own clients
        import torch.distributed as dist
        dist.all_reduce(metrics)
        pa = getattr(sim, "_peer_agg", None)
        if pa is not None:
            pa.check()   # a peer that never flagged its chunks: raise instead of training on a partial aggregate
    counts = torch.stack([data.nsamp[t], data.nsamp[t + 1] if t + 1 < T1 else torch.zeros_like(data.nsamp[t])], 1).float()
    return {"metrics": metrics, "counts": counts}


def _world_rank(sim):
    import torch.distributed as dist
    if getattr(sim, "shard_clients", False) and dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def _peer_aggregate(sim, world, rank):
    """Multi-GPU aggregation + broadcast of the cluster models in ONE kernel over NVLink peer memory
    (``parallel/peer_aggregate.py``): this rank contributes the rows of its own clients, read IN PLACE from the client arena
    (no gather / pad copies), and the model bank lives in the kernel's symmetric θ buffer (no copy back)."""
    from ..parallel.peer_aggregate import PeerAggregator
    pa = getattr(sim, "_peer_agg", None)
    if pa is None:
        pa = sim._peer_agg = PeerAggregator(sim.M, sim.bank.P, sim.device, sim.bank.theta)
        if pa.world > 1:
            sim.bank.rebind_storage(pa.theta_full)          # the kernel's all-gather target IS the bank from now on
            sim.evaluator.bank = sim.bank
        mine = [c for c in range(sim.C) if c % world == rank]
        sim._peer_mine = (mine, torch.tensor(mine, dtype=torch.int32, device=sim.device))
    mine, cidx = sim._peer_mine
    pa.aggregate(sim.clients.params, sim.clients.n[mine], cidx)
    if sim.bank.theta.data_ptr() != pa.theta.data_ptr():    # world == 1 fallback / unpadded rows: plain copy
        sim.bank.theta.copy_(pa.theta)


def _nhwc(x: torch.Tensor) -> torch.Tensor:
    """Opt-in (``FDB_NHWC=1``) channels_last activations for conv nets.  With NCHW activations 28 % of a ResNet-18 step's
    GPU time is cuDNN's nchwToNhwc / nhwcToNchw conversion kernels (tools/profile_generic.py), but NHWC kernels need
    16-byte aligned weight pointers (the arena now aligns every big tensor, models/utils.py::flat_spec); the first
    end-to-end attempt with the aligned arena did not finish within its GPU time box, so this stays opt-in (DESIGN §9)."""
    if os.environ.get("FDB_NHWC") == "1" and x.is_cuda and x.dim() == 4:
        return x.contiguous(memory_format=torch.channels_last)
    return x


def _lazy_client_xy(Xc_all, data, c, T1, S):
    cache = []

    def xy():
        if not cache:
            cache.append((Xc_all[:, c].reshape(T1 * S, *data.X.shape[3:]), data.Y[:, c].reshape(T1 * S)))
        return cache[0]
    return xy


def _cpu(x: Optional[torch.Tensor]):
    return x.cpu() if isinstance(x, torch.Tensor) else x


class _GraphedStep:
    """Local training captured as a CUDA graph over static buffers.

    * per-step mode (``indexed=False``): ONE step (zero-grad → forward → CE → backward → fused optimizer row update);
      the caller copies each minibatch into ``x`` / ``y`` and replays;
    * per-pair mode (``indexed=True``): ALL ``steps`` local steps of a (client, model) pair in one graph; every step
      starts with a gather node that pulls its minibatch out of the device-resident dataset through the static index
      buffer ``idx[e]`` (global sample ids), so a pair costs one index upload, one multi-tensor state load, ONE replay
      and one multi-tensor state store on the host side."""

    def __init__(self, sim, batch_shape, use_adam: bool, lr: float, wd: float, steps: int = 1, indexed: bool = False):
        import copy
        bank, dev = sim.bank, sim.device
        P = bank.P
        z = lambda: torch.zeros(P, dtype=torch.float32, device=dev)  # noqa: E731
        self.row, self.g, self.m, self.v, self.vmax = z(), z(), z(), z(), z()
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.x = torch.zeros(batch_shape, dtype=sim.data.X.dtype, device=dev)
        self.y = torch.zeros(batch_shape[0], dtype=torch.long, device=dev)
        self.steps, self.indexed = int(steps), bool(indexed)
        if self.indexed:
            self.idx = torch.zeros(self.steps, batch_shape[0], dtype=torch.long, device=dev)
            self.Xf = sim.data.X.reshape(-1, *sim.data.X.shape[3:])      # [T1·C·S, …] view of the resident dataset
            self.Yf = sim.data.Y.reshape(-1)
        self.row.copy_(bank.theta[0])
        self.mod = copy.deepcopy(bank.template).to(dev)
        _bind(self.mod, bank, self.row)
        self.mod.train()
        from ..models.utils import unflatten_to_state_dict
        gviews = unflatten_to_state_dict(self.g, bank.spec)
        for name, p_ in self.mod.named_parameters():
            p_.grad = gviews[name]          # backward accumulates straight into the flat gradient row
        self.use_adam, self.lr, self.wd = use_adam, lr, wd
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(2):              # warm-up (cuDNN autotune, lazy inits) outside the capture
                self._body()
        torch.cuda.current_stream(dev).wait_stream(side)
        # a DEDICATED capture stream per graph: cuBLAS keeps one workspace per (handle, stream), and torch.cuda.graph's
        # default capture stream is shared by all captures — graphs captured there would share a split-K workspace and
        # race when they are replayed concurrently on the slot streams
        self._capture_stream = torch.cuda.Stream(device=dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self._capture_stream):
            self._body()
        self.launches = 0

    def _body(self):
        for e in range(self.steps if self.indexed else 1):
            if self.indexed:
                x, y = self.Xf.index_select(0, self.idx[e]), self.Yf.index_select(0, self.idx[e]).long()
            else:
                x, y = self.x, self.y
            self.g.zero_()
            F.cross_entropy(self.mod(_nhwc(x)), y).backward()
            if self.use_adam:
                ops.adam_amsgrad_rows_(self.row.view(1, -1), self.g.view(1, -1), self.m.view(1, -1), self.v.view(1, -1),
                                       self.vmax.view(1, -1), self.step, self.lr, self.wd)
            else:
                ops.sgd_rows_(self.row.view(1, -1), self.g.view(1, -1), self.lr, 0.0)

    def load(self, cl, c, m):
        if self.use_adam:   # one multi-tensor copy kernel instead of four
            torch._foreach_copy_([self.row, self.m, self.v, self.vmax], [cl.params[c, m], cl.m[c, m], cl.v[c, m], cl.vmax[c, m]])
            self.step.copy_(cl.step[c, m].reshape(1))
        else:
            self.row.copy_(cl.params[c, m])

    def store(self, cl, c, m):
        if self.use_adam:
            torch._foreach_copy_([cl.params[c, m], cl.m[c, m], cl.v[c, m], cl.vmax[c, m]], [self.row, self.m, self.v, self.vmax])
            cl.step[c, m].copy_(self.step[0])
        else:
            cl.params[c, m].copy_(self.row)

    def run_pair(self, gidx_cpu: torch.Tensor):
        """Per-pair mode: upload the [steps, B] global sample ids and replay the whole local training of the pair."""
        self.idx.copy_(gidx_cpu, non_blocking=True)
        self.graph.replay()
        self.launches += 1

    def run(self, xb, yb):
        self.x.copy_(xb)
        self.y.copy_(yb)
        self.graph.replay()
        self.launches += 1


def _stream_slots(sim):
    """Side streams for concurrent pair execution (CUDA + graphed module path only).  A federated local step is ~60
    small dependent kernels, i.e. latency-bound even inside a CUDA graph; replaying K pairs' graphs on K streams lets the
    SMs overlap them.  ``FDB_GRAPH_STREAMS`` (default 8; 1 disables) sets K."""
    if sim.device.type != "cuda" or sim.bank.mlp is not None or os.environ.get("FDB_NO_GRAPHS") == "1":
        return []
    k = int(os.environ.get("FDB_GRAPH_STREAMS", "8"))
    if k <= 1:
        return []
    slots = sim.__dict__.get("_slot_streams")
    if slots is None or len(slots) != k:
        slots = sim._slot_streams = [torch.cuda.Stream(device=sim.device) for _ in range(k)]
    main = torch.cuda.current_stream(sim.device)
    for s_ in slots:                        # the side streams must see θ / data produced on the main stream
        s_.wait_stream(main)
    return slots


def _join_slots(sim, slots):
    if slots:
        main = torch.cuda.current_stream(sim.device)
        for s_ in slots:
            main.wait_stream(s_)


def _graphed_step(sim, batch_shape, use_adam, lr, wd, slot: int = 0, steps: int = 1, indexed: bool = False):
    """Cached ``_GraphedStep`` for this (batch shape, optimizer, lr) or None when graphs are unavailable."""
    if sim.device.type != "cuda" or sim.bank.mlp is not None or os.environ.get("FDB_NO_GRAPHS") == "1" \
            or getattr(sim, "_graphs_broken", False):
        return None
    cache = sim.__dict__.setdefault("_step_graphs", {})
    key = (tuple(batch_shape), bool(use_adam), float(lr), float(wd), int(slot), int(steps), bool(indexed))
    gs = cache.get(key)
    if gs is None:
        nslots = max(1, len(sim.__dict__.get("_slot_streams") or [1]))
        if len(cache) >= 2 * nslots:        # e.g. Adaptive-FedAvg changes lr every round: keep the pool small
            cache.pop(next(iter(cache)))
        try:
            gs = cache[key] = _GraphedStep(sim, batch_shape, use_adam, lr, wd, steps, indexed)
        except Exception as exc:  # noqa: BLE001  (capture is an optimisation; the eager path is always valid)
            import logging
            logging.warning("CUDA-graph capture of the local step failed (%s); running eagerly", exc)
            sim._graphs_broken = True
            torch.cuda.synchronize()
            return None
    return gs


def _local_steps(sim, c, m, xy, sampler, seed, rnd, E, use_adam, lr, wd, feat_mask, slot: int = 0, s: Optional[int] = None):
    """``xy()`` lazily materialises the client's flattened samples (only the non-indexed paths need that copy).  Client c's
    data trains arena row ``[s, m]`` (worker slot s; default s = c)."""
    Xc = Yc = None
    bank, cl = sim.bank, sim.clients
    s = c if s is None else s
    row = cl.params[s, m]
    mlp = bank.mlp
    idxs = []
    for step in range(E):
        h1 = batch_hash(seed, rnd, c, m, step)
        idxs.append(sampler(h1, mix32(h1 ^ 0x68E31DA4)))
    # one H2D + one gather for all E minibatches of this pair when they have equal length (the common case)
    same = all(i.numel() == idxs[0].numel() for i in idxs)
    if same and feat_mask is None and mlp is None and sim.device.type == "cuda" and os.environ.get("FDB_NO_PAIR_GRAPH") != "1":
        # per-pair graph: the minibatch gathers are graph nodes reading the resident dataset through global sample ids
        S_, C_ = sim.data.X.shape[2], sim.C
        loc = torch.stack(idxs)                                              # [E, B] ids into the client's [T1·S] axis
        gidx = (loc // S_) * (C_ * S_) + c * S_ + (loc % S_)
        gs = _graphed_step(sim, (loc.shape[1],) + tuple(sim.data.X.shape[3:]), use_adam, lr, wd, slot, steps=E, indexed=True)
        if gs is not None:
            gs.load(cl, s, m)
            gs.run_pair(gidx)
            gs.store(cl, s, m)
            return
    if Xc is None:
        Xc, Yc = xy()
    if same:
        idx_all = torch.stack(idxs).to(Xc.device, non_blocking=True)
        xs, ys = Xc[idx_all], Yc[idx_all].long()
        if feat_mask is not None:
            xs = xs * feat_mask[m].reshape((1, 1) + tuple(xs.shape[2:]))
        batches = [(xs[e], ys[e]) for e in range(E)]
    else:
        batches = []
        for i in idxs:
            i = i.to(Xc.device)
            xb = Xc[i]
            if feat_mask is not None:
                xb = xb * feat_mask[m].reshape((1,) + tuple(xb.shape[1:]))
            batches.append((xb, Yc[i].long()))
    gs = _graphed_step(sim, batches[0][0].shape, use_adam, lr, wd, slot) if same else None
    if gs is not None:
        gs.load(cl, s, m)
        for xb, yb in batches:
            gs.run(xb, yb)
        gs.store(cl, s, m)
        return
    if mlp is None:
        mod = _scratch_module(sim)
        _bind(mod, bank, row)
        mod.train()
    for xb, yb in batches:
        if mlp is not None:
            th = row.detach().clone().requires_grad_(True)
            logits = ops.mlp_forward(th, xb.reshape(xb.shape[0], -1), mlp["kind"], mlp["in"], mlp["hidden"], mlp["out"])
            (g,) = torch.autograd.grad(F.cross_entropy(logits, yb), th)
        else:
            for p_ in mod.parameters():
                p_.grad = None
            F.cross_entropy(mod(_nhwc(xb)), yb).backward()
            g = _flat_grads(mod, bank, row)
        r2 = row.reshape(1, -1)
        if use_adam:
            ops.adam_amsgrad_rows_(r2, g.reshape(1, -1), cl.m[s, m].reshape(1, -1), cl.v[s, m].reshape(1, -1),
                                   cl.vmax[s, m].reshape(1, -1), cl.step[s, m].reshape(1), lr, wd)
        else:
            ops.sgd_rows_(r2, g.reshape(1, -1), lr, 0.0)


def _scratch_module(sim):
    mod = getattr(sim, "_scratch_mod", None)
    if mod is None:
        import copy
        mod = sim._scratch_mod = copy.deepcopy(sim.bank.template).to(sim.device)
    return mod


def _bind(mod, bank, row):
    """Point the module's parameters/buffers at ``row`` (views, no copy)."""
    from ..parallel.arena import _set_tensor
    from ..models.utils import unflatten_to_state_dict
    views = unflatten_to_state_dict(row, bank.spec)
    for name, p in list(mod.named_parameters()):
        _set_tensor(mod, name, torch.nn.Parameter(views[name], requires_grad=True))
    for name, b in list(mod.named_buffers()):
        if name in views and views[name].dtype == b.dtype:
            _set_tensor(mod, name, views[name], buffer=True)


def _flat_grads(mod, bank, row):
    from ..models.utils import flat_view
    g = torch.zeros_like(row)
    grads = dict(mod.named_parameters())
    for k, shape, dtype, off, n in bank.spec:
        p = grads.get(k)
        if p is not None and p.grad is not None:
            g[off:off + n] = flat_view(p.grad)
    return g


def _eval_grouped(sim, tt: int, models, clients, out, col: int):
    """Score client c with model ``models[c]`` on its time-``tt`` data for every c in ``clients``: ONE batched forward per
    distinct model (chunked to ≤ ~8k samples), per-client (correct, loss-sum) by masked reduction → ``out[c, col:col+2]``."""
    data, bank = sim.data, sim.bank
    S = data.X.shape[2]
    nsamp = sim.data_host.nsamp[tt]
    by_model: Dict[int, list] = {}
    for c in clients:
        if int(nsamp[c]) > 0:
            by_model.setdefault(int(models[c]), []).append(c)
    per_chunk = max(1, 8192 // max(S, 1))
    ar = torch.arange(S, device=sim.device)
    for m, cs in by_model.items():
        for i in range(0, len(cs), per_chunk):
            ck = cs[i:i + per_chunk]
            ct = torch.tensor(ck, device=sim.device)
            X = data.X[tt].index_select(0, ct)
            Y = data.Y[tt].index_select(0, ct).long()
            mask = (ar[None, :] < nsamp[ck].to(sim.device)[:, None]).float()
            logits = bank.forward(m, X.reshape(len(ck) * S, *X.shape[2:])).float()
            loss = F.cross_entropy(logits, Y.reshape(-1), reduction="none").reshape(len(ck), S)
            hit = (logits.argmax(-1) == Y.reshape(-1)).float().reshape(len(ck), S)
            out[ct, col] = (hit * mask).sum(1)
            out[ct, col + 1] = (loss * mask).sum(1)


def _evaluate(sim, plan, st, r, metrics, ens_mode):
    data, bank, t, C = sim.data, sim.bank, sim.t, sim.C
    pick = st["W"][t].argmax(dim=0)
    etr, ete = plan.get("eval_train_model"), plan.get("eval_test_model")
    world, rank = _world_rank(sim)
    mine = [c for c in range(C) if world == 1 or c % world == rank]
    mtr = [int(etr[c]) if etr is not None and int(etr[c]) >= 0 else int(pick[c]) for c in range(C)]
    mte = [int(ete[c]) if ete is not None and int(ete[c]) >= 0 else int(pick[c]) for c in range(C)]
    with torch.no_grad():
        _eval_grouped(sim, t, mtr, mine, metrics[r], 0)
        if ens_mode == 0 and t + 1 < data.steps:
            _eval_grouped(sim, t + 1, mte, mine, metrics[r], 2)
    if ens_mode == 0 or t + 1 >= data.steps:
        return
    _eval_ensemble_grouped(sim, plan, t + 1, mine, metrics[r], ens_mode)


def _eval_ensemble_grouped(sim, plan, tt: int, clients, out, ens_mode: int):
    """Ensemble test metric (AUE / AUE-PC weighted hard vote, KUE weighted soft vote) with ONE batched forward per
    ensemble member over all clients (chunked) instead of a forward per (client, member): per-sample tallies
    ``Σ_k w[c,k]·onehot(pred_k)`` (hard) or ``Σ_k w[c,k]·softmax_k`` (soft) are accumulated on device, the vote is the
    arg-max class, correct counts go to ``out[c, 2]``."""
    data, bank, dev = sim.data, sim.bank, sim.device
    S, classes = data.X.shape[2], int(data.class_num)
    nsamp = sim.data_host.nsamp[tt]
    cs = [c for c in clients if int(nsamp[c]) > 0]
    if not cs:
        return
    Wc = torch.as_tensor(plan["ens_w"]).double().cpu()[cs].clamp(min=0).to(dev)     # [n, M]; non-positive weights do not vote
    members = [k for k in range(bank.num_models) if bool((Wc[:, k] > 0).any())]
    per_chunk = max(1, 8192 // max(S, 1))
    ar = torch.arange(S, device=dev)
    with torch.no_grad():
        for i in range(0, len(cs), per_chunk):
            ck = cs[i:i + per_chunk]
            ct = torch.tensor(ck, device=dev)
            X = data.X[tt].index_select(0, ct)
            Y = data.Y[tt].index_select(0, ct).long()
            mask = ar[None, :] < nsamp[ck].to(dev)[:, None]
            tally = torch.zeros(len(ck), S, classes, dtype=torch.float64, device=dev)
            wck = Wc[i:i + per_chunk]
            for k in members:
                logits = bank.forward(k, X.reshape(len(ck) * S, *X.shape[2:])).float()
                wk = wck[:, k][:, None, None]
                if ens_mode == 1:
                    pred = logits.argmax(-1).reshape(len(ck), S, 1)
                    tally.scatter_add_(2, pred, wk.expand(len(ck), S, 1).contiguous())
                else:
                    tally += wk * torch.softmax(logits, 1).reshape(len(ck), S, classes).double()
            hit = (tally.argmax(-1) == Y) & mask
            out[ct, 2] = hit.sum(1).float()
