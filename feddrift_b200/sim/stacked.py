"""Pair-stacked local training of convolutional federations: EVERY (client, model) pair of a GPU advances one local step in the
SAME forward / backward pass (reference semantic: ``FedAvgEnsTrainerSoftCluster.py:97-113`` trains the pairs one after the
other; round 1 of this framework replayed one CUDA graph per pair).

The template network is rewritten into a *channel-stacked* network that evaluates ``npairs`` independent copies at once:

* activations are ``[B, npairs·C, H, W]`` (channels_last memory ⇒ every pixel holds the pairs' channel vectors back to back),
  so all the per-sample layers — ReLU, pooling, dropout, residual adds, flatten — are unchanged;
* ``Conv2d`` → :class:`StackedConv2d`: a grouped convolution with one group per pair — on CUDA the implicit-GEMM tcgen05 kernels
  in grouped mode (``csrc/gemm_tc.cu`` conv modes: the TMA-im2col producer addresses channel chunk ``pair·C + c``), a grouped
  library convolution for the 1/3-channel stems and on CPU;
* ``Linear`` → :class:`StackedLinear` (one batched GEMM), ``BatchNorm2d`` / ``GroupNorm`` → the same normalisation over
  ``npairs·C`` channels (per-channel batch statistics are per-pair statistics), ``Softmax(dim=1)`` → per-pair softmax.

Parameters are NOT copied per step: a round stages the pairs' rows ``[npairs, P]`` (parameters + Adam moments) once, the
stacked layers' parameters are strided VIEWS ``stage[:, off:off+n]`` of those rows and their ``.grad`` are the same views of the
gradient rows, one ``adam_amsgrad_rows`` launch updates all pairs, and the rows go back to the client arena at the end of the
round.  The counter-hash batch selection is the shared RNG stream of every executor; dropout masks come from one generator
for all pairs (statistically, not bitwise, the per-pair executor's masks).

Used by ``sim/generic.py`` when the template is a stackable conv net and every pair draws the same batch size.
"""
from __future__ import annotations

import copy
import os
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from .. import ops
from ..models.utils import ohwi_stored
from ..ops.reference import batch_hash, mix32

_GRAPH_DEFAULT = "0"      # FDB_STACKED_GRAPH: capture the stacked E-step training as one CUDA graph

_PASS = (nn.ReLU, nn.MaxPool2d, nn.AvgPool2d, nn.AdaptiveAvgPool2d, nn.Dropout, nn.Dropout2d, nn.Flatten, nn.Identity)


class _Stacked(nn.Module):
    """Base of the stacked layers: parameters are bound later to strided views of the staged rows."""
    param_names: tuple = ()

    def bind(self, prefix: str, spec: Dict, stage: torch.Tensor, grads: torch.Tensor) -> None:
        n = stage.shape[0]
        for attr in self.param_names:
            key = f"{prefix}.{attr}" if prefix else attr
            if key not in spec:
                self._parameters[attr] = None
                continue
            shape, off, numel = spec[key]

            def view(t):
                seg = t[:, off:off + numel]
                if ohwi_stored(shape):
                    # flat rows hold conv weights as (O, kh, kw, I): models.utils.flat_view / unflatten_to_state_dict
                    return seg.view(n, shape[0], shape[2], shape[3], shape[1]).permute(0, 1, 4, 2, 3)
                return seg.view(n, *shape)
            p = nn.Parameter(view(stage), requires_grad=True)
            p.grad = view(grads)
            self._parameters[attr] = p


class StackedConv2d(_Stacked):
    param_names = ("weight", "bias")

    def __init__(self, conv, npairs: int):
        super().__init__()
        self.npairs = npairs
        self.in_channels, self.out_channels = conv.in_channels, conv.out_channels
        pair = lambda v: (int(v), int(v)) if isinstance(v, int) else (int(v[0]), int(v[1]))  # noqa: E731
        self.kernel_size, self.stride, self.padding = pair(conv.kernel_size), pair(conv.stride), pair(conv.padding)
        self.dilation, self.groups = pair(conv.dilation), int(conv.groups)
        self.activation = getattr(conv, "activation", "none")
        self.register_parameter("weight", None)
        self.register_parameter("bias", None)

    def forward(self, x):
        n = self.npairs
        relu = self.activation == "relu"
        from ..ops import conv as C
        if C.stacked_eligible(self, x):
            return C._StackedConvFn.apply(x, self.weight, self.bias, self.stride, self.padding, relu, n)
        w = self.weight.reshape(n * self.out_channels, self.in_channels // self.groups, *self.kernel_size)
        b = self.bias.reshape(-1) if self.bias is not None else None
        y = F.conv2d(x, w, b, self.stride, self.padding, self.dilation, n * self.groups)
        return F.relu(y) if relu else y


class StackedLinear(_Stacked):
    param_names = ("weight", "bias")

    def __init__(self, lin, npairs: int):
        super().__init__()
        self.npairs, self.in_features, self.out_features = npairs, lin.in_features, lin.out_features
        self.activation = getattr(lin, "activation", "none")
        self.register_parameter("weight", None)
        self.register_parameter("bias", None)

    def forward(self, x):                                     # [B, npairs·in] → [B, npairs·out]
        n, B = self.npairs, x.shape[0]
        xv = x.reshape(B, n, self.in_features).transpose(0, 1)                   # [n, B, in]
        wt = self.weight.transpose(1, 2)                                          # [n, in, out] (strided view of the rows)
        y = torch.baddbmm(self.bias.unsqueeze(1), xv, wt) if self.bias is not None else torch.bmm(xv, wt)
        if self.activation == "relu":
            y = F.relu(y)
        return y.transpose(0, 1).reshape(B, n * self.out_features)


class StackedBatchNorm2d(_Stacked):
    param_names = ("weight", "bias")

    def __init__(self, bn, npairs: int):
        super().__init__()
        if bn.momentum is None and bn.track_running_stats:
            raise TypeError("cumulative-average BatchNorm (momentum=None) is not pair-stacked")   # per-pair path keeps its semantics
        self.npairs, self.num_features, self.eps, self.momentum = npairs, bn.num_features, bn.eps, bn.momentum
        self.track = bn.track_running_stats
        self.register_parameter("weight", None)
        self.register_parameter("bias", None)
        if self.track:
            self.register_buffer("running_mean", torch.zeros(npairs * bn.num_features))
            self.register_buffer("running_var", torch.ones(npairs * bn.num_features))
        self.steps = 0                                         # num_batches_tracked increments of this round

    def forward(self, x):
        if self.training:
            self.steps += 1
        mom = self.momentum if self.momentum is not None else 0.1
        if (self.training and x.is_cuda and x.dim() == 4 and self.weight is not None and os.environ.get("FDB_NO_BN_KERNEL") != "1"
                and ops.native(x) and hasattr(ops._ext.load(), "bn_nhwc_fwd")):
            # npairs·C channels, few rows: the coalesced NHWC kernels (cuDNN needs 200–300 µs per call at 16 k channels)
            return ops.batch_norm_train_nhwc(x, self.weight, self.bias, self.running_mean if self.track else None,
                                             self.running_var if self.track else None, self.eps, mom)
        w = self.weight.reshape(-1) if self.weight is not None else None
        b = self.bias.reshape(-1) if self.bias is not None else None
        return F.batch_norm(x, self.running_mean if self.track else None, self.running_var if self.track else None, w, b,
                            self.training or not self.track, mom, self.eps)


class StackedGroupNorm(_Stacked):
    param_names = ("weight", "bias")

    def __init__(self, gn, npairs: int):
        super().__init__()
        self.npairs, self.eps = npairs, gn.eps
        self.num_groups = gn.num_groups
        self.register_parameter("weight", None)
        self.register_parameter("bias", None)

    def forward(self, x):
        w = self.weight.reshape(-1) if self.weight is not None else None
        b = self.bias.reshape(-1) if self.bias is not None else None
        g = self.npairs * self.num_groups
        if x.is_cuda and w is not None:
            return ops.group_norm(x, g, w, b, self.eps)
        return F.group_norm(x, g, w, b, self.eps)


class StackedSoftmax(nn.Module):
    def __init__(self, npairs: int):
        super().__init__()
        self.npairs = npairs

    def forward(self, x):
        B = x.shape[0]
        return F.softmax(x.reshape(B, self.npairs, -1), dim=2).reshape(B, -1)


def _convert(mod: nn.Module, npairs: int) -> nn.Module:
    from ..models.group_norm import _GroupNorm
    from ..ops.conv import TcConv2d
    from ..ops.linear import TcLinear
    for name, child in list(mod.named_children()):
        if isinstance(child, (nn.Conv2d, TcConv2d)):
            if isinstance(child, nn.Conv2d) and (child.padding_mode != "zeros" or isinstance(child.padding, str)):
                raise TypeError("padding mode")
            new = StackedConv2d(child, npairs)
        elif isinstance(child, (nn.Linear, TcLinear)):
            new = StackedLinear(child, npairs)
        elif isinstance(child, nn.BatchNorm2d):
            new = StackedBatchNorm2d(child, npairs)
        elif isinstance(child, (_GroupNorm, nn.GroupNorm)):
            new = StackedGroupNorm(child, npairs)
        elif isinstance(child, nn.Softmax):
            if child.dim not in (1, -1):
                raise TypeError("softmax dim")
            new = StackedSoftmax(npairs)
        elif isinstance(child, _PASS):
            continue
        else:
            if any(True for _ in child.parameters(recurse=False)) or any(True for _ in child.buffers(recurse=False)):
                raise TypeError(f"layer {type(child).__name__} cannot be pair-stacked")
            _convert(child, npairs)
            continue
        setattr(mod, name, new)
    return mod


def stack_module(template: nn.Module, npairs: int) -> nn.Module:
    """Channel-stacked copy of ``template`` (raises ``TypeError`` when a layer type has no stacked counterpart)."""
    if any(True for _ in template.parameters(recurse=False)):
        raise TypeError("top-level parameters")
    return _convert(copy.deepcopy(template), npairs)


def stack_input(template: nn.Module, x: torch.Tensor) -> torch.Tensor:
    """``x``: ``[npairs, B, *features]`` → the stacked network's input ``[B, npairs·C, H, W]`` (channels_last)."""
    if hasattr(template, "stack_input"):
        x = template.stack_input(x)
    if x.dim() != 5:
        raise TypeError("stacked training needs image-shaped samples")
    n, B, C, H, W = x.shape
    x = x.permute(1, 0, 2, 3, 4).reshape(B, n * C, H, W)
    return x.contiguous(memory_format=torch.channels_last) if x.is_cuda else x


def stackable(template: nn.Module) -> bool:
    """Architectures whose ``forward`` is channel-count agnostic (audited): the MNIST CNNs, the CIFAR / GN / torchvision ResNets."""
    from ..models import cnn, resnet
    ok = [cnn.CNN_DropOut, cnn.CNN_OriginalFedAvg, resnet.ResNet]
    try:
        import torchvision
        ok.append(torchvision.models.ResNet)
    except Exception:  # noqa: BLE001
        pass
    try:
        from ..models import resnet_gn
        ok.append(resnet_gn.ResNet)
    except Exception:  # noqa: BLE001
        pass
    if not isinstance(template, tuple(ok)):
        return False
    if getattr(template, "KD", False) or getattr(template, "return_stem_features", False):
        return False
    try:
        stack_module(template, 2)
    except TypeError:
        return False
    return True


def applicable(sim, feat_mask) -> bool:
    if os.environ.get("FDB_STACKED", "1") == "0" or feat_mask is not None or sim.bank.mlp is not None:
        return False
    ok = sim.__dict__.get("_stackable")
    if ok is None:
        ok = bool(sim.data.X.dtype.is_floating_point and stackable(sim.bank.template))
        if ok and sim.device.type == "cuda" and os.environ.get("FDB_STACKED") != "force":
            # on the GPU stacking pays when the body convolutions run on the grouped tcgen05 kernels; a body layer they do not
            # cover (e.g. the MNIST CNN's 32→64 conv) would fall to the library's grouped convolution, which loops over the
            # groups (profiles/cfg3_stacked_profile_r2.txt) — the per-pair graph executor is faster there
            for mod in stack_module(sim.bank.template, 2).modules():
                if isinstance(mod, StackedConv2d) and mod.in_channels >= 16 and not (
                        mod.in_channels % 64 == 0 and mod.out_channels % 64 == 0 and mod.groups == 1 and mod.dilation == (1, 1)
                        and mod.kernel_size[0] == mod.kernel_size[1] and mod.padding[0] == mod.padding[1] and mod.stride[0] == mod.stride[1]):
                    ok = False
        sim._stackable = ok
    return ok


class _Stage:
    """Round-local staging of ``npairs`` rows + the stacked network bound to them (cached per pair count)."""

    def __init__(self, sim, npairs: int):
        bank, dev = sim.bank, sim.device
        P = bank.P
        z = lambda: torch.zeros(npairs, P, dtype=torch.float32, device=dev)  # noqa: E731
        self.params, self.grads, self.m, self.v, self.vmax = z(), z(), z(), z(), z()
        self.step = torch.zeros(npairs, dtype=sim.clients.step.dtype, device=dev)
        self.net = stack_module(bank.template, npairs).to(dev)
        self.spec = {k: (tuple(shape), off, n) for k, shape, _, off, n in bank.spec}
        self.bns: List = []
        for name, mod in self.net.named_modules():
            if isinstance(mod, _Stacked):
                mod.bind(name, self.spec, self.params, self.grads)
            if isinstance(mod, StackedBatchNorm2d) and mod.track:
                self.bns.append((name, mod))
        self.net.train()
        self.npairs = npairs

    def load_buffers(self) -> None:
        for name, bn in self.bns:
            C = bn.num_features
            for attr in ("running_mean", "running_var"):
                _, off, _ = self.spec[f"{name}.{attr}"]
                getattr(bn, attr).copy_(self.params[:, off:off + C].reshape(-1))
            bn.steps = 0

    def store_buffers(self, steps: Optional[int] = None) -> None:
        """``steps``: BatchNorm forward passes of this round (a replayed CUDA graph does not run the Python counter)."""
        for name, bn in self.bns:
            C = bn.num_features
            for attr in ("running_mean", "running_var"):
                _, off, _ = self.spec[f"{name}.{attr}"]
                self.params[:, off:off + C].copy_(getattr(bn, attr).view(self.npairs, C))
            key = f"{name}.num_batches_tracked"
            if key in self.spec:
                self.params[:, self.spec[key][1]] += float(bn.steps if steps is None else steps)


def max_pairs_per_pass(P: int) -> int:
    """How many pairs are stacked at once: the staged rows (parameters, gradients, three Adam moments) of one pass stay below
    ``FDB_STACKED_MAX_GB`` (default 24 GB of the 180 GB HBM; activations scale with the same count)."""
    budget = float(os.environ.get("FDB_STACKED_MAX_GB", "24")) * (1 << 30)
    return max(1, int(budget // (5 * 4 * max(P, 1))))


def train_pairs(sim, pairs: List, seed: int, rnd: int, E: int, use_adam: bool, lr: float, wd: float) -> bool:
    """``pairs``: list of ``(s, c, m, sampler)``: client c's data trains arena row ``[s, m]`` (worker slot s).  Runs the E local
    steps of every pair; returns False (nothing done) when the pairs
    draw different batch sizes — the caller then takes the per-pair path.  Large federations are processed in passes of at most
    :func:`max_pairs_per_pass` pairs (equal-sized passes, so at most two staging sets are ever alive)."""
    cap = max_pairs_per_pass(sim.bank.P)
    if len(pairs) > cap:
        npass = (len(pairs) + cap - 1) // cap
        per = (len(pairs) + npass - 1) // npass
        chunks = [pairs[i:i + per] for i in range(0, len(pairs), per)]
        if not _train_pass(sim, chunks[0], seed, rnd, E, use_adam, lr, wd):
            return False                                  # nothing was modified: the caller takes the per-pair path for all pairs
        for ch in chunks[1:]:
            if not _train_pass(sim, ch, seed, rnd, E, use_adam, lr, wd):
                raise RuntimeError("pair-stacked training: batch sizes differ between passes of one round")
        return True
    return _train_pass(sim, pairs, seed, rnd, E, use_adam, lr, wd)


def _train_pass(sim, pairs: List, seed: int, rnd: int, E: int, use_adam: bool, lr: float, wd: float) -> bool:
    bank, cl, dev = sim.bank, sim.clients, sim.device
    C, M, P = sim.C, sim.M, bank.P
    npairs = len(pairs)
    if npairs == 0:
        return True
    S = sim.data.X.shape[2]
    sel = []
    for (_, c, m, sampler) in pairs:
        row = []
        for e in range(E):
            h1 = batch_hash(seed, rnd, c, m, e)
            loc = sampler(h1, mix32(h1 ^ 0x68E31DA4)).numpy()
            row.append((loc // S) * (C * S) + c * S + (loc % S))          # ids into the flattened [T1·C·S] sample axis
        sel.append(row)
    B = len(sel[0][0])
    if B == 0 or any(len(a) != B for row in sel for a in row):
        return False
    gidx = torch.from_numpy(np.asarray(sel, dtype=np.int64).transpose(1, 0, 2).copy()).to(dev, non_blocking=True)   # [E, npairs, B]
    stages = sim.__dict__.setdefault("_stack_stages", {})           # per pair count (a chunked round has ≤ 2 distinct counts)
    st: Optional[_Stage] = stages.get(npairs)
    if st is None:
        if len(stages) >= 2:
            stages.clear()
        st = stages[npairs] = _Stage(sim, npairs)
    sim._stack_stage = st
    rows = torch.tensor([s * M + m for s, _, m, _ in pairs], dtype=torch.int64, device=dev)
    ms = torch.tensor([m for _, _, m, _ in pairs], dtype=torch.int64, device=dev)
    CM = C * M
    torch.index_select(bank.theta, 0, ms, out=st.params)                 # broadcast: every pair starts from its cluster model
    if use_adam:
        torch.index_select(cl.m.view(CM, P), 0, rows, out=st.m)
        torch.index_select(cl.v.view(CM, P), 0, rows, out=st.v)
        torch.index_select(cl.vmax.view(CM, P), 0, rows, out=st.vmax)
        st.step.copy_(cl.step.view(-1).index_select(0, rows))
    st.load_buffers()
    Xf = sim.data.X.reshape(-1, *sim.data.X.shape[3:])
    Yf = sim.data.Y.reshape(-1)
    tmpl = bank.template

    def steps(idx: torch.Tensor) -> None:
        for e in range(E):
            x = Xf[idx[e]]                                                    # [npairs, B, *features]
            y = Yf[idx[e]].long()                                             # [npairs, B]
            st.grads.zero_()
            logits = st.net(stack_input(tmpl, x))                             # [B, npairs·K]
            K = logits.shape[1] // npairs
            # Σ_pairs mean_B CE: every pair's gradient is exactly its own mean-reduced loss gradient
            loss = F.cross_entropy(logits.reshape(B * npairs, K), y.t().reshape(-1), reduction="sum") / B
            loss.backward()
            if use_adam:
                ops.adam_amsgrad_rows_(st.params, st.grads, st.m, st.v, st.vmax, st.step, lr, wd)
            else:
                ops.sgd_rows_(st.params, st.grads, lr, 0.0)

    # The whole E-step training of all pairs as ONE CUDA graph over the staged rows (the eager stacked step is ≈ 400 launches
    # for a ResNet-18 and host-bound).  First call with a given shape runs eagerly (warm-up: lazy inits, autotuning), the
    # second captures, later ones replay; any capture failure falls back to eager execution for good.
    key = (npairs, B, E, bool(use_adam), float(lr), float(wd), tuple(gidx.shape))
    use_graph = (dev.type == "cuda" and os.environ.get("FDB_STACKED_GRAPH", _GRAPH_DEFAULT) == "1" and os.environ.get("FDB_NO_GRAPHS") != "1"
                 and not sim.__dict__.get("_stack_graph_broken", False))
    g = st.__dict__.get("graph") if use_graph else None
    if g is not None and g["key"] == key:
        g["idx"].copy_(gidx, non_blocking=True)
        g["graph"].replay()
    elif use_graph and st.__dict__.get("warm_key") == key:
        st.captures = st.__dict__.get("captures", 0) + 1
        if st.captures > 4:                        # e.g. Adaptive-FedAvg changes lr every round: re-capturing would cost more than it saves
            sim._stack_graph_broken = True
        try:
            idx_static = gidx.clone()
            cs = torch.cuda.Stream(device=dev)
            cs.wait_stream(torch.cuda.current_stream(dev))
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=cs):
                steps(idx_static)
            torch.cuda.current_stream(dev).wait_stream(cs)
            st.graph = {"key": key, "graph": graph, "idx": idx_static, "stream": cs}
            graph.replay()
        except Exception as exc:  # noqa: BLE001  (capture is an optimisation; the eager path is always valid)
            import logging
            logging.warning("CUDA-graph capture of the stacked step failed (%s); running eagerly", exc)
            sim._stack_graph_broken = True
            torch.cuda.synchronize()
            st.load_buffers()                      # a failed capture executed nothing: restart this round's steps eagerly
            torch.index_select(bank.theta, 0, ms, out=st.params)
            if use_adam:
                torch.index_select(cl.m.view(CM, P), 0, rows, out=st.m)
                torch.index_select(cl.v.view(CM, P), 0, rows, out=st.v)
                torch.index_select(cl.vmax.view(CM, P), 0, rows, out=st.vmax)
                st.step.copy_(cl.step.view(-1).index_select(0, rows))
            steps(gidx)
    else:
        st.warm_key = key
        st.graph = None
        steps(gidx)
    st.store_buffers(E)
    cl.params.view(CM, P).index_copy_(0, rows, st.params)
    if use_adam:
        cl.m.view(CM, P).index_copy_(0, rows, st.m)
        cl.v.view(CM, P).index_copy_(0, rows, st.v)
        cl.vmax.view(CM, P).index_copy_(0, rows, st.vmax)
        cl.step.view(-1).index_copy_(0, rows, st.step)
    return True
