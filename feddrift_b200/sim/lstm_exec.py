"""Batched local training of an LSTM federation: EVERY (client, model) pair of a GPU advances one local step in the same
handful of launches (reference semantic: ``FedAvgEnsTrainerSoftCluster.py:97-113`` runs the pairs one after the other, and
``model/nlp/rnn.py:18-33`` runs each through ~10 cuDNN kernels per timestep).

Per local step, for all pairs at once:

  1. ``lstm2_fwd_kernel``   one thread-block cluster per (pair, 16-row chunk); weights are read straight from the pair's
                            ``ClientArena`` row (no parameter copies, no ``load_state_dict``);
  2. ``lstm_head_kernel``   fc + softmax-CE + dlogits + dW_fc / db_fc / dh;
  3. ``lstm2_bwd_kernel``   BPTT;
  4. three batched tcgen05 GEMMs (``gemm_batched_mn``: one batch entry per chunk) for dW_hh1 / dW_ih2 / dW_hh2, a few
     batched reductions for the small tensors (biases, W_ih1, embedding);
  5. gradient rows → ``adam_amsgrad_rows`` over the arena rows of the active pairs (one launch).

Host work per ROUND (not per pair and step): the counter-hash batch selection of every pair (the same RNG stream as every other
executor) and ONE index upload.  Used by ``sim/generic.py`` when the bank's template is ``RNN_OriginalFedAvg``.
"""
from __future__ import annotations

from typing import Dict, List

import numpy as np
import torch

from .. import ops
from ..ops import lstm as L
from ..ops.reference import batch_hash, mix32

_KEYS = {"emb": "embeddings.weight", "w_ih1": "lstm.weight_ih_l0", "w_hh1": "lstm.weight_hh_l0", "b_ih1": "lstm.bias_ih_l0",
         "b_hh1": "lstm.bias_hh_l0", "w_ih2": "lstm.weight_ih_l1", "w_hh2": "lstm.weight_hh_l1", "b_ih2": "lstm.bias_ih_l1",
         "b_hh2": "lstm.bias_hh_l1", "fc_w": "fc.weight", "fc_b": "fc.bias"}


def applicable(sim, feat_mask) -> bool:
    """The batched path handles ``RNN_OriginalFedAvg`` (last-step head) on CUDA with token inputs."""
    import os
    from ..models.rnn import RNN_OriginalFedAvg
    from ..ops import _ext
    if os.environ.get("FDB_LSTM_BATCHED", "1") == "0" or os.environ.get("FDB_NO_FUSED_LSTM") == "1":
        return False
    t = sim.bank.template
    if not (isinstance(t, RNN_OriginalFedAvg) and not t.per_position and sim.device.type == "cuda" and feat_mask is None):
        return False
    if not (_ext.available() and hasattr(_ext.load(), "lstm2_forward") and hasattr(_ext.load(), "lstm_head")):
        return False
    X = sim.data.X
    return (X.dim() == 4 and not X.dtype.is_floating_point and t.lstm.hidden_size == L.H and t.lstm.num_layers == 2
            and t.embeddings.embedding_dim <= 16 and t.fc.out_features <= 96)


def _layout(sim) -> Dict:
    lay = sim.__dict__.get("_lstm_layout")
    if lay is None:
        spec = {k: (off, n, shape) for k, shape, _, off, n in sim.bank.spec}
        lay = {name: spec[key] for name, key in _KEYS.items()}
        lay["offs9"] = [lay[k][0] for k in L.PARAM_ORDER]
        sim._lstm_layout = lay
    return lay


def train_pairs(sim, pairs: List, seed: int, rnd: int, E: int, use_adam: bool, lr: float, wd: float) -> None:
    """``pairs``: list of ``(s, c, m, sampler)``; runs the E local steps of every pair (models start from ``bank.theta[m]``) on
    client c's data in arena row ``[s, m]`` (worker slot s)."""
    bank, cl, dev = sim.bank, sim.clients, sim.device
    C, M, P = sim.C, sim.M, bank.P
    npairs = len(pairs)
    if npairs == 0:
        return
    lay = _layout(sim)
    S, T = sim.data.X.shape[2], sim.data.X.shape[3]
    V, Eemb = lay["fc_b"][1], lay["emb"][2][1]
    # ---- host: the batch of every (step, pair) from the shared counter-hash RNG; one upload per round
    sel = [[None] * npairs for _ in range(E)]
    bmax = 1
    for j, (_, c, m, sampler) in enumerate(pairs):
        for e in range(E):
            h1 = batch_hash(seed, rnd, c, m, e)
            loc = sampler(h1, mix32(h1 ^ 0x68E31DA4)).numpy()
            sel[e][j] = (loc // S) * (C * S) + c * S + (loc % S)          # ids into the flattened [T1·C·S] sample axis
            bmax = max(bmax, len(loc))
    nc = (bmax + L.NB - 1) // L.NB
    gidx = np.full((E, npairs, nc * L.NB), -1, dtype=np.int64)
    for e in range(E):
        for j in range(npairs):
            gidx[e, j, :len(sel[e][j])] = sel[e][j]
    gidx_d = torch.from_numpy(gidx).to(dev, non_blocking=True)
    valid = gidx_d >= 0
    safe = gidx_d.clamp(min=0)
    Xf = sim.data.X.reshape(-1, T)
    Yf = sim.data.Y.reshape(-1)
    tokens_all = torch.where(valid.unsqueeze(-1), Xf[safe], torch.zeros((), dtype=Xf.dtype, device=dev)).to(torch.int32)  # [E, np, nc·16, T]
    labels_all = torch.where(valid, Yf[safe], torch.full((), -1, dtype=Yf.dtype, device=dev)).to(torch.int32)            # [E, np, nc·16]
    cnt = valid.sum(-1).clamp(min=1).float()                                                                              # [E, np]
    scale_all = (1.0 / cnt).repeat_interleave(nc, dim=1).contiguous()                                                     # [E, np·nc]
    rows_h = [s * M + m for s, _, m, _ in pairs]
    rows = torch.tensor(rows_h, dtype=torch.int64, device=dev)
    ms = torch.tensor([m for _, _, m, _ in pairs], dtype=torch.int64, device=dev)
    chunk_rows = rows.repeat_interleave(nc)
    chunk_off = (chunk_rows * P).contiguous()
    nch = npairs * nc

    params2 = cl.params.view(C * M, P)
    params2.index_copy_(0, rows, bank.theta.index_select(0, ms))         # broadcast: every pair starts from its cluster model
    arena = cl.params.view(-1)
    G = sim.__dict__.get("_grad_arena")
    if G is None or G.shape != params2.shape:
        G = sim._grad_arena = torch.zeros_like(params2)
    mask = torch.zeros(C * M, dtype=torch.uint8, device=dev)
    mask[rows] = 1
    key = (nch, T)
    ws = sim.__dict__.get("_lstm_ws")
    if ws is None or sim.__dict__.get("_lstm_ws_key") != key:
        ws = sim._lstm_ws = L.Lstm2Workspace(nch, T, dev, train=True)
        sim._lstm_ws_key = key
    from ..ops import _ext
    ext = _ext.load(required=True)
    o_emb, n_emb, _ = lay["emb"]
    o_wih1 = lay["w_ih1"][0]

    def put(name: str, t: torch.Tensor) -> None:                         # per-pair gradient block → its slot in the gradient rows
        off, n, _ = lay[name]
        t = t.reshape(npairs, nc, n).sum(1) if nc > 1 else t.reshape(npairs, n)
        G[:, off:off + n].index_copy_(0, rows, t)

    for e in range(E):
        tok = tokens_all[e].reshape(nch, L.NB, T).contiguous()
        L.lstm2_pairs_forward(arena, chunk_off, lay["offs9"], tok, Eemb, ws)
        dh, dWfc, dbfc, _ = L.lstm_head(arena, chunk_off, lay["fc_w"][0], lay["fc_b"][0], ws.hlast,
                                        labels_all[e].reshape(nch, L.NB).contiguous(), scale_all[e], V)
        L.lstm2_pairs_backward(arena, chunk_off, lay["offs9"], tok, Eemb, ws, dh)
        big = L.lstm2_weight_grads_per_chunk(ws)
        # small tensors (biases, W_ih1, embedding): one fused pass over the bf16 gate-gradient histories
        b1, b2, dWih1, demb = ext.lstm_small_grads(arena, chunk_off, o_emb, o_wih1, tok, ws.dgates, Eemb, n_emb // Eemb)
        demb[:, 0] = 0                                                   # nn.Embedding(padding_idx=0)
        put("w_hh1", big["w_hh1"]); put("w_ih2", big["w_ih2"]); put("w_hh2", big["w_hh2"])
        put("b_ih1", b1); put("b_hh1", b1); put("b_ih2", b2); put("b_hh2", b2)
        put("w_ih1", dWih1); put("emb", demb); put("fc_w", dWfc); put("fc_b", dbfc)
        if use_adam:
            ops.adam_amsgrad_rows_(params2, G, cl.m.view(C * M, P), cl.v.view(C * M, P), cl.vmax.view(C * M, P), cl.step.view(-1),
                                   lr, wd, row_mask=mask)
        else:
            params2.index_add_(0, rows, G.index_select(0, rows), alpha=-lr)
