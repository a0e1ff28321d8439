"""Plain-PyTorch fp32 reference implementations of every native op.

These are (a) the CPU fallbacks and (b) the numerics oracle the GPU tests
compare the sm_100a kernels against.  Nothing here is tuned; clarity wins.
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import numpy as np
import torch
import torch.nn.functional as F

M32 = 0xFFFFFFFF


# --------------------------------------------------------------------------- RNG
def mix32(x: int) -> int:
    """lowbias32 integer finaliser — the device RNG is the same function (csrc/common.cuh)."""
    x &= M32
    x ^= x >> 16
    x = (x * 0x7FEB352D) & M32
    x ^= x >> 15
    x = (x * 0x846CA68B) & M32
    x ^= x >> 16
    return x


def batch_hash(seed: int, rnd: int, client: int, model: int, step: int) -> int:
    h = mix32((seed + 0x9E3779B9 * (rnd + 1)) & M32)
    h = mix32(h ^ ((client * 0x85EBCA6B + 0x165667B1) & M32))
    h = mix32(h ^ ((model * 0xC2B2AE35 + 0x27D4EB2F) & M32))
    h = mix32(h ^ ((step * 0x2545F491 + 1) & M32))
    return h


def hash_choice(h: int, n: int) -> int:
    """Unbiased-enough index in [0, n): high 32 bits of h·n (no modulo)."""
    return (h * n) >> 32


# --------------------------------------------------------------------------- small MLP family
def mlp_param_count(kind: str, din: int, hid: int, dout: int) -> int:
    if kind == "lr":
        return dout * din + dout
    return hid * din + hid + dout * hid + dout


def mlp_unpack(theta: torch.Tensor, kind: str, din: int, hid: int, dout: int):
    """theta [..., P] -> weight/bias views in state_dict order."""
    if kind == "lr":
        w = theta[..., : dout * din].reshape(*theta.shape[:-1], dout, din)
        b = theta[..., dout * din:]
        return w, b
    o = 0
    w1 = theta[..., o:o + hid * din].reshape(*theta.shape[:-1], hid, din); o += hid * din
    b1 = theta[..., o:o + hid]; o += hid
    w2 = theta[..., o:o + dout * hid].reshape(*theta.shape[:-1], dout, hid); o += dout * hid
    b2 = theta[..., o:o + dout]
    return w1, b1, w2, b2


def mlp_forward(theta: torch.Tensor, x: torch.Tensor, kind: str, din: int, hid: int, dout: int) -> torch.Tensor:
    """theta [P], x [B, din] -> logits-as-fed-to-CE [B, dout] (lr applies the sigmoid first)."""
    if kind == "lr":
        w, b = mlp_unpack(theta, kind, din, hid, dout)
        return torch.sigmoid(x @ w.t() + b)
    w1, b1, w2, b2 = mlp_unpack(theta, kind, din, hid, dout)
    return torch.relu(x @ w1.t() + b1) @ w2.t() + b2


def mlp_loss_grad(theta, x, y, kind, din, hid, dout):
    th = theta.detach().clone().requires_grad_(True)
    loss = F.cross_entropy(mlp_forward(th, x, kind, din, hid, dout), y.long())
    (g,) = torch.autograd.grad(loss, th)
    return loss.detach(), g


def adam_amsgrad_update(p, g, m, v, vmax, step: int, lr, wd, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam(amsgrad=True, weight_decay=wd) single-tensor semantics; in place; returns new step."""
    step += 1
    g = g + wd * p
    m.mul_(b1).add_(g, alpha=1 - b1)
    v.mul_(b2).addcmul_(g, g, value=1 - b2)
    torch.maximum(vmax, v, out=vmax)
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    denom = vmax.sqrt() / math.sqrt(bc2) + eps
    p.addcdiv_(m, denom, value=-(lr / bc1))
    return step


def mlp_eval(theta, x, y, n, kind, din, hid, dout) -> Tuple[float, float]:
    """-> (correct, loss_sum) over the first n samples."""
    if n == 0:
        return 0.0, 0.0
    logits = mlp_forward(theta, x[:n], kind, din, hid, dout)
    loss = F.cross_entropy(logits, y[:n].long(), reduction="sum")
    correct = (logits.argmax(-1) == y[:n]).sum()
    return float(correct), float(loss)


def mlp_eval_matrix(theta, X, Y, nsamp, kind, din, hid, dout):
    """theta [M,P]; X [C,S,din]; Y [C,S]; nsamp [C] -> correct [M,C], loss_sum [M,C] (fp32)."""
    M, C = theta.shape[0], X.shape[0]
    correct = torch.zeros(M, C, dtype=torch.float32, device=theta.device)
    loss = torch.zeros(M, C, dtype=torch.float32, device=theta.device)
    for m in range(M):
        for c in range(C):
            k, l = mlp_eval(theta[m], X[c], Y[c], int(nsamp[c]), kind, din, hid, dout)
            correct[m, c], loss[m, c] = k, l
    return correct, loss


def _np_view(st, nb):
    """Host-side numpy mirrors of the plan tensors (built once per `st`): scalar indexing of torch tensors costs a few
    µs per access, which dominated the per-pair sampler of the generic executor."""
    cache = st.get("_np")
    if cache is None or cache["W_id"] is not st["W"]:
        cache = st["_np"] = {"W_id": st["W"], "W": st["W"].detach().cpu().double().numpy(),
                             "nsamp": st["nsamp"].detach().cpu().numpy().astype(np.int64),
                             "nb": nb.detach().cpu().numpy().astype(np.int64),
                             "tc": st["train_count"].detach().cpu().numpy() if st.get("train_count") is not None else None}
    return cache


def _pair_plan(st, c, m, t, nb, B):
    """-> (n_cm, sampler) for (client c, model m); sampler(h1, h2) -> (sample index tensor into X[·, c])."""
    v = _np_view(st, nb)
    Wn, nsn, nbn = v["W"], v["nsamp"], v["nb"]
    mode = st.get("sample_mode", "pool")
    if mode == "index":
        cnt = int(v["tc"][m, c])
        if cnt <= 0:
            return 0.0, None
        lst = st["train_index"][m, c, :cnt].long()
        nbm = (cnt + B - 1) // B

        def sampler(h1, h2):
            b = hash_choice(h1, nbm)
            return lst[b * B:min((b + 1) * B, cnt)]
        return float(cnt), sampler
    S = st["X"].shape[2]
    wcol = Wn[: t + 1, m, c]
    nbc, nsc = nbn[: t + 1, c], nsn[: t + 1, c]
    if mode == "time":
        tot = float(wcol.sum())
        if tot <= 0:
            return 0.0, None
        n_cm = float(nbc.sum())
        cum = np.cumsum(wcol.astype(np.float32), dtype=np.float32)

        def sampler(h1, h2):
            u = np.float32(h1 >> 8) * np.float32(1.0 / 16777216.0) * np.float32(cum[-1])
            tt = min(int((cum <= u).sum()), t)
            while int(nbc[tt]) == 0 and tt > 0:
                tt -= 1
            b = hash_choice(h2, max(int(nbc[tt]), 1))
            lo, hi = b * B, min((b + 1) * B, int(nsc[tt]))
            return torch.from_numpy(np.arange(tt * S + lo, tt * S + hi, dtype=np.int64))
        return n_cm, sampler
    n_cm = float((wcol * nbc).sum())
    if n_cm <= 0:
        return 0.0, None
    pool = [(tt, b) for tt in range(t + 1) if wcol[tt] * nbc[tt] > 0 for b in range(int(nbc[tt]))]
    if st.get("n_mode", "batches") == "samples":
        n_cm = float((wcol * nsc).sum())

    def sampler(h1, h2):
        tt, b = pool[hash_choice(h1, len(pool))]
        lo, hi = b * B, min((b + 1) * B, int(nsc[tt]))
        return torch.from_numpy(np.arange(tt * S + lo, tt * S + hi, dtype=np.int64))
    return n_cm, sampler


def fed_round_small(st: Dict, rounds: int = 1) -> Dict[str, torch.Tensor]:
    """Reference semantics of the fused persistent round kernel (csrc/fed_round_small.cu).

    ``st`` keys — spec: kind,din,hid,dout; data: X [T1,C,S,din], Y [T1,C,S] int, nsamp [T1,C] int;
    batch_size; W [T,M,C] float (T ≥ t_cur+1); theta [M,P]; opt_m/opt_v/opt_vmax [C,M,P]; opt_step [C,M] int;
    hyper: lr (float or 1-elem tensor), wd, epochs, optimizer ('adam'|'sgd'), seed, round0, t_cur.
    Training-set selection (``sample_mode``):
      'pool'  — uniform over the batches of every past step t' with W[t',m,c]·nb > 0; n = Σ W·nb
                (``FedAvgEnsTrainerSoftCluster.py:72-113``); ``n_mode='samples'`` weights by Σ W·nsamp instead;
      'time'  — t' ~ W[·,m,c], then a uniform batch of t'; n = Σ_t' nb (``FedAvgEnsTrainerExp.py:55-75``);
      'index' — explicit per-(m,c) sample lists ``train_index [M,C,L]`` / ``train_count [M,C]`` (window concat,
                replication, Poisson bootstrap, client-select); batches are chunks of the list; n = list length
                (``FedAvgEnsTrainer.py:54-75``).
    Optional: ``feat_mask [M,din]`` (training inputs only, KUE), ``recluster_hard`` (IFCA per-round argmax
    re-clustering), ``eval_train_model``/``eval_test_model`` [C] int (-1 → argmax_m W[t,m,c]),
    ``ens_mode`` 0|1 (weighted hard vote)|2 (weighted soft vote) with ``ens_w [C,M]`` for the TEST metric.
    Partial participation: ``participants [rows, K]`` int — round ``round0 + r`` trains only the clients of row
    ``(round0 + r) % rows``; the s-th of them is worker slot s and uses optimizer-state row ``[s, m]`` (the state follows
    the slot across rounds, like the reference's per-worker optimizers); each model is the weighted mean of the slots that
    trained it, in slot order; evaluation still covers all C clients.
    Mutates theta / opt state / W (if recluster) in place; returns ``metrics [rounds, C, 4]`` =
    (train_correct, train_loss_sum, test_correct, test_loss_sum) and ``counts [C, 2]`` = (n_train, n_test).
    """
    kind, din, hid, dout = st["kind"], st["din"], st["hid"], st["dout"]
    X, Y, nsamp, W, theta = st["X"], st["Y"], st["nsamp"], st["W"], st["theta"]
    B, E, t = int(st["batch_size"]), int(st["epochs"]), int(st["t_cur"])
    T1, C, S = X.shape[0], X.shape[1], X.shape[2]
    M, P = theta.shape
    wd = float(st["wd"])
    use_adam = st.get("optimizer", "adam") != "sgd"
    seed, round0 = int(st["seed"]), int(st["round0"])
    nb = (nsamp.to(torch.int64) + B - 1) // B  # [T1, C] batches per (t, c)
    metrics = torch.zeros(rounds, C, 4, dtype=torch.float32)
    feat_mask = st.get("feat_mask")
    ens_mode = int(st.get("ens_mode", 0) or 0)
    Xflat = X.reshape(T1, C, S, -1)
    part = st.get("participants")
    for r in range(rounds):
        rnd = round0 + r
        cur_lr = float(st["lr"])
        Wt = W[t]
        if st.get("sample_mode", "pool") == "index":
            active = (st["train_count"] > 0).any(dim=1)
        else:
            active = (Wt != 0).any(dim=1)  # [M]
        acc_w = torch.zeros(M, dtype=torch.float64)
        locals_: Dict[Tuple[int, int], Tuple[torch.Tensor, float]] = {}   # keyed by (slot, model)
        sampled = range(C) if part is None else [int(c) for c in part[rnd % part.shape[0]]]
        for s, c in enumerate(sampled):
            Xc = Xflat[:, c].reshape(T1 * S, -1)
            Yc = Y[:, c].reshape(T1 * S)
            for m in range(M):
                if not bool(active[m]):
                    continue
                n_cm, sampler = _pair_plan(st, c, m, t, nb, B)
                if n_cm <= 0:
                    continue
                p = theta[m].clone()
                for step in range(E):
                    h1 = batch_hash(seed, rnd, c, m, step)
                    idx = sampler(h1, mix32(h1 ^ 0x68E31DA4))
                    xb, yb = Xc[idx], Yc[idx]
                    if feat_mask is not None:
                        xb = xb * feat_mask[m]
                    _, g = mlp_loss_grad(p, xb, yb, kind, din, hid, dout)
                    if use_adam:
                        st["opt_step"][s, m] = adam_amsgrad_update(
                            p, g, st["opt_m"][s, m], st["opt_v"][s, m], st["opt_vmax"][s, m],
                            int(st["opt_step"][s, m]), cur_lr, wd)
                    else:
                        p.add_(g, alpha=-cur_lr)
                locals_[(s, m)] = (p, n_cm)
                acc_w[m] += n_cm
        for m in range(M):
            if acc_w[m] <= 0:
                continue
            tot = np.float32(acc_w[m])
            out = torch.zeros(P, dtype=torch.float32)
            for s in range(len(sampled)):
                if (s, m) in locals_:
                    p, n_cm = locals_[(s, m)]
                    out += p * (np.float32(n_cm) / tot)
            theta[m] = out
        if st.get("recluster_hard", False):
            corr, _ = mlp_eval_matrix(theta, Xflat[t], Y[t], nsamp[t], kind, din, hid, dout)
            accm = corr / nsamp[t].clamp(min=1).float()
            best = accm.argmax(dim=0)  # first max == np.argmax tie-break
            W[t].zero_()
            W[t][best, torch.arange(C)] = 1.0
            st.pop("_np", None)   # the numpy mirror of W is stale
        pick = W[t].argmax(dim=0)
        etr, ete = st.get("eval_train_model"), st.get("eval_test_model")
        for c in range(C):
            mtr = int(etr[c]) if etr is not None and int(etr[c]) >= 0 else int(pick[c])
            mte = int(ete[c]) if ete is not None and int(ete[c]) >= 0 else int(pick[c])
            k, l = mlp_eval(theta[mtr], Xflat[t, c], Y[t, c], int(nsamp[t, c]), kind, din, hid, dout)
            metrics[r, c, 0], metrics[r, c, 1] = k, l
            if t + 1 < T1:
                n1 = int(nsamp[t + 1, c])
                if ens_mode == 0:
                    k, l = mlp_eval(theta[mte], Xflat[t + 1, c], Y[t + 1, c], n1, kind, din, hid, dout)
                elif n1 > 0:
                    tally = torch.zeros(n1, dout, dtype=torch.float32)
                    for m in range(M):
                        w = float(st["ens_w"][c, m])
                        if w <= 0:
                            continue
                        lg = mlp_forward(theta[m], Xflat[t + 1, c, :n1], kind, din, hid, dout)
                        if ens_mode == 1:
                            tally[torch.arange(n1), lg.argmax(-1)] += np.float32(w)
                        else:
                            tally += np.float32(w) * F.softmax(lg, dim=1)
                    k, l = float((tally.argmax(-1) == Y[t + 1, c, :n1]).sum()), 0.0
                else:
                    k, l = 0.0, 0.0
                metrics[r, c, 2], metrics[r, c, 3] = k, l
    counts = torch.stack([nsamp[t], nsamp[t + 1] if t + 1 < T1 else torch.zeros_like(nsamp[t])], dim=1).float()
    st["round0"] = round0 + rounds
    return {"metrics": metrics, "counts": counts}


# --------------------------------------------------------------------------- K1 / K8 / K10 / K11 / K12
def cluster_aggregate_(theta: torch.Tensor, client_params: torch.Tensor, n: torch.Tensor) -> torch.Tensor:
    """theta [M,P] <- per-model weighted mean of client_params [C,M,P] with weights n [C,M]
    (models whose total weight is 0 are left untouched).  Returns totals [M]."""
    tot = n.double().sum(0)  # [M]
    for m in range(theta.shape[0]):
        if tot[m] > 0:
            w = (n[:, m].double() / tot[m]).float()
            theta[m] = (client_params[:, m, :] * w[:, None]).sum(0)
    return tot.float()


def weighted_average(rows: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
    """rows [n,P], weights [n] -> Σ w_i/Σw · row_i  (plain FedAvg, K1)."""
    w = (weights.double() / weights.double().sum()).to(rows.dtype)
    return (rows * w[:, None]).sum(0)


def _mix32_np(x):
    import numpy as np
    x = x.astype(np.uint32)
    x ^= x >> np.uint32(16)
    x *= np.uint32(0x7FEB352D)
    x ^= x >> np.uint32(15)
    x *= np.uint32(0x846CA68B)
    x ^= x >> np.uint32(16)
    return x


def gauss_hash(seed: int, R: int, P: int) -> torch.Tensor:
    """[R, P] standard-normal noise: Box–Muller on lowbias32 hashes of (seed, row, element) — bit-compatible inputs
    with ``gauss_hash`` in csrc/aggregate.cu (P < 2³²)."""
    import numpy as np
    with np.errstate(over="ignore"):
        i = np.arange(P, dtype=np.uint32)[None, :]
        r = np.arange(R, dtype=np.uint32)[:, None]
        base = _mix32_np(np.uint32(seed & M32) ^ _mix32_np(r * np.uint32(0x9E3779B9) + np.uint32(0x7F4A7C15)))
        h1 = _mix32_np(base ^ (i * np.uint32(2) + np.uint32(1)))
        h2 = _mix32_np(base ^ (i * np.uint32(2) + np.uint32(2)) ^ np.uint32(0x68E31DA4))
    u1 = ((h1 >> np.uint32(8)).astype(np.float64) + 1.0) / 16777216.0
    u2 = (h2 >> np.uint32(8)).astype(np.float64) / 16777216.0
    return torch.from_numpy((np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)).astype(np.float32))


def robust_clip_(rows: torch.Tensor, global_row: torch.Tensor, bound: float, weight_mask=None, stddev: float = 0.0,
                 seed: int = 0) -> torch.Tensor:
    """rows[i] <- global + (rows[i]-global)/max(1, ‖diff‖/bound) (+ stddev·N(0,1)); mask=False entries pass through (K10)."""
    diff = rows - global_row
    d = diff if weight_mask is None else diff * weight_mask
    norm = d.norm(dim=1, keepdim=True)
    scale = 1.0 / torch.clamp(norm / bound, min=1.0)
    new = global_row + diff * scale
    if stddev:
        new = new + stddev * gauss_hash(seed, rows.shape[0], rows.shape[1]).to(rows.device)
    if weight_mask is not None:
        new = torch.where(weight_mask.bool(), new, rows)
    rows.copy_(new)
    return norm.squeeze(1)


def server_opt_step_(theta, avg, state: Dict, opt: str, lr: float, momentum=0.0, b1=0.9, b2=0.999, eps=1e-8):
    """FedOpt (K11): pseudo-gradient g = theta - avg, then one server-optimizer step in place."""
    g = theta - avg
    if opt == "sgd":
        if momentum:
            buf = state.setdefault("momentum", torch.zeros_like(theta))
            buf.mul_(momentum).add_(g)
            g = buf
        theta.add_(g, alpha=-lr)
    elif opt == "adam":
        state["step"] = state.get("step", 0) + 1
        m = state.setdefault("m", torch.zeros_like(theta))
        v = state.setdefault("v", torch.zeros_like(theta))
        m.mul_(b1).add_(g, alpha=1 - b1)
        v.mul_(b2).addcmul_(g, g, value=1 - b2)
        bc1, bc2 = 1 - b1 ** state["step"], 1 - b2 ** state["step"]
        theta.addcdiv_(m, v.sqrt() / math.sqrt(bc2) + eps, value=-lr / bc1)
    elif opt == "adagrad":
        s = state.setdefault("sum", torch.zeros_like(theta))
        s.addcmul_(g, g)
        theta.addcdiv_(g, s.sqrt() + eps, value=-lr)
    elif opt == "yogi":
        state["step"] = state.get("step", 0) + 1
        m = state.setdefault("m", torch.zeros_like(theta))
        v = state.setdefault("v", torch.full_like(theta, 1e-6))
        m.mul_(b1).add_(g, alpha=1 - b1)
        g2 = g * g
        v.sub_((1 - b2) * torch.sign(v - g2) * g2)
        theta.addcdiv_(m, v.sqrt() + eps, value=-lr)
    else:
        raise ValueError(opt)
    return theta


def ada_stats(theta: torch.Tensor, prev_muh: torch.Tensor) -> float:
    """mean((θ - μ̂_{t-1})²) — the only O(P) term of Adaptive-FedAvg's LR rule (K8)."""
    return float(((theta - prev_muh) ** 2).mean())


def gossip_mix(X: torch.Tensor, Wmix: torch.Tensor) -> torch.Tensor:
    """x_i <- Σ_j W_ij x_j over rows (K12)."""
    return Wmix.to(X.dtype) @ X


def merge_axpby_(theta: torch.Tensor, base: int, second: int, w1: float, w2: float) -> None:
    theta[base] = theta[base] * w1 + theta[second] * w2


# --------------------------------------------------------------------------- K4 / K7 (big models: from logits)
def eval_logits(logits: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """-> tensor [3] (correct, loss_sum, count) accumulated on device, no host sync."""
    loss = F.cross_entropy(logits.float(), target.long(), reduction="sum")
    correct = (logits.argmax(-1) == target).sum()
    return torch.stack([correct.float(), loss.float(), torch.tensor(float(target.numel()), device=logits.device)])


def aue_sqerr(logits: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """Σ (1 - softmax(logits)[y])²  (AUE MSE_i numerator)."""
    p = F.softmax(logits.float(), dim=1).gather(1, target.long()[:, None]).squeeze(1)
    return ((1.0 - p) ** 2).sum()


def ensemble_vote(preds: torch.Tensor, weights: torch.Tensor, num_classes: int) -> torch.Tensor:
    """preds [K,B] int hard votes, weights [K] -> argmax_c Σ_k w_k·[pred_k == c]  ([B])."""
    K, B = preds.shape
    tally = torch.zeros(B, num_classes, dtype=torch.float64, device=preds.device)
    for k in range(K):
        tally[torch.arange(B, device=preds.device), preds[k].long()] += float(weights[k])
    return tally.argmax(-1)


def soft_vote(probs: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
    """probs [K,B,C], weights [K] (≤0 entries skipped) -> argmax Σ w_k p_k  (KUE)."""
    w = torch.clamp(weights.to(probs.dtype), min=0)
    return (probs * w[:, None, None]).sum(0).argmax(-1)


def confusion_matrix(pred: torch.Tensor, target: torch.Tensor, num_classes: int) -> torch.Tensor:
    idx = target.long() * num_classes + pred.long()
    return torch.bincount(idx, minlength=num_classes * num_classes).reshape(num_classes, num_classes).double()


def cohen_kappa(A: torch.Tensor) -> float:
    n = float(A.sum())
    left = float(torch.diagonal(A).sum())
    right = float((A.sum(1) * A.sum(0)).sum())
    den = n * n - right
    return (n * left - right) / den if den != 0 else 0.0


# --------------------------------------------------------------------------- K5 / K6
def cluster_distance(acc: np.ndarray, kind: str = "A") -> np.ndarray:
    """FedDrift cluster distance from the L×L cross-accuracy matrix (a_ij = acc of model i on data j)."""
    a = np.asarray(acc, dtype=np.float64)
    d = np.diag(a)
    if kind == "A":
        D = np.maximum(d[:, None] - a, (d[:, None] - a).T)
    else:
        D = np.maximum(d[:, None] - a.T, (d[:, None] - a.T).T)
    return np.maximum(D, 0.0)


def gram_cosine(U: torch.Tensor, eps: float = 1e-12):
    """U [n,P] -> (cosine-similarity [n,n], norms [n])  (CFL, K6)."""
    G = U.double() @ U.double().t()
    nrm = torch.sqrt(torch.diagonal(G))
    return (G / (nrm[:, None] * nrm[None, :] + eps)), nrm


# --------------------------------------------------------------------------- K13..K16
def modp_matmul(A: torch.Tensor, B: torch.Tensor, p: int) -> torch.Tensor:
    """(A @ B) mod p, exact for any p < 2**63 (python-int arithmetic when products could overflow int64)."""
    A, B = A.to(torch.int64) % p, B.to(torch.int64) % p
    if p < (1 << 31):
        out = torch.zeros(A.shape[0], B.shape[1], dtype=torch.int64)
        for k in range(A.shape[1]):  # products < 2^62: reduce per term
            out = (out + (A[:, k:k + 1] * B[k:k + 1, :]) % p) % p
        return out
    An, Bn = A.numpy().astype(object), B.numpy().astype(object)
    return torch.from_numpy((An.dot(Bn) % p).astype(np.int64))


def kd_kl_loss(student_logits, teacher_logits, temperature: float = 1.0):
    """FedGKT distillation loss: T² · KL(softmax(t/T) ‖ softmax(s/T)), batch-mean (K14)."""
    T = temperature
    ls = F.log_softmax(student_logits / T, dim=1)
    pt = F.softmax(teacher_logits / T, dim=1) + 1e-7
    return (T * T) * (pt * (torch.log(pt) - ls)).sum(1).mean()


def vfl_bce_grad(logit_parts: torch.Tensor, y: torch.Tensor):
    """logit_parts [K,B,1] -> (mean BCE-with-logits loss, dL/dlogit [B,1]) for the summed logit (K15)."""
    z = logit_parts.sum(0)
    loss = F.binary_cross_entropy_with_logits(z, y.float(), reduction="mean")
    grad = (torch.sigmoid(z) - y.float()) / z.shape[0]
    return loss, grad


def group_norm(x: torch.Tensor, groups: int, weight=None, bias=None, eps: float = 1e-5):
    return F.group_norm(x, groups, weight, bias, eps)
