"""Python side of the fused persistent round kernel (``csrc/fed_round_small.cu``): packs the state dict
into the launch arguments, keeps the metrics on device, and (multi-GPU) wires the symmetric inbox/flag
buffers.  One call == one kernel launch == ``rounds`` complete FL rounds."""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _ext

KIND_ID = {"lr": 0, "fnn": 1}
MODE_ID = {"pool": 0, "time": 1, "index": 2}
LAUNCH_COUNT = {"fed_round_small": 0}


def supported(kind: str, din: int, hid: int, dout: int) -> bool:
    ext = _ext.load()
    return ext is not None and bool(ext.fed_round_small_supported(KIND_ID[kind], din, hid, dout))


def fits(kind: str, din: int, hid: int, dout: int, C: int, M: int, t_cur: int) -> bool:
    """True when the fused kernel can run this federation at time step ``t_cur`` (instantiated MLP shape, ``t_cur`` below
    the kernel's plan-table limit, shared-memory layout within 227 KB); otherwise route to the generic executor."""
    ext = _ext.load()
    if ext is None:
        return True   # CPU reference has no such limits
    return bool(ext.fed_round_small_fits(KIND_ID[kind], din, hid, dout, int(C), int(M), int(t_cur)))


def spin_timeout_ms(st: Dict) -> int:
    """Cross-GPU spin bound: generous by default (a peer may legitimately be busy for seconds in host-side clustering or
    a CUDA-graph build); ``FDB_SPIN_TIMEOUT_MS`` / ``st['spin_timeout_ms']`` override it."""
    import os
    return int(st.get("spin_timeout_ms") or os.environ.get("FDB_SPIN_TIMEOUT_MS", 60000))


def _i32(t: Optional[torch.Tensor], dev) -> Optional[torch.Tensor]:
    if t is None:
        return None
    return t.to(device=dev, dtype=torch.int32).contiguous()


def _f32(t: Optional[torch.Tensor], dev) -> Optional[torch.Tensor]:
    if t is None:
        return None
    return t.to(device=dev, dtype=torch.float32).contiguous()


def check_participants(table, C: int) -> None:
    """Raise ``ValueError`` unless ``table`` is a valid partial-participation table for ``C`` clients: int32 ``[rows, K]``
    with ``1 ≤ K ≤ C``, every id in ``[0, C)`` and the ids of each row distinct."""
    if not isinstance(table, torch.Tensor) or table.dtype != torch.int32 or table.dim() != 2:
        raise ValueError("participants must be an int32 tensor of shape [rows, K]")
    rows, K = table.shape
    if rows < 1 or not 1 <= K <= C:
        raise ValueError(f"participants table of shape {tuple(table.shape)}: need at least one row and 1 <= K <= {C}")
    h = table.detach().cpu()
    if int(h.min()) < 0 or int(h.max()) >= C:
        raise ValueError(f"participants table holds client ids outside [0, {C})")
    if K > 1 and bool((h.sort(dim=1).values.diff(dim=1) == 0).any()):
        raise ValueError("participants table lists a client twice in one round")


def prepare(st: Dict) -> Dict:
    """Build (once per time step) the device views the kernel reads: fp32 X, int32 Y / nsamp / index tables."""
    cache = st.setdefault("_native", {})
    if not cache:
        theta = st["theta"]
        dev = theta.device
        X = st["X"]
        T1, C, S = X.shape[0], X.shape[1], X.shape[2]
        cache["X"] = X.reshape(T1, C, S, -1).to(torch.float32).contiguous()
        cache["Y"] = _i32(st["Y"], dev)
        cache["nsamp"] = _i32(st["nsamp"], dev)
        cache["train_index"] = _i32(st.get("train_index"), dev)
        cache["train_count"] = _i32(st.get("train_count"), dev)
        cache["feat_mask"] = _f32(st.get("feat_mask"), dev)
        cache["eval_train_model"] = _i32(st.get("eval_train_model"), dev)
        cache["eval_test_model"] = _i32(st.get("eval_test_model"), dev)
        part = st.get("participants")
        if part is not None:
            check_participants(part, C)
            cache["participants"] = part.to(dev).contiguous()
        # launch shape hints: warps per pair from the mini-batch size, cluster size from the active pair count
        B, t = int(st["batch_size"]), int(st["t_cur"])
        bmax = min(B, int(cache["nsamp"].max()))
        cache["wpp"] = 4 if bmax > 64 else (2 if bmax > 32 else 1)
        P = theta.shape[1]
        nwarps = 16 if P <= 24 else (12 if P <= 40 else 8)
        groups = max(1, nwarps // cache["wpp"])
        if st.get("recluster_hard"):
            npairs = C * theta.shape[0]
        elif st.get("sample_mode", "pool") == "index":
            npairs = int((cache["train_count"] > 0).sum())
        else:
            Wc = st["W"][: t + 1].detach().float().cpu()
            active = (Wc[t] != 0).any(dim=1)
            npairs = int(((Wc.sum(0) > 0) & active[:, None]).sum())
        if part is not None:   # at most K·M pairs train in a round
            npairs = min(npairs, int(part.shape[1]) * theta.shape[0])
        mg = st.get("multi_gpu")
        if mg:
            npairs = -(-npairs // int(mg["world"]))
        G = 1
        while G < 8 and G * groups < npairs:
            G *= 2
        cache["cluster"] = G
        cache["counts"] = torch.stack(
            [cache["nsamp"][st["t_cur"]],
             cache["nsamp"][st["t_cur"] + 1] if st["t_cur"] + 1 < T1 else torch.zeros_like(cache["nsamp"][0])],
            dim=1).float()
    return cache


def run_native(st: Dict, rounds: int, metrics_out: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    ext = _ext.load(required=True)
    theta = st["theta"]
    dev = theta.device
    X, W = st["X"], st["W"]
    T1, C, S = X.shape[0], X.shape[1], X.shape[2]
    M = theta.shape[0]
    cache = prepare(st)
    if not (W.is_cuda and W.dtype == torch.float32 and W.is_contiguous()):
        st["W"] = W = W.to(device=dev, dtype=torch.float32).contiguous()
    ens_w = _f32(st.get("ens_w"), dev)
    use_adam = st.get("optimizer", "adam") != "sgd"
    if metrics_out is None:
        metrics_out = torch.zeros(rounds, C, 4, dtype=torch.float32, device=dev)
    lr = st["lr"]
    lr_dev = lr if isinstance(lr, torch.Tensor) else None
    Lmax = int(cache["train_index"].shape[2]) if cache["train_index"] is not None else 0
    mg = st.get("multi_gpu")  # dict(world, rank, inbox_ptrs, metrics_ptrs, flag_base, error_flag)
    world = int(mg["world"]) if mg else 1
    icfg = [T1, C, S, M, Lmax, int(st["batch_size"]), int(st["epochs"]), int(st["t_cur"]), int(rounds), int(st["round0"]),
            int(st["seed"]) & 0xFFFFFFFF, int(use_adam), MODE_ID[st.get("sample_mode", "pool")],
            1 if st.get("n_mode", "batches") == "samples" else 0, int(bool(st.get("recluster_hard", False))),
            int(st.get("ens_mode", 0) or 0), int(bool(st.get("skip_aggregate", False))), world,
            int(mg["rank"]) if mg else 0, int(mg["flag_base"]) if mg else 0, int(st.get("cluster", 0) or cache["cluster"]),
            spin_timeout_ms(st), int(st.get("warps_per_pair", 0) or cache["wpp"])]
    fcfg = [float(lr) if lr_dev is None else 0.0, float(st["wd"]), 0.9, 0.999, 1e-8]
    peer_metrics = []
    if mg and mg.get("metrics_ptrs") is not None:
        # every rank's LL staging area (symmetric); the kernel compacts this launch's rows into the plain metrics_out
        assert rounds <= int(mg["metrics_rounds"]), "block larger than the symmetric metrics staging area"
        peer_metrics = list(mg["metrics_ptrs"])
    info = ext.fed_round_small(
        KIND_ID[st["kind"]], int(st["din"]), int(st["hid"]), int(st["dout"]), cache["X"], cache["Y"], cache["nsamp"], W, theta,
        int(st.get("theta_stride", theta.stride(0))), st.get("opt_m"), st.get("opt_v"), st.get("opt_vmax"), st["opt_step"],
        cache["train_index"], cache["train_count"], cache["feat_mask"], cache["eval_train_model"], cache["eval_test_model"],
        ens_w, st.get("client_out"), lr_dev, metrics_out, st.get("timers"), fcfg, icfg,
        list(mg["inbox_ptrs"]) if mg else [], mg.get("error_flag") if mg else None,
        st.get("counters"), peer_metrics, [int(v) for v in st["host_io"]] if st.get("host_io") else [],
        cache.get("participants"))
    if mg:
        mg["flag_base"] = int(mg["flag_base"]) + rounds
    if st.get("counters") is not None:
        st["_counter_rounds"] = st.get("_counter_rounds", 0) + rounds
    LAUNCH_COUNT["fed_round_small"] += 1
    st["round0"] = int(st["round0"]) + rounds
    st["_launch_info"] = info
    return {"metrics": metrics_out, "counts": cache["counts"]}
