"""Drift algorithms as *planners* for the device engine.

Each algorithm owns its state machine (``drift/softcluster.py``, ``drift/states.py``) and, per time step,
emits a training plan for the fused round kernel: the weight tensor ``W[t', m, c]`` (or explicit sample
lists), how batches are sampled, how clients are weighted in the aggregation, which model each client is
evaluated with, and optional ensemble weights.  That one representation covers every algorithm of the
reference's ``FedML_FedAvgEns_data_loader`` dispatch (``FedAvgEnsAPI.py:31-60``) plus the single-model
window baselines of ``fedavg_cont_one`` (README names ``win-1``, ``win-2``, ``all``, SURVEY Appendix A).

| ``--concept_drift_algo``                      | planner            | reference server / client classes            |
| softcluster, softclusterwin-1, softclusterreset| SoftClusterAlgo    | AggregatorSoftCluster / TrainerSoftCluster   |
| win-k / all / weight-* (``--retrain_data``)   | WindowAlgo         | fedavg FedAVGAggregator / FedAVGTrainer      |
| lin, exp                                       | LinExpAlgo         | AggregatorVanilla / TrainerLin, TrainerExp   |
| ada                                            | AdaAlgo            | AggregatorAda / TrainerAda                   |
| aue, auepc                                     | AueAlgo            | AggregatorAue(Pc) / Trainer                  |
| kue                                            | KueAlgo            | AggregatorKue / TrainerKue                   |
| driftsurf                                      | DriftSurfAlgo      | AggregatorDriftSurf / Trainer                |
| mmacc, mmgeni, mmgeniex                        | MultiModelAlgo     | AggregatorMultiModelAcc / Trainer            |
| clusterfl                                      | ClusterFLAlgo      | AggregatorClusterFL / TrainerClusterFL       |
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch

from .. import ops
from ..data import changepoints as cpmod
from ..data.drift import DEFAULT_DELTAS, select_iterations, poisson_bootstrap_index
from ..drift.softcluster import SoftClusterState
from ..drift.states import AdaState, DriftSurfState, KueState, MultiModelAccState, aue_model_num

BIG = 1 << 30


class DriftAlgo:
    """Planner interface."""

    def __init__(self, args, sim):
        self.args, self.sim = args, sim

    # sizing -----------------------------------------------------------------------
    def num_model_slots(self) -> int:
        return 1

    def fused_ok(self) -> bool:
        return True

    def block_size(self, round_in_step: int, remaining: int) -> int:
        """How many rounds may run back-to-back on the device before the host must look."""
        return remaining

    # hooks ------------------------------------------------------------------------
    def begin_step(self, t: int) -> None:
        ...

    def plan(self, t: int) -> Dict:
        raise NotImplementedError

    def after_block(self, t: int, round_in_step: int) -> None:
        ...

    def absorb_weights(self, t: int, W: torch.Tensor) -> None:
        ...

    def end_step(self, t: int) -> None:
        ...

    def state_dict(self) -> Dict:
        return {}

    def load_state_dict(self, d: Dict) -> None:
        ...

    # helpers ----------------------------------------------------------------------
    def _index_plan(self, t: int, per_model_iters, poisson: bool = False) -> Dict:
        """Explicit sample lists: model m at client c trains on the concatenated, shuffled samples of the
        iterations ``per_model_iters[m](c)`` (with multiplicity).  Mirrors ``load_retrain_table_data`` +
        ``batch_data`` (``common/retrain.py``, ``sea/data_loader.py:15-35``)."""
        data = self.sim.data_host
        S = data.X.shape[2]
        M, C = len(per_model_iters), data.client_num
        lists = [[None] * C for _ in range(M)]
        L = 1
        rng = self.sim.rng
        for m in range(M):
            for c in range(C):
                idx: List[np.ndarray] = []
                for it in per_model_iters[m](c):
                    n = int(data.nsamp[it, c])
                    base = np.arange(n, dtype=np.int64)
                    if poisson:
                        pb = poisson_bootstrap_index(n, rng)
                        if pb is not None:
                            base = pb.numpy()
                    idx.append(it * S + base)
                flat = np.concatenate(idx) if idx else np.zeros(0, dtype=np.int64)
                flat = flat[rng.permutation(len(flat))] if len(flat) else flat
                lists[m][c] = flat
                L = max(L, len(flat))
        ti = torch.zeros(M, C, L, dtype=torch.int32)
        tc = torch.zeros(M, C, dtype=torch.int32)
        for m in range(M):
            for c in range(C):
                n = len(lists[m][c])
                ti[m, c, :n] = torch.from_numpy(lists[m][c].astype(np.int32))
                tc[m, c] = n
        W = torch.zeros(t + 1, M, C)
        W[t] = (tc > 0).float()  # only used for "model active" + default eval routing
        dev = self.sim.device
        return {"W": W, "sample_mode": "index", "train_index": ti.to(dev), "train_count": tc.to(dev)}


# =============================================================================== soft-cluster family
class SoftClusterAlgo(DriftAlgo):
    def __init__(self, args, sim):
        super().__init__(args, sim)
        cps = None
        if args.concept_drift_algo_arg == "geni":
            cps = cpmod.load(args.change_points, args.total_train_iteration, args.client_num_in_total,
                             bool(args.drift_together), args.time_stretch)
        self.state = SoftClusterState.from_args(args, cps, rng=np.random.RandomState(int(args.dummy_arg)),
                                                sink=sim.sink, max_steps=args.total_train_iteration + 2)
        self.arg = args.concept_drift_algo_arg

    def num_model_slots(self) -> int:
        return int(self.args.concept_num)

    def fused_ok(self) -> bool:
        return "cfl" not in self.arg  # CFL inspects raw client updates before aggregating

    def block_size(self, round_in_step, remaining):
        return 1 if "cfl" in self.arg else remaining

    def begin_step(self, t: int) -> None:
        sim, st, a = self.sim, self.state, self.args
        bank, ev = sim.bank, sim.evaluator
        arg = self.arg
        if "H" in arg:
            st.cluster_init() if t == 0 else st.cluster_hierarchical(t, bank, ev)
        elif "cfl" in arg:
            st.cluster_init() if t == 0 else st.cluster_cfl_init(t)
        elif "hard" in arg:
            if t == 0:  # IFCA needs distinct starting models
                g = torch.Generator().manual_seed(int(a.dummy_arg) + 12345)
                for m in range(bank.num_models):
                    bank.reset_parameters_random(m, g)
            st.cluster(ev.acc_matrix(list(range(bank.num_models)), t), t, 0)
        elif "mmacc" in arg:
            st.cluster_init() if t == 0 else st.cluster_mmacc2(t, bank, ev)
        else:
            if t == 0:
                st.cluster_init()
            else:
                acc = ev.acc_matrix(list(range(bank.num_models)), t)
                if a.concept_drift_algo == "softclusterreset":
                    deleted: List[int] = []
                    for m in reversed(range(bank.num_models)):
                        rest = np.delete(acc, deleted + [m], axis=0)
                        if rest.shape[0] > 0 and np.all(acc[m] < np.max(rest, axis=0) + 0.01):
                            deleted.append(m)
                            sim.sink.set_summary(f"Reset-{m}", 1)
                            st.set_weights_zero_model(m)
                            bank.reinit(m)
                    if deleted:
                        acc = ev.acc_matrix(list(range(bank.num_models)), t)
                st.cluster(acc, t, 0)
        if a.concept_drift_algo == "softclusterwin-1":
            st.set_weights_win1(t)
        if t == 0:  # initialise the drift detector's reference accuracies
            pick = st.test_model_indices(0)
            acc = ev.acc_matrix(sorted(set(int(p) for p in pick)), 0)
            rows = {m: r for r, m in enumerate(sorted(set(int(p) for p in pick)))}
            for c in range(st.client_num):
                st.set_acc(c, acc[rows[int(pick[c])], c])

    def plan(self, t: int) -> Dict:
        return {"W": self.state.weights_tensor(t), "sample_mode": "pool", "n_mode": "batches",
                "recluster_hard": self.arg == "hard-r"}

    def absorb_weights(self, t: int, W: torch.Tensor) -> None:
        self.state.W[t] = W[t].detach().cpu().double().numpy()

    def state_dict(self):
        return {"sc_state": self.state.state_dict()}

    def load_state_dict(self, d):
        self.state.load_state_dict(d["sc_state"])


# =============================================================================== single-model baselines
class WindowAlgo(DriftAlgo):
    """``fedavg_cont_one``: one model, ``--retrain_data`` ∈ all | win-k | weight-linear | weight-exp | sel-…"""

    def plan(self, t: int) -> Dict:
        method = self.args.retrain_data
        return self._index_plan(t, [lambda c, m=method: select_iterations(m, t, c)])


class LinExpAlgo(DriftAlgo):
    def plan(self, t: int) -> Dict:
        C = self.sim.C
        w = torch.tensor([2.0 ** i if self.args.concept_drift_algo == "exp" else float(i + 1)
                          for i in range(t + 1)])
        return {"W": w[:, None, None].expand(t + 1, 1, C).contiguous(), "sample_mode": "time"}


class AdaAlgo(DriftAlgo):
    def __init__(self, args, sim):
        super().__init__(args, sim)
        self.state = AdaState(init_lr=args.lr)
        parts = args.concept_drift_algo_arg.split("_")
        self.retrain = parts[0]
        if parts[1] not in ("round", "iter"):
            raise NameError("ada config")
        self.each_round = parts[1] == "round"
        self.lr_dev: Optional[torch.Tensor] = None

    def block_size(self, round_in_step, remaining):
        if self.each_round:
            return 1
        gate = self.args.comm_round - 5  # update once per iteration at round R-5
        if round_in_step <= gate:
            return min(remaining, gate - round_in_step + 1)
        return remaining

    def plan(self, t: int) -> Dict:
        p = self._index_plan(t, [lambda c: select_iterations(self.retrain, t, c)])
        p["optimizer"] = "sgd"  # TrainerAda forces SGD
        p["lr"] = self.state.current_lr()
        return p

    def after_block(self, t: int, round_in_step: int) -> None:
        a = self.args
        r = round_in_step - 1
        if self.each_round:
            self.state.update(self.sim.bank.theta[0], r + t * a.comm_round)
        elif r == a.comm_round - 5:
            self.state.update(self.sim.bank.theta[0], t)
        if self.sim._small is not None:
            self.sim._small["lr"] = self.state.current_lr()

    def state_dict(self):
        s = self.state
        return {"ada": {"eta": s.eta, "mu": s.mu, "s": s.s, "gam": s.gam, "init_lr": s.init_lr}}

    def load_state_dict(self, d):
        for k, v in d["ada"].items():
            setattr(self.state, k, v)


# =============================================================================== ensembles
class AueAlgo(DriftAlgo):
    EPS = 1e-20

    def __init__(self, args, sim):
        super().__init__(args, sim)
        self.per_client = args.concept_drift_algo == "auepc"
        self.ens_w: Optional[torch.Tensor] = None
        self.K = 1

    def num_model_slots(self) -> int:
        return int(self.args.ensemble_window)

    def block_size(self, round_in_step, remaining):
        R = self.args.comm_round
        if round_in_step > R - 10:
            return 1
        nxt = (round_in_step // 10) * 10  # weights refresh after rounds 0, 10, 20, …
        nxt = nxt if nxt >= round_in_step else nxt + 10
        return max(1, min(remaining, nxt - round_in_step + 1, (R - 10) - round_in_step + 1))

    def begin_step(self, t: int) -> None:
        bank = self.sim.bank
        self.K = aue_model_num(t, self.args.ensemble_window)
        if t > 0 and not self.args.reset_models:  # circular shift: model k ← previous model k-1; slot 0 fresh
            for k in range(self.K - 1, 0, -1):
                bank.copy(k, k - 1)
        bank.reinit(0)
        mser = (1 - 1.0 / self.sim.data.class_num) ** 2
        w = torch.zeros(self.sim.C, bank.num_models)
        w[:, : self.K] = 1.0 / (mser + self.EPS)
        self.ens_w = w / w.sum(1, keepdim=True)

    def plan(self, t: int) -> Dict:
        iters = [(lambda c, k=k: select_iterations(f"win-{k + 1}", t, c)) if k < self.K else (lambda c: [])
                 for k in range(self.sim.bank.num_models)]
        p = self._index_plan(t, iters)
        C = self.sim.C
        p.update(ens_mode=1, ens_w=self.ens_w.to(self.sim.device),
                 eval_train_model=torch.zeros(C, dtype=torch.int32, device=self.sim.device))
        return p

    def after_block(self, t: int, round_in_step: int) -> None:
        r, R = round_in_step - 1, self.args.comm_round
        if not (r % 10 == 0 or r > R - 10):
            return
        sim = self.sim
        s = sim.spec
        C, mser = sim.C, (1 - 1.0 / sim.data.class_num) ** 2
        sq = torch.zeros(self.K, C, dtype=torch.float64)
        for k in range(1, self.K):  # MSE_i of every older model on the newest data
            for c in range(C):
                n = int(sim.data.nsamp[t, c])
                logits = sim.bank.forward(k, sim.data.X[t, c, :n])
                sq[k, c] = float(ops.aue_sqerr(logits, sim.data.Y[t, c, :n]))
        ns = sim.data.nsamp[t].double().cpu()
        w = torch.zeros(C, sim.bank.num_models, dtype=torch.float64)
        w[:, 0] = 1.0 / (mser + self.EPS)  # the newest model gets the "perfect" score
        for k in range(1, self.K):
            if self.per_client:
                msei = torch.where(ns > 0, sq[k] / ns.clamp(min=1), torch.zeros_like(ns))
            else:
                tot = ns.sum()
                msei = torch.full_like(ns, float(sq[k].sum() / tot) if tot > 0 else 0.0)
            w[:, k] = 1.0 / (mser + msei + self.EPS)
        if getattr(self.args, "strict_ref", 0) and self.K > 1:
            # reference off-by-one (FedAvgEnsAggregatorAue.py:65-79): model k's weight lands on index k-1,
            # index 0 is then overwritten by the perfect score and index K-1 keeps its previous value
            shifted = w.clone()
            shifted[:, : self.K - 1] = w[:, 1: self.K]
            shifted[:, 0] = 1.0 / (mser + self.EPS)
            shifted[:, self.K - 1] = self.ens_w[:, self.K - 1].double()
            w = shifted
        w = w / w.sum(1, keepdim=True)
        self.ens_w = w.float()
        if sim._small is not None:
            sim._small["ens_w"] = self.ens_w.to(sim.device)


class KueAlgo(DriftAlgo):
    def __init__(self, args, sim):
        super().__init__(args, sim)
        self.state = KueState(args.concept_num, sim.data_host.feature_num, np.random.RandomState(int(args.dummy_arg)))
        self.kappa = np.ones(args.concept_num)

    def num_model_slots(self) -> int:
        return int(self.args.concept_num)

    block_size = AueAlgo.block_size

    def begin_step(self, t: int) -> None:
        if t != 0:
            worst = self.state.get_worst_idx()
            self.state.initialize_mask(worst)
            self.sim.bank.reinit(worst)

    def _ens(self) -> torch.Tensor:
        w = torch.tensor(self.kappa, dtype=torch.float32).clamp(min=0)
        w[self.state.get_worst_idx()] = 0.0
        return w[None, :].expand(self.sim.C, -1).contiguous()

    def plan(self, t: int) -> Dict:
        M = self.sim.bank.num_models
        p = self._index_plan(t, [lambda c: [t]] * M, poisson=True)
        self._train_lists = (p["train_index"], p["train_count"])
        dev = self.sim.device
        p.update(feat_mask=self.state.masks_tensor(dev), ens_mode=2, ens_w=self._ens().to(dev),
                 eval_train_model=torch.zeros(self.sim.C, dtype=torch.int32, device=dev))
        return p

    def after_block(self, t: int, round_in_step: int) -> None:
        r, R = round_in_step - 1, self.args.comm_round
        if not (r % 10 == 0 or r > R - 10):
            return
        sim, K = self.sim, sim_classes(self.sim)
        ti, tc = self._train_lists
        masks = self.state.masks_tensor(sim.device)
        S = sim.data.X.shape[2]
        for m in range(sim.bank.num_models):
            A = torch.zeros(K, K, dtype=torch.float64)
            for c in range(sim.C):
                n = int(tc[m, c])
                if n == 0:
                    continue
                idx = ti[m, c, :n].long()
                Xc = sim.data.X[:, c].reshape(-1, sim.data.feature_num)
                Yc = sim.data.Y[:, c].reshape(-1)
                logits = sim.bank.forward(m, Xc[idx] * masks[m])
                A += ops.confusion_matrix(logits.argmax(-1), Yc[idx], K).cpu()
            self.kappa[m] = ops.cohen_kappa(A)
        if t != 0:
            self.state.set_worst_idx(int(np.argmin(self.kappa)))
        if sim._small is not None:
            sim._small["ens_w"] = self._ens().to(sim.device)

    def state_dict(self):
        # the mask RNG is part of the state: a resumed run must draw the same feature subspaces as an uninterrupted one
        return {"kue": {"masks": self.state.masks.copy(), "worst": self.state.worst_idx, "kappa": self.kappa.copy(),
                        "rng": self.state.rng.get_state()}}

    def load_state_dict(self, d):
        self.state.masks, self.state.worst_idx, self.kappa = d["kue"]["masks"], d["kue"]["worst"], d["kue"]["kappa"]
        if d["kue"].get("rng") is not None:
            self.state.rng.set_state(d["kue"]["rng"])


def sim_classes(sim) -> int:
    return int(sim.data.class_num)


# =============================================================================== DriftSurf
class DriftSurfAlgo(DriftAlgo):
    DELTAS = {"sea": 0.02, "sine": 0.10, "circle": 0.05}

    def __init__(self, args, sim):
        super().__init__(args, sim)
        d = 0.01 * float(args.concept_drift_algo_arg or 0)
        if d == 0:
            d = self.DELTAS.get(args.dataset, 0.05)
        self.state = DriftSurfState(delta=d)
        self.test_idx = 0

    def num_model_slots(self) -> int:
        return 3  # two trained models + one scratch row for scoring snapshots

    def begin_step(self, t: int) -> None:
        st, bank = self.state, self.sim.bank
        if t > 0:
            st.run_ds_algo(bank, self.sim.evaluator, t, scratch_row=2)
            if not self.args.reset_models:
                for idx, key in enumerate(st.get_train_keys()):
                    snap = st.snapshots[key]
                    if snap is not None:
                        bank.theta[idx].copy_(snap.to(bank.device))
                    else:
                        bank.reinit(idx)
        self.keys = list(st.get_train_keys())
        self.test_idx = self.keys.index(st.get_model_key()) if st.get_model_key() in self.keys else 0

    def plan(self, t: int) -> Dict:
        st = self.state
        lists = [st.get_train_data(k) or [] for k in self.keys]
        if t == 0:
            lists = [[0], [0]]
        iters = [(lambda c, l=l: list(l)) for l in lists] + [lambda c: []]
        p = self._index_plan(t, iters)
        ev = torch.full((self.sim.C,), self.test_idx, dtype=torch.int32, device=self.sim.device)
        p.update(eval_train_model=ev, eval_test_model=ev.clone())
        return p

    def end_step(self, t: int) -> None:
        for idx, key in enumerate(self.keys):
            self.state.set_snapshot(key, self.sim.bank.theta[idx])

    def state_dict(self):
        s = self.state
        return {"ds": {k: getattr(s, k) for k in ("snapshots", "train_data_dict", "train_keys", "acc_best", "acc_dict",
                                                 "reac_ctr", "state", "model_key")}}

    def load_state_dict(self, d):
        for k, v in d["ds"].items():
            setattr(self.state, k, v)


# =============================================================================== legacy multi-model + oracles
class MultiModelAlgo(DriftAlgo):
    def __init__(self, args, sim):
        super().__init__(args, sim)
        delta = DEFAULT_DELTAS.get(args.dataset, 0.1)
        self.state = MultiModelAccState(args.client_num_in_total, args.concept_num, delta)
        self.cps = None
        if args.concept_drift_algo in ("mmgeni", "mmgeniex"):
            self.cps = cpmod.load(args.change_points, args.total_train_iteration, args.client_num_in_total,
                                  bool(args.drift_together), args.time_stretch)

    def num_model_slots(self) -> int:
        return int(self.args.concept_num)

    def begin_step(self, t: int) -> None:
        algo, st = self.args.concept_drift_algo, self.state
        if algo == "mmacc":
            st.run_model_select(self.sim.evaluator if t > 0 else None, t)
        elif algo == "mmgeni":
            st.model_select_geni(t, self.cps, self.args.time_stretch)
        else:
            st.model_select_geniex(t, self.cps, self.args.time_stretch)
        for m in range(self.args.concept_num):
            if st.get_train_data_by_model(m) != "":
                st.set_model(m)

    def plan(self, t: int) -> Dict:
        st = self.state
        iters = [(lambda c, m=m: list(st.train_data_dict[m][c])) for m in range(self.args.concept_num)]
        p = self._index_plan(t, iters)
        dev = self.sim.device
        p["eval_train_model"] = torch.tensor([st.get_train_model_idx(c) for c in range(self.sim.C)],
                                             dtype=torch.int32, device=dev)
        p["eval_test_model"] = torch.tensor([st.get_test_model_idx(c) for c in range(self.sim.C)],
                                            dtype=torch.int32, device=dev)
        return p

    def end_step(self, t: int) -> None:
        # the per-client training accuracy of the last tested round is the detector's baseline (…MultiModelAcc.py:143)
        hist = self.sim.sink
        for c in range(self.sim.C):
            v = hist.last(f"Train/Acc-CL-{c}")
            if v is not None and v >= 0:
                self.state.set_acc(c, v)

    def state_dict(self):
        s = self.state
        return {"mm": {k: getattr(s, k) for k in ("train_data_dict", "models", "train_model_idx", "test_model_idx",
                                                 "acc_dict")}}

    def load_state_dict(self, d):
        for k, v in d["mm"].items():
            setattr(self.state, k, v)


class ClusterFLAlgo(DriftAlgo):
    """Legacy one-shot CFL (``FedAvgEnsAggregatorClusterFL.py``): a single split check after round 100."""

    def __init__(self, args, sim):
        super().__init__(args, sim)
        self.assign = np.zeros(args.client_num_in_total, dtype=np.int64)
        self.split_done = False
        self.split_round = 100

    def num_model_slots(self) -> int:
        return int(self.args.concept_num)

    def fused_ok(self) -> bool:
        return self.split_done or self.sim.round_in_step != self.split_round

    def block_size(self, round_in_step, remaining):
        if self.split_done:
            return remaining
        if round_in_step < self.split_round:
            return min(remaining, self.split_round - round_in_step)
        return 1

    def plan(self, t: int) -> Dict:
        retrain = self.args.concept_drift_algo_arg or "win-1"
        iters = [(lambda c, m=m: select_iterations(retrain, t, c) if self.assign[c] == m else [])
                 for m in range(self.args.concept_num)]
        return self._index_plan(t, iters)

    def state_dict(self):
        return {"clusterfl": {"assign": self.assign.copy(), "split_done": bool(self.split_done)}}

    def load_state_dict(self, d):
        if "clusterfl" in d:
            self.assign = np.asarray(d["clusterfl"]["assign"], dtype=np.int64).copy()
            self.split_done = bool(d["clusterfl"]["split_done"])

    def on_client_updates(self, t: int, client_params: torch.Tensor, n: torch.Tensor,
                          clients: Optional[List[int]] = None) -> bool:
        """Called by the generic path at the split round with raw local models; returns True if split.  Under partial
        participation row s holds the update of client ``clients[s]`` and only those clients can move (``None``: row c is
        client c)."""
        from ..drift.hclust import complete_linkage_bipartition
        self.split_done = True
        if clients is None:
            members = np.nonzero(self.assign == 0)[0]
            rows = members.tolist()
        else:
            rows = [s for s, c in enumerate(clients) if self.assign[c] == 0]
            members = np.asarray([clients[s] for s in rows], dtype=np.int64)
        if len(members) < 2 or self.args.concept_num < 2:
            return False
        U = client_params[rows, 0, :] - self.sim.bank.theta[0][None, :]
        S, norms = ops.gram_cosine(U)
        self.sim.sink.log({"Max_Norm": float(norms.max()), "Mean_Norm": float(U.mean(0).norm()),
                           "round": self.sim.round_in_step})
        g1, g2 = complete_linkage_bipartition(S.cpu().numpy())
        for i in g2:
            self.assign[members[i]] = 1
        self.sim.bank.copy(1, 0)
        self.sim.invalidate_plan()  # re-plan with the new assignment
        return True


# =============================================================================== factory
def make_algo(args, sim) -> DriftAlgo:
    name = args.concept_drift_algo
    if name in ("softcluster", "softclusterwin-1", "softclusterreset"):
        return SoftClusterAlgo(args, sim)
    if name in ("win", "window", "fedavg", "all", "") or name.startswith("win-") or name.startswith("weight-"):
        if name.startswith("win-") or name.startswith("weight-") or name == "all":
            args.retrain_data = name
        return WindowAlgo(args, sim)
    if name in ("lin", "exp"):
        return LinExpAlgo(args, sim)
    if name == "ada":
        return AdaAlgo(args, sim)
    if name in ("aue", "auepc"):
        return AueAlgo(args, sim)
    if name == "kue":
        return KueAlgo(args, sim)
    if name == "driftsurf":
        return DriftSurfAlgo(args, sim)
    if name in ("mmacc", "mmgeni", "mmgeniex"):
        return MultiModelAlgo(args, sim)
    if name == "clusterfl":
        return ClusterFLAlgo(args, sim)
    raise NameError("concept_drift_algo")
