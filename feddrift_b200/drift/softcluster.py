"""Soft-cluster drift state — the FedDrift brain.

Behavioural parity with ``SoftClusterState`` (``fedml_api/distributed/fedavg_ens/FedAvgEnsDataLoader.py:581-1269``)
and its arg-string grammar (``SoftCluster_data_loader`` ``:1272-1341``), re-designed around a dense weight
tensor ``W[t, m, c]`` (time × model × client) that is mirrored to the device for the fused round kernel,
and around a :class:`ModelBank` (flat parameter rows) instead of lists of ``nn.Module``:

* clone-on-drift = one row copy, merge = one fused axpby over rows (``ops.merge_axpby_``, K5),
  re-initialise = one row copy from the cached init row;
* every accuracy the algorithms look at comes from :class:`Evaluator` (one K4 launch per matrix).

Algorithms: ``hard`` / ``hard-r`` (IFCA), ``softmax_α``, ``mmacc_δ`` (FedDrift-Eager), ``gmm``, ``geni``
(oracle), ``cfl_γ_{win-1|all}`` (Clustered FL), ``H_{A|B}_{C|D|E|F}_W_δ_δ'`` (FedDrift hierarchical).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import ops
from ..data.drift import DEFAULT_DELTAS
from ..parallel.arena import ModelBank
from ..utils.metrics import MetricsSink, get_sink
from .evaluator import Evaluator
from .hclust import complete_linkage_bipartition, linkage_fcluster

_FRESH = -42  # "no drift seen yet this step" marker for the eager variant


def parse_algo_arg(cluster_alg: str, dataset: str = "", change_points: Optional[np.ndarray] = None,
                   time_stretch: int = 1) -> Dict:
    """Decode ``--concept_drift_algo_arg`` (grammar: SURVEY §2.3 / reference ``:1292-1313``)."""
    cfg = dict(cluster_alg=cluster_alg, mmacc_delta=0.0, softmax_alpha=0, geni_change_points=None, geni_stretch=1,
               h_delta=0.0, h_deltap=0.0, h_w=0, h_distance="", h_cluster="", cfl_gamma=0.0, cfl_retrain="")
    parts = cluster_alg.split("_")
    default = DEFAULT_DELTAS.get(dataset)
    if "mmacc" in cluster_alg:
        d = 0.01 * float(parts[-1])
        cfg["mmacc_delta"] = default if (d == 0 and default is not None) else d
    elif "softmax" in cluster_alg:
        cfg["softmax_alpha"] = int(parts[-1])
    elif cluster_alg == "geni":
        cfg["geni_change_points"], cfg["geni_stretch"] = change_points, time_stretch
    elif "H" in cluster_alg:
        cfg["h_distance"], cfg["h_cluster"], cfg["h_w"] = parts[1], parts[2], int(parts[3])
        d = 0.01 * float(parts[4])
        cfg["h_delta"] = default if (d == 0 and default is not None) else d
        dp = 0.01 * float(parts[5])
        cfg["h_deltap"] = cfg["h_delta"] if dp == 0 else dp
    elif "cfl" in cluster_alg:
        cfg["cfl_gamma"], cfg["cfl_retrain"] = float(parts[1]), parts[2]
    return cfg


class SoftClusterState:
    def __init__(self, client_num: int, model_num: int = 2, cluster_alg: str = "softmax_0", mmacc_delta: float = 0.1,
                 softmax_alpha: int = 0, geni_change_points=None, geni_stretch: int = 1, h_delta: float = 0.1,
                 h_deltap: float = 0.1, h_w: int = 1, h_distance: str = "A", h_cluster: str = "C",
                 cfl_gamma: float = 0.1, cfl_retrain: str = "win-1", max_steps: int = 64,
                 rng: Optional[np.random.RandomState] = None, sink: Optional[MetricsSink] = None):
        self.client_num, self.model_num = client_num, model_num
        self.W = np.zeros((max_steps, model_num, client_num), dtype=np.float64)  # train_data_weights
        self.steps: set = set()  # time steps that have a weight matrix ("dict keys" of the reference)
        self.cluster_alg = cluster_alg
        self.mmacc_delta, self.softmax_alpha = mmacc_delta, softmax_alpha
        self.prev_acc: Dict[int, float] = {}  # mmacc_acc_dict
        self.geni_change_points, self.geni_stretch = geni_change_points, geni_stretch
        self.h_delta, self.h_deltap, self.h_w = h_delta, h_deltap, h_w
        self.h_distance, self.h_cluster = h_distance, h_cluster
        self.h_marked: Dict[int, Tuple[int, int]] = {}  # client -> (private model, time to unmark)
        self.h_next_free_model = 1
        self.cfl_gamma, self.cfl_retrain = cfl_gamma, cfl_retrain
        self.cfl_norm, self.cfl_eps1, self.cfl_eps2 = 0.0, 0.0, 10000.0
        self.rng = rng if rng is not None else np.random.RandomState(0)
        self._sink = sink
        self.last_distance: Optional[np.ndarray] = None
        self.last_cluster_acc: Optional[np.ndarray] = None

    @classmethod
    def from_args(cls, args, change_points=None, **kw) -> "SoftClusterState":
        cfg = parse_algo_arg(args.concept_drift_algo_arg, getattr(args, "dataset", ""), change_points,
                             getattr(args, "time_stretch", 1))
        return cls(args.client_num_in_total, args.concept_num, **cfg, **kw)

    # ------------------------------------------------------------------ helpers
    @property
    def sink(self) -> MetricsSink:
        return self._sink if self._sink is not None else get_sink()

    def _ensure(self, t: int) -> None:
        if t >= self.W.shape[0]:
            grow = np.zeros((max(t + 1, 2 * self.W.shape[0]),) + self.W.shape[1:], dtype=np.float64)
            grow[: self.W.shape[0]] = self.W
            self.W = grow

    def _new_step(self, t: int) -> np.ndarray:
        self._ensure(t)
        self.W[t] = 0.0
        self.steps.add(t)
        return self.W[t]

    def get_weights(self) -> Dict[int, np.ndarray]:
        return {t: self.W[t] for t in sorted(self.steps)}

    def weights_tensor(self, t_cur: int, device="cpu") -> torch.Tensor:
        self._ensure(t_cur)
        return torch.from_numpy(self.W[: t_cur + 1].astype(np.float32)).to(device)

    def set_acc(self, client: int, acc: float) -> None:
        self.prev_acc[client] = float(acc)

    def get_test_model_idx(self, t: int, c: int) -> int:
        return int(np.argmax(self.W[t][:, c]))

    def test_model_indices(self, t: int) -> np.ndarray:
        return np.argmax(self.W[t], axis=0)

    def set_weights_win1(self, t_cur: int) -> None:
        self.W[:t_cur] = 0.0

    def set_weights_zero_model(self, m: int) -> None:
        self.W[:, m, :] = 0.0

    def _used_before(self, t_cur: int) -> np.ndarray:
        """bool[M]: model had positive weight at some step < t_cur."""
        return (self.W[:t_cur] > 0).any(axis=(0, 2)) if t_cur > 0 else np.zeros(self.model_num, dtype=bool)

    def _log_plurality(self, t: int, round_idx: int) -> None:
        best = self.test_model_indices(t)
        for c in range(self.client_num):
            self.sink.log({f"Plurality/CL-{c}": int(best[c]), "round": round_idx})

    # ------------------------------------------------------------------ t = 0
    def cluster_init(self) -> None:
        w = self._new_step(0)
        s = self.sink
        if self.h_cluster == "F":  # every client starts on its own model (needs model_num ≥ client_num)
            for c in range(self.client_num):
                w[c, c] = 1.0
                s.log({f"Plurality/CL-{c}": c, "round": 0})
                s.set_summary(f"Contribute/CL-{c}", 1)
            s.set_summary("num_models", self.client_num)
            s.set_summary("local_models", self.client_num)
            return
        w[0, :] = 1.0
        for c in range(self.client_num):
            s.log({f"Plurality/CL-{c}": 0, "round": 0})
            s.set_summary(f"Contribute/CL-{c}", 1)
        s.set_summary("num_models", 1)
        s.set_summary("local_models", 0)

    # ------------------------------------------------------------------ accuracy-matrix clusterings
    def cluster(self, acc_matrix: np.ndarray, t: int, round_idx: int) -> None:
        alg = self.cluster_alg
        if alg in ("hard", "hard-r"):
            self.cluster_hard(acc_matrix, t)
        elif "softmax" in alg:
            self.cluster_softmax(acc_matrix, t)
        elif "mmacc" in alg:
            if round_idx == 0:
                self.cluster_mmacc(acc_matrix, t)
            else:
                self.cluster_hard_among_existing(acc_matrix, t)
        elif alg == "gmm":
            self.cluster_gmm(acc_matrix, t)
        elif alg == "geni":
            if round_idx == 0:
                self.cluster_geni(t)
        else:
            raise NameError("cluster alg")
        self._log_plurality(t, round_idx)
        if "softmax" in alg:
            for c in range(self.client_num):
                self.sink.log({f"Weight-All/CL-{c}": np.array2string(self.W[t][:, c]), "round": round_idx})

    def cluster_hard(self, acc_matrix: np.ndarray, t: int) -> None:
        w = self._new_step(t)
        w[np.argmax(acc_matrix, axis=0), np.arange(self.client_num)] = 1.0

    def cluster_softmax(self, acc_matrix: np.ndarray, t: int) -> None:
        z = np.asarray(acc_matrix, dtype=np.float64) * (2 ** self.softmax_alpha)
        z = z - z.max(axis=0, keepdims=True)
        e = np.exp(z)
        self._ensure(t)
        self.W[t] = e / e.sum(axis=0, keepdims=True)
        self.steps.add(t)

    def cluster_hard_among_existing(self, acc_matrix: np.ndarray, t: int) -> None:
        in_use = [m for m in range(self.model_num) if (self.W[t][m] > 0).any()]
        w = self._new_step(t)
        best = np.argmax(acc_matrix[in_use, :], axis=0)
        w[np.asarray(in_use)[best], np.arange(self.client_num)] = 1.0

    def cluster_gmm(self, acc_matrix: np.ndarray, t: int) -> None:
        from sklearn.mixture import GaussianMixture
        w = self._new_step(t)
        gm = GaussianMixture(n_components=2, random_state=0).fit(acc_matrix.T)
        probs = gm.predict_proba(acc_matrix.T).T
        a, b = (0, 1) if gm.means_[0][0] > gm.means_[0][1] else (1, 0)
        w[0], w[1] = probs[a], probs[b]

    def cluster_geni(self, t: int) -> None:
        w = self._new_step(t)
        row = self.geni_change_points[t // self.geni_stretch]
        w[np.asarray(row[: self.client_num], dtype=np.int64), np.arange(self.client_num)] = 1.0

    # ------------------------------------------------------------------ FedDrift-Eager
    def _eager(self, acc_matrix: np.ndarray, t: int, bank: Optional[ModelBank]) -> None:
        in_use = np.nonzero(self._used_before(t))[0]
        w = self._new_step(t)
        best_rows = np.argmax(acc_matrix[in_use, :], axis=0)
        best_models = in_use[best_rows]
        w[best_models, np.arange(self.client_num)] = 1.0
        slot = _FRESH
        for c in range(self.client_num):
            bm = int(best_models[c])
            newest = float(acc_matrix[bm][c])
            if self.prev_acc[c] - newest > self.mmacc_delta:
                if slot == _FRESH:  # ONE shared new model per time step
                    slot = self.find_unused_model_lru(t, bank, bm)
                if slot != -1:
                    w[:, c] = 0.0
                    w[slot, c] = 1.0
            self.set_acc(c, newest)

    def cluster_mmacc(self, acc_matrix: np.ndarray, t: int) -> None:
        self._eager(acc_matrix, t, None)
        self.log_models(t)

    def cluster_mmacc2(self, t: int, bank: ModelBank, ev: Evaluator) -> None:
        acc = ev.acc_matrix(list(range(self.model_num)), t)
        self._eager(acc, t, bank)
        self._log_plurality(t, 0)
        self.log_models(t)

    # ------------------------------------------------------------------ FedDrift (hierarchical)
    def cluster_hierarchical(self, t: int, bank: ModelBank, ev: Evaluator) -> None:
        if self.h_cluster == "E":  # keep ONE random model among those created last step
            created = [m for (m, _) in self.h_marked.values()]
            if created:
                keep = self.rng.choice(created)
                for mm in created:
                    if mm != keep:
                        bank.reinit(mm)
                        self.set_weights_zero_model(mm)
        self.update_marking(t)
        isolated = {m for (m, _) in self.h_marked.values()}
        used = self._used_before(t)
        in_use = [m for m in range(self.model_num) if used[m] and m not in isolated]
        acc = ev.acc_matrix(in_use, t)  # [len(in_use), C]

        w = self._new_step(t)
        for c, (m, _) in self.h_marked.items():
            w[m, c] = 1.0
        free = [c for c in range(self.client_num) if c not in self.h_marked]
        best_row = np.argmax(acc, axis=0) if len(in_use) else np.zeros(self.client_num, dtype=np.int64)
        for c in free:  # park everybody on their best model first so LRU never evicts a live one
            w[in_use[best_row[c]], c] = 1.0
        for c in free:
            row = int(best_row[c])
            best_model = in_use[row]
            newest = float(acc[row][c])
            if self.prev_acc[c] - newest > self.h_delta:
                slot = self.find_unused_model_lru(t, bank, best_model)
                if slot != -1:
                    self.h_marked[c] = (slot, t + self.h_w)
                    w[:, c] = 0.0
                    w[slot, c] = 1.0
            self.set_acc(c, newest)

        if len(in_use) > 1:
            L = len(in_use)
            pools = {m: [(c, tt) for c in range(self.client_num) for tt in range(t + 1) if self.W[tt][m][c] == 1]
                     for m in in_use}
            cacc = np.zeros((L, L))
            for j, mj in enumerate(in_use):
                # one shuffled subset per data pool, shared by all models (the reference shuffles per pool)
                state = self.rng.get_state()
                for i, mi in enumerate(in_use):
                    self.rng.set_state(state)
                    cacc[i, j] = ev.pooled_acc(mi, pools[mj], 20, self.rng)
            D = ops.cluster_distance(cacc, "A" if self.h_distance == "A" else "B")
            self.last_cluster_acc, self.last_distance = cacc, D
            method = "average" if self.h_cluster == "D" else "complete"
            labels = linkage_fcluster(D, method, self.h_deltap)
            groups: Dict[int, List[int]] = {}
            for i, lab in enumerate(labels):
                groups.setdefault(int(lab), []).append(in_use[i])
            merged = ["(" + ", ".join(str(e) for e in g) + ")" for g in groups.values() if len(g) > 1]
            if merged:
                self.sink.set_summary("Merge", ", ".join(merged))
            for g in groups.values():
                for second in g[1:]:
                    self.merge(t, bank, g[0], second)
        self._log_plurality(t, 0)
        self.log_models(t)

    def update_marking(self, t: int) -> None:
        for c in [c for c, (_, tu) in self.h_marked.items() if tu == t]:
            del self.h_marked[c]

    def merge(self, t: int, bank: ModelBank, base: int, second: int) -> None:
        w1 = float(self.W[: t + 1, base, :].sum())
        w2 = float(self.W[: t + 1, second, :].sum())
        s = w1 + w2
        bank.merge(base, second, w1 / s, w2 / s)
        bank.reinit(second)
        self.W[: t + 1, base, :] += self.W[: t + 1, second, :]
        self.set_weights_zero_model(second)

    # ------------------------------------------------------------------ model-slot allocation policies
    def find_unused_model_capped(self) -> int:
        if self.h_next_free_model < self.model_num:
            self.h_next_free_model += 1
            return self.h_next_free_model - 1
        return -1

    def find_unused_model(self, t: int, bank: Optional[ModelBank]) -> int:
        if self.h_next_free_model < self.model_num:
            self.h_next_free_model += 1
            return self.h_next_free_model - 1
        slot = 0
        for i in range(self.model_num):
            m = (i + self.h_next_free_model) % self.model_num
            if not (self.W[t - 1][m].any() or self.W[t][m].any()):
                slot = m
        self.h_next_free_model = self.model_num + slot + 1
        self.set_weights_zero_model(slot)
        if bank is not None:
            bank.reinit(slot)
        return slot

    def find_unused_model_lru(self, t: int, bank: Optional[ModelBank] = None, original_model: int = 0) -> int:
        if self.h_next_free_model < self.model_num:
            slot = self.h_next_free_model
            self.h_next_free_model += 1
        else:
            used = self.W[: t + 1].any(axis=2)  # [t+1, M]
            last = np.where(used.any(axis=0), (used * np.arange(t + 1)[:, None]).max(axis=0), -1).astype(float)
            lru = np.where(last == last.min())[0]
            slot = int(self.rng.choice(lru))
            if last[slot] == t:
                return -1
            self.set_weights_zero_model(slot)
        if bank is not None:  # start the new concept's model from the client's previous best model
            bank.copy(slot, original_model)
        return slot

    # ------------------------------------------------------------------ Clustered FL
    def cluster_cfl_init(self, t: int) -> None:
        self._ensure(t)
        self.W[t] = self.W[t - 1]
        self.steps.add(t)
        if self.cfl_retrain == "win-1":
            self.set_weights_win1(t)
        self._log_plurality(t, 0)

    def cluster_cfl(self, t: int, round_idx: int, bank: ModelBank, client_params: torch.Tensor,
                    n: torch.Tensor, clients: Optional[Sequence[int]] = None) -> bool:
        """``client_params [C, M, P]`` local models, ``n [C, M]`` their sample weights (0 = did not train).  Under partial
        participation row s holds the update of client ``clients[s]`` (``None``: row c is client c)."""
        did_split = False
        row_of = None if clients is None else {int(c): s for s, c in enumerate(clients)}
        in_use = [m for m in range(self.model_num) if (self.W[t][m] > 0).any()]
        for m in in_use:
            members = np.nonzero(self.W[t][m])[0]
            if row_of is None:
                trained = [int(c) for c in members if float(n[c, m]) != 0]
                rows = trained
            else:
                trained = [int(c) for c in members if int(c) in row_of and float(n[row_of[int(c)], m]) != 0]
                rows = [row_of[c] for c in trained]
            if not trained:
                continue
            U = client_params[rows, m, :] - bank.theta[m][None, :]
            S, norms = ops.gram_cosine(U)
            max_norm = float(norms.max())
            mean_norm = float(U.mean(dim=0).norm())
            self.sink.log({"Max_Norm": max_norm, "Mean_Norm": mean_norm, "round": round_idx})
            if mean_norm > self.cfl_norm:
                self.cfl_norm = mean_norm
                self.cfl_eps1 = self.cfl_norm / 10.0
                self.cfl_eps2 = 6 * self.cfl_eps1
            elif mean_norm < self.cfl_eps1 and max_norm > self.cfl_eps2 and len(trained) >= 2:
                Sn = S.cpu().numpy()
                g1, g2 = complete_linkage_bipartition(Sn)
                alpha_cross = max(Sn[i, j] for i in g1 for j in g2)
                if ((1 - alpha_cross) / 2.0) ** 0.5 > self.cfl_gamma:
                    slot = self.find_unused_model_capped()
                    if slot != -1:
                        did_split = True
                        bank.reinit(m)
                        self.W[t][m] = 0.0
                        # g1/g2 index the clients that uploaded an update; idle members stay on m
                        for c in members:
                            if int(c) not in trained:
                                self.W[t][m][c] = 1.0
                        for i in g1:
                            self.W[t][m][trained[i]] = 1.0
                        for i in g2:
                            self.W[t][slot][trained[i]] = 1.0
        if did_split:
            self._log_plurality(t, round_idx)
            if self.cfl_retrain == "all":
                for tt in range(t):
                    self.W[tt] = self.W[t]
        return did_split

    # ------------------------------------------------------------------ bookkeeping / summaries
    def log_models(self, t: int) -> None:
        s = self.sink
        if self.h_cluster == "E":
            num = int(self._used_before(t).sum()) + (1 if self.h_marked else 0)
        else:
            num = int((self.W[: t + 1] > 0).any(axis=(0, 2)).sum())
        s.set_summary("num_models", num)
        trained_by = (self.W[: t + 1] > 0).any(axis=0)  # [M, C]
        counts = trained_by.sum(axis=1)
        s.set_summary("local_models", int((counts == 1).sum()))
        shared = trained_by[counts != 1]
        for c in range(self.client_num):
            s.set_summary(f"Contribute/CL-{c}", int(shared[:, c].sum()) if shared.size else 0)

    # ------------------------------------------------------------------ (de)serialisation
    def state_dict(self) -> Dict:
        d = {k: v for k, v in self.__dict__.items() if k not in ("rng", "_sink", "W")}
        d["W"] = self.W.copy()
        d["steps"] = sorted(self.steps)
        d["rng_state"] = self.rng.get_state()
        return d

    def load_state_dict(self, d: Dict) -> None:
        d = dict(d)
        self.rng.set_state(d.pop("rng_state"))
        self.steps = set(d.pop("steps"))
        self.W = np.array(d.pop("W"))
        self.h_marked = {int(k): tuple(v) for k, v in d.pop("h_marked").items()}
        self.prev_acc = {int(k): float(v) for k, v in d.pop("prev_acc").items()}
        self.__dict__.update(d)
