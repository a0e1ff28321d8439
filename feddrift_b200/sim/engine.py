"""DriftSim — the device-resident continual-FL engine (the B200-native replacement of
``run_fedavg_distributed_pytorch.sh`` + ``main_fedavg.py`` + Server/ClientManager FSM).

The reference launches ``mpirun -np N+1`` once per time step, ships every model to every rank every
round as pickles, trains with eager per-client optimizers and evaluates with per-batch ``.item()`` syncs
(SURVEY §3).  Here ONE process owns the whole experiment:

* all time steps' data live in HBM (``DriftData`` tensors), all model slots in a :class:`ModelBank` row
  arena, all per-(client, model) optimizer state in a :class:`ClientArena`;
* a drift algorithm (``sim/algos.py``) turns its state machine into a *training plan*: the dense weight
  tensor ``W[t', m, c]`` (which past time steps' data of client c train model m), sampling/weighting
  modes, test-model routing and optional ensemble weights — all device tensors;
* a whole block of rounds (broadcast → E local steps per (client, model) → per-cluster weighted
  aggregation → evaluation of every client on train/test data) runs in ONE launch of the fused
  persistent kernel ``fed_round_small`` (small MLPs) with zero host synchronisation; per-round metrics
  are accumulated on device and flushed to the wandb-compatible sink once per block;
* host logic only runs at time-step boundaries (clustering decisions on a tiny accuracy matrix) or at
  the sparse per-round hooks some algorithms need (CFL split checks, AUE weight refresh every 10 rounds).

Models that are not small MLPs run through ``sim/generic.py`` (bank-bound ``nn.Module`` + fused arena
optimizer + K1 aggregation kernel) behind the same interface.
"""
from __future__ import annotations

import os
import time
from types import SimpleNamespace
from typing import Dict, List, Optional

import numpy as np
import torch

from .. import ops
from ..data.drift import DriftData, generate_drift_data
from ..drift.evaluator import Evaluator
from ..models import utils as mutils
from ..models.utils import create_model
from ..parallel.arena import ClientArena, ModelBank
from ..utils.metrics import MetricsSink, get_sink
from . import checkpoint as ckpt

DEFAULTS = dict(
    model="fnn", dataset="sea", client_num_in_total=10, client_num_per_round=10, batch_size=500,
    client_optimizer="adam", lr=0.01, wd=0.001, epochs=5, comm_round=200, frequency_of_the_test=1,
    total_train_iteration=10, curr_train_iteration=0, drift_together=0, report_client=1, retrain_data="win-1",
    concept_drift_algo="softcluster", concept_drift_algo_arg="H_A_C_1_10_0", ensemble_window=4, concept_num=4,
    change_points="A", time_stretch=1, reset_models=0, noise_prob=0.0, dummy_arg=0, sample_num=100, ci=0,
    is_mobile=0, gpu_num_per_server=1, data_dir=None, checkpoint_dir=None, rounds_per_launch=0,
)


def make_args(**kw) -> SimpleNamespace:
    d = dict(DEFAULTS)
    d.update(kw)
    return SimpleNamespace(**d)


from ..ops.small_round import LAUNCH_COUNT as _SMALL_LAUNCHES  # noqa: E402


def client_sampling(round_idx: int, client_num_in_total: int, client_num_per_round: int) -> List[int]:
    """The clients that train in round ``round_idx`` of a time step (``--client_num_per_round`` K of
    ``--client_num_in_total`` C): all of them when K ≥ C, otherwise the reference's draw
    ``np.random.seed(round_idx); np.random.choice(range(C), K, replace=False)`` taken from a private ``RandomState`` so that
    the engine's own random streams are left alone.  The s-th entry is worker slot s."""
    C, K = int(client_num_in_total), int(client_num_per_round)
    if K >= C:
        return list(range(C))
    return [int(c) for c in np.random.RandomState(round_idx).choice(range(C), K, replace=False)]


class DriftSim:
    def __init__(self, args, data: Optional[DriftData] = None, device=None, sink: Optional[MetricsSink] = None,
                 algo=None):
        self.args = args
        self.device = torch.device(device) if device is not None else torch.device(
            "cuda" if torch.cuda.is_available() else "cpu")
        self.sink = sink if sink is not None else get_sink()
        seed = int(getattr(args, "dummy_arg", 0))
        np.random.seed(seed)
        torch.manual_seed(seed)
        mutils.torch_seed = seed
        self.rng = np.random.RandomState(seed)
        if data is None:
            data = generate_drift_data(args.dataset, args.total_train_iteration, args.client_num_in_total,
                                       args.sample_num, args.noise_prob, args.time_stretch, args.change_points,
                                       bool(args.drift_together), seed=0, data_dir=getattr(args, "data_dir", None))
        self.data_host = data
        self.data = data.to(self.device)
        self.C = data.client_num
        from .algos import make_algo
        self.algo = algo if algo is not None else make_algo(args, self)
        self.M = self.algo.num_model_slots()
        mkw = {"small_input": True} if (args.model in ("resnet", "resnet18") and data.X.shape[-1] <= 64) else {}
        template = create_model(args.model, data.class_num, data.feature_num, **mkw)
        self.bank = ModelBank(template, self.M, self.device)
        self.spec = self.bank.mlp
        self.evaluator = Evaluator(self.bank, self.data, args.batch_size)
        self.t = -1
        self.round_in_step = 0
        self.global_round = 0
        self.history: List[Dict] = []
        self._small: Optional[Dict] = None
        self._plan: Optional[Dict] = None
        self._last_counts = None
        self.multi = None
        self.shard_clients = False   # generic path: shard clients over torch.distributed ranks + PeerAggregator
        self.clients = ClientArena(self.C, self.M, self.bank.P, self.device,
                                   adam=(args.client_optimizer != "sgd"))
        # partial participation: [comm_round, K] sampled client ids per round of a time step (None = every client trains)
        self.K = min(int(getattr(args, "client_num_per_round", self.C)), self.C)
        self.participants_table: Optional[torch.Tensor] = None
        self._participant_rows: List[List[int]] = []
        if self.K < self.C:
            self._participant_rows = [client_sampling(r, self.C, self.K) for r in range(max(int(args.comm_round), 1))]
            self.participants_table = torch.tensor(self._participant_rows, dtype=torch.int32, device=self.device)
        self.timings = {"cluster_s": 0.0, "rounds_s": 0.0}

    # ------------------------------------------------------------------ experiment driver
    def run(self, start_iteration: int = 0, end_iteration: Optional[int] = None) -> Dict:
        end = self.args.total_train_iteration if end_iteration is None else end_iteration
        for t in range(start_iteration, end):
            self.run_time_step(t)
        return self.summary()

    def run_time_step(self, t: int, rounds: Optional[int] = None) -> Dict:
        self.begin_time_step(t)
        R = self.args.comm_round if rounds is None else rounds
        out = self.run_rounds(R)
        self.end_time_step()
        return out

    def begin_time_step(self, t: int) -> None:
        """Clustering / state machine for time step t (runs BEFORE round 0 with models trained at t-1 —
        ``FedAvgEnsAggregatorSoftCluster.py:46-118``) and optimizer-state reset (new process in the reference)."""
        t0 = time.perf_counter()
        self.t = t
        self.args.curr_train_iteration = t
        self.round_in_step = 0
        if getattr(self.args, "reset_models", 0) and t > 0:
            for m in range(self.M):
                self.bank.reinit(m)
        self.clients.reset_optimizer()
        self.algo.begin_step(t)
        self._small = None
        self._plan = None
        self._counts_host = None
        self.timings["cluster_s"] += time.perf_counter() - t0

    def end_time_step(self) -> None:
        self.algo.end_step(self.t)
        cdir = getattr(self.args, "checkpoint_dir", None)
        if cdir:
            ckpt.save(self, os.path.join(cdir, f"step_{self.t:04d}.fdck"))

    # ------------------------------------------------------------------ rounds
    def participants(self, r: int) -> List[int]:
        """Client ids of the worker slots of round ``r`` of the current time step: slot s trains client ``[s]`` and owns row
        s of the client arena.  The table has ``comm_round`` rows (the reference never runs more rounds in a time step);
        rounds past that, which only benchmarks and graph replay reach, reuse row ``r % comm_round``."""
        if self.participants_table is None:
            return list(range(self.C))
        return self._participant_rows[r % len(self._participant_rows)]

    def _check_partial_participation(self) -> None:
        if self.participants_table is not None and (self.multi is not None or getattr(self, "shard_clients", False)):
            raise ValueError(f"partial participation (client_num_per_round={self.K} < {self.C} clients) is single-GPU only; "
                             "run with client_num_per_round >= client_num_in_total on several GPUs")

    def current_plan(self) -> Dict:
        """The algorithm's training plan for the current time step (built once; sample lists are randomised)."""
        if self._plan is None:
            self._plan = self.algo.plan(self.t)
        return self._plan

    def invalidate_plan(self) -> None:
        self._plan = None
        self._small = None

    def _small_state(self) -> Dict:
        """Device-side argument block of the fused round kernel for the current time step."""
        if self._small is None:
            a, s, plan = self.args, self.spec, self.current_plan()
            X = self.data.X.reshape(self.data.steps, self.C, self.data.X.shape[2], -1)
            self._small = dict(
                kind=s["kind"], din=s["in"], hid=s["hidden"], dout=s["out"],
                X=X, Y=self.data.Y.to(torch.int32) if self.device.type == "cuda" else self.data.Y,
                nsamp=self.data.nsamp, batch_size=a.batch_size,
                W=plan["W"].to(self.device), theta=self.bank.theta,
                opt_m=self.clients.m, opt_v=self.clients.v, opt_vmax=self.clients.vmax, opt_step=self.clients.step,
                lr=a.lr, wd=a.wd if a.client_optimizer != "sgd" else 0.0, epochs=a.epochs,
                optimizer=("sgd" if a.client_optimizer == "sgd" else "adam"),
                seed=int(a.dummy_arg) * 7919 + 13 + 1000003 * self.t, round0=0, t_cur=self.t,
                recluster_hard=bool(plan.get("recluster_hard", False)),
                sample_mode=plan.get("sample_mode", "pool"), n_mode=plan.get("n_mode", "batches"),
            )
            for k in ("feat_mask", "train_index", "train_count", "ens_mode", "ens_w", "eval_train_model",
                      "eval_test_model", "optimizer", "lr"):
                if plan.get(k) is not None:
                    self._small[k] = plan[k]
            if self._small["optimizer"] == "sgd":
                self._small["wd"] = 0.0
            if self.participants_table is not None:
                self._small["participants"] = self.participants_table
            if getattr(self, "multi", None) is not None:
                self._small["multi_gpu"] = self.multi
            if self.device.type == "cuda":  # device-resident round / epoch counters (CUDA-graph replay friendly)
                self._small["counters"] = torch.tensor(
                    [self.round_in_step, int(self.multi["flag_base"]) if self.multi else 0], dtype=torch.int32, device=self.device)
            self._graph = None
            if self.bank.stride != self.bank.P:
                self._small["theta_stride"] = self.bank.stride
        return self._small

    def run_rounds(self, rounds: int) -> Dict:
        """Run ``rounds`` FL rounds of the current time step; returns the last round's aggregate metrics."""
        self._check_partial_participation()
        t0 = time.perf_counter()
        done, last = 0, {}
        while done < rounds:
            block = self.algo.block_size(self.round_in_step, rounds - done)
            rpl = int(getattr(self.args, "rounds_per_launch", 0) or 0)
            if rpl > 0:
                block = min(block, rpl)
            if self.multi is not None:
                block = min(block, int(self.multi["metrics_rounds"]))
            if self._use_fused():
                st = self._small_state()
                st["round0"] = self.round_in_step
                out = ops.fed_round_small(st, block)
                if st.get("recluster_hard"):
                    self.algo.absorb_weights(self.t, st["W"])
            else:
                from .generic import run_rounds_generic
                out = run_rounds_generic(self, block)
            last = self._flush_metrics(out, self.round_in_step, block)
            self.round_in_step += block
            self.global_round += block
            done += block
            self.algo.after_block(self.t, self.round_in_step)
        self.timings["rounds_s"] += time.perf_counter() - t0
        return last

    def _use_fused(self) -> bool:
        """Route a block of rounds: the fused persistent kernel when the federation is a small MLP it can hold (shape
        instantiated, ``t < 64`` plan-table limit, shared-memory layout within 227 KB), the generic executor otherwise."""
        if self.spec is None or not self.algo.fused_ok() or getattr(self, "shard_clients", False):
            return False
        if self.device.type != "cuda":
            return True
        from ..ops import small_round
        s = self.spec
        return small_round.fits(s["kind"], s["in"], s["hidden"], s["out"], self.C, self.M, self.t)

    def _check_peer_error(self) -> None:
        if self.multi is not None and self.multi["error_np"][0] != 0:
            from ..parallel.symm import check_error
            check_error(self)

    # ------------------------------------------------------------------ device-only / end-to-end single rounds
    def run_rounds_device(self, n: int) -> torch.Tensor:
        """Launch ``n`` fused rounds and leave the per-round metrics ON DEVICE (no host sync, no logging).
        Returns the device metrics view ``[n, C, 4]``."""
        self._check_partial_participation()
        st = self._small_state()
        st["round0"] = self.round_in_step
        if self.device.type == "cuda":
            from ..ops import small_round
            buf = getattr(self, "_metrics_buf", None)
            if buf is None or buf.shape[0] < n:
                buf = self._metrics_buf = torch.zeros(max(n, 64), self.C, 4, dtype=torch.float32, device=self.device)
            # multi-GPU: the owners push their rows into every rank's LL staging area; the kernel compacts them into buf
            out = small_round.run_native(st, n, buf[:n])
        else:
            out = ops.fed_round_small(st, n)
        self.round_in_step += n
        self.global_round += n
        self._last_counts = out["counts"]
        return out["metrics"]

    def run_round_device(self) -> torch.Tensor:
        return self.run_rounds_device(1)

    def make_host_round_inputs(self) -> Dict[str, torch.Tensor]:
        """Pinned host copies of what one round consumes: the clients' time-t training data and time-(t+1)
        test data (features + labels) — in a deployment these arrive from the data plane every round."""
        t = self.t
        hi = min(t + 2, self.data_host.steps)
        pin = self.device.type == "cuda"
        X = self.data_host.X[t:hi].reshape(hi - t, self.C, self.data_host.X.shape[2], -1).float().contiguous()
        Y = self.data_host.Y[t:hi].to(torch.int32).contiguous()
        out = {"X": X.pin_memory() if pin else X, "Y": Y.pin_memory() if pin else Y}
        self._host_metrics = torch.zeros(self.C, 4, dtype=torch.float32)
        if pin:
            self._host_metrics = self._host_metrics.pin_memory()
        return out

    def host_round_bytes(self):
        hi = min(self.t + 2, self.data_host.steps)
        n = (hi - self.t) * self.C * self.data_host.X.shape[2]
        return int(n * (self.data_host.feature_num * 4 + 4)), int(self.C * 4 * 4)

    def _build_round_graph(self, host_inputs: Dict[str, torch.Tensor]):
        """Capture one end-to-end round into ONE CUDA graph (replayed once per round).

        The graph is a single kernel node — ``fed_round_small_kernel`` itself copies the round's inputs from the pinned
        host tensors into the device arena (16-byte system-scope loads over PCIe) and mirrors the metric rows into the
        pinned host buffer (fused H2D / D2H, ``host_io``); with several GPUs every rank copies its own inputs in and
        mirrors the complete rows after the end-of-launch peer handshake.  Non-pinned inputs fall back to
        [H2D memcpy nodes → kernel → D2H memcpy node]."""
        from ..ops import small_round
        st = self._small_state()
        cache = small_round.prepare(st)
        t = self.t
        hi = t + host_inputs["X"].shape[0]
        hm = self._host_metrics
        fused_io = (host_inputs["X"].is_pinned() and host_inputs["Y"].is_pinned() and hm.is_pinned()
                    and host_inputs["X"].dtype == torch.float32 and host_inputs["Y"].dtype == torch.int32
                    and host_inputs["X"].is_contiguous() and host_inputs["Y"].is_contiguous())
        # warm-up launch outside the capture (lazy allocations, function attributes) — on a snapshot: building the graph
        # must not advance the experiment (models, optimizer state, RNG round counter are restored afterwards; only the
        # cross-GPU epoch stays advanced because the peers have seen it)
        cl = self.clients
        snap = [(x, x.clone()) for x in (self.bank.theta, cl.m, cl.v, cl.vmax, cl.step, st.get("W")) if isinstance(x, torch.Tensor)]
        cnt = st.get("counters")
        cnt0 = cnt[0:1].clone() if isinstance(cnt, torch.Tensor) else None
        r0, g0, l0 = self.round_in_step, self.global_round, small_round.LAUNCH_COUNT["fed_round_small"]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self.run_rounds_device(1)
        torch.cuda.current_stream().wait_stream(side)
        for dst, src in snap:
            dst.copy_(src)
        if cnt0 is not None:
            cnt[0:1].copy_(cnt0)
        self.round_in_step, self.global_round = r0, g0
        small_round.LAUNCH_COUNT["fed_round_small"] = l0
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        if fused_io:
            st["host_io"] = (host_inputs["X"].data_ptr(), host_inputs["Y"].data_ptr(), hm.data_ptr(), t, hi - t)
        try:
            with torch.cuda.graph(g):
                if not fused_io:
                    cache["X"][t:hi].copy_(host_inputs["X"], non_blocking=True)
                    cache["Y"][t:hi].copy_(host_inputs["Y"], non_blocking=True)
                met = self.run_rounds_device(1)
                if not fused_io:
                    hm.copy_(met[0], non_blocking=True)
        finally:
            st.pop("host_io", None)
        self.round_in_step -= 1   # the capture itself executed nothing
        self.global_round -= 1
        small_round.LAUNCH_COUNT["fed_round_small"] -= 1
        if self.multi is not None:
            self.multi["flag_base"] = int(self.multi["flag_base"]) - 1
        self._graph_keep = (host_inputs, hm)   # the graph holds raw host pointers: keep the pinned tensors alive
        return g

    def run_round(self, host_inputs: Optional[Dict[str, torch.Tensor]] = None, log: bool = False,
                  use_graph: bool = False) -> Dict:
        """ONE end-to-end FL round through the public API: (optional) host→device copy of the round's inputs
        from pinned memory, the fused round kernel, device→host copy of the per-client metrics, host reduction.
        Synchronises (the caller gets real numbers back).

        ``use_graph=True`` replays a captured graph that holds the ADDRESSES of ``host_inputs``' pinned tensors: write each
        round's new data into the same ``host_inputs`` buffers (``make_host_round_inputs`` allocates them once per time
        step); passing a different dict rebuilds the graph."""
        if use_graph and host_inputs is not None and self.device.type == "cuda":
            gr = getattr(self, "_graph", None)
            if gr is None or gr[1] is not host_inputs:
                if getattr(self, "_host_metrics", None) is None or not self._host_metrics.is_pinned():
                    self._host_metrics = torch.zeros(self.C, 4, dtype=torch.float32).pin_memory()
                g = self._build_round_graph(host_inputs)
                fast = None
                try:   # one C++ call per round (graph launch + stream sync, GIL released) when the raw handle is exposed
                    from ..ops import _ext
                    ext = _ext.load()
                    if ext is not None and hasattr(ext, "graph_launch_sync") and hasattr(g, "raw_cuda_graph_exec"):
                        handle = int(g.raw_cuda_graph_exec())
                        fast = (ext.graph_launch_sync, handle)
                except Exception:  # noqa: BLE001  (older torch: fall back to replay() + synchronize())
                    fast = None
                gr = self._graph = (g, host_inputs, self._host_metrics.numpy(), torch.cuda.current_stream(), fast)
            if gr[4] is not None:
                gr[4][0](gr[4][1], True)
            else:
                gr[0].replay()
                gr[3].synchronize()
            self.round_in_step += 1
            self.global_round += 1
            _SMALL_LAUNCHES["fed_round_small"] += 1
            if self.multi is not None:
                self.multi["flag_base"] = int(self.multi["flag_base"]) + 1
            return self._round_result(gr[2], log)
        st = self._small_state()
        t = self.t
        if host_inputs is not None:
            if self.device.type == "cuda":
                from ..ops import small_round
                cache = small_round.prepare(st)
                hi = t + host_inputs["X"].shape[0]
                cache["X"][t:hi].copy_(host_inputs["X"], non_blocking=True)
                cache["Y"][t:hi].copy_(host_inputs["Y"], non_blocking=True)
            else:
                hi = t + host_inputs["X"].shape[0]
                st["X"][t:hi].copy_(host_inputs["X"].reshape(st["X"][t:hi].shape))
                st["Y"][t:hi].copy_(host_inputs["Y"])
        met = self.run_rounds_device(1)   # multi-GPU: every rank already holds all clients' rows (peer stores)
        hm = getattr(self, "_host_metrics", None)
        if hm is None:
            hm = self._host_metrics = torch.zeros(self.C, 4, dtype=torch.float32)
        hm.copy_(met[0], non_blocking=True)
        if self.device.type == "cuda":
            torch.cuda.current_stream().synchronize()
        return self._round_result(hm.numpy(), log)

    def _round_result(self, m, log: bool) -> Dict:
        self._check_peer_error()
        t = self.t
        nn_ = getattr(self, "_counts_tot", None)
        if nn_ is None or nn_[0] != t:
            c = self._last_counts.cpu().numpy()
            nn_ = self._counts_tot = (t, max(float(c[:, 0].sum()), 1.0), max(float(c[:, 1].sum()), 1.0))
        ntr, nte = nn_[1], nn_[2]
        tot = m.sum(0).tolist()     # one reduction over the [C, 4] host buffer
        res = {"round": self.round_in_step - 1, "iteration": t, "train_acc": tot[0] / ntr, "train_loss": tot[1] / ntr,
               "test_acc": tot[2] / nte, "test_loss": tot[3] / nte}
        if log:
            for k_, key in (("train_acc", "Train/Acc"), ("train_loss", "Train/Loss"), ("test_acc", "Test/Acc"),
                            ("test_loss", "Test/Loss")):
                self.sink.log({key: res[k_], "round": res["round"]})
        return res

    def _flush_metrics(self, out: Dict[str, torch.Tensor], r0: int, n: int) -> Dict:
        """One D2H copy per block; emits the reference's wandb keys for every tested round."""
        met = out["metrics"].detach().to("cpu", torch.float64).numpy()  # [n, C, 4]
        self._check_peer_error()
        cnt = out["counts"].detach().to("cpu", torch.float64).numpy()   # [C, 2]
        a = self.args
        ntr, nte = max(cnt[:, 0].sum(), 1.0), max(cnt[:, 1].sum(), 1.0)
        last: Dict = {}
        for i in range(n):
            r = r0 + i
            if not (r % a.frequency_of_the_test == 0 or r == a.comm_round - 1):
                continue
            tr_acc, tr_loss = met[i, :, 0].sum() / ntr, met[i, :, 1].sum() / ntr
            te_acc, te_loss = met[i, :, 2].sum() / nte, met[i, :, 3].sum() / nte
            if a.report_client:
                for c in range(self.C):
                    self.sink.log({f"Train/Acc-CL-{c}": (met[i, c, 0] / cnt[c, 0]) if cnt[c, 0] else -1, "round": r})
                    self.sink.log({f"Test/Acc-CL-{c}": (met[i, c, 2] / cnt[c, 1]) if cnt[c, 1] else -1, "round": r})
            self.sink.log({"Train/Acc": tr_acc, "round": r})
            self.sink.log({"Train/Loss": tr_loss, "round": r})
            self.sink.log({"Test/Acc": te_acc, "round": r})
            self.sink.log({"Test/Loss": te_loss, "round": r})
            last = {"round": r, "train_acc": tr_acc, "train_loss": tr_loss, "test_acc": te_acc,
                    "test_loss": te_loss, "iteration": self.t}
        if last:
            self.history.append(last)
        return last

    def summary(self) -> Dict:
        return {"history": self.history, "summary": dict(self.sink.run.summary), "timings": dict(self.timings),
                "rounds": self.global_round}
