#!/usr/bin/env python
"""Headline benchmark: FL rounds/sec of SEA-4 / fnn / 10-client FedDrift (softcluster H_A_C_1_10_0, change
points A, 5 local Adam-amsgrad steps, batch 500, 100 samples/client/step) — BASELINE.json's metric.

  python bench.py --gpus N --steps K --warmup W            # this framework (default arm)
  python bench.py --impl reference --gpus N --steps K ...   # the unmodified reference through baseline/

A *step* is one complete FL round: broadcast of the cluster models, 5 local optimizer steps on every
participating (client, model) pair, per-cluster weighted aggregation, train+test evaluation of every client
(``frequency_of_the_test = 1`` like the reference's run script).  Timing: CUDA events around every round on the
launching stream, L2 flushed (256 MiB write) between rounds outside the event brackets, max over ranks; the
``e2e`` number drives the public ``DriftSim.run_round`` API: every round the round's inputs travel from pinned host
memory to the device and the round's metrics come back to pinned host memory inside the timed region (the round kernel
performs both transfers itself — fused host I/O — so the whole round is one CUDA-graph node).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASELINE_ROUNDS_PER_S = None  # the reference publishes no number (BASELINE.md)

HEADLINE = dict(model="fnn", dataset="sea", client_num_in_total=10, client_num_per_round=10, batch_size=500, lr=0.01,
                epochs=5, comm_round=200, sample_num=100, total_train_iteration=10, concept_num=4,
                concept_drift_algo="softcluster", concept_drift_algo_arg="H_A_C_1_10_0", change_points="A",
                noise_prob=0.0, time_stretch=1, dummy_arg=0, report_client=1, frequency_of_the_test=1)
BENCH_TIME_STEP = 5  # timed rounds run at time step 5 of change-point matrix A (two concepts live)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from feddrift_b200.ops import small_round
    from feddrift_b200.sim import DriftSim, make_args
    from baseline import headline_config

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, max(args.warmup, 3)

    sim_args = make_args(**HEADLINE)
    sim = DriftSim(sim_args, device=dev)
    if world > 1:
        from feddrift_b200.parallel.symm import attach_multi_gpu
        attach_multi_gpu(sim, world, rank)
    # untimed: play the experiment up to the benchmark time step so real cluster state exists
    for t in range(BENCH_TIME_STEP):
        sim.run_time_step(t, rounds=20)
    sim.begin_time_step(BENCH_TIME_STEP)
    sim.args.rounds_per_launch = 1
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-level (device-timed) number: one fused launch per round, L2 flushed between rounds
    clocks = ClockSampler(local_rank)
    clocks.start()
    time.sleep(0.5)  # nvidia-smi start-up (outside every timed region)
    for _ in range(Wm):
        sim.run_round_device()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    l0 = small_round.LAUNCH_COUNT["fed_round_small"]
    barrier()
    for i in range(K):
        flush.fill_(i & 0xFF)
        ev[i][0].record()
        metrics = sim.run_round_device()
        ev[i][1].record()
    barrier()
    launches = small_round.LAUNCH_COUNT["fed_round_small"] - l0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    # what the last timed round handed back, copied before the informational phases below advance the experiment
    outputs = {"round_metrics": metrics[0].cpu().numpy(), "cluster_models": sim.bank.theta.cpu().numpy()} if args.dump_outputs else {}

    # ---- persistent mode (all K rounds inside ONE launch; no flush possible between rounds) — informational
    sim.args.rounds_per_launch = 0
    sim.run_rounds_device(Wm)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sim.run_rounds_device(K)
    e1.record()
    barrier()
    persistent_ms = e0.elapsed_time(e1)

    # ---- end-to-end through the public API: pinned H2D of the round's inputs + D2H of the round's metrics
    sim.args.rounds_per_launch = 1
    host_inputs = sim.make_host_round_inputs()
    for _ in range(Wm):
        sim.run_round(host_inputs, use_graph=True)
    barrier()
    e2e_s = 0.0
    for i in range(K):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = sim.run_round(host_inputs, use_graph=True)  # one CUDA-graph replay: H2D → fused round → D2H; syncs
        e2e_s += time.perf_counter() - t0
    barrier()
    clk = clocks.stop()
    # ---- correctness gate: a fast wrong answer is not a result
    assert res["train_acc"] == res["train_acc"] and 0.5 < res["train_acc"] <= 1.0 and 0.5 < res["test_acc"] <= 1.0, res
    assert res["train_loss"] > 0.0 and res["test_loss"] > 0.0, res
    if world > 1:
        from feddrift_b200.parallel.symm import check_error
        check_error(sim)
        th = sim.bank.theta.detach().double()
        sig = torch.stack([th.sum(), (th * th).sum(), th.abs().max()])
        sigs = [torch.zeros_like(sig) for _ in range(world)]
        dist.all_gather(sigs, sig)
        for g_, s_ in enumerate(sigs):   # the peer-inbox sum runs in rank order on every rank: models must be BIT-identical
            assert torch.equal(s_, sigs[0]), f"cluster models diverged between rank 0 and rank {g_}: {s_.tolist()} vs {sigs[0].tolist()}"

    # ---- BASELINE.json's other named configs in the same bench line (device-timed, max over ranks; informational)
    extra = {}
    if os.environ.get("FDB_BENCH_EXTRA", "1") != "0":
        from feddrift_b200.experiments.configs import measure_config
        names = os.environ.get("FDB_BENCH_EXTRA_CONFIGS", "cfg2_sea_fnn_100clients_feddrift,cfg3_mnist_cnn_64clients_ifca,"
                               "cfg4_cifar_resnet18_32clients_aue,cfg5_shakespeare_lstm_128clients_win1").split(",")
        t_extra = time.perf_counter()
        for name in [n for n in names if n]:
            spent = torch.tensor([time.perf_counter() - t_extra], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(spent, op=dist.ReduceOp.MAX)   # rank-consistent decision
            if float(spent) > float(os.environ.get("FDB_BENCH_EXTRA_SECONDS", 150)):
                extra[name] = {"skipped": "extra-config time budget spent"}
                continue
            try:
                r_ = measure_config(name, dev, world, rank)
                extra[name] = {k: r_[k] for k in ("rounds_per_s", "ms_per_round", "rounds", "clients", "P", "fused_kernel", "last")}
            except Exception as e:  # noqa: BLE001 — an extra config must never take the headline down
                extra[name] = {"error": repr(e)[:200]}
            barrier()

    t = torch.tensor([dev_ms, persistent_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, persistent_ms, e2e_ms = [float(x) for x in t.tolist()]
    if rank == 0:
        value = K / (dev_ms / 1e3)
        out = {
            "metric": "fl_rounds_per_sec", "value": value, "unit": "rounds/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": (value / BASELINE_ROUNDS_PER_S) if BASELINE_ROUNDS_PER_S else None,
            "dtype": "fp32", "data": "synthetic",
            "config": headline_config(world),
            "arm_details": {"parallelism": f"clients-sharded x{world}" if world > 1 else "1gpu",
                            "l2": "256 MiB flush write between timed rounds, outside the event brackets",
                            "timing": "CUDA events per round on the launching stream, summed; max over ranks",
                            "e2e_path": ("DriftSim.run_round(host_inputs, use_graph=True): one CUDA-graph replay per round + stream "
                                         "sync; the round kernel itself copies the pinned host inputs in (PCIe loads) and mirrors "
                                         "the metrics into pinned host memory (single graph node)")},
            "e2e": {"value": K / (e2e_ms / 1e3), "unit": "rounds/s", "h2d_bytes_per_step": sim.host_round_bytes()[0],
                    "d2h_bytes_per_step": sim.host_round_bytes()[1]},
            "gpu_launches": launches,
            "persistent_rounds_per_s": K / (persistent_ms / 1e3),
            "clocks": clk,
            "extra": extra,
            "impl": "feddrift_b200",
        }
        try:   # the reference arm ran first on this box (driver order): quote its sleep-removed rate next to ours
            with open(os.path.join(ROOT, "baseline", "_ref_last.json")) as fh:
                ref_last = json.load(fh)
            ns = ref_last.get("no_sleep", {}).get("value")
            if ns and ref_last.get("n_gpus") == world:
                out["reference_no_sleep"] = {"rounds_per_s": ns, "e2e_ratio_vs_no_sleep": out["e2e"]["value"] / ns,
                                             "reference_as_shipped_rounds_per_s": ref_last.get("value")}
        except (OSError, ValueError):
            pass
        if outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr.astype(np.float32))
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-sleep", dest="no_sleep", action="store_true",
                    help="reference arm only: report the sleep-removed variant as the main value (the as-shipped run always "
                         "carries it as the extra key 'no_sleep')")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed round computed as DIR/<name>.npy (float32): "
                         "round_metrics [clients, 4] (train correct, train loss sum, test correct, test loss sum) and "
                         "cluster_models [model slots, parameters]")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        from baseline.run_reference import main as ref_main
        return ref_main(args)
    run_ours(args)


if __name__ == "__main__":
    main()
