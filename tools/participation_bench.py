"""Rounds/s of the named large-federation configs with every client training (K = C) and with partial participation
(``client_num_per_round`` K < C), one executor per config:

  cfg2  fused round kernel, 100 SEA-fnn clients        K = 100 | 10
  cfg3  per-pair CUDA graphs, 64 MNIST-CNN clients     K = 64  | 16
  cfg4  pair-stacked ResNet-18, 32 CIFAR clients       K = 32  | 8
  cfg5  batched LSTM, 128 Shakespeare clients          K = 128 | 32

Each number is device-timed with CUDA events by ``experiments.configs.measure_config`` (time step 1 after a one-round warm-up);
the two K settings of a config alternate ``--repeat`` times so that the spread is visible.  Every round still evaluates all C
clients, which bounds what sampling can save: for the fused kernel the script also reads the kernel's per-phase timers
(train / aggregate / evaluate of CTA 0) and reports the evaluation share of a round.  One JSON line per run, with the card
name and power limit read in the same process, goes to ``--out``.

  python tools/participation_bench.py --out profiles/participation_bench.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RUNS = [("cfg2_sea_fnn_100clients_feddrift", 100, 10, 400),
        ("cfg3_mnist_cnn_64clients_ifca", 64, 16, None),
        ("cfg4_cifar_resnet18_32clients_aue", 32, 8, None),
        ("cfg5_shakespeare_lstm_128clients_win1", 128, 32, None)]


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in q.split(",")[:2]]
    except Exception:  # noqa: BLE001 — the power limit is informational; the device name still comes from torch
        name, power = None, None
    return {"gpu": torch.cuda.get_device_name(0), "smi_name": name, "power_limit": power}


def fused_phases(name: str, K: int, rounds: int):
    """Mean per-round (train, aggregate, evaluate) nanoseconds from the fused kernel's globaltimer stamps, one launch."""
    import torch
    from feddrift_b200.experiments.configs import CONFIGS
    from feddrift_b200.ops import small_round
    from feddrift_b200.sim import DriftSim, make_args
    from feddrift_b200.utils.metrics import MetricsSink
    kw = dict(CONFIGS[name])
    kw.update(total_train_iteration=2, epochs=5, lr=0.01, report_client=0, client_num_per_round=K)
    sim = DriftSim(make_args(**kw), device="cuda", sink=MetricsSink())
    sim.run_time_step(0, rounds=1)
    sim.begin_time_step(1)
    sim.run_rounds(1)
    st = sim._small_state()
    st["round0"] = sim.round_in_step
    st["timers"] = torch.zeros(rounds, 4, dtype=torch.int64, device="cuda")
    try:
        small_round.run_native(st, rounds)
        torch.cuda.synchronize()
        ts = st["timers"].cpu().double()
    finally:
        st.pop("timers")
    train = (ts[1:, 0] - ts[:-1, 2]).mean().item()   # round r's training starts when round r-1's evaluation ends
    agg = (ts[1:, 1] - ts[1:, 0]).mean().item()
    ev = (ts[1:, 2] - ts[1:, 1]).mean().item()
    del sim
    return {"train_ns": train, "aggregate_ns": agg, "evaluate_ns": ev, "evaluate_share": ev / max(train + agg + ev, 1.0)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "participation_bench.jsonl"))
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--configs", default="", help="comma-separated subset of the config names")
    a = ap.parse_args()
    import torch
    from feddrift_b200.experiments.configs import measure_config
    assert torch.cuda.is_available(), "participation_bench measures on a GPU"
    hw = card()
    runs = [r for r in RUNS if not a.configs or r[0] in a.configs.split(",")]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        for name, C, K, rounds in runs:
            for rep in range(a.repeat):
                for k in (C, K):
                    res = measure_config(name, "cuda", rounds=rounds, overrides={"client_num_per_round": k})
                    res.update(hw, clients_per_round=k, repeat=rep)
                    if res["fused_kernel"] and rep == 0:
                        res["phases"] = fused_phases(name, k, rounds or 40)
                    line = json.dumps(res)
                    print(line, flush=True)
                    f.write(line + "\n")


if __name__ == "__main__":
    main()
