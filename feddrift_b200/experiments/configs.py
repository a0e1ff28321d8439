"""BASELINE.json's named configurations (synthetic data of the named shapes, random-init weights) as ``make_args`` keyword
sets, shared by ``bench.py`` (extra keys of the bench line) and ``tools/config_bench.py``."""
from __future__ import annotations

import time
from typing import Dict, Optional

CONFIGS = {
    # config 2: SEA-4 fnn, 100 clients packed on the box, FedDrift hierarchical soft-cluster
    "cfg2_sea_fnn_100clients_feddrift": dict(model="fnn", dataset="sea", client_num_in_total=100, client_num_per_round=100,
                                             concept_drift_algo="softcluster", concept_drift_algo_arg="H_A_C_1_10_0", concept_num=4,
                                             change_points="A", sample_num=100, batch_size=500, comm_round=40),
    # config 3: MNIST 2-conv CNN, 4 concepts, 64 clients, IFCA hard-r
    "cfg3_mnist_cnn_64clients_ifca": dict(model="cnn", dataset="MNIST", client_num_in_total=64, client_num_per_round=64,
                                          concept_drift_algo="softclusterwin-1", concept_drift_algo_arg="hard-r", concept_num=4,
                                          change_points="B", sample_num=64, batch_size=32, comm_round=3),
    # config 4: CIFAR-10 ResNet-18, 2 concepts, 32 clients, AUE ensemble
    "cfg4_cifar_resnet18_32clients_aue": dict(model="resnet18", dataset="cifar10", client_num_in_total=32, client_num_per_round=32,
                                              concept_drift_algo="aue", concept_drift_algo_arg="", concept_num=2, ensemble_window=2,
                                              change_points="A", sample_num=32, batch_size=32, comm_round=2),
    # config 5: fed_shakespeare char-LSTM, 128 clients, win-1 vs FedDrift
    "cfg5_shakespeare_lstm_128clients_win1": dict(model="rnn", dataset="shakespeare", client_num_in_total=128, client_num_per_round=128,
                                                  concept_drift_algo="win-1", concept_drift_algo_arg="", concept_num=2,
                                                  change_points="A", sample_num=32, batch_size=16, comm_round=2),
    "cfg5_shakespeare_lstm_128clients_feddrift": dict(model="rnn", dataset="shakespeare", client_num_in_total=128, client_num_per_round=128,
                                                      concept_drift_algo="softcluster", concept_drift_algo_arg="H_A_C_1_10_0", concept_num=2,
                                                      change_points="A", sample_num=32, batch_size=16, comm_round=2),
}


def measure_config(name: str, device, world: int = 1, rank: int = 0, rounds: Optional[int] = None,
                   overrides: Optional[Dict] = None) -> Dict:
    """Rounds/s of one named config at time step 1 after a one-round warm-up, device-timed with CUDA events on the launching
    stream (max over ranks is taken by the caller).  Under ``world > 1`` the clients are sharded over the ranks: the fused
    kernel uses its NVLink peer-inbox mode, the generic executor ``sim.shard_clients`` + the peer aggregation kernel.
    ``overrides`` replaces keys of the named config (e.g. ``client_num_per_round``)."""
    import torch
    from ..sim import DriftSim, make_args
    from ..utils.metrics import MetricsSink
    kw = dict(CONFIGS[name])
    kw.update(total_train_iteration=2, epochs=5, lr=0.01, report_client=0)
    kw.update(overrides or {})
    t0 = time.perf_counter()
    sim = DriftSim(make_args(**kw), device=device, sink=MetricsSink())
    fused = bool(sim.spec is not None and sim.algo.fused_ok())
    if world > 1:
        import torch.distributed as dist
        if fused:
            from ..parallel.symm import attach_multi_gpu
            attach_multi_gpu(sim, world, rank)
        else:
            sim.shard_clients = True
    sim.run_time_step(0, rounds=1)
    sim.begin_time_step(1)
    sim.run_rounds(1)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    setup = time.perf_counter() - t0
    R = int(rounds or kw["comm_round"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = sim.run_rounds(R)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt)
    res = {"config": name, "world": world, "rounds": R, "rounds_per_s": R / (ms / 1e3), "ms_per_round": ms / R,
           "setup_s": round(setup, 2), "fused_kernel": fused, "P": sim.bank.P, "clients": sim.C,
           "last": {k: round(v, 4) for k, v in out.items() if isinstance(v, float)},
           "theta_sq_sum": float(sim.bank.theta.detach().double().square().sum())}   # fingerprint of the trained models
    del sim
    torch.cuda.empty_cache()
    return res
