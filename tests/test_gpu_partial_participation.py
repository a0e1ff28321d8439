"""Partial client participation on the GPU: the fused round kernel with a participants table vs its CPU oracle, the K == C
table vs no table (bit for bit), graph replay vs a plain launch under sampling, and the batched executors vs the per-pair
path when only K of C clients train."""
import copy
import os

import pytest
import torch

from feddrift_b200 import ops
from feddrift_b200.ops import reference as ref
from feddrift_b200.sim.engine import client_sampling
from test_gpu_small_round import make_state, to_cuda

pytestmark = pytest.mark.gpu

C37 = 37


def _with_table(st, K, rows=2):
    C = st["X"].shape[1]
    st["participants"] = torch.tensor([client_sampling(r, C, K) for r in range(rows)], dtype=torch.int32)
    return st


def _compare(st_cpu, rounds):
    st_gpu = to_cuda(copy.deepcopy(st_cpu))
    out_ref = ref.fed_round_small(st_cpu, rounds)
    out_gpu = ops.fed_round_small(st_gpu, rounds)
    torch.cuda.synchronize()
    return st_gpu, out_gpu, out_ref


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
@pytest.mark.parametrize("mode", ["pool", "time", "index"])
@pytest.mark.parametrize("K", [1, 3, C37 - 1])
def test_fused_round_with_participants_matches_reference(optimizer, mode, K):
    cfg = dict(C=C37, M=4, optimizer=optimizer, mode=mode)
    if mode == "index":
        cfg["B"] = 64
    st_cpu = _with_table(make_state(**cfg), K)   # 2 table rows, 3 rounds: the third round wraps to row 0
    st_gpu, out_gpu, out_ref = _compare(st_cpu, 3)
    assert torch.allclose(st_gpu["theta"].cpu(), st_cpu["theta"], rtol=2e-4, atol=2e-5), \
        (st_gpu["theta"].cpu() - st_cpu["theta"]).abs().max()
    assert torch.equal(st_gpu["opt_step"].cpu(), st_cpu["opt_step"])
    assert not st_cpu["opt_step"][K:].any()
    if optimizer == "adam":
        assert st_cpu["opt_step"][:K].any()
        assert torch.allclose(st_gpu["opt_m"].cpu(), st_cpu["opt_m"], rtol=1e-3, atol=1e-6)
    mg, mr = out_gpu["metrics"].cpu(), out_ref["metrics"]
    assert (mg[..., 0] - mr[..., 0]).abs().max() <= 1.0
    assert torch.allclose(mg[..., 1], mr[..., 1], rtol=1e-3, atol=1e-2)
    assert (mg[..., 2] - mr[..., 2]).abs().max() <= 1.0


def test_fused_round_with_participants_ifca_recluster():
    st_cpu = _with_table(make_state(M=3), 4)
    st_cpu["recluster_hard"] = True
    st_gpu, _, _ = _compare(st_cpu, 2)
    assert torch.equal(st_gpu["opt_step"].cpu(), st_cpu["opt_step"])
    Wg = st_gpu["W"][st_gpu["t_cur"]].cpu()
    assert torch.all(Wg.sum(0) == 1)       # re-clustering still assigns every client, sampled or not
    agree = (Wg.argmax(0) == st_cpu["W"][st_cpu["t_cur"]].argmax(0)).float().mean()
    assert agree >= 0.8


@pytest.mark.parametrize("mode", ["pool", "index"])
def test_identity_table_is_bit_identical_to_no_table(mode):
    cfg = dict(C=C37, M=4, mode=mode, B=64 if mode == "index" else 500)
    a = to_cuda(make_state(**cfg))
    b = to_cuda(make_state(**cfg))
    b["participants"] = torch.arange(C37, dtype=torch.int32, device="cuda")[None].repeat(3, 1)
    oa = ops.fed_round_small(a, 3)
    ob = ops.fed_round_small(b, 3)
    torch.cuda.synchronize()
    for k in ("theta", "opt_m", "opt_v", "opt_vmax", "opt_step"):
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(oa["metrics"], ob["metrics"])


def test_graph_replay_and_device_launch_agree_under_sampling():
    """N end-to-end rounds through the captured graph (the kernel reads the round counter on device, so every replay picks
    up its own row of the table) and N rounds in one launch leave the same models, bit for bit."""
    from feddrift_b200.sim import DriftSim, make_args

    def make():
        sim = DriftSim(make_args(client_num_in_total=10, client_num_per_round=4, comm_round=6, total_train_iteration=4),
                       device="cuda")
        for t in range(2):
            sim.run_time_step(t, rounds=6)
        sim.begin_time_step(2)
        sim.run_rounds(2)
        return sim

    a, b = make(), make()
    assert a.participants_table is not None and torch.equal(a.bank.theta, b.bank.theta)
    n = 8                                     # past comm_round: rows wrap
    ha = a.make_host_round_inputs()
    for _ in range(n):
        a.run_round(ha, use_graph=True)
    b.run_rounds_device(n)
    torch.cuda.synchronize()
    assert a.round_in_step == b.round_in_step == 2 + n
    assert torch.equal(a.bank.theta, b.bank.theta)
    assert torch.equal(a.clients.step, b.clients.step) and not a.clients.step[4:].any()


def _run_env(env, kw, rounds):
    from feddrift_b200.sim import DriftSim, make_args
    from feddrift_b200.utils.metrics import MetricsSink
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        sim = DriftSim(make_args(**kw), device="cuda", sink=MetricsSink())
        for name in ("dropout_1", "dropout_2"):
            if hasattr(sim.bank.template, name):
                getattr(sim.bank.template, name).p = 0.0
        init = sim.bank.theta.clone()
        out = sim.run_time_step(0, rounds=rounds)
        torch.cuda.synchronize()
        assert sim.participants_table is not None
        return init, sim.bank.theta.clone(), out, sim
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_stacked_executor_matches_per_pair_under_sampling():
    kw = dict(model="cnn", dataset="MNIST", client_num_in_total=6, client_num_per_round=3, concept_drift_algo="win-1",
              concept_drift_algo_arg="", concept_num=2, change_points="A", sample_num=16, batch_size=8, comm_round=3,
              total_train_iteration=2, epochs=2, lr=0.05, report_client=0, client_optimizer="sgd")
    _, th_s, _, sim = _run_env({"FDB_STACKED": "force", "FDB_STACKED_GRAPH": "0"}, kw, 3)
    assert sim.__dict__.get("_stack_stage") is not None, "stacked executor did not run"
    _, th_p, _, _ = _run_env({"FDB_STACKED": "0"}, kw, 3)
    scale = th_p.abs().max().item()
    assert (th_s - th_p).abs().max().item() < 2e-2 * scale


def test_batched_lstm_matches_per_pair_under_sampling():
    from feddrift_b200.ops import lstm as fused
    kw = dict(model="rnn", dataset="shakespeare", client_num_in_total=6, client_num_per_round=3, concept_drift_algo="win-1",
              concept_drift_algo_arg="", concept_num=2, change_points="A", sample_num=32, batch_size=16, comm_round=2,
              total_train_iteration=2, epochs=2, lr=0.05, client_optimizer="sgd", report_client=0)
    n0 = fused.CALLS["bwd"]
    init, th_b, out_b, _ = _run_env({"FDB_LSTM_BATCHED": "1"}, kw, 2)
    assert fused.CALLS["bwd"] > n0, "batched executor did not run the fused BPTT kernel"
    _, th_r, out_r, _ = _run_env({"FDB_LSTM_BATCHED": "0", "FDB_NO_FUSED_LSTM": "1"}, kw, 2)
    upd_b, upd_r = th_b - init, th_r - init
    scale = upd_r.abs().max().item()
    assert scale > 1e-4
    assert (upd_b - upd_r).abs().max().item() / scale < 6e-2
    assert abs(out_b["train_loss"] - out_r["train_loss"]) < 5e-2 * max(1.0, abs(out_r["train_loss"]))
