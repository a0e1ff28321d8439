"""Partial client participation (``client_num_per_round`` K < ``client_num_in_total`` C) in the device engine: the
per-round client draw, worker-slot optimizer state in the CPU oracle of the fused round kernel, every drift algorithm
through ``DriftSim`` on CPU, CFL splits that address the sampled clients, and the multi-GPU refusal."""
import copy

import numpy as np
import pytest
import torch

from feddrift_b200.ops import reference as ref
from feddrift_b200.sim import DriftSim, make_args
from feddrift_b200.sim.engine import client_sampling
from feddrift_b200.utils.metrics import MetricsSink


@pytest.mark.parametrize("C,K,r", [(10, 3, 0), (10, 3, 7), (100, 10, 0), (100, 10, 39), (6, 5, 2), (37, 1, 11)])
def test_client_sampling_matches_facade_and_reference_draw(C, K, r):
    from feddrift_b200.drift.fedavg_ens import _BaseAggregator
    state = np.random.get_state()
    try:
        facade = [int(c) for c in _BaseAggregator.client_sampling(None, r, C, K)]
        np.random.seed(r)
        direct = [int(c) for c in np.random.choice(range(C), K, replace=False)]
    finally:
        np.random.set_state(state)
    before = np.random.get_state()[1].copy()
    mine = client_sampling(r, C, K)
    assert mine == facade == direct
    assert np.array_equal(np.random.get_state()[1], before), "client_sampling must not touch the global RNG"


@pytest.mark.parametrize("C,K", [(6, 6), (6, 9)])
def test_client_sampling_full_participation(C, K):
    assert client_sampling(3, C, K) == list(range(C))


def _state(C, M=2, S=40, B=64, epochs=3, optimizer="adam", seed=0, T1=2, t=0):
    g = torch.Generator().manual_seed(seed)
    din, hid, dout = 3, 6, 2
    P = ref.mlp_param_count("fnn", din, hid, dout)
    X = torch.rand(T1, C, S, din, generator=g) * 10.0
    Y = (X[..., 1] + X[..., 2] > 10.0).long()
    nsamp = torch.full((T1, C), S, dtype=torch.int32)
    W = torch.zeros(t + 1, M, C)
    W[t, 0, :] = 1.0                      # model 0 trained by every client, model 1 idle
    theta = torch.randn(M, P, generator=g) * 0.3
    z = lambda: torch.zeros(C, M, P)      # noqa: E731
    return dict(kind="fnn", din=din, hid=hid, dout=dout, X=X, Y=Y, nsamp=nsamp, batch_size=B, W=W, theta=theta,
                opt_m=z(), opt_v=z(), opt_vmax=z(), opt_step=torch.zeros(C, M, dtype=torch.int32), lr=0.01, wd=0.001,
                epochs=epochs, optimizer=optimizer, seed=77, round0=0, t_cur=t, sample_mode="pool")


def _subset(st, clients):
    """The same federation restricted to ``clients`` (a smaller, fully participating one)."""
    out = copy.deepcopy(st)
    out.pop("participants", None)
    idx = torch.tensor(clients)
    for k in ("X", "Y"):
        out[k] = st[k][:, idx].clone()
    out["nsamp"] = st["nsamp"][:, idx].clone()
    out["W"] = st["W"][:, :, idx].clone()
    K, M, P = len(clients), st["theta"].shape[0], st["theta"].shape[1]
    out["opt_m"], out["opt_v"], out["opt_vmax"] = (torch.zeros(K, M, P) for _ in range(3))
    out["opt_step"] = torch.zeros(K, M, dtype=torch.int32)
    return out


def test_oracle_fixed_sample_equals_smaller_full_federation():
    """Clients {0, 2, 4} of 6 with one batch per client (so batch selection does not depend on the client-keyed hash) must
    train exactly like a 3-client federation of those clients: same models and Adam state, bit for bit."""
    sampled = [0, 2, 4]
    st = _state(C=6)
    st["participants"] = torch.tensor([sampled], dtype=torch.int32)
    small = _subset(st, sampled)
    out_p = ref.fed_round_small(st, 3)
    out_s = ref.fed_round_small(small, 3)
    assert torch.equal(st["theta"], small["theta"])
    for k in ("opt_m", "opt_v", "opt_vmax", "opt_step"):
        assert torch.equal(st[k][:3], small[k]), k
        assert not st[k][3:].any(), k       # rows of idle worker slots stay untouched
    assert out_p["metrics"].shape == (3, 6, 4)
    assert torch.equal(out_p["metrics"][:, sampled], out_s["metrics"])


@pytest.mark.parametrize("optimizer", ["adam", "sgd"])
def test_oracle_rotating_samples_slot_state_and_full_evaluation(optimizer):
    C, K, R, E = 6, 3, 4, 2
    st = _state(C=C, B=16, epochs=E, optimizer=optimizer, seed=1)
    st["participants"] = torch.tensor([client_sampling(r, C, K) for r in range(R)], dtype=torch.int32)
    theta1 = st["theta"][1].clone()
    out = ref.fed_round_small(st, R)
    if optimizer == "adam":
        assert torch.equal(st["opt_step"][:K, 0], torch.full((K,), E * R, dtype=torch.int32))
        assert not st["opt_m"][K:].any() and not st["opt_step"][K:].any()
    assert not st["opt_step"][:, 1].any()
    assert torch.equal(st["theta"][1], theta1)        # a model nobody trains keeps its parameters
    m = out["metrics"]
    assert m.shape == (R, C, 4)
    assert (m[..., 1] > 0).all() and (m[..., 3] > 0).all()   # every client is evaluated every round


def test_oracle_explicit_identity_table_is_full_participation():
    st = _state(C=5, B=16, seed=2)
    st_id = copy.deepcopy(st)
    st_id["participants"] = torch.arange(5, dtype=torch.int32)[None].repeat(3, 1)
    a = ref.fed_round_small(st, 3)
    b = ref.fed_round_small(st_id, 3)
    for k in ("theta", "opt_m", "opt_v", "opt_vmax", "opt_step"):
        assert torch.equal(st[k], st_id[k]), k
    assert torch.equal(a["metrics"], b["metrics"])


def test_participants_table_validation():
    from feddrift_b200.ops.small_round import check_participants
    check_participants(torch.tensor([[0, 2, 4], [5, 1, 3]], dtype=torch.int32), 6)
    bad = [torch.tensor([[0, 2]], dtype=torch.int64), torch.tensor([0, 2], dtype=torch.int32),
           torch.tensor([[0, 6]], dtype=torch.int32), torch.tensor([[-1, 2]], dtype=torch.int32),
           torch.tensor([[1, 1]], dtype=torch.int32), torch.zeros(1, 7, dtype=torch.int32), torch.zeros(1, 0, dtype=torch.int32)]
    for b in bad:
        with pytest.raises(ValueError):
            check_participants(b, 6)


ALGOS = [("softcluster", "H_A_C_1_10_0"), ("softcluster", "hard-r"), ("win-1", ""), ("aue", ""), ("kue", ""),
         ("driftsurf", "0"), ("ada", "win-1_round"), ("softcluster", "cfl_0.1_win-1")]


def _sim(algo, arg, C=6, K=3, **kw):
    a = dict(model="fnn", dataset="sea", client_num_in_total=C, client_num_per_round=K, concept_drift_algo=algo,
             concept_drift_algo_arg=arg, concept_num=2, change_points="A", sample_num=30, batch_size=16, comm_round=3,
             total_train_iteration=2, epochs=1, ensemble_window=2)
    a.update(kw)
    return DriftSim(make_args(**a), device="cpu", sink=MetricsSink())


@pytest.mark.parametrize("algo,arg", ALGOS)
def test_drift_sim_cpu_partial_participation(algo, arg):
    C, K = 6, 3
    sim = _sim(algo, arg, C, K)
    assert sim.participants_table is not None and tuple(sim.participants_table.shape) == (3, K)
    for r in range(5):   # rounds past comm_round reuse row r % comm_round
        assert sim.participants(r) == client_sampling(r % 3, C, K)
    out = sim.run()
    assert out["rounds"] == 2 * 3 and out["history"]
    for c in range(C):   # evaluation covers every client, sampled or not
        assert sim.sink.last(f"Train/Acc-CL-{c}") is not None
    assert not sim.clients.params[K:].any() and not sim.clients.step[K:].any()   # idle worker slots
    h = out["history"][-1]
    assert 0.0 <= h["test_acc"] <= 1.0 and h["train_loss"] == h["train_loss"]


def test_full_participation_keeps_no_table():
    sim = _sim("softcluster", "H_A_C_1_10_0", C=6, K=6)
    assert sim.participants_table is None and sim.participants(4) == list(range(6))
    sim.begin_time_step(0)
    assert "participants" not in sim._small_state()


def test_cfl_split_assigns_sampled_client_columns():
    """Slot-indexed raw updates: a split must move the W columns of the clients that uploaded, not of the slot numbers."""
    from feddrift_b200.drift.softcluster import SoftClusterState
    from feddrift_b200.parallel.arena import ModelBank
    torch.manual_seed(0)
    C, M = 6, 2
    bank = ModelBank(torch.nn.Linear(3, 2), M, "cpu")
    st = SoftClusterState(C, M, cluster_alg="cfl_0.1_win-1", cfl_gamma=0.1, cfl_retrain="win-1")
    st.cluster_init()
    clients = [5, 0, 3, 2]                                  # slot s uploaded the update of client clients[s]
    d = torch.randn(bank.P, generator=torch.Generator().manual_seed(1))
    params = torch.zeros(C, M, bank.P)
    n = torch.zeros(C, M)
    n[:4, 0] = 10
    params[:4, 0] = bank.theta[0] + d                       # warm-up round: common direction sets the CFL thresholds
    assert not st.cluster_cfl(0, 1, bank, params, n, clients=clients)
    sign = torch.tensor([1.0, 1.0, -1.0, -1.0])             # clients 5, 0 vs clients 3, 2
    params[:4, 0] = bank.theta[0] + sign[:, None] * d
    assert st.cluster_cfl(0, 2, bank, params, n, clients=clients)
    on0 = set(np.nonzero(st.W[0][0])[0].tolist())
    on1 = set(np.nonzero(st.W[0][1])[0].tolist())
    assert {1, 4} <= on0                                    # idle members stay on the split model
    assert on1 in ({5, 0}, {3, 2}) and on0 == set(range(C)) - on1


def test_clusterfl_split_moves_sampled_clients():
    sim = _sim("clusterfl", "win-1", C=6, K=4)
    algo = sim.algo
    clients = [4, 1, 5, 0]
    P = sim.bank.P
    d = torch.randn(P, generator=torch.Generator().manual_seed(2))
    params = torch.zeros(6, sim.M, P)
    params[:4, 0] = sim.bank.theta[0] + torch.tensor([1.0, -1.0, 1.0, -1.0])[:, None] * d
    assert algo.on_client_updates(0, params, torch.ones(6, sim.M), clients=clients)
    moved = set(np.nonzero(algo.assign == 1)[0].tolist())
    assert moved in ({4, 5}, {1, 0})


@pytest.mark.parametrize("how", ["multi", "shard"])
def test_multi_gpu_partial_participation_is_refused(how):
    sim = _sim("softcluster", "H_A_C_1_10_0")
    sim.begin_time_step(0)
    if how == "multi":
        sim.multi = {"world": 2, "rank": 0, "flag_base": 0, "metrics_rounds": 8}
    else:
        sim.shard_clients = True
    theta = sim.bank.theta.clone()
    with pytest.raises(ValueError, match="single-GPU"):
        sim.run_rounds(1)
    with pytest.raises(ValueError, match="single-GPU"):
        sim.run_rounds_device(1)
    assert sim.round_in_step == 0 and torch.equal(sim.bank.theta, theta)   # refused before anything ran
