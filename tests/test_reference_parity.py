"""Parity of the FedDrift brain against the ACTUAL reference implementation (microsoft/FedDrift).

Every test drives ``feddrift_b200`` through a scripted scenario and compares what it computes with what the unmodified
reference computed on the same inputs: drift detection, LRU slot allocation with parameter copy, the marking window, the
A/B distances, complete/average linkage with the δ' cut, merges and the identical re-initialisation, through the
reference's own ``cluster_hierarchical`` / ``cluster`` code paths (``FedAvgEnsDataLoader.py:640-978``), and the other
state machines, aggregator scores and wire formats below.

The reference's side of every scenario (the ``_ref_*`` functions) was run once against the reference sources and its
observations are stored in ``tests/golden/reference_parity.json``; its change-point data files are stored verbatim under
``tests/golden/changepoints``.  The suite therefore needs no copy of the reference.  To record them again from a FedDrift
checkout::

    python tests/test_reference_parity.py --reference /path/to/FedDrift
"""
import json
import os
import shutil
import sys

import numpy as np
import pytest
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden", "reference_parity.json")
GOLDEN_CP_DIR = os.path.join(HERE, "golden", "changepoints")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _plain(o):
    if isinstance(o, (np.ndarray, torch.Tensor)):
        return o.tolist()
    if isinstance(o, np.generic):
        return o.item()
    raise TypeError(f"not JSON-serialisable: {type(o)}")


def _canon(x):
    """JSON-normal form (dict keys → str, tuples → lists, numpy / torch → Python numbers), applied to both sides."""
    return json.loads(json.dumps(x, default=_plain))


@pytest.fixture(autouse=True)
def _default_reinit_seed(monkeypatch):
    """Model slots are initialised from ``models.utils.torch_seed``, which every experiment resets to its own seed; the
    golden data was recorded with the default."""
    from feddrift_b200.models import utils as mutils
    monkeypatch.setattr(mutils, "torch_seed", 42)


_GOLD = None


def _gold(name):
    global _GOLD
    if _GOLD is None:
        with open(GOLDEN) as fh:
            _GOLD = json.load(fh)
    return _GOLD[name]


C, T, S, M = 5, 5, 16, 8
# concept k: label = [x0 > 0.5] XOR flip_k on half-plane pairs; 0/1 are opposites, 2/3 use the other axis
CONCEPT_W = {0: ([8.0, 0.0], -4.0), 1: ([-8.0, 0.0], 4.0), 2: ([0.0, 8.0], -4.0), 3: ([0.0, -8.0], 4.0)}
HIER_SEEDS = [0, 1, 2, 3, 4, 5]
HIER_VARIANTS = ["H_A_C", "H_B_D"]
MATRIX_ALGS = ["hard", "softmax_2", "mmacc_10"]
DRIFTSURF_SEEDS = [0, 1, 2, 3]
MMACC_SEEDS = [0, 1, 2]
CFL_RETRAIN = ["win-1", "all"]
RETRAIN_METHODS = ["all", "win-1", "win-3", "sel-0,2,4", "weight-linear", "weight-exp", 'clientsel-[[0,1],[2],[1,4]]']
TOPOLOGIES = ((6, 2), (8, 4), (5, 2))
MPC_P = 2 ** 15 - 19


def _label(x, k):
    w, b = CONCEPT_W[k]
    return ((x @ torch.tensor(w)) + b > 0).long()


def _ideal_state_dict(k):
    w, b = CONCEPT_W[k]
    # 2-class logistic regression: class-1 logit = w·x + b, class-0 logit = 0
    return {"linear.weight": torch.tensor([[0.0, 0.0], w]), "linear.bias": torch.tensor([0.0, b])}


class _LR(nn.Module):
    """Plain linear 2-class model (no sigmoid) used on BOTH sides."""

    def __init__(self):
        super().__init__()
        self.linear = nn.Linear(2, 2)

    def forward(self, x):
        return self.linear(x)


def _schedule(seed):
    """[T+1, C] concept ids with staggered drifts (some clients drift to the same new concept at different times)."""
    rng = np.random.RandomState(seed)
    cp = np.zeros((T + 1, C), dtype=np.int64)
    for c in range(C):
        k, t_change = 0, rng.randint(1, T)
        for t in range(T + 1):
            if t == t_change:
                k = rng.choice([1, 2, 3])
            cp[t, c] = k
        if rng.rand() < 0.4:   # a second drift back or onwards
            t2 = min(T, t_change + rng.randint(1, 3))
            cp[t2:, c] = rng.choice([0, 1, 2, 3])
    return cp


def _hier_scenario(seed):
    """Scripted drifting federation shared by both sides: concept schedule, data, our model bank and evaluator."""
    from feddrift_b200.data.drift import DriftData
    from feddrift_b200.drift.evaluator import Evaluator
    from feddrift_b200.parallel.arena import ModelBank
    cp = _schedule(seed)
    g = torch.Generator().manual_seed(100 + seed)
    X = torch.rand(T + 1, C, S, 2, generator=g)
    X = torch.where((X - 0.5).abs() < 0.06, X + 0.12 * torch.sign(X - 0.5 + 1e-9), X)   # keep a margin around the boundaries
    Y = torch.stack([torch.stack([_label(X[t, c], int(cp[t, c])) for c in range(C)]) for t in range(T + 1)])
    nsamp = torch.full((T + 1, C), S, dtype=torch.int32)
    data = DriftData("parity", X, Y, nsamp, cp, 2)
    torch.manual_seed(7)
    bank = ModelBank(_LR(), M, "cpu")
    return cp, X, Y, bank, Evaluator(bank, data, batch_size=S)


def _hier_train(t, W_t, cp, bank, models):
    """Emulated local training + aggregation: every model used at t becomes the ideal classifier of the majority
    concept of its clients (identical on both sides)."""
    for m in range(M):
        cs = np.nonzero(W_t[m] > 0)[0]
        if len(cs) == 0:
            continue
        sd = _ideal_state_dict(int(np.bincount(cp[t, cs]).argmax()))
        if bank is not None:
            bank.load_state_dict(m, sd)
        if models is not None:
            models[m].load_state_dict(sd)


@pytest.mark.parametrize("seed", HIER_SEEDS)
@pytest.mark.parametrize("variant", HIER_VARIANTS)
def test_hierarchical_feddrift_matches_reference_implementation(seed, variant):
    from feddrift_b200.drift.softcluster import SoftClusterState
    gold = _gold("hierarchical")[f"{variant}/{seed}"]
    dist_kind, link = variant.split("_")[1], variant.split("_")[2]
    cp, X, Y, bank, ev = _hier_scenario(seed)
    mine = SoftClusterState(C, M, "H", h_delta=0.15, h_deltap=0.15, h_w=1, h_distance=dist_kind, h_cluster=link)
    mine.cluster_init()

    def check(t):
        want = gold[t]
        for tt in range(t + 1):
            assert np.array_equal(mine.W[tt], np.asarray(want["W"][tt])), (seed, variant, t, tt, mine.W[tt], want["W"][tt])
        assert _canon({c: tuple(v) for c, v in mine.h_marked.items()}) == want["marked"]
        for m in range(M):
            assert torch.allclose(bank.theta[m], torch.tensor(want["theta"][m]), atol=1e-6), (seed, variant, t, m)

    _hier_train(0, mine.W[0], cp, bank, None)
    acc0 = ev.acc_matrix([0], 0)[0]
    for c in range(C):   # the aggregator records the t = 0 accuracies for the drift detector (SoftCluster.py:107-116)
        mine.set_acc(c, float(acc0[c]))
    check(0)
    for t in range(1, T + 1):
        mine.cluster_hierarchical(t, bank, ev)
        check(t)
        _hier_train(t, mine.W[t], cp, bank, None)
    # the scenario must actually exercise the algorithm: new models were spawned, and usually some were merged
    assert max(int((mine.W[t].sum(1) > 0).sum()) for t in range(T + 1)) >= 2


def _ref_hierarchical(ref_mod, seed, variant):
    from feddrift_b200.models import utils as mutils
    dist_kind, link = variant.split("_")[1], variant.split("_")[2]
    cp, X, Y, bank, ev = _hier_scenario(seed)
    init_sd = {k: v.clone() for k, v in bank.state_dict(0).items()}
    models = [_LR() for _ in range(M)]
    for mod in models:
        mod.load_state_dict(init_sd)
    ref_mod.reinitialize = lambda model: model.load_state_dict(init_sd)      # "every re-init is identical" on both sides
    all_data = [[[(X[t, c], Y[t, c])] for t in range(T + 1)] for c in range(C)]   # [client][iter] -> list of batches
    theirs = ref_mod.SoftClusterState(C, M, "H", h_delta=0.15, h_deltap=0.15, h_w=1, h_distance=dist_kind, h_cluster=link)
    theirs.cluster_init()
    out = []

    def observe(t):
        out.append(_canon({"W": [theirs.train_data_weights[tt] for tt in range(t + 1)],
                           "marked": {c: tuple(v) for c, v in theirs.h_marked.items()},
                           "theta": [mutils.flatten_state_dict(models[m].state_dict()) for m in range(M)]}))

    _hier_train(0, theirs.train_data_weights[0], cp, bank, models)
    acc0 = ev.acc_matrix([0], 0)[0]
    for c in range(C):
        theirs.set_acc(c, float(acc0[c]))
    observe(0)
    for t in range(1, T + 1):
        theirs.cluster_hierarchical(t, models, all_data, torch.device("cpu"))
        observe(t)
        _hier_train(t, theirs.train_data_weights[t], cp, bank, models)
    return out


def _matrix_kw(alg):
    kw = dict(cluster_alg=alg.split("_")[0] if alg.startswith("mmacc") else alg)
    if alg.startswith("softmax"):
        kw = dict(cluster_alg=alg, softmax_alpha=2)
    if alg.startswith("mmacc"):
        kw = dict(cluster_alg=alg, mmacc_delta=0.10)
    return kw


def _matrix_run(state, weights_attr):
    """`cluster()` on the scripted accuracy matrices; returns W[t] for t = 1..4."""
    state.cluster_init()
    rng = np.random.RandomState(3)
    for c in range(6):
        state.set_acc(c, 0.9)
    out = []
    for t in range(1, 5):
        acc = rng.rand(4, 6) * 0.3 + 0.6
        acc[:, rng.randint(0, 6)] -= 0.35      # one client's data drifted: every model is bad on it
        state.cluster(acc.copy(), t, 0)
        out.append(np.array(getattr(state, weights_attr)[t]))
    return out


@pytest.mark.parametrize("alg", MATRIX_ALGS)
def test_matrix_driven_clustering_matches_reference_implementation(alg):
    """`cluster()` on scripted accuracy matrices: IFCA hard, softmax_α and FedDrift-Eager (mmacc_δ with LRU slots)."""
    from feddrift_b200.drift.softcluster import SoftClusterState
    want = _gold("matrix")[alg]
    got = _matrix_run(SoftClusterState(6, 4, **_matrix_kw(alg)), "W")
    for t in range(1, 5):
        assert np.allclose(got[t - 1], np.asarray(want[t - 1])), (alg, t)


def _ada_run(state, as_numpy):
    g = torch.Generator().manual_seed(0)
    theta = torch.randn(5000, generator=g)
    out = []
    for t in range(12):
        theta = theta + 0.3 * torch.randn(5000, generator=g) * (3.0 if t in (5, 9) else 1.0)   # two "drifts"
        state.update(theta.double().numpy() if as_numpy else theta.clone(), t)
        out.append(float(state.current_lr()))
    return out


def test_ada_state_matches_reference_implementation():
    """Adaptive-FedAvg server learning-rate schedule (EMA mean / variance / ratio) on the same parameter trajectory."""
    from feddrift_b200.drift.states import AdaState
    want = _gold("ada")
    got = _ada_run(AdaState(init_lr=0.05), as_numpy=False)
    for t in range(12):
        assert abs(got[t] - want[t]) <= 1e-5 * want[t] + 1e-9, t


def _driftsurf_run(state, seed, device):
    rng = np.random.RandomState(seed)
    cur = {}
    state._score = lambda key, *a, **k: cur[key]
    out = []
    for it in range(1, 16):
        base = 0.9 - (0.3 if rng.rand() < 0.3 else 0.0)          # occasional accuracy collapse of the predictive model
        cur.update(pred=base + 0.02 * rng.randn(), stab=0.88 + 0.05 * rng.randn(), reac=0.7 + 0.25 * rng.rand())
        state.run_ds_algo(None, device, it)
        out.append(_canon({"state": state.state, "model_key": state.model_key, "train_keys": state.get_train_keys(),
                           "data": {key: state.train_data_dict[key] or [] for key in ("pred", "stab", "reac")},
                           "acc_best": state.acc_best, "reac_ctr": state.reac_ctr}))
    return out


@pytest.mark.parametrize("seed", DRIFTSURF_SEEDS)
def test_driftsurf_state_machine_matches_reference_implementation(seed):
    """DriftSurf stable/reactive transitions, training windows, model switch — same scripted accuracy stream."""
    from feddrift_b200.drift.states import DriftSurfState
    want = _gold("driftsurf")[str(seed)]
    got = _driftsurf_run(DriftSurfState(delta=0.1, r=3, wl=4), seed, None)
    for it, (a, b) in enumerate(zip(got, want), start=1):
        assert a["state"] == b["state"] and a["model_key"] == b["model_key"], it
        assert a["train_keys"] == b["train_keys"], it
        for key in ("pred", "stab", "reac"):
            assert a["data"][key] == b["data"][key], (it, key)
        assert abs(a["acc_best"] - b["acc_best"]) < 1e-12
        assert a["reac_ctr"] == b["reac_ctr"]
    assert len(got) == len(want)


def test_change_point_matrices_equal_the_reference_data_files():
    """Every named change-point matrix (A–F, W–Z, R0–R9) equals ``data/changepoints/<name>.cp`` of the reference."""
    from feddrift_b200.data import changepoints
    names = sorted(f[:-3] for f in os.listdir(GOLDEN_CP_DIR) if f.endswith(".cp"))
    assert len(names) >= 20
    for name in names:
        want = np.loadtxt(os.path.join(GOLDEN_CP_DIR, name + ".cp"), dtype=np.int64)
        got = changepoints.named(name)
        assert got.shape == want.shape and np.array_equal(got, want), name


def _retrain_cases():
    for t_cur in (0, 2, 4):
        for method in RETRAIN_METHODS:
            if method.startswith("clientsel") and t_cur < 4:
                continue
            yield method, t_cur


def test_retrain_window_selector_matches_reference_csv_loader():
    """`select_iterations` (all / win-k / sel-… / clientsel-… / weight-linear|exp) vs the iterations the reference's
    ``common/retrain.py`` actually reads, observed by giving every (client, iteration) CSV a unique marker row."""
    from feddrift_b200.data.drift import select_iterations
    gold = _gold("retrain")
    cases = list(_retrain_cases())
    assert len(gold) == len(cases)
    for method, t_cur in cases:
        for c, want in enumerate(gold[f"{method}|{t_cur}"]):
            got = list(select_iterations(method, t_cur, c))
            assert sorted(got) == sorted(want), (method, t_cur, c, got, want)


def _ref_retrain(tmp_dir):
    import pandas as pd
    from fedml_api.data_preprocessing.common import retrain as ref_retrain
    if not hasattr(pd.DataFrame, "append"):   # pandas ≥ 2 removed it; the reference arm restores it the same way
        pd.DataFrame.append = (lambda self, other, ignore_index=False, **kw:
                               pd.concat([self, other], ignore_index=ignore_index) if len(self) else other.reset_index(drop=True))
    C_, T_ = 3, 5
    for c in range(C_):
        for it in range(T_ + 2):
            pd.DataFrame({"f1": [float(it)], "label": [c]}).to_csv(os.path.join(tmp_dir, f"client_{c}_iter_{it}.csv"), index=False)
    out = {}
    for method, t_cur in _retrain_cases():
        train, _ = ref_retrain.load_retrain_table_data(tmp_dir + "/", C_, t_cur, "client_{}_iter_{}.csv", method)
        out[f"{method}|{t_cur}"] = [[int(v) for v in train[c]["f1"].tolist()] for c in range(C_)]
    return out


def _mpc_run(mod):
    """The deterministic TurboAggregate entry points on fixed inputs, every result reduced mod p."""
    p = MPC_P
    rng = np.random.RandomState(0)
    modp = lambda v: (np.asarray(v, dtype=np.int64) % p).tolist()   # noqa: E731
    out = {"modular_inv": [int(mod.modular_inv(a, p)) for a in (3, 17, 12345, p - 2)],
           "divmod": [int(mod.divmod(a, 7, p)) for a in (3, 17, 12345, p - 2)]}
    vals = [int(v) for v in rng.randint(1, p, 6)]
    out["PI"] = int(mod.PI(vals, p))
    alpha, beta = np.arange(1, 8), np.arange(8, 12)
    out["lagrange"] = modp(mod.gen_Lagrange_coeffs(alpha, beta, p))
    out["bgw"] = modp(mod.gen_BGW_lambda_s(alpha, p))
    N, K, T_ = 8, 2, 1
    X = rng.randint(0, p, (4, 6)).astype(np.int64)
    R_ = rng.randint(0, p, (T_, 2, 6)).astype(np.int64)
    enc = np.asarray(mod.LCC_encoding_w_Random(X, R_, N, K, T_, p), dtype=np.int64) % p
    out["enc"] = enc.tolist()
    widx = np.arange(K + T_)
    flat = enc[widx].reshape(len(widx), -1)   # [workers, m/K · d]
    out["dec"] = modp(mod.LCC_decoding(flat, 1, N, K, T_, widx, p))
    out["X"] = (X % p).tolist()
    # small secrets: the reference computes g ** sk in numpy int64 (it overflows for real key sizes; ours uses pow(g, sk, p))
    out["pk"] = int(mod.my_pk_gen(11, p, 5))
    out["key_agreement"] = int(mod.my_key_agreement(7, 3, p, 5))
    return out


def test_mpc_primitives_match_reference_implementation():
    """TurboAggregate finite-field primitives vs ``turboaggregate/mpc_function.py`` (deterministic entry points)."""
    from feddrift_b200.fl import turboaggregate as ours
    got, want = _mpc_run(ours), _gold("mpc")
    for key in ("modular_inv", "divmod", "PI", "lagrange", "bgw", "enc", "dec", "pk", "key_agreement"):
        assert got[key] == want[key], key
    assert np.array_equal(np.asarray(got["dec"]).reshape(2, 2, 6).reshape(4, 6), np.asarray(got["X"]))   # the decode recovers X


def _topology_run(cls):
    out = {}
    for n, k in TOPOLOGIES:
        a = cls(n, k)
        a.generate_topology()
        out[f"{n},{k}"] = {"topology": np.asarray(a.topology).tolist(),
                           "in_idx": [list(a.get_in_neighbor_idx_list(i)) for i in range(n)],
                           "in_w": [np.asarray(a.get_in_neighbor_weights(i)).tolist() for i in range(n)]}
    return _canon(out)


def _message_json(cls):
    msg = cls(3, 1, 0)
    msg.add_params("client_idx", "4")
    msg.add_params("num_samples", 17)
    return msg.to_json()


def test_symmetric_topology_and_message_wire_format_match_reference():
    from feddrift_b200.core.message import Message
    from feddrift_b200.core.topology import SymmetricTopologyManager
    got, want = _topology_run(SymmetricTopologyManager), _gold("topology")
    for name in want:
        a, b = got[name], want[name]
        assert np.allclose(np.asarray(a["topology"]), np.asarray(b["topology"])), name
        assert a["in_idx"] == b["in_idx"], name
        for wa, wb in zip(a["in_w"], b["in_w"]):
            assert np.allclose(wa, wb), name
    ref_json = _gold("message_json")
    assert json.loads(_message_json(Message)) == json.loads(ref_json)
    back = Message()   # and the reference's wire bytes read back through ours
    back.init_from_json_string(ref_json)
    assert back.get_type() == 3 and back.get_sender_id() == 1 and back.get("num_samples") == 17


def _mmacc_run(state, seed, reference):
    """Legacy FedDrift-Eager (mmacc) then oracle (mmgeniex) model selection on scripted accuracies.  The reference
    scores a model through ``_score`` and keeps real models in ``models`` / accuracies in ``acc_dict``; ours takes an
    evaluator and ``set_model`` / ``set_acc``."""
    C_, M_ = 5, 3
    rng = np.random.RandomState(seed)
    table, cur_t = {}, [0]

    class FakeEvaluator:
        def acc_matrix(self, models, t):
            return np.array([[table[(m, c, t)] for c in range(C_)] for m in models])

    if reference:
        state._score = lambda m, data, device: table[(m, data, cur_t[0])]      # `data` is the client id in this harness
        select = lambda t: state.run_model_select({c: c for c in range(C_)} if t else None, "cpu", t)   # noqa: E731
        set_model = lambda m: state.models.__setitem__(m, object())             # noqa: E731
        set_acc = state.acc_dict.__setitem__
    else:
        select = lambda t: state.run_model_select(FakeEvaluator() if t else None, t)   # noqa: E731
        set_model, set_acc = state.set_model, state.set_acc
    select(0)
    set_model(0)
    for c in range(C_):
        set_acc(c, 0.9)
    steps = []
    for t in range(1, 6):
        cur_t[0] = t
        for m in range(M_):
            for c in range(C_):
                table[(m, c, t)] = float(np.clip(0.9 - (0.4 if rng.rand() < 0.25 else 0.0) + 0.03 * rng.randn(), 0, 1))
        select(t)
        steps.append(_canon({"data": state.train_data_dict, "train_idx": state.train_model_idx,
                             "test_idx": state.test_model_idx}))
        for m in {state.train_model_idx[c] for c in range(C_)}:   # models that got data this step exist from now on
            set_model(m)
        for c in range(C_):
            set_acc(c, table[(state.train_model_idx[c], c, t)])
    cp = (rng.rand(4, C_) < 0.5).astype(np.int64)
    cp[0] = 0
    return steps, cp


def _geniex_run(state, cp):
    out = []
    for t in range(6):
        state.model_select_geniex(t, cp, 2)
        out.append(_canon({"train_idx": state.train_model_idx, "test_idx": state.test_model_idx}))
    return out, _canon(state.train_data_dict)


@pytest.mark.parametrize("seed", MMACC_SEEDS)
def test_multi_model_acc_state_matches_reference_implementation(seed):
    """Legacy FedDrift-Eager (mmacc) and oracle (mmgeni / mmgeniex) model selection on scripted accuracies."""
    from feddrift_b200.drift.states import MultiModelAccState
    want = _gold("mmacc")[str(seed)]
    steps, cp = _mmacc_run(MultiModelAccState(5, 3, 0.1), seed, reference=False)
    assert len(steps) == len(want["steps"])
    for t, (a, b) in enumerate(zip(steps, want["steps"]), start=1):
        assert a["data"] == b["data"], t
        assert a["train_idx"] == b["train_idx"] and a["test_idx"] == b["test_idx"], t
    genie, genie_data = _geniex_run(MultiModelAccState(5, 2, 0.1), cp)
    assert genie == want["geniex"]
    assert genie_data == want["geniex_data"]


def _ensemble_inputs_kue():
    torch.manual_seed(0)
    C_, M_, classes, feat = 3, 3, 3, 6
    models = [nn.Linear(feat, classes) for _ in range(M_)]
    masks = [(torch.rand(feat) > 0.3).float().numpy() for _ in range(M_)]
    data = {m: {c: [(torch.randn(10, feat), torch.randint(0, classes, (10,))) for _ in range(2)] for c in range(C_)}
            for m in range(M_)}
    return C_, M_, classes, models, masks, data


def test_kue_kappa_weights_match_reference_aggregator_code():
    """KUE ensemble weights: the reference's ``FedAvgEnsAggregatorKue.update_ens_weights`` (masked confusion matrices →
    Cohen's κ per model, worst-model index) executed on a stand-in ``self`` vs ops.confusion_matrix + cohen_kappa."""
    from feddrift_b200 import ops
    from feddrift_b200.ops import reference as oref
    C_, M_, classes, models, masks, data = _ensemble_inputs_kue()
    want = _gold("kue")
    mine = []
    for m in range(M_):
        A = torch.zeros(classes, classes, dtype=torch.float64)
        for c in range(C_):
            for x, y in data[m][c]:
                with torch.no_grad():
                    pred = models[m](x * torch.from_numpy(masks[m])).argmax(-1)
                A += ops.confusion_matrix(pred, y, classes).double()
        mine.append(oref.cohen_kappa(A))
    assert np.allclose(mine, want["ens_weights"], atol=1e-12)
    assert int(np.argmin(mine)) == want["worst"]


def _ref_kue():
    from types import SimpleNamespace
    from fedml_api.distributed.fedavg_ens.FedAvgEnsAggregatorKue import FedAvgEnsAggregatorKue as RefKue
    C_, M_, classes, models, masks, data = _ensemble_inputs_kue()
    state = SimpleNamespace(get_masks=lambda: masks, worst=None)
    state.set_worst_idx = lambda i: setattr(state, "worst", int(i))
    fake = SimpleNamespace(models=models, class_num=classes, device=torch.device("cpu"), kue_state=state,
                           train_data_local_dicts=data, ens_weights=np.ones(M_),
                           args=SimpleNamespace(client_num_in_total=C_, curr_train_iteration=1))
    fake._confusion_matrix = lambda model, d, mask: RefKue._confusion_matrix(fake, model, d, mask)
    RefKue.update_ens_weights(fake)
    return {"ens_weights": fake.ens_weights, "worst": state.worst}


def _ensemble_inputs_aue():
    torch.manual_seed(1)
    C_, K_, classes, feat = 4, 4, 3, 5
    models = [nn.Linear(feat, classes) for _ in range(K_)]
    newest = {c: [(torch.randn(12, feat), torch.randint(0, classes, (12,))) for _ in range(2)] for c in range(C_)}
    return C_, K_, classes, models, newest


def test_aue_model_scores_match_reference_aggregator_code():
    """AUE weights 1/(MSE_r + MSE_i + ε): the reference's ``update_ens_weights`` run on a stand-in ``self``.  The reference
    stores the score of model k+1 at index k (``enumerate(self.models[1:])``, DESIGN §8) — we compare score by score."""
    from feddrift_b200 import ops
    C_, K_, classes, models, newest = _ensemble_inputs_aue()
    mser = (1 - 1.0 / classes) ** 2
    ours = np.zeros(K_)
    ours[0] = 1.0 / (mser + 1e-20)
    n = sum(y.shape[0] for c in range(C_) for _, y in newest[c])
    for k in range(1, K_):
        with torch.no_grad():
            sq = sum(float(ops.aue_sqerr(models[k](x), y)) for c in range(C_) for x, y in newest[c])
        ours[k] = 1.0 / (mser + sq / n + 1e-20)
    ref_w = np.asarray(_gold("aue"))
    ref_w = ref_w / ref_w[0]                                # undo the normalisation: index 0 is the "perfect" score
    for k in range(2, K_):                                  # reference index k-1 holds model k's score
        assert abs(ref_w[k - 1] - ours[k] / ours[0]) < 1e-6, k


def _ref_aue():
    from types import SimpleNamespace
    from fedml_api.distributed.fedavg_ens.FedAvgEnsAggregatorAue import FedAvgEnsAggregatorAue as RefAue
    C_, K_, classes, models, newest = _ensemble_inputs_aue()
    fake = SimpleNamespace(models=models, class_num=classes, device=torch.device("cpu"), ens_weights=np.ones(K_),
                           train_data_local_dicts={0: newest}, args=SimpleNamespace(client_num_in_total=C_))
    fake._mse = lambda model, d: RefAue._mse(fake, model, d)
    RefAue.update_ens_weights(fake)
    return fake.ens_weights


def _cfl_scenario():
    from feddrift_b200.parallel.arena import ModelBank
    C_, M_ = 6, 4
    torch.manual_seed(3)
    bank = ModelBank(_LR(), M_, "cpu")
    g = torch.Generator().manual_seed(9)
    direction = torch.randn(bank.P, generator=g)

    def round_updates(kind):
        """kind 'warm': everybody moves the same way (large mean norm → sets ε); 'split': two opposed groups."""
        ups = []
        for c in range(C_):
            if kind == "warm":
                ups.append(direction * 1.0 + 0.01 * torch.randn(bank.P, generator=g))
            else:
                sign = 1.0 if c < 3 else -1.0
                ups.append(sign * direction * 0.9 + 0.01 * torch.randn(bank.P, generator=g))
        return ups
    return C_, M_, bank, round_updates


CFL_ROUNDS = ["warm", "split", "warm", "split"]


@pytest.mark.parametrize("retrain", CFL_RETRAIN)
def test_cfl_split_logic_matches_reference_implementation(retrain):
    """Clustered FL: adaptive ε₁/ε₂ from the observed update norms, cosine-similarity bipartition (complete linkage),
    γ test, capped slot allocation, weight rewrite — the reference's ``cluster_cfl`` vs ours on the same client updates."""
    from feddrift_b200.drift.softcluster import SoftClusterState
    C_, M_, bank, round_updates = _cfl_scenario()
    gold = _gold("cfl")[retrain]
    mine = SoftClusterState(C_, M_, cluster_alg="cfl", cfl_gamma=0.1, cfl_retrain=retrain)
    mine.cluster_init()
    mine.cluster_cfl_init(1)
    split_seen = False
    for rnd, kind in enumerate(CFL_ROUNDS):
        ups = round_updates(kind)
        client_params = torch.zeros(C_, M_, bank.P)
        n = torch.zeros(C_, M_)
        for c in range(C_):
            for m in range(M_):
                if mine.W[1][m][c] > 0:
                    client_params[c, m], n[c, m] = bank.theta[m] + ups[c], 10
        a = mine.cluster_cfl(1, rnd, bank, client_params, n)
        want = gold[rnd]
        assert a == want["split"], (rnd, kind)
        split_seen = split_seen or a
        for tt in (0, 1):
            assert np.array_equal(mine.W[tt], np.asarray(want["W"][tt])), (rnd, tt)
        assert abs(mine.cfl_norm - want["norm"]) < 1e-5 and abs(mine.cfl_eps2 - want["eps2"]) < 1e-5
        for m in range(M_):
            assert torch.allclose(bank.theta[m], torch.tensor(want["theta"][m]), atol=1e-6)
    assert split_seen


def _ref_cfl(ref_mod, retrain):
    import sklearn.cluster as skc
    from feddrift_b200.models import utils as mutils

    def agglo(affinity=None, linkage="ward", **kw):   # sklearn renamed `affinity` → `metric` (same shim as the reference arm)
        return skc.AgglomerativeClustering(metric=affinity or "euclidean", linkage=linkage, **kw)
    ref_mod.AgglomerativeClustering = agglo
    C_, M_, bank, round_updates = _cfl_scenario()
    init_sd = {k: v.clone() for k, v in bank.state_dict(0).items()}
    models = [_LR() for _ in range(M_)]
    for mod in models:
        mod.load_state_dict(init_sd)
    ref_mod.reinitialize = lambda model: model.load_state_dict(init_sd)
    theirs = ref_mod.SoftClusterState(C_, M_, cluster_alg="cfl", cfl_gamma=0.1, cfl_retrain=retrain)
    theirs.cluster_init()
    theirs.cluster_cfl_init(1)
    out = []
    for rnd, kind in enumerate(CFL_ROUNDS):
        ups = round_updates(kind)
        weights_dict = {}
        for c in range(C_):
            weights_dict[c] = {}
            for m in range(M_):
                if theirs.train_data_weights[1][m][c] > 0:
                    row = mutils.flatten_state_dict(models[m].state_dict()) + ups[c]
                    weights_dict[c][m] = (mutils.unflatten_to_state_dict(row.clone(), bank.spec), 10)
                else:
                    weights_dict[c][m] = (None, 0)
        b = theirs.cluster_cfl(1, rnd, models, weights_dict)
        out.append(_canon({"split": bool(b), "W": [theirs.train_data_weights[tt] for tt in (0, 1)], "norm": float(theirs.cfl_norm),
                           "eps2": float(theirs.cfl_eps2), "theta": [mutils.flatten_state_dict(md.state_dict()) for md in models]}))
    return out


class _SD(dict):   # the reference calls both `.items()` and `.state_dict()` on the local model argument
    def state_dict(self):
        return self


def _robust_inputs():
    from types import SimpleNamespace
    # the reference's vectorize_weight concatenates the tensors un-flattened (torch.cat fails on mixed ranks), so the
    # comparison uses 1-D parameters; ours flattens and therefore also handles real conv / linear state_dicts
    torch.manual_seed(0)
    glob = {"l1.weight": torch.randn(12), "l1.bias": torch.randn(4), "bn.running_mean": torch.randn(4),
            "bn.num_batches_tracked": torch.tensor([3.0]), "l2.weight": torch.randn(7)}
    local = _SD({k: v + 0.7 * torch.randn_like(v) for k, v in glob.items()})
    return SimpleNamespace(defense_type="norm_diff_clipping", norm_bound=0.5, stddev=0.01), glob, local


def test_robust_aggregator_clipping_matches_reference_implementation():
    from feddrift_b200.core.robustness import RobustAggregator
    args, glob, local = _robust_inputs()
    ours, theirs = RobustAggregator(args).norm_diff_clipping(local, glob), _gold("robust")
    assert list(ours.keys()) == theirs["keys"]
    for k in ours:
        assert torch.allclose(ours[k].float(), torch.tensor(theirs["values"][k]).float(), atol=1e-6), k
    diff = torch.cat([(ours[k] - glob[k]).reshape(-1) for k in ours if "running" not in k and "num_batches" not in k])
    assert abs(diff.norm().item() - 0.5) < 1e-4


def _ref_robust():
    from fedml_core.robustness.robust_aggregation import RobustAggregator as RefRA
    args, glob, local = _robust_inputs()
    theirs = RefRA(args).norm_diff_clipping(local, glob)
    return {"keys": list(theirs.keys()), "values": dict(theirs)}


def _load_reference(ref_root):
    """Import the unmodified reference from a FedDrift checkout under the library-compatibility shims of the reference arm."""
    os.environ.setdefault("WANDB_MODE", "disabled")
    os.environ.setdefault("WANDB_SILENT", "true")
    for p in (os.path.join(ROOT, "baseline", "shims"), ref_root):
        if p not in sys.path:
            sys.path.insert(0, p)
    import wandb
    if wandb.run is None:
        wandb.init(mode="disabled")
    from fedml_api.distributed.fedavg_ens import FedAvgEnsDataLoader as ref_mod
    return ref_mod


def record(ref_root):
    """Run the reference's side of every scenario and store its observations (and its change-point files) as golden data."""
    import tempfile
    import networkx as nx
    ref_mod = _load_reference(ref_root)
    if not hasattr(nx, "to_numpy_matrix"):
        nx.to_numpy_matrix = nx.to_numpy_array          # removed in networkx 3 (same shim as the reference arm)
    from fedml_api.distributed.turboaggregate import mpc_function as ref_mpc
    from fedml_core.distributed.communication.message import Message as RefMessage
    from fedml_core.distributed.topology.symmetric_topology_manager import SymmetricTopologyManager as RefTopo
    gold = {"hierarchical": {f"{v}/{s}": _ref_hierarchical(ref_mod, s, v) for v in HIER_VARIANTS for s in HIER_SEEDS},
            "matrix": {a: _matrix_run(ref_mod.SoftClusterState(6, 4, **_matrix_kw(a)), "train_data_weights") for a in MATRIX_ALGS},
            "ada": _ada_run(ref_mod.AdaState(init_lr=0.05), as_numpy=True),
            "driftsurf": {str(s): _driftsurf_run(ref_mod.DriftSurfState(delta=0.1, r=3, wl=4), s, "cpu") for s in DRIFTSURF_SEEDS},
            "mpc": _mpc_run(ref_mpc), "topology": _topology_run(RefTopo), "message_json": _message_json(RefMessage),
            "mmacc": {}, "kue": _ref_kue(), "aue": _ref_aue(),
            "cfl": {r: _ref_cfl(ref_mod, r) for r in CFL_RETRAIN}, "robust": _ref_robust()}
    for s in MMACC_SEEDS:
        steps, cp = _mmacc_run(ref_mod.MultiModelAccState(5, 3, 0.1), s, reference=True)
        genie, genie_data = _geniex_run(ref_mod.MultiModelAccState(5, 2, 0.1), cp)
        gold["mmacc"][str(s)] = {"steps": steps, "geniex": genie, "geniex_data": genie_data}
    with tempfile.TemporaryDirectory() as tmp:
        gold["retrain"] = _ref_retrain(tmp)
    os.makedirs(GOLDEN_CP_DIR, exist_ok=True)
    cp_src = os.path.join(ref_root, "data", "changepoints")
    for f in sorted(os.listdir(cp_src)):
        if f.endswith(".cp"):
            shutil.copyfile(os.path.join(cp_src, f), os.path.join(GOLDEN_CP_DIR, f))
    def entry(v):   # one line per scenario keeps the file diffable
        if isinstance(v, dict) and any(isinstance(x, (dict, list)) for x in v.values()):
            return "{\n" + ",\n".join(f"  {json.dumps(k)}: {json.dumps(x)}" for k, x in v.items()) + "\n }"
        return json.dumps(v)
    with open(GOLDEN, "w") as fh:
        fh.write("{\n" + ",\n".join(f" {json.dumps(k)}: {entry(_canon(v))}" for k, v in gold.items()) + "\n}\n")
    print("wrote", GOLDEN)


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reference", required=True, help="root of a microsoft/FedDrift checkout (holds fedml_api/ and data/)")
    record(os.path.abspath(ap.parse_args().reference))
