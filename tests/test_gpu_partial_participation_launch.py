"""GPU: the fused round kernel with a participants table for a large federation with few sampled clients (small cluster,
full-size evaluation), and IFCA re-clustering under sampling checked model by model against the CPU oracle."""
import copy

import pytest
import torch

from feddrift_b200 import ops
from feddrift_b200.ops import reference as ref
from feddrift_b200.sim.engine import client_sampling
from test_gpu_small_round import make_state, to_cuda

pytestmark = pytest.mark.gpu


def _table(C, K, rows=2):
    return torch.tensor([client_sampling(r, C, K) for r in range(rows)], dtype=torch.int32)


def _assert_models_match(st_gpu, st_cpu):
    assert torch.allclose(st_gpu["theta"].cpu(), st_cpu["theta"], rtol=2e-4, atol=2e-5), \
        (st_gpu["theta"].cpu() - st_cpu["theta"]).abs().max()
    assert torch.equal(st_gpu["opt_step"].cpu(), st_cpu["opt_step"])


@pytest.mark.parametrize("C,K,B", [(1000, 10, 32), (1000, 2, 500)])
def test_large_federation_few_sampled_clients_matches_reference(C, K, B):
    st_cpu = make_state(C=C, M=4, B=B, epochs=2)
    st_cpu["participants"] = _table(C, K)
    st_gpu = to_cuda(copy.deepcopy(st_cpu))
    out_ref = ref.fed_round_small(st_cpu, 1)
    out_gpu = ops.fed_round_small(st_gpu, 1)
    torch.cuda.synchronize()
    assert st_gpu["_launch_info"][2] <= 227 * 1024
    _assert_models_match(st_gpu, st_cpu)
    assert torch.allclose(st_gpu["opt_m"].cpu(), st_cpu["opt_m"], rtol=1e-3, atol=1e-6)
    mg, mr = out_gpu["metrics"].cpu(), out_ref["metrics"]
    assert (mg[..., 0] - mr[..., 0]).abs().max() <= 1.0
    assert torch.allclose(mg[..., 1], mr[..., 1], rtol=1e-3, atol=1e-2)


def test_ifca_recluster_under_sampling_models_match_reference():
    """Round 1 aggregates before it re-clusters, so its models must match the oracle; round 2 then starts both sides from
    the oracle's assignment and must match again (the per-round pair list is rebuilt from the rewritten W and the table)."""
    st_cpu = make_state(M=3)
    st_cpu["recluster_hard"] = True
    st_cpu["participants"] = _table(10, 4)
    st_gpu = to_cuda(copy.deepcopy(st_cpu))
    t = st_cpu["t_cur"]
    for _ in range(2):
        ref.fed_round_small(st_cpu, 1)
        ops.fed_round_small(st_gpu, 1)
        torch.cuda.synchronize()
        _assert_models_match(st_gpu, st_cpu)
        Wg = st_gpu["W"][t].cpu()
        assert torch.all(Wg.sum(0) == 1)
        assert (Wg.argmax(0) == st_cpu["W"][t].argmax(0)).float().mean() >= 0.8
        st_gpu["W"].copy_(st_cpu["W"])        # same assignment on both sides for the next round
    assert st_cpu["round0"] == st_gpu["round0"] == 2
