"""Launch shape of the fused round kernel for large federations: the cluster size the host picks (from the trained pair
count, which sampling makes small) and the kernel's shared-memory layout must fit 227 KB whenever the federation is routed
to the fused kernel.  Host-side only: the built extension answers without a GPU."""
import pytest
import torch

from feddrift_b200.ops import _ext, small_round
from feddrift_b200.sim.engine import client_sampling
from test_partial_participation import _state

SEA = (small_round.KIND_ID["fnn"], 3, 6, 2)
SMEM_MAX = 227 * 1024


def _ext_or_fail():
    ext = _ext.load()
    assert ext is not None, "the sm_100a extension is not built (run __graft_entry__.build())"
    return ext


@pytest.mark.parametrize("C,K,B", [(1000, 10, 32), (500, 5, 32), (1000, 2, 500), (1000, 1000, 32), (100, 10, 500)])
def test_large_federation_small_sample_fits(C, K, B):
    ext = _ext_or_fail()
    M = 4
    st = _state(C=C, M=M, S=100, B=B)
    if K < C:
        st["participants"] = torch.tensor([client_sampling(r, C, K) for r in range(2)], dtype=torch.int32)
    assert small_round.fits("fnn", 3, 6, 2, C, M, 0)            # routed to the fused kernel
    cache = small_round.prepare(st)
    G, smem = ext.fed_round_small_launch_shape(*SEA, C, M, min(K, C), cache["cluster"], cache["wpp"])
    assert 1 <= G <= 8 and smem <= SMEM_MAX, (G, smem)


def test_small_requested_cluster_grows_until_layout_fits():
    """Few trained pairs ask for a small cluster, but the per-CTA staging scales with ceil(slots·M / G)."""
    ext = _ext_or_fail()
    G, smem = ext.fed_round_small_launch_shape(*SEA, 1000, 4, 1000, 1, 1)
    assert G == 8 and smem <= SMEM_MAX
    G, smem = ext.fed_round_small_launch_shape(*SEA, 1000, 4, 10, 1, 1)   # 10 sampled slots: one CTA is enough
    assert G == 1 and smem <= SMEM_MAX
    G, _ = ext.fed_round_small_launch_shape(*SEA, 10, 4, 10, 2, 4)        # small federations keep the requested cluster
    assert G == 2
