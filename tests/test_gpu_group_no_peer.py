"""The device-group ctx on a host without peer access.  With ACCMSM_NO_PEER=1 at accmsm_init_multi no two children count as
peers, even contexts of one GPU: every child leaves its partials in its own scratch, copied into child 0's gather buffer
afterwards, and the cyclic key layouts of sharded openings are gathered through a local copy of each shard.  The group
scenarios of test_gpu_multi.py, test_gpu_nark.py, test_gpu_group_open.py and test_gpu_ipa_open_zk.py re-run on such a
group, against the oracle and the single-device ctx."""
import pytest

import accumulation_b200 as ab
from oracle import cref
from tests import test_gpu_group_open as tgo
from tests import test_gpu_ipa_open_zk as tzk
from tests import test_gpu_msm as tm
from tests import test_gpu_multi as tmu
from tests import test_gpu_nark as tn

pytestmark = pytest.mark.gpu

MIN_SHARD = 16


@pytest.fixture(scope="module")
def gctx():
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("ACCMSM_NO_PEER", "1")
        c = ab.Context(devices=[0, 0, 0], min_shard=MIN_SHARD)
    yield c
    c.close()


@pytest.fixture(scope="module")
def gkeys(gctx):
    out = {}
    for curve in (0, 1):
        pts = cref.gen_points(curve, 100 + curve, 1 << 14)
        out[curve] = (pts, gctx.register_bases(curve, pts))
    yield out
    for _, b in out.values():
        b.release()


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("n", [1, 33, 5000, 1 << 14])
def test_no_peer_msm_sizes(gctx, gkeys, curve, n):
    tm.test_msm_sizes_vs_oracle(gctx, gkeys, curve, n)


@pytest.mark.parametrize("curve", [0, 1])
def test_no_peer_commit_hiding_generator_in_any_shard(gctx, gkeys, curve):
    tmu.test_group_commit_hiding_generator_in_any_shard(gctx, gkeys, curve)


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("n,k,precompute", [(300, 10, False), (6000, 8, True)])
def test_no_peer_msm_batch(gctx, curve, n, k, precompute):
    tmu.test_group_msm_batch(gctx, curve, n, k, precompute)


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("k", [4, 14])
def test_no_peer_ipa_decide_tail(gctx, gkeys, curve, k):
    tmu.test_group_ipa_decide_tail(gctx, gkeys, curve, k)


@pytest.mark.parametrize("curve,L,zk", [(0, 1 << 16, True), (1, 3000, True), (0, 1, True)])
def test_no_peer_hp_as_decide(gctx, curve, L, zk):
    tmu.test_group_hp_as_decide(gctx, curve, L, zk)


@pytest.mark.parametrize("curve,n_in,L,zk", [(0, 2, 1 << 16, False), (0, 3, 5000, True), (0, 6, 300, False)])
def test_no_peer_hp_as_product_poly_comm(gctx, curve, n_in, L, zk):
    tmu.test_group_hp_as_product_poly_comm(gctx, curve, n_in, L, zk)


@pytest.mark.parametrize("dense,zk", [(False, True), (True, True)])
def test_no_peer_r1cs_nark_matvec_commit(gctx, dense, zk):
    tmu.test_group_r1cs_nark_matvec_commit(gctx, dense, zk)


@pytest.mark.parametrize("long_key", [False, True])
def test_no_peer_nark_is_bit_identical(ctx, long_key, monkeypatch):
    """the NARK test builds its own group of three contexts; with the long key the last child owns only the hiding generator"""
    monkeypatch.setenv("ACCMSM_NO_PEER", "1")
    tn.test_group_is_bit_identical(ctx, [0, 0, 0], long_key)


@pytest.mark.parametrize("curve", [0, 1])
def test_no_peer_sharded_open(ctx, gctx, curve):
    tgo.test_group_open_parity(ctx, gctx, curve, 10, True, False, True)


@pytest.mark.parametrize("curve", [0, 1])
def test_no_peer_zk_open(ctx, gctx, curve):
    try:
        tzk.test_zk_group_parity(ctx, gctx, curve, 10, None, True)
    finally:
        gctx.set_min_shard(MIN_SHARD)
