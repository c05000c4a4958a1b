"""CPU checks of oracle/screen_oracle.py: the float64 reference of the tensor-core screen agrees with the FINCH and
retrieval oracles, breaks ties as np.argmin does, flags exactly the rows it should, and every input generator delivers
the property the GPU tests rely on."""
import math

import numpy as np
import pytest

from oracle import finch_oracle as fo
from oracle import retrieval_oracle as ro
from oracle import screen_oracle as so


def test_top1_agrees_with_finch_oracle_float64():
    rng = np.random.default_rng(1)
    x = fo._unit_rows(rng.standard_normal((300, 40)))
    idx, dist, amb = so.reference_top1(x, x, self_offset=0)
    nn, full = fo.first_neighbors_dense(x)
    assert not amb.any()
    assert np.array_equal(idx, nn)
    np.testing.assert_allclose(dist, full[np.arange(300), nn], rtol=0, atol=1e-15)
    # rectangular, float32: the blocked oracle with the same float32 arithmetic
    x32 = fo._unit_rows(rng.standard_normal((500, 24)).astype(np.float32))
    idx, dist, amb = so.reference_top1(x32[100:200], x32, self_offset=100, block=37)
    enn, ed, gap = fo.first_neighbors_blocked(x32, rows=np.arange(100, 200))
    clear = gap > 2e-6
    assert clear.mean() > 0.9 and np.array_equal(idx[clear], enn[clear])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_topk_agrees_with_retrieval_oracle(dtype):
    rng = np.random.default_rng(2)
    q = fo._unit_rows(rng.standard_normal((50, 32))).astype(dtype)
    x = fo._unit_rows(rng.standard_normal((400, 32))).astype(dtype)
    idx, dist, amb = so.reference_topk(q, x, 10)
    dm = ro.distance_matrix(q.astype(np.float64), x.astype(np.float64))
    ref = ro.closest_data_mat(dm, 10)
    assert amb.sum() <= 1
    assert np.array_equal(idx[~amb], ref[~amb])
    np.testing.assert_allclose(dist, np.take_along_axis(dm, idx, 1), rtol=0, atol=1e-6 if dtype == np.float32 else 1e-15)


def test_hand_built_ties():
    """Equal after float32 rounding -> lowest index; self excluded; zero rows (s = 0 everywhere, distance 1)."""
    q = np.zeros((4, 3), dtype=np.float32)
    x = np.zeros((6, 3), dtype=np.float32)
    q[0] = [1, 0, 0]
    x[2] = [1, 0, 0]
    x[4] = [1, 0, 0]                                        # exact tie with 2
    q[1] = [0, 1, 0]
    x[1] = [0, 1, 0]                                        # self column of query 1 (self_offset 0): excluded
    x[5] = [0, np.float32(1 - 2 ** -24), np.float32(2 ** -12)]     # s differs from 1 below float32 resolution near 1
    x[3] = [0, np.float32(math.sqrt(1 - 2 ** -20)), np.float32(2 ** -10)]
    # q[2], q[3] are zero rows
    idx, dist, amb = so.reference_top1(q, x, self_offset=0, delta=0)
    assert idx[0] == 2 and dist[0] == 0
    assert idx[1] == 5 and dist[1] == np.float32(1) - np.float32(np.float64(x[5, 1]))
    assert idx[2] == 0 and dist[2] == 1                     # all distances 1, self (column 2) excluded
    assert idx[3] == 0 and dist[3] == 1
    assert not amb.any()
    # two columns whose float64 s differ but whose float32 distances are equal: the lower index wins
    q = np.array([[1.0, 0.0]], dtype=np.float32)
    x = np.array([[0.0, 1.0], [np.float32(0.75), 0.0], [np.float32(0.75) + np.float32(2 ** -24), 0.0]], dtype=np.float32)
    s = x[:, 0].astype(np.float64)
    assert s[2] > s[1] and np.float32(1) - np.float32(s[2]) != np.float32(1) - np.float32(s[1])
    x[2, 0] = np.float32(0.75)
    x[2, 1] = np.float32(2 ** -13)                         # same s in float32 arithmetic, larger norm
    idx, dist, amb = so.reference_top1(q, x, delta=0)
    assert idx[0] == 1
    # top-k: the tie group is taken in index order, self excluded
    x = np.tile(np.array([[1.0, 0.0]], dtype=np.float32), (8, 1))
    idx, _, amb = so.reference_topk(x[:3], x, 4, self_offset=0, delta=0)
    assert idx.tolist() == [[1, 2, 3, 4], [0, 2, 3, 4], [0, 1, 3, 4]] and not amb.any()


def test_ambiguity_mask_flags_a_midpoint_and_nothing_else():
    """Row 0: two columns at s = c +- delta / 2 - their order can swap under a perturbation of delta.  Row 1: the same
    pair 8 delta apart.  Row 2: s lies exactly on a float32 rounding midpoint - the float32 distance bits can change."""
    import torch
    delta = 2.0 ** -40
    s = torch.tensor([[0.5 - 0.5 * delta, 0.5 + 0.5 * delta, 0.1],
                      [0.5 - 4 * delta, 0.5 + 4 * delta, 0.1],
                      [0.1, 0.75 + 2.0 ** -25, 0.2]], dtype=torch.float64)
    idx, _, amb = so._block_topk(s, torch.float64, 1, torch.arange(3), -1, delta)
    assert idx[:, 0].tolist() == [1, 1, 1] and amb.tolist() == [True, False, False]
    # float32: rows 0 and 1 are exact ties after rounding (lowest index, stable), row 2 is ambiguous
    idx, _, amb = so._block_topk(s, torch.float32, 1, torch.arange(3), -1, delta)
    assert idx[:, 0].tolist() == [0, 0, 1] and amb.tolist() == [False, False, True]
    # top-k: a swap at the k / k+1 boundary and inside the list
    s = np.array([[0.9, 0.5 + 2 ** -45, 0.5, 0.1], [0.9, 0.5 + 2 ** -30, 0.5, 0.1]])
    s = torch.from_numpy(s)
    _, _, amb = so._block_topk(s, torch.float64, 2, torch.arange(2), -1, 2.0 ** -44)
    assert amb.tolist() == [True, False]
    _, _, amb = so._block_topk(s, torch.float64, 3, torch.arange(2), -1, 2.0 ** -44)
    assert amb.tolist() == [True, False]


@pytest.mark.parametrize("m,d", [(1, 1), (1, 3), (64, 64), (64, 65), (256, 513), (256, 1000), (1024, 2048), (4096, 4096), (64, 6000)])
def test_sign_rows_are_exact(m, d):
    rng = np.random.default_rng(m + d)
    x = so.sign_rows(300, d, m, rng, zero_rows=(5, 77))
    assert np.array_equal((x != 0).sum(1), np.where(np.isin(np.arange(300), [5, 77]), 0, m))
    nz = np.ones(300, bool)
    nz[[5, 77]] = False
    assert np.all(np.einsum("ij,ij->i", x[nz].astype(np.float64), x[nz].astype(np.float64)) == 1.0)
    assert np.array_equal(x.astype(np.float16).astype(np.float32), x)           # exact in float16
    assert np.array_equal(fo._unit_rows(x), x)                                    # normalisation leaves them alone
    s = x.astype(np.float64) @ x.astype(np.float64).T
    assert np.array_equal(s * m, np.round(s * m))                                 # integer / m
    assert np.array_equal(x.astype(np.float32) @ x.astype(np.float32).T, s)       # float32 arithmetic is exact too
    _, _, amb = so.reference_top1(x, x, self_offset=0)                            # default delta: nothing ambiguous
    assert not amb.any()


def test_boundary_groups_and_left_pairs_lie_where_claimed():
    n = 16384 + 255
    groups = so.boundary_groups(n)
    assert [g[1] for g in groups] == [1, 2, 31, 32, 33, 100]
    for start, size in groups[1:]:
        assert start // 256 != (start + size - 1) // 256                       # straddles a tile / row-unit boundary
    rng = np.random.default_rng(0)
    x = so.plant_duplicates(so.sign_rows(n, 64, 64, rng), groups)
    for start, size in groups:
        assert (x[start:start + size] == x[start]).all()
    for j, i in so.left_pairs(n, 20, rng):
        assert j < i and i // 256 > j // 256


def test_cone_queries_have_negative_best_scores():
    rng = np.random.default_rng(3)
    x = so.cone_rows(4000, 512, 64, 48, rng, 1.0)
    q = so.cone_rows(300, 512, 64, 48, rng, -1.0)
    assert np.all(np.einsum("ij,ij->i", x.astype(np.float64), x.astype(np.float64)) == 1.0)
    s = q.astype(np.float64) @ x.astype(np.float64).T
    assert s.max() < 0 and np.array_equal(s * 64, np.round(s * 64))
    idx, dist, amb = so.reference_top1(q, x)
    assert not amb.any() and np.all(dist > 1)


def test_ladder_steps():
    q, cols, s = so.ladder(4096, 4096, 1200)
    got = cols.astype(np.float64) @ q.astype(np.float64)
    assert np.array_equal(got, s) and np.all(np.diff(s) == 2.0 ** -11)
    assert 2.0 ** -11 < so.default_eps(4096) / 5 and 2.0 ** -11 > so.default_eps(4096) / 7     # about eps / 6
    rng = np.random.default_rng(4)
    qf = so._unit64(rng.standard_normal(256))
    eps = float(so.default_eps(256))
    fl = so.fine_ladder(qf, 200, eps / 64, 0.6, rng)
    np.testing.assert_allclose(np.linalg.norm(fl, axis=1), 1, atol=1e-15)
    np.testing.assert_allclose(np.diff(fl @ qf), eps / 64, atol=1e-14)


def test_gaussian_planted_pairs():
    rng = np.random.default_rng(5)
    x, info = so.gaussian_planted(3000, 96, rng, near_pairs=64, round_ties=16)
    assert x.dtype == np.float32 and len(info["near"]) == 64 and len(info["round_ties"]) == 16
    np.testing.assert_allclose(np.linalg.norm(x.astype(np.float64), axis=1), 1, atol=1e-6)
    # at least a quarter of the planted near pairs are ordered the wrong way by the float16 product
    assert so.f16_order_reversals(x, info["near"]) >= 16
    x64 = x.astype(np.float64)
    idx, dist, amb = so.reference_top1(x, x, self_offset=0)
    assert amb.sum() <= 1
    for q, a, b in info["round_ties"]:
        sa, sb = x64[q] @ x64[a], x64[q] @ x64[b]
        assert a < b and sa < sb and np.float32(sa) == np.float32(sb)
        assert idx[q] == a                         # lower index, although b is closer in float64
    for q, a, b in info["near"]:
        assert idx[q] in (a, b) or amb[q]


def test_f16_equal_rows():
    rng = np.random.default_rng(6)
    x = so.f16_equal_rows(2000, 64, rng)
    assert len(np.unique(x, axis=0)) == 2000
    x16 = x.astype(np.float16)
    assert np.all(x16[:, 0] == 1)
    sub = np.abs(x16[:, 1:]) < np.float16(2 ** -14)
    assert sub.mean() > 0.9                       # float16's subnormal range
    sc = so.f16_product(x16[:100], x16).astype(np.float32)
    assert np.all(np.abs(sc - 1) <= 2 ** -23)     # every screened score is 1 to float32 accuracy: all within eps


def test_default_eps_matches_the_derivation():
    assert so.default_eps(64) == so.default_eps(4096) == np.float32(2 ** -9 + 2 ** -10 + 2 ** -16)
    prev = so.default_eps(4096)
    for d_pad in (4160, 6016, 8192, 16384, 65536, 1 << 20):
        e = so.default_eps(d_pad)
        assert e > prev and e >= 2 * so.screen_error_bound(d_pad)
        prev = e
    for d_pad in range(64, 4097, 64):
        assert so.default_eps(d_pad) >= 2 * so.screen_error_bound(d_pad)
