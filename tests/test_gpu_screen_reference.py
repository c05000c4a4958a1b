"""-m gpu: every instantiation of the float16 tensor-core screen (nn_screen_kernel<TOPK, ARES, SYM>, csrc/nn_screen_tc.cu)
against the float64 reference of oracle/screen_oracle.py, bit for bit - indices and float32 distance bits - on every row
the reference does not flag as ambiguous, and the tests bound how many it flags.

Which kernel a case runs is decided by the input alone:
  ARES   d_pad <= 512 keeps the A rows resident in shared memory; wider rows stream A and B
  SYM    slic_nn_top1 with q is x (same pointers), nq == n, self_offset == 0 and n >= 16384
  rect   any other slic_nn_top1 call: a different query set, or a row slice with self_offset = r0
  TOPK   slic_topk_cosine_tc
The tests call slic_nn_top1 / slic_topk_cosine_tc directly, so the backend's routing of small inputs to the exact
kernels (n < 2048) does not apply.

  case                                        kernel <TOPK, ARES, SYM>        dtypes
  test_rect_top1_sign_rows  d <= 512          <0, 1, 0>                       f32, f64
  test_rect_top1_sign_rows  d >= 513          <0, 0, 0>                       f32, f64
  test_rect_top1_gaussian   d = 96 / >= 1000  <0, 1, 0> / <0, 0, 0>           f32, f64
  test_rect_top1_negative_best                <0, 1, 0>, <0, 0, 0>            f32
  test_ladders                                <0, 1, 0>, <0, 0, 0>            f32
  test_sym_top1_sign_rows   d <= 512          <0, 1, 1>                       f32, f64
  test_sym_top1_sign_rows   d >= 513          <0, 0, 1>                       f32, f64
  test_sym_top1_cone_outlier                  <0, 1, 1>                       f32
  test_sym_top1_gaussian                      <0, 1, 1>                       f32
  test_sym_log_overflow                       <0, 1, 1> then <0, 1, 0>        f32
  test_sym_parts_and_two_phase                <0, 1, 1>                       f32
  test_topk_sign_rows       d <= 512          <1, 1, 0>                       f32, f64
  test_topk_sign_rows       d >= 513          <1, 0, 0>                       f32, f64
  test_topk_gaussian                          <1, 1, 0>, <1, 0, 0>            f32, f64
  test_raw_scores                             <0, 0, 0> (d_pad >= 576)        f16 operands
  test_default_eps_plumbing                   <0, 1, 0>, <1, 0, 0>            f32
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import screen_oracle as so

pytestmark = pytest.mark.gpu

TIE_MARGIN_F64 = 1e-12     # test_gpu_kernels.py: float64 rows whose best two distances are closer are ties


@pytest.fixture(scope="module")
def be():
    from video_similarity_search_b200.backend import CudaBackend
    return CudaBackend()


def _lib():
    from video_similarity_search_b200 import _lib as lib
    return lib


def d_pad_of(d):
    return (d + 63) // 64 * 64


def upload(be, a):
    """Unit rows exactly as given (no normalisation) and their float16 copy, zero padded to d_pad."""
    u = torch.from_numpy(np.ascontiguousarray(a)).to(be.device)
    n, d = u.shape
    f = torch.zeros((n, d_pad_of(d)), dtype=torch.float16, device=be.device)
    f[:, :d] = u.to(torch.float16)
    return u, f


def normalized(be, a):
    """slic_normalize_rows of exact-arithmetic rows: the unit rows and their float16 copy must be the rows themselves."""
    u, f = be.normalize_rows(be.to_device(a))
    assert torch.equal(u.cpu(), torch.from_numpy(a))
    assert torch.equal(f[:, :a.shape[1]].to(u.dtype).cpu(), torch.from_numpy(a))
    return u, f


def top1(be, q, qb, x, xb, off, eps=0.0):
    idx, dist = be.nn_top1(q, qb, x, xb, self_offset=off, eps=eps)
    return idx.cpu().numpy(), dist.cpu().numpy(), be.last_stats.cpu().numpy()


def topk(be, q, qb, x, xb, k, off, eps=0.0):
    nq, d = q.shape
    idx = torch.empty((nq, k), dtype=torch.int32, device=be.device)
    val = torch.empty((nq, k), dtype=x.dtype, device=be.device)
    stats = torch.zeros(4, dtype=torch.int32, device=be.device)
    dt = 0 if x.dtype == torch.float32 else 1
    _lib().call("slic_topk_cosine_tc", q.data_ptr(), qb.data_ptr(), nq, x.data_ptr(), xb.data_ptr(), x.shape[0], d,
                xb.shape[1], dt, k, off, float(eps), idx.data_ptr(), val.data_ptr(), stats.data_ptr(), be._stream())
    return idx.cpu().numpy(), val.cpu().numpy(), stats.cpu().numpy()


def assert_matches(idx, dist, ref, max_amb, exact_dist=True):
    """Device result against the reference on every unambiguous row: indices equal, distances bit for bit (float32, or
    float64 on exact-arithmetic inputs) or to 1e-14 (float64 otherwise)."""
    ri, rv, amb = ref
    assert int(amb.sum()) <= max_amb, "ambiguous rows: %d" % int(amb.sum())
    ok = ~amb
    idx, dist = idx.reshape(ri.shape), dist.reshape(rv.shape)
    bad = np.flatnonzero((idx != ri).reshape(len(ok), -1).any(1) & ok)
    assert bad.size == 0, ("rows differ", bad[:8].tolist(), idx[bad[:8]].tolist(), ri[bad[:8]].tolist())
    if exact_dist:
        assert np.array_equal(dist[ok].view(np.uint8), rv[ok].view(np.uint8))
    else:
        np.testing.assert_allclose(dist[ok], rv[ok], rtol=0, atol=1e-14)


def f64_delta(d):
    return max(so.sum_delta(d), TIE_MARGIN_F64 / 2)


def max_amb(n):
    return max(1, n // 10000)


def ran_symmetric(be):
    """True if the last profiled screen launch computed only about half of the square (the symmetric kernel)."""
    lib = be.lib
    fl, ex, ms = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_float(0)
    assert lib.slic_last_screen_time(ctypes.byref(ms), ctypes.byref(fl)) == 0
    assert lib.slic_last_screen_exec_flop(ctypes.byref(ex)) == 0
    return ex.value < 0.8 * fl.value


def sign_database(n, d, m, seed, dtype=np.float32, zero=True):
    """Sign rows with duplicate groups across the 256-row boundaries and a few zero rows."""
    rng = np.random.default_rng(seed)
    zeros = (3, n // 2 + 1) if zero and n > 8 else ()
    x = so.sign_rows(n, d, m, rng, dtype, zero_rows=zeros)
    so.plant_duplicates(x, so.boundary_groups(n))
    for j, i in (so.left_pairs(n, 24, rng) if n > 512 else ()):
        x[i] = x[j]
    return x


# ---------------------------------------------------------------------------------------------------------------------
# rectangular top-1
# ---------------------------------------------------------------------------------------------------------------------
RECT = [  # d, m, nq, n, self_offset (-1: a separate query set)
    (1, 1, 1, 2, -1), (3, 1, 127, 255, -1), (64, 64, 128, 257, -1), (65, 64, 129, 4096, 300),
    (512, 256, 255, 16383, 1001), (512, 64, 257, 16385, 0),
    (513, 256, 257, 2048, 77), (1000, 256, 129, 16384 + 255, -1), (2048, 1024, 128, 4097, 3333),
    (4096, 4096, 127, 2049, -1), (6000, 64, 200, 3000, 1500),
]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("d,m,nq,n,off", RECT)
def test_rect_top1_sign_rows(be, dtype, d, m, nq, n, off):
    x = sign_database(n, d, m, d + n, dtype)
    ux, xb = normalized(be, x)
    if off >= 0:
        uq, qb = ux[off:off + nq], xb[off:off + nq]
    else:
        rng = np.random.default_rng(n)
        q = so.sign_rows(nq, d, m, rng, dtype)
        q[: nq // 3] = x[rng.integers(0, n, nq // 3)]          # queries equal to database rows: exact ties
        uq, qb = normalized(be, q)
    idx, dist, stats = top1(be, uq, qb, ux, xb, off)
    # exact arithmetic: the float64 reference needs no perturbation; in float32 nothing is ambiguous at the default one
    # either (a perturbed float64 distance separates exact ties, so float64 is compared with delta = 0 alone)
    assert_matches(idx, dist, so.reference_top1(uq, ux, off, delta=0), 0)
    if dtype == np.float32:
        assert not so.reference_top1(uq, ux, off)[2].any()
    assert stats[0] >= nq - stats[1]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("d,n,r0,nq,seed", [(96, 3000, 129, 2500, 96), (1000, 4000, 0, 3999, 1000),
                                             (6000, 2500, 1, 2499, 6002)])
def test_rect_top1_gaussian(be, dtype, d, n, r0, nq, seed):
    """Planted near pairs (Delta 1e-7 .. 1e-4, many ordered wrongly by the float16 product) and pairs whose float32
    distances are equal although their float64 s differ (the lower index must win: np.argmin on float32 distances)."""
    x, info = so.gaussian_planted(n, d, np.random.default_rng(seed), near_pairs=64, round_ties=24)
    assert so.f16_order_reversals(x, info["near"]) >= 8
    ux, xb = upload(be, x.astype(dtype))
    idx, dist, stats = top1(be, ux[r0:r0 + nq], xb[r0:r0 + nq], ux, xb, r0)
    if dtype == np.float32:
        ref = so.reference_top1(ux[r0:r0 + nq], ux, r0)
        assert_matches(idx, dist, ref, max_amb(n))
        ties = [(q, a) for q, a, b in info["round_ties"] if r0 <= q < r0 + nq and not ref[2][q - r0]]
        assert len(ties) >= 16
        assert all(idx[q - r0] == a for q, a in ties)
    else:
        assert_matches(idx, dist, so.reference_top1(ux[r0:r0 + nq], ux, r0, delta=f64_delta(d)), max_amb(n),
                       exact_dist=False)
    assert stats[1] <= nq // 100


@pytest.mark.parametrize("d,m,c", [(512, 64, 48), (1000, 64, 48)])
def test_rect_top1_negative_best(be, d, m, c):
    """A query set in the cone opposite the database: every row's best score is negative (enc_score / dec_score of
    negative floats, distances above 1)."""
    rng = np.random.default_rng(d)
    x = so.cone_rows(5000, d, m, c, rng, 1.0)
    q = so.cone_rows(300, d, m, c, rng, -1.0)
    ux, xb = normalized(be, x)
    uq, qb = normalized(be, q)
    idx, dist, stats = top1(be, uq, qb, ux, xb, -1)
    ref = so.reference_top1(uq, ux, -1)
    assert np.all(ref[1] > 1)
    assert_matches(idx, dist, ref, 0)


def test_ladders(be):
    """Columns of rising score in column order.  A step of about eps / 6 (2^-11, exact sign rows at m = 4096, streaming
    kernel) or 2^-7 (m = 256, A-resident kernel) keeps the candidate list alive by compaction: stats[2] > 0 and no row
    needs the exact finisher.  A step of eps / 64 (float rows) puts 64 columns inside eps: the list overflows and the
    exact finisher settles the row."""
    for d, m, steps, n in ((4096, 4096, 1200, 16384), (512, 256, 250, 2048)):
        rng = np.random.default_rng(m)
        q, cols, _ = so.ladder(d, m, steps)
        x = so.sign_rows(n, d, m, rng)
        pos = np.sort(rng.choice(n, steps, replace=False))
        x[pos] = cols
        qs = np.tile(q, (4, 1))
        ux, xb = normalized(be, x)
        uq, qb = normalized(be, qs)
        idx, dist, stats = top1(be, uq, qb, ux, xb, -1)
        assert_matches(idx, dist, so.reference_top1(uq, ux, -1, delta=0), 0)
        assert idx[0] == pos[-1]
        assert stats[2] >= 4 and stats[1] == 0, stats
    rng = np.random.default_rng(7)
    d, n = 256, 2048
    x = so._unit64(rng.standard_normal((n, d)))
    q = x[0].copy()
    pos = np.sort(rng.choice(np.arange(1, n), 200, replace=False))
    x[pos] = so.fine_ladder(q, 200, float(so.default_eps(256)) / 64, 0.6, rng)
    ux, xb = upload(be, x.astype(np.float32))
    idx, dist, stats = top1(be, ux[:64], xb[:64], ux, xb, 0)
    assert_matches(idx, dist, so.reference_top1(ux[:64], ux, 0), 1)
    assert stats[1] >= 1


# ---------------------------------------------------------------------------------------------------------------------
# symmetric self-search
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,d,m,n", [
    (np.float32, 64, 64, 16384), (np.float32, 512, 256, 16384 + 255), (np.float64, 512, 64, 16385),
    (np.float32, 1000, 256, 16385), (np.float64, 513, 256, 16384 + 255), (np.float32, 4096, 1024, 16384),
])
def test_sym_top1_sign_rows(be, dtype, d, m, n):
    """Duplicate groups across tile boundaries and on diagonal tiles, pairs whose only copy lies to the LEFT (found only
    through the column role of an upper-triangle tile), zero rows."""
    x = sign_database(n, d, m, n + d, dtype, zero=False)   # (a zero row logs every column: kept to the other tests)
    ux, xb = normalized(be, x)
    be.lib.slic_profile_screen(1)
    try:
        idx, dist, stats = top1(be, ux, xb, ux, xb, 0)
        assert ran_symmetric(be)
    finally:
        be.lib.slic_profile_screen(0)
    assert_matches(idx, dist, so.reference_top1(ux, ux, 0, delta=0), 0)
    assert stats[1] < n // 20


def test_sym_top1_cone_outlier(be):
    """A self-search in a cone plus one row antipodal to a member: that row's best score is negative."""
    rng = np.random.default_rng(11)
    n = 16384 + 100
    x = so.cone_rows(n, 512, 256, 128, rng, 1.0)
    x[9000] = -x[123]
    ux, xb = normalized(be, x)
    idx, dist, stats = top1(be, ux, xb, ux, xb, 0)
    ref = so.reference_top1(ux, ux, 0)
    assert ref[1][9000] > 1
    assert_matches(idx, dist, ref, 0)


def test_sym_top1_gaussian(be):
    x, info = so.gaussian_planted(16384 + 255, 96, np.random.default_rng(12), near_pairs=128, round_ties=24)
    ux, xb = upload(be, x)
    idx, dist, stats = top1(be, ux, xb, ux, xb, 0)
    ref = so.reference_top1(ux, ux, 0)
    assert_matches(idx, dist, ref, max_amb(len(x)))
    assert all(idx[q] == a for q, a, b in info["round_ties"] if not ref[2][q])


@pytest.mark.parametrize("kind", ["f16_equal", "sign_d1"])
def test_sym_log_overflow(be, kind):
    """Every pair within eps of every row's best: the symmetric screen's candidate log overflows.  The parts API must
    say so (keys[n] == 0); slic_nn_top1 falls back to the full square, whose lists overflow too, and the exact finisher
    must settle every row."""
    n = 16385
    rng = np.random.default_rng(13)
    if kind == "f16_equal":
        x = so.f16_equal_rows(n, 64, rng)
        ux, xb = upload(be, x)
    else:
        x = so.sign_rows(n, 1, 1, rng, zero_rows=(0, 5000))
        ux, xb = normalized(be, x)
    d = x.shape[1]
    keys = torch.empty(n + 1, dtype=torch.int64, device=be.device)
    st = torch.zeros(4, dtype=torch.int32, device=be.device)
    _lib().call("slic_nn_top1_sym_part", ux.data_ptr(), xb.data_ptr(), n, d, xb.shape[1], 0, 1, None, 0.0,
                keys.data_ptr(), st.data_ptr(), be._stream())
    assert int(keys[n]) == 0
    idx, dist, stats = top1(be, ux, xb, ux, xb, 0)
    ref = so.reference_top1(ux, ux, 0)
    assert_matches(idx, dist, ref, 0 if kind == "sign_d1" else 1)
    assert stats[1] > n // 2


def test_sym_parts_and_two_phase(be):
    """slic_nn_top1_sym_part: the element-wise MIN of the parts' keys must be the reference's (distance bits, index)
    key of every row, single-phase and two-phase (row bests merged by MAX first); every part is complete."""
    n, d, parts = 16384 + 255, 64, 3
    x = sign_database(n, d, 64, 14, zero=False)
    bounds = [n * p // parts for p in range(1, parts)]
    for b in bounds:                        # duplicates on both sides of the parts' row boundaries
        x[b + 3] = x[b - 700]
        x[b - 2] = x[min(n - 1, b + 900)]
    ux, xb = normalized(be, x)
    ri, rv, amb = so.reference_top1(ux, ux, 0, delta=0)
    assert not amb.any()
    want = (rv.view(np.uint32).astype(np.int64) << 32) | ri
    bests = None
    for p in range(parts):
        b = torch.empty(n, dtype=torch.int32, device=be.device)
        _lib().call("slic_sym_row_bests", ux.data_ptr(), xb.data_ptr(), n, d, xb.shape[1], p, parts, b.data_ptr(),
                    be._stream())
        bests = b if bests is None else torch.maximum(bests, b)
    for seeded in (None, bests):
        merged = None
        for p in range(parts):
            keys = torch.empty(n + 1, dtype=torch.int64, device=be.device)
            _lib().call("slic_nn_top1_sym_part", ux.data_ptr(), xb.data_ptr(), n, d, xb.shape[1], p, parts,
                        None if seeded is None else seeded.data_ptr(), 0.0, keys.data_ptr(), None, be._stream())
            assert int(keys[n]) == 1
            merged = keys if merged is None else torch.minimum(merged, keys)
        assert np.array_equal(merged[:n].cpu().numpy(), want)


# ---------------------------------------------------------------------------------------------------------------------
# top-k
# ---------------------------------------------------------------------------------------------------------------------
TOPK = [  # d, m, nq, n, k, self_offset
    (64, 64, 65, 65, 64, 0),                  # k = n - 1
    (64, 16, 129, 3000, 63, -1), (512, 64, 257, 4096, 32, 1001), (512, 256, 255, 2048, 1, -1),
    (513, 256, 128, 3000, 2, 0), (1000, 64, 257, 16384 + 255, 64, -1), (4096, 1024, 127, 2049, 32, 100),
    (6000, 64, 129, 2500, 64, 7),
]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("d,m,nq,n,k,off", TOPK)
def test_topk_sign_rows(be, dtype, d, m, nq, n, k, off):
    """Exact ties everywhere, including a group of more than 255 identical rows (saturates the 8-bit score
    histograms): the top k must be the first k columns in (distance, index) order."""
    x = sign_database(n, d, m, n + k, dtype)
    if n > 2000:
        x[1000:1300] = x[1000]
    ux, xb = normalized(be, x)
    if off >= 0:
        uq, qb = ux[off:off + nq], xb[off:off + nq]
    else:
        rng = np.random.default_rng(k)
        q = so.sign_rows(nq, d, m, rng, dtype)
        q[: nq // 2] = x[rng.integers(0, n, nq // 2)]
        if n > 2000:
            q[nq // 2: nq // 2 + 20] = x[1000]
        uq, qb = normalized(be, q)
    idx, dist, stats = topk(be, uq, qb, ux, xb, k, off)
    assert_matches(idx, dist, so.reference_topk(uq, ux, k, off, delta=0), 0)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("d,n,k", [(96, 5000, 50), (1000, 3000, 16)])
def test_topk_gaussian(be, dtype, d, n, k):
    x, info = so.gaussian_planted(n, d, np.random.default_rng(d + k), near_pairs=64, round_ties=8)
    ux, xb = upload(be, x.astype(dtype))
    idx, dist, stats = topk(be, ux, xb, ux, xb, k, 0)
    if dtype == np.float32:
        assert_matches(idx, dist, so.reference_topk(ux, ux, k, 0), max_amb(n))
    else:
        assert_matches(idx, dist, so.reference_topk(ux, ux, k, 0, delta=f64_delta(d)), max_amb(n), exact_dist=False)


# ---------------------------------------------------------------------------------------------------------------------
# raw scores and eps
# ---------------------------------------------------------------------------------------------------------------------
def _subnormal_heavy(n, d, rng):
    """One large component per row, the rest of magnitude 1e-6 .. 6e-5 (float16 subnormals)."""
    x = rng.standard_normal((n, d)) * np.exp(rng.uniform(np.log(1e-6), np.log(6e-5), (n, d)))
    x[np.arange(n), rng.integers(0, d, n)] = 1.0
    return so._unit64(x).astype(np.float32)


@pytest.mark.parametrize("d_pad", [576, 1024, 4096, 6016])
def test_raw_scores(be, d_pad):
    """screen_scores_debug: sign rows equal the float64 product of the float16 operands exactly; Gaussian and
    subnormal-heavy rows stay within the float32 accumulation bound of it and within eps / 2 of the float64 product of
    the float32 unit rows - the premise of the eps derivation, tested directly."""
    nq, n, d = 129, 300, d_pad - 13
    rng = np.random.default_rng(d_pad)
    q = so.sign_rows(nq, d, 256, rng)
    x = so.sign_rows(n, d, 256, rng)
    x[:40] = q[:40]
    _, qb = normalized(be, q)
    _, xb = normalized(be, x)
    got = be.screen_scores_debug(qb, xb).cpu().numpy().astype(np.float64)
    assert np.array_equal(got, so.f16_product(qb.cpu().numpy(), xb.cpu().numpy()))
    half_eps = float(so.default_eps(d_pad)) / 2
    for gen in (lambda k: so._unit64(rng.standard_normal((k, d))).astype(np.float32),
                lambda k: _subnormal_heavy(k, d, rng)):
        q, x = gen(nq), gen(n)
        x[:40] = q[:40]
        uq, qb = be.normalize_rows(be.to_device(q))
        ux, xb = be.normalize_rows(be.to_device(x))
        got = be.screen_scores_debug(qb, xb).cpu().numpy().astype(np.float64)
        f16 = so.f16_product(qb.cpu().numpy(), xb.cpu().numpy())
        acc = d_pad * 2.0 ** -23 * (1 + 2.0 ** -9)
        assert np.abs(got - f16).max() <= acc
        exact = uq.cpu().numpy().astype(np.float64) @ ux.cpu().numpy().astype(np.float64).T
        assert np.abs(got - exact).max() <= half_eps


def test_default_eps_plumbing(be):
    """eps = 4 x the default gives the same answer and re-ranks at least as many candidates; eps <= 0 is the default."""
    x = sign_database(4000, 512, 256, 21)
    ux, xb = normalized(be, x)
    a = top1(be, ux[:1000], xb[:1000], ux, xb, 0, eps=0.0)
    b = top1(be, ux[:1000], xb[:1000], ux, xb, 0, eps=4 * float(so.default_eps(512)))
    c = top1(be, ux[:1000], xb[:1000], ux, xb, 0, eps=float(so.default_eps(512)))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and b[2][0] >= a[2][0]
    assert np.array_equal(a[0], c[0]) and np.array_equal(a[2], c[2])
    x, _ = so.gaussian_planted(3000, 1000, np.random.default_rng(22), near_pairs=32, round_ties=4)
    ux, xb = upload(be, x)
    a = topk(be, ux, xb, ux, xb, 20, 0, eps=0.0)
    b = topk(be, ux, xb, ux, xb, 20, 0, eps=4 * float(so.default_eps(1024)))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and b[2][0] >= a[2][0]
