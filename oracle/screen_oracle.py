"""Float64 reference of the tensor-core screen's contract, and inputs that stress the screen.  TEST INFRASTRUCTURE ONLY.

slic_nn_top1 and slic_topk_cosine_tc (include/slic_b200.h) promise, for unit query rows q and unit database rows x held
by the device in float32 or float64:
  s[r, j]    = <q_r, x_j>, evaluated in float64
  dist[r, j] = clip(float32(1) - float32(s), 0, 2) in float32 arithmetic (cosine_distance_from_sim<float>), or
               clip(1 - s, 0, 2) in float64
  column r + self_offset is excluded (self_offset >= 0);
  top-1 = smallest dist, ties to the lowest j; top-k = the first k columns in (dist, j) order.
The functions here restate exactly that, starting from the rows the device holds (the caller reads them back), so that
a test can compare bit for bit: indices and float32 distance bits, no tolerances, no tie margins.

The device adds the float64 products in another order than this module does, so a row's float64 s may differ by up to
delta = d * 2^-52.  A row is AMBIGUOUS if its answer could change when every s of the row moves by up to delta; only
ambiguous rows may be left out of a comparison, and the tests bound how many there are.  For inputs on which every
product and partial sum is exact (sign_rows below) delta can be 0 - the device's s is then the same number whatever the
order of the additions.

Small cases are computed with numpy on the host; large ones as a blocked float64 GEMM with torch (cuBLAS) on the
device of the inputs.  Nothing here calls the project's own kernels.
"""
import math

import numpy as np
import torch

TC_CAP = 32            # candidate slots per (split, column half, row) of the top-1 screen (nn_screen_tc.cu)
TILE = 256             # column tile and row unit of the screen
TC_DEFAULT_EPS = 2.0 ** -9 + 2.0 ** -10 + 2.0 ** -16


def default_eps(d_pad):
    """screen_default_eps(d_pad) of nn_screen_tc.cu, as float32."""
    if d_pad <= 4096:
        return np.float32(TC_DEFAULT_EPS)
    return np.float32(2.0 ** -9 + d_pad * (2.0 ** -22 + 2.0 ** -28))


def screen_error_bound(d_pad):
    """Worst case |f16 screen score - float64 score of the unit rows| the eps derivation allows (eps must be >= twice it)."""
    return (2.0 ** -10 + 2.0 ** -22) + 2.0 ** -24 * math.sqrt(d_pad) + d_pad * 2.0 ** -23 * (1 + 2.0 ** -9)


def sum_delta(d):
    """Largest difference between two float64 evaluations of <q, x> for unit rows of width d (any addition order)."""
    return d * 2.0 ** -52


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------
def _as_torch(a):
    return a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))


def _dist(s, dtype):
    """cosine_distance_from_sim<T>: the distance in the reference dtype from float64 similarities."""
    if dtype == torch.float32:
        return torch.clamp(torch.ones((), dtype=torch.float32, device=s.device) - s.to(torch.float32), 0.0, 2.0)
    return torch.clamp(1.0 - s, 0.0, 2.0)


def _block_topk(s, dtype, k, rows, self_offset, delta):
    """Top-k and ambiguity flags of one block of rows.  s: float64 [b, n]; rows: int64 [b] global query rows."""
    b, n = s.shape
    dev = s.device
    cols = torch.arange(n, device=dev)
    dist = _dist(s, dtype)
    lo = _dist(s + delta, dtype)         # the smallest distance a perturbation of s can give
    hi = _dist(s - delta, dtype)         # the largest
    if self_offset >= 0:
        sc = rows + self_offset
        ok = (sc >= 0) & (sc < n)
        r_ok, c_ok = torch.nonzero(ok).flatten(), sc[ok]
        inf = torch.tensor(float("inf"), dtype=dist.dtype, device=dev)
        for t in (dist, lo, hi):
            t[r_ok, c_ok] = inf
    if k == 1:
        m = dist.min(dim=1, keepdim=True).values
        idx = torch.where(dist == m, cols, n).min(dim=1, keepdim=True).values
    else:
        idx = torch.sort(dist, dim=1, stable=True).indices[:, :k]      # (dist, j) order
    val = dist.gather(1, idx)
    lo_s, hi_s = lo.gather(1, idx), hi.gather(1, idx)
    amb = torch.zeros(b, dtype=torch.bool, device=dev)
    if dtype == torch.float32:                                          # the distance bits are part of the answer
        amb |= (lo_s != hi_s).any(dim=1)
    if k > 1:                                                           # order inside the top k
        a, c = hi_s[:, :-1], lo_s[:, 1:]
        amb |= ((c < a) | ((c == a) & (idx[:, 1:] < idx[:, :-1]))).any(dim=1)
    # boundary: a column outside the top k that could enter it
    H = hi_s[:, -1:]
    M = torch.where(hi_s == H, idx, -1).max(dim=1, keepdim=True).values
    outside = torch.ones_like(dist, dtype=torch.bool).scatter_(1, idx, False)
    amb |= (outside & ((lo < H) | ((lo == H) & (cols < M)))).any(dim=1)
    return idx, val, amb


def reference_topk(q, x, k, self_offset=-1, delta=None, block=2048):
    """Top-k of every query row (see the module docstring).  q [nq, d], x [n, d]: the unit rows the device holds
    (float32 or float64, numpy or torch; torch tensors on a CUDA device are searched there with cuBLAS).
    delta: perturbation of s for the ambiguity flags (default sum_delta(d)).
    -> (idx int64 [nq, k], dist [nq, k] in the rows' dtype, ambiguous bool [nq]) as numpy arrays."""
    qt, xt = _as_torch(q), _as_torch(x)
    dtype = xt.dtype
    assert qt.dtype == dtype and dtype in (torch.float32, torch.float64)
    nq, d = qt.shape
    delta = sum_delta(d) if delta is None else float(delta)
    on_dev = xt.is_cuda
    x64 = xt.to(torch.float64)
    xn = None if on_dev else x64.numpy()
    out_i, out_v, out_a = [], [], []
    for r0 in range(0, nq, block):
        r1 = min(nq, r0 + block)
        q64 = qt[r0:r1].to(torch.float64)
        s = q64 @ x64.T if on_dev else torch.from_numpy(q64.numpy() @ xn.T)
        rows = torch.arange(r0, r1, device=s.device)
        i, v, a = _block_topk(s, dtype, k, rows, self_offset, delta)
        out_i.append(i.cpu())
        out_v.append(v.cpu())
        out_a.append(a.cpu())
    return (torch.cat(out_i).numpy(), torch.cat(out_v).numpy(), torch.cat(out_a).numpy())


def reference_top1(q, x, self_offset=-1, delta=None, block=2048):
    """First neighbour: -> (idx int64 [nq], dist [nq], ambiguous bool [nq])."""
    i, v, a = reference_topk(q, x, 1, self_offset, delta, block)
    return i[:, 0], v[:, 0], a


def f16_product(q16, x16):
    """float64 product of float16 rows (what the screen computes before its float32 accumulation rounds)."""
    return q16.astype(np.float64) @ x16.astype(np.float64).T


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def sign_rows(n, d, m, rng, dtype=np.float32, zero_rows=()):
    """Exact-arithmetic rows: m non-zero entries +-1/sqrt(m) (m a power of 4, so the entries are powers of two) at random
    positions among d columns; rows listed in zero_rows are all zero.  Every row is an exact unit vector in float32,
    float64 and float16, every product and partial sum of two rows is exact, and every score is an integer / m."""
    assert m >= 1 and m <= d and (m & (m - 1)) == 0 and int(math.log2(m)) % 2 == 0, "m must be a power of 4 <= d"
    x = _scatter_signs(n, d, m, 1.0 / math.sqrt(m), rng, dtype)
    x[list(zero_rows)] = 0
    return x


def _scatter_signs(n, d, cnt, v, rng, dtype):
    """[n, d] rows with cnt entries +-v at random positions."""
    x = np.zeros((n, d), dtype=dtype)
    if cnt == 0:
        return x
    if cnt == d:
        pos = np.broadcast_to(np.arange(d), (n, d))
    else:
        pos = np.argpartition(rng.random((n, d), dtype=np.float32), cnt - 1, axis=1)[:, :cnt]
    np.put_along_axis(x, pos, np.where(rng.random((n, cnt)) < 0.5, -v, v).astype(dtype), axis=1)
    return x


def plant_duplicates(x, groups):
    """groups: (start, size) - rows start .. start + size - 1 become copies of row `start`."""
    for start, size in groups:
        x[start:start + size] = x[start]
    return x


def boundary_groups(n, sizes=(1, 2, 31, 32, 33, 100), spacing=3):
    """Duplicate groups of the given sizes, each centred on a 256-row boundary (a row unit of the screen, a column tile,
    and for a self-search the edge of a diagonal tile), every `spacing`-th boundary.  -> [(start, size)]."""
    out, t = [], 1
    for size in sizes:
        c = TILE * t
        start = c - size // 2
        if start + size > n:
            break
        out.append((start, size))
        t += spacing
    return out


def left_pairs(n, count, rng):
    """Pairs (j, i), j < i in different column tiles: copying row j to row i makes i's best neighbour lie to its LEFT
    (a symmetric self-search finds it only through the column role of tile (unit of j, tile of i))."""
    out = []
    while len(out) < count:
        j, i = sorted(rng.choice(n, 2, replace=False).tolist())
        if i // TILE > j // TILE:
            out.append((j, i))
    return out


def cone_rows(n, d, m, c, rng, sign=1.0, dtype=np.float32):
    """Sign rows that share their first c entries (+-1/sqrt(m) with the given sign) and have m - c random entries in the
    other d - c columns.  Rows of opposite cones have s = (-c + small overlap) / m < 0: a query set from the cone
    opposite the database has a negative best score on every row."""
    assert (m & (m - 1)) == 0 and int(math.log2(m)) % 2 == 0 and c <= m and m - c <= d - c
    v = 1.0 / math.sqrt(m)
    head = np.full((n, c), sign * v, dtype=dtype)
    return np.concatenate([head, _scatter_signs(n, d - c, m - c, v, rng, dtype)], axis=1)


def ladder(d, m, steps, dtype=np.float32):
    """A query row q (m entries 1/sqrt(m) in the first m columns) and `steps` columns of rising score: column t flips
    the sign of the first steps - t entries, s_t = 1 - 2 (steps - t) / m - a step of 2 / m (2^-11 at m = 4096, about
    eps / 6).  Exact arithmetic.  -> (q [d], cols [steps, d], s [steps])."""
    assert steps <= m
    v = 1.0 / math.sqrt(m)
    q = np.zeros(d, dtype=dtype)
    q[:m] = v
    cols = np.tile(q, (steps, 1))
    for t in range(steps):
        cols[t, :steps - t] = -v
    s = 1.0 - 2.0 * (steps - np.arange(steps)) / m
    return q, cols, s


def _unit64(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def fine_ladder(q, steps, step, s0, rng):
    """Columns of float rows whose score against the unit row q rises by `step` in column order from s0 (step < eps / 32
    puts more than 32 columns inside eps of the best: the top-1 list overflows).  float64 [steps, d]."""
    d = q.shape[0]
    u = rng.standard_normal((steps, d))
    u -= np.outer(u @ q, q)
    u = _unit64(u)
    c = s0 + step * np.arange(steps)
    return c[:, None] * q[None, :] + np.sqrt(1 - c * c)[:, None] * u


def gaussian_planted(n, d, rng, near_pairs=64, round_ties=16):
    """float32 unit rows: Gaussian background plus planted structure.
    near:       triples (q, a, b), s(q, a) - s(q, b) = Delta in [1e-7, 1e-4] (log-uniform), both far above the background.
    round_ties: triples (q, a, b), a < b, float32(s(q, a)) == float32(s(q, b)) (so the float32 distances are equal) but
                s(q, a) < s(q, b) in float64: np.argmin on float32 distances takes a, the lower index, although b is
                closer in exact arithmetic.
    -> (x float32 [n, d], {"near": [(q, a, b)], "round_ties": [(q, a, b)]})."""
    x = _unit64(rng.standard_normal((n, d)))
    slots = rng.permutation(n)
    take = iter(slots.tolist())
    near, ties = [], []
    for _ in range(near_pairs):
        q, a, b = next(take), next(take), next(take)
        c = 0.7 + 0.25 * rng.random()
        delta = 10 ** rng.uniform(-7, -4)
        ua, ub = _unit64(rng.standard_normal((2, d)))
        for row, cc, u in ((a, c + delta, ua), (b, c, ub)):
            u = _unit64(u - (u @ x[q]) * x[q])
            x[row] = cc * x[q] + math.sqrt(1 - cc * cc) * u
        near.append((q, a, b))
    x32 = x.astype(np.float32)
    while len(ties) < round_ties:
        q, a, b = next(take), next(take), next(take)
        a, b = min(a, b), max(a, b)
        u = _unit64(rng.standard_normal(d))
        u = _unit64(u - (u @ x32[q]) * x32[q].astype(np.float64))
        c = 0.8 + 0.15 * rng.random()
        vb = (c * x32[q] + math.sqrt(1 - c * c) * u).astype(np.float32)
        qv = x32[q].astype(np.float64)
        sb = float(qv @ vb.astype(np.float64))
        # row a = row b with one component moved by one ulp against the query: s drops by ~1e-9, inside one float32 ulp
        k = int(np.argmax(np.abs(qv * vb)))
        va = vb.copy()
        va[k] = np.nextafter(va[k], np.float32(-np.inf) if qv[k] > 0 else np.float32(np.inf))
        sa = float(qv @ va.astype(np.float64))
        if not (sa < sb and np.float32(sa) == np.float32(sb)):
            continue
        x32[a], x32[b] = va, vb
        ties.append((q, a, b))
    return x32, {"near": near, "round_ties": ties}


def f16_order_reversals(x, triples):
    """How many planted triples (q, a, b) have the order of s(q, a), s(q, b) reversed (or tied) in the float64 product of
    the float16-rounded rows - the pairs only the exact re-rank can order."""
    x16 = x.astype(np.float16).astype(np.float64)
    x64 = x.astype(np.float64)
    rev = 0
    for q, a, b in triples:
        exact = x64[q] @ x64[a] - x64[q] @ x64[b]
        screened = x16[q] @ x16[a] - x16[q] @ x16[b]
        rev += int(np.sign(exact) != np.sign(screened))
    return rev


def f16_equal_rows(n, d, rng, noise=3e-5):
    """float32 unit rows e_0 + noise: distinct in float32, every pair's float16 score rounds to the same float32 value
    (components of ~noise lie in float16's subnormal range, the first one rounds to 1).  Every pair lies within eps of
    every row's best, so every candidate list and the symmetric screen's log overflow."""
    x = np.zeros((n, d))
    x[:, 0] = 1.0
    x[:, 1:] = noise * rng.standard_normal((n, d - 1))
    return _unit64(x).astype(np.float32)
