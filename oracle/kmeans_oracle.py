"""numpy restatement of spherecluster 0.1.x SphericalKMeans(...).fit(X) over scikit-learn 0.22 helpers
(the reference's fit_cluster(method='spherical_kmeans'), clustering/cluster_masks.py:23,38-98).

Neither package installs next to a current scikit-learn, so the algorithm is written out here.  Adapted from
scikit-learn 1.9 `sklearn/cluster/_kmeans.py` and `sklearn/preprocessing/_data.py`:
  * `_kmeans_plusplus` -> k_init.  0.22's `_k_init` is the same loop; 1.9 draws the first seed with
    `sample_weight`-weighted `choice` and weights the potentials, 0.22 (and this file) uses `randint(n)` and plain
    sums.  Potentials are summed in float64 here (0.22 sums the float32 distances).
  * `_tolerance` -> tolerance: mean(var(X, axis=0)) * tol (unchanged since 0.22).
  * `_kmeans_single_lloyd` -> lloyd.  1.9 runs Cython chunks with a strict-convergence check on the labels; 0.22 (and
    this file) loops E-step, `_centers_dense` (with the empty-cluster relocation restated in centers_dense), keeps the
    best inertia seen, stops on the centre shift and repeats the E-step against the best centres if the last shift is
    above zero.  spherecluster adds `normalize(centers)` after every update.
  * `_labels_inertia` -> labels_inertia: squared-Euclidean argmin (ties -> lowest centre).  1.9 works in the array
    dtype; here |x|^2 + |c|^2 - 2 x.c is evaluated in float64 and rounded to float32 (0.22's float32 upcast path).
  * `normalize` -> normalize: row L2 normalisation, zero rows stay zero.

Deliberate differences from spherecluster (the device code follows them too; DESIGN section 1, row a17):
  * centre sums in float64 (accumulate='float64'); accumulate='float32' sums in float32 in row order as spherecluster;
  * an explicit init array is normalised before the first E-step;
  * relocation sort: among equal distances the higher row index comes first (a reversed stable ascending sort);
  * a zero row goes to centre 0;
  * a zero centre (a zero row drawn as a seed) is at cosine distance 1 from every row, so it takes the rows whose
    similarity to every other centre is below 0; the reference's squared-Euclidean rule (|x - 0|^2 = 1 = 2 - 2 * 0.5)
    gives it every row below similarity 0.5.  mindist and the inertia keep the squared-Euclidean value.
Diagnostics for the tests: per iteration, the number of rows whose top-1 / top-2 mindist gap is below TIE_MARGIN, the
relocation events, and per k-means++ step whether a pick was within 1e-6 (relative) of a candidate-potential tie or a
cumsum boundary.
"""
import numpy as np

TIE_MARGIN = 2e-6   # the project's float32 tie margin (DESIGN section 2)
_CHUNK = 16384


def normalize(x):
    """Rows / float32 norm (the norm from a float64 sum of squares, as csrc/prep.cu); zero rows stay zero."""
    x = np.asarray(x, dtype=np.float32)
    nrm = np.sqrt(np.einsum("ij,ij->i", x.astype(np.float64), x.astype(np.float64)).astype(np.float32))
    nrm[nrm == 0] = 1
    return x / nrm[:, None]


def check_random_state(seed):
    if seed is None:
        return np.random.mtrand._rand
    if isinstance(seed, np.random.RandomState):
        return seed
    return np.random.RandomState(seed)


def draws(random_state, n, k, n_init):
    """Runs share one RandomState: per run randint(n), then random_sample(L) per later seed, L = 2 + int(log(k))."""
    L = 2 + int(np.log(k))
    rs = check_random_state(random_state)
    first, uni = [], []
    for _ in range(n_init):
        first.append(rs.randint(n))
        uni.append(np.concatenate([rs.random_sample(L) for _ in range(k - 1)]) if k > 1 else np.zeros(0))
    return np.array(first, dtype=np.int64), np.array(uni, dtype=np.float64).reshape(n_init, -1), L


def sqdist(a, X, xn=None):
    """max(|a|^2 + |x|^2 - 2 a.x, 0) in float64, rounded to float32; a [m, d] -> [m, n]."""
    a64 = np.atleast_2d(a).astype(np.float64)
    X64 = X.astype(np.float64)
    an = np.einsum("ij,ij->i", a64, a64)
    xn = np.einsum("ij,ij->i", X64, X64) if xn is None else xn
    q = (an[:, None] + xn[None, :]) - 2.0 * (a64 @ X64.T)
    return np.maximum(q, 0.0).astype(np.float32)


def k_init(X, k, first, uniforms, L):
    """_k_init of 0.22 on unit rows X with the given draws.  -> (seed indices int64 [k], near_ties: steps whose pick
    lay within 1e-6 relative of a candidate-potential tie or of a cumsum boundary)."""
    n = X.shape[0]
    xn = np.einsum("ij,ij->i", X.astype(np.float64), X.astype(np.float64))
    seeds = [int(first)]
    closest = sqdist(X[first], X, xn)[0]
    pot = closest.astype(np.float64).sum()
    near = []
    for c in range(1, k):
        u = uniforms[(c - 1) * L:c * L]
        vals = u * pot
        cs = np.cumsum(closest.astype(np.float64))
        ids = np.minimum(np.searchsorted(cs, vals), n - 1)
        m = np.minimum(closest[None, :], sqdist(X[ids], X, xn))
        pots = m.astype(np.float64).sum(axis=1)
        best = int(np.argmin(pots))
        scale = max(pot, 1e-300)
        lo = np.where(ids > 0, cs[np.maximum(ids - 1, 0)], 0.0)
        boundary = np.any(np.minimum(np.abs(cs[ids] - vals), np.abs(vals - lo)) <= 1e-6 * scale)
        others = [pots[l] for l in range(L) if ids[l] != ids[best]]
        pot_tie = bool(others) and min(others) - pots[best] <= 1e-6 * abs(pots[best])
        if boundary or pot_tie:
            near.append(c)
        seeds.append(int(ids[best]))
        closest = m[best]
        pot = pots[best]
    return np.array(seeds, dtype=np.int64), near


def labels_inertia(X, centers):
    """-> (labels int32, mindist float32, inertia float64 (fixed-order float64 sum), rows inside TIE_MARGIN)."""
    n = X.shape[0]
    X64 = X.astype(np.float64)
    C64 = centers.astype(np.float64)
    cn = np.einsum("ij,ij->i", C64, C64)
    labels = np.empty(n, dtype=np.int32)
    mind = np.empty(n, dtype=np.float32)
    ties = 0
    for s in range(0, n, _CHUNK):
        x = X64[s:s + _CHUNK]
        xn = np.einsum("ij,ij->i", x, x)
        D = ((xn[:, None] + cn[None, :]) - 2.0 * (x @ C64.T)).astype(np.float32)
        # the choice is by cosine distance: a zero centre competes as a unit centre orthogonal to the row would
        S = D.copy()
        S[:, cn == 0] = (xn[:, None] + 1.0).astype(np.float32)
        lab = np.argmin(S, axis=1)
        lab[xn == 0] = 0
        labels[s:s + _CHUNK] = lab
        mind[s:s + _CHUNK] = D[np.arange(D.shape[0]), lab]
        if D.shape[1] > 1:
            two = np.partition(S, 1, axis=1)[:, :2].astype(np.float64)
            ties += int(np.sum((two[:, 1] - two[:, 0] < TIE_MARGIN) & (xn > 0)))
    return labels, mind, mind.astype(np.float64).sum(), ties


def centers_dense(X, labels, distances, k, accumulate="float64"):
    """_centers_dense of 0.22 followed by spherecluster's normalize.  -> (centres float32 [k, d], relocations
    [(cluster, row)])."""
    acc = np.float64 if accumulate == "float64" else np.float32
    counts = np.bincount(labels, minlength=k)
    sums = np.zeros((k, X.shape[1]), dtype=acc)
    np.add.at(sums, labels, X.astype(acc))
    relocations = []
    empty = np.where(counts == 0)[0]
    if len(empty):
        far = np.argsort(distances, kind="stable")[::-1]
        for i, c in enumerate(empty):
            sums[c] = X[far[i]]
            counts[c] = 1
            relocations.append((int(c), int(far[i])))
    if accumulate == "float64":
        mean = sums / counts[:, None]
        nrm = np.sqrt((mean * mean).sum(axis=1))
        nrm[nrm == 0] = 1
        return (mean / nrm[:, None]).astype(np.float32), relocations
    mean = (sums / counts[:, None].astype(np.float32)).astype(np.float32)
    nrm = np.sqrt(np.einsum("ij,ij->i", mean, mean))
    nrm[nrm == 0] = 1
    return (mean / nrm[:, None]).astype(np.float32), relocations


def tolerance(X, tol):
    return float(np.mean(np.var(X.astype(np.float64), axis=0)) * tol)


def lloyd(X, centers, max_iter, tol_abs, accumulate="float64"):
    """One run from unit centres.  -> dict(labels, inertia, centers, n_iter, ties [per E-step], relocations)."""
    k = centers.shape[0]
    best = None
    ties, relocs = [], []
    shift = 0.0
    for i in range(max_iter):
        old = centers
        labels, mind, inertia, t = labels_inertia(X, centers)
        ties.append(t)
        centers, rel = centers_dense(X, labels, mind, k, accumulate)
        relocs.append(rel)
        if best is None or inertia < best[1]:
            best = [labels.copy(), inertia, centers.copy()]
        shift = float(((old.astype(np.float64) - centers.astype(np.float64)) ** 2).sum())
        if shift <= tol_abs:
            break
    if shift > 0:
        labels, _, inertia, t = labels_inertia(X, best[2])
        ties.append(t)
        best[0], best[1] = labels, inertia
    return dict(labels=best[0], inertia=best[1], centers=best[2], n_iter=i + 1, ties=ties, relocations=relocs)


def spherical_kmeans(X, k, init=None, n_init=10, max_iter=300, tol=1e-4, random_state=None, first_ids=None,
                     uniforms=None, accumulate="float64"):
    """SphericalKMeans(n_clusters=k, init, n_init, max_iter, tol, random_state).fit(X) as the module docstring states.
    Explicit draws (first_ids [n_init], uniforms [n_init, (k - 1) * L]) may replace random_state.
    -> dict(labels, inertia, centers, n_iter, ties (all runs), relocations (all runs), seeds, seed_near_ties,
    run_inertias: the inertia of every run, so that a caller can tell runs that tie on the inertia)."""
    U = normalize(X)
    n = U.shape[0]
    if n < k:
        raise ValueError("n_samples=%d should be >= n_clusters=%d" % (n, k))
    tol_abs = tolerance(U, tol)
    L = 2 + int(np.log(k))
    if init is not None:
        n_init = 1
    elif first_ids is None:
        first_ids, uniforms, L = draws(random_state, n, k, n_init)
    out, ties, relocs, seeds, near, inertias = None, [], [], [], [], []
    for r in range(n_init):
        if init is not None:
            c0 = centers_dense(np.asarray(init, np.float32), np.arange(k), np.zeros(k, np.float32), k, "float64")[0]
        else:
            s, nt = k_init(U, k, first_ids[r], uniforms[r], L)
            seeds.append(s)
            near.extend(nt)
            c0 = U[s].copy()
        res = lloyd(U, c0, max_iter, tol_abs, accumulate)
        ties.extend(res["ties"])
        relocs.extend(res["relocations"])
        inertias.append(res["inertia"])
        if out is None or res["inertia"] < out["inertia"]:
            out = res
    out = dict(out)
    out.update(ties=ties, relocations=relocs, seeds=seeds, seed_near_ties=near, unit=U, tol_abs=tol_abs,
               run_inertias=inertias)
    return out
