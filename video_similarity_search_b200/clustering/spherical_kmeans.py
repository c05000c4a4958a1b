"""Spherical k-means on B200 - the estimator behind fit_cluster(method='spherical_kmeans').

The reference imports it from spherecluster (clustering/cluster_masks.py:23), a package built on private modules of
scikit-learn 0.22 that later releases removed.  This class keeps its constructor, fit / fit_predict and fitted
attributes; the algorithm is restated in oracle/kmeans_oracle.py and runs on the device in one call
(slic_spherical_kmeans, csrc/skmeans.cu).  The random draws are made here, on the host, in the reference's order, so a
given random_state picks the same seeds as spherecluster.

Deliberate differences from spherecluster (DESIGN section 1, row a17):
  * centre sums and the inertia are accumulated in float64 (spherecluster: float32, row order);
  * an explicit `init` array is normalised before the first assignment (spherecluster uses it raw in the first E-step,
    which is Euclidean to non-unit centres);
  * empty-cluster relocation takes the farthest rows with ties going to the higher row index;
  * a zero row is assigned to centre 0 (every cosine distance from it is 1);
  * rows are assigned by cosine distance, so a zero centre (a zero row drawn as a seed) takes only the rows whose
    similarity to every other centre is negative (spherecluster's Euclidean rule: below 0.5);
  * the rows are processed in float32 (a float64 input is rounded once).
There is no `predict`: spherecluster inherits scikit-learn's Euclidean predict on unnormalised rows, which no caller uses.
"""
import warnings

import numpy as np
import torch

from .. import backend as _backend


def check_random_state(seed):
    """scikit-learn's check_random_state: None -> numpy's global RandomState, int -> a new one, RandomState -> itself."""
    if seed is None or seed is np.random:
        return np.random.mtrand._rand
    if isinstance(seed, (int, np.integer)):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError("%r cannot be used to seed a numpy.random.RandomState instance" % (seed,))


def n_local_trials(k):
    """Candidates per k-means++ step, as scikit-learn 0.22's _k_init draws them."""
    return 2 + int(np.log(k))


def draw_seeding(random_state, n, k, n_init):
    """The draws of n_init k-means++ runs that share one RandomState, in the reference's order: per run randint(n) for
    the first seed, then random_sample(L) for each of the k - 1 later seeds.
    -> (first_ids int64 [n_init], uniforms float64 [n_init, (k - 1) * L], L)."""
    L = n_local_trials(k)
    first = np.empty(n_init, dtype=np.int64)
    uniforms = np.empty((n_init, (k - 1) * L), dtype=np.float64)
    for r in range(n_init):
        first[r] = random_state.randint(n)
        for c in range(k - 1):
            uniforms[r, c * L:(c + 1) * L] = random_state.random_sample(L)
    return first, uniforms, L


class SphericalKMeans:
    """spherecluster.SphericalKMeans(n_clusters, init, n_init, max_iter, tol, random_state) on the device.

    X: numpy array or torch tensor [N, D], on the CPU or the GPU.  After fit: cluster_centers_ (float32 [k, D], unit
    rows), labels_ (int32 [N]), inertia_ (float), n_iter_ (int); last_stats_ holds the screen's counters of the fit
    (candidates re-ranked, rows finished by the exact kernel, list compactions, screened assignments)."""

    def __init__(self, n_clusters=8, init='k-means++', n_init=10, max_iter=300, tol=1e-4, random_state=None,
                 backend=None):
        self.n_clusters = n_clusters
        self.init = init
        self.n_init = n_init
        self.max_iter = max_iter
        self.tol = tol
        self.random_state = random_state
        self.backend = backend

    def _check(self, n):
        k = self.n_clusters
        if not isinstance(k, (int, np.integer)) or k < 1:
            raise ValueError("n_clusters must be a positive integer, got %r" % (k,))
        if n < k:
            raise ValueError("n_samples=%d should be >= n_clusters=%d" % (n, k))
        if self.n_init < 1:
            raise ValueError("Invalid number of initializations. n_init=%d must be bigger than zero." % self.n_init)
        if self.max_iter < 1:
            raise ValueError("Number of iterations should be a positive number, got %d instead" % self.max_iter)
        if self.tol < 0:
            raise ValueError("tol must be >= 0, got %r" % (self.tol,))

    def fit(self, X, y=None):
        be = self.backend or _backend.default_backend()
        if isinstance(X, torch.Tensor):
            X = X.detach()
        if len(X.shape) != 2:
            raise ValueError("X must be a 2-d matrix [n_samples, n_features]")
        n, d = int(X.shape[0]), int(X.shape[1])
        self._check(n)
        k = int(self.n_clusters)
        n_init = int(self.n_init)
        init = None
        if isinstance(self.init, str):
            if self.init != 'k-means++':
                raise ValueError("init must be 'k-means++' or an array of shape (n_clusters, n_features), got %r"
                                 % (self.init,))
        else:
            init = self.init.detach() if isinstance(self.init, torch.Tensor) else np.asarray(self.init)
            if tuple(init.shape) != (k, d):
                raise ValueError("init has shape %r, expected (%d, %d)" % (tuple(init.shape), k, d))
            if n_init != 1:
                warnings.warn("Explicit initial center position passed: performing only one init in k-means instead "
                              "of n_init=%d" % n_init, RuntimeWarning, stacklevel=2)
                n_init = 1
        x = be.to_device(X, torch.float32).contiguous()
        if init is not None:
            init_dev = be.to_device(init, torch.float32).contiguous()
            first, uniforms, L = None, None, 0
        else:
            init_dev = None
            first, uniforms, L = draw_seeding(check_random_state(self.random_state), n, k, n_init)
        labels, centres, inertia, n_iter, stats = be.spherical_kmeans(
            x, k, init=init_dev, first_ids=first, uniforms=uniforms, n_local_trials=L, n_init=n_init,
            max_iter=int(self.max_iter), tol=float(self.tol))
        self.labels_ = be.to_host(labels).astype(np.int32, copy=False)
        self.cluster_centers_ = be.to_host(centres).astype(np.float32, copy=False)
        self.inertia_ = float(inertia)
        self.n_iter_ = int(n_iter)
        self.last_stats_ = stats
        return self

    def fit_predict(self, X, y=None):
        return self.fit(X).labels_
