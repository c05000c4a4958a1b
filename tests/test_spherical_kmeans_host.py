"""Spherical k-means without a GPU: the oracle (oracle/kmeans_oracle.py), the host logic of SphericalKMeans (the
random draws it hands to the device, warnings, argument errors), fit_cluster's spherical_kmeans branch and the argument
checks of the two C entries.  The device code itself is checked by tests/test_gpu_spherical_kmeans.py."""
import ctypes
import io
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

from oracle import kmeans_oracle as ko
from video_similarity_search_b200 import _lib
from video_similarity_search_b200 import synth
from video_similarity_search_b200.clustering import cluster_masks as cm
from video_similarity_search_b200.clustering import spherical_kmeans as skm


class RecordingBackend:
    """Stand-in for CudaBackend.spherical_kmeans: records what the estimator passes and returns fixed results."""

    def __init__(self):
        self.calls = []

    def to_device(self, array, dtype=None):
        t = torch.as_tensor(array)
        return (t.to(dtype) if dtype is not None else t).contiguous()

    def to_host(self, t):
        return t.cpu().numpy()

    def spherical_kmeans(self, x, k, init=None, first_ids=None, uniforms=None, n_local_trials=1, n_init=1,
                         max_iter=300, tol=1e-4):
        self.calls.append(dict(x=x, k=k, init=init, first_ids=first_ids, uniforms=uniforms, L=n_local_trials,
                               n_init=n_init, max_iter=max_iter, tol=tol))
        n, d = x.shape
        return (torch.arange(n, dtype=torch.int32) % k, torch.zeros((k, d), dtype=torch.float32), 1.5, 3,
                np.zeros(4, dtype=np.int64))


@pytest.mark.parametrize("n,d,k,seed", [(1200, 64, 12, 3), (777, 200, 9, 13)])
def test_oracle_reaches_a_fixed_point(n, d, k, seed):
    x = synth.gaussian_mixture(n, d, k, seed)
    res = ko.spherical_kmeans(x, k, n_init=1, max_iter=300, tol=0.0, random_state=0)
    assert res["n_iter"] < 300                      # converged: the last shift was 0
    U = res["unit"]
    lab, _, inertia, _ = ko.labels_inertia(U, res["centers"])
    assert np.array_equal(lab, res["labels"])       # labels are the argmin against the final centres
    assert inertia == pytest.approx(res["inertia"], rel=1e-12)
    means = np.zeros((k, d))
    np.add.at(means, lab, U.astype(np.float64))
    means /= np.linalg.norm(means, axis=1, keepdims=True)
    np.testing.assert_allclose(res["centers"], means, atol=1e-6)   # centres are the normalised means of their members


def relocation_case():
    """Rows in the positive orthant, three centres on rows and a fourth at -(1, ..., 1): no row is nearest to it."""
    x = np.abs(synth.gaussian_mixture(400, 16, 3, 5))
    init = np.vstack([x[0], x[1], x[2], -np.ones(16)]).astype(np.float32)
    return x, init


def test_oracle_relocates_an_empty_cluster():
    x, init = relocation_case()
    U = ko.normalize(x)
    lab, mind, _, _ = ko.labels_inertia(U, ko.normalize(init))
    assert not np.any(lab == 3)
    res = ko.spherical_kmeans(x, 4, init=init, max_iter=1, tol=0.0)
    order = np.argsort(mind, kind="stable")[::-1]
    assert res["relocations"][0] == [(3, int(order[0]))]   # the farthest row becomes the empty cluster's centre
    assert res["n_iter"] == 1


def test_oracle_relocation_tie_goes_to_higher_row():
    X = np.array([[1, 0], [1, 0], [0, 1], [0, 1]], dtype=np.float32)
    dist = np.array([0.5, 0.5, 0.5, 0.1], dtype=np.float32)
    centres, rel = ko.centers_dense(X, np.array([0, 0, 0, 0]), dist, 3)
    assert rel == [(1, 2), (2, 1)]
    np.testing.assert_array_equal(centres[1], X[2])


def _replay(seed, n, k, n_init):
    rs = np.random.RandomState(seed)
    L = 2 + int(np.log(k))
    first, uni = [], []
    for _ in range(n_init):
        first.append(rs.randint(n))
        u = []
        for _ in range(k - 1):
            u.append(rs.random_sample(L))
        uni.append(np.concatenate(u))
    return np.array(first), np.array(uni), L


def test_estimator_hands_the_reference_draws_to_the_device():
    be = RecordingBackend()
    x = synth.gaussian_mixture(500, 16, 7, 2)
    est = skm.SphericalKMeans(n_clusters=20, n_init=3, random_state=11, backend=be).fit(x)
    call = be.calls[-1]
    first, uni, L = _replay(11, 500, 20, 3)
    assert call["L"] == L == 2 + int(np.log(20)) and call["n_init"] == 3 and call["init"] is None
    assert np.array_equal(call["first_ids"], first)
    assert np.array_equal(call["uniforms"], uni)
    assert call["x"].dtype == torch.float32 and tuple(call["x"].shape) == (500, 16)
    assert est.labels_.dtype == np.int32 and est.labels_.shape == (500,)
    assert est.cluster_centers_.dtype == np.float32 and est.cluster_centers_.shape == (20, 16)
    assert est.inertia_ == 1.5 and est.n_iter_ == 3
    # the oracle's own draws are the same sequence
    f2, u2, _ = ko.draws(11, 500, 20, 3)
    assert np.array_equal(f2, first) and np.array_equal(u2, uni)
    # a shared RandomState advances across fits; None draws from numpy's global state
    rs = np.random.RandomState(4)
    skm.SphericalKMeans(n_clusters=5, n_init=2, random_state=rs, backend=be).fit(x)
    f3, _, _ = _replay(4, 500, 5, 4)
    assert np.array_equal(be.calls[-1]["first_ids"], f3[:2])
    skm.SphericalKMeans(n_clusters=5, n_init=2, random_state=rs, backend=be).fit(x)
    assert np.array_equal(be.calls[-1]["first_ids"], f3[2:])
    np.random.seed(9)
    skm.SphericalKMeans(n_clusters=5, n_init=1, backend=be).fit(torch.from_numpy(x))
    assert be.calls[-1]["first_ids"][0] == np.random.RandomState(9).randint(500)


def test_explicit_init_warns_and_runs_once():
    be = RecordingBackend()
    x = synth.gaussian_mixture(300, 8, 4, 1)
    init = x[:4]
    with pytest.warns(RuntimeWarning, match="performing only one init"):
        skm.SphericalKMeans(n_clusters=4, init=init, n_init=10, backend=be).fit(x)
    call = be.calls[-1]
    assert call["n_init"] == 1 and call["first_ids"] is None and call["uniforms"] is None
    assert np.array_equal(call["init"].numpy(), init)
    with pytest.raises(ValueError):
        skm.SphericalKMeans(n_clusters=4, init=x[:3], n_init=1, backend=be).fit(x)


@pytest.mark.parametrize("kw,n", [(dict(n_clusters=11), 10), (dict(n_clusters=0), 10), (dict(n_clusters=3, n_init=0), 10),
                                  (dict(n_clusters=3, max_iter=0), 10), (dict(n_clusters=3, init="random"), 10)])
def test_estimator_argument_errors(kw, n):
    be = RecordingBackend()
    with pytest.raises(ValueError):
        skm.SphericalKMeans(backend=be, **kw).fit(np.ones((n, 4), dtype=np.float32))
    assert not be.calls


def test_fit_cluster_spherical_kmeans(monkeypatch):
    from video_similarity_search_b200 import backend as bk
    be = RecordingBackend()
    monkeypatch.setattr(bk, "_default", be)
    x = synth.gaussian_mixture(600, 32, 5, 3)
    buf = io.StringIO()
    with redirect_stdout(buf):
        lab = cm.fit_cluster(torch.from_numpy(x), method="spherical_kmeans", k=7)
    assert lab.dtype == np.int32 and lab.shape == (600,)
    assert buf.getvalue().strip().splitlines() == ["Clustering with spherical_kmeans...",
                                                   "Fitted 7 clusters with spherical_kmeans"]
    call = be.calls[-1]
    assert call["k"] == 7 and call["n_init"] == 10 and call["max_iter"] == 300 and call["tol"] == 1e-4
    with pytest.raises(NotImplementedError), redirect_stdout(io.StringIO()):
        cm.fit_cluster(torch.from_numpy(x), method="kmeans")


def test_c_entries_refuse_bad_arguments_without_a_device():
    lib = _lib.load()
    buf = ctypes.create_string_buffer(1 << 12)
    ids = (ctypes.c_int64 * 2)(0, 0)
    inertia, n_iter = ctypes.c_double(), ctypes.c_int32()
    out = [ctypes.addressof(inertia), ctypes.addressof(n_iter), None, None]

    def fit(n, k, n_init, max_iter):
        return lib.slic_spherical_kmeans(buf, n, 4, k, None, ctypes.addressof(ids), buf, 3, n_init, max_iter, 1e-4,
                                         buf, buf, *out)
    assert fit(5, 6, 1, 10) == -1 and b"n >= k" in lib.slic_last_error()
    assert fit(5, 0, 1, 10) == -1 and b"k >= 1" in lib.slic_last_error()
    assert fit(5, 2, 0, 10) == -1 and b"n_init" in lib.slic_last_error()
    assert fit(5, 2, 1, 0) == -1 and b"max_iter" in lib.slic_last_error()
    assert lib.slic_spherical_kmeans(buf, 5, 4, 2, buf, None, None, 0, 2, 10, 1e-4, buf, buf, *out) == -1   # init + n_init 2
    assert lib.slic_kmeans_plusplus(buf, 5, 4, 6, 0, buf, 3, buf, None) == -1 and b"kmeans_plusplus" in lib.slic_last_error()
    assert lib.slic_kmeans_plusplus(buf, 5, 4, 2, 7, buf, 3, buf, None) == -1                  # first_id outside [0, n)
    assert lib.slic_kmeans_plusplus(buf, 5, 4, 2, 0, buf, 40, buf, None) == -1                 # too many candidates
