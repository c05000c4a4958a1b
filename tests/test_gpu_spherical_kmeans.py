"""Spherical k-means on the B200 (csrc/skmeans.cu) against the numpy restatement in oracle/kmeans_oracle.py."""
import numpy as np
import pytest
import torch

from oracle import kmeans_oracle as ko
from tests.golden.make_golden import CASES, make_input
from video_similarity_search_b200 import _lib, synth
from video_similarity_search_b200.clustering.spherical_kmeans import SphericalKMeans

pytestmark = pytest.mark.gpu

FIT_CASES = {"gmm_3000x128": (3000, 128, 30, 7), "c1_9537x512": (9537, 512, 101, 0), "gmm_777x200_odd": (777, 200, 9, 13)}


@pytest.fixture(scope="module")
def be():
    from video_similarity_search_b200.backend import CudaBackend
    return CudaBackend()


@pytest.fixture(params=["exact", "screen"])
def path(request, monkeypatch):
    """The assignment on the exact kernel (k below the screen threshold) or forced onto the tcgen05 screen."""
    if request.param == "screen":
        monkeypatch.setenv("SLIC_SKMEANS_SCREEN_MIN_K", "2")
    return request.param


@pytest.mark.parametrize("shape", [(3000, 128, 30, 7), (9537, 512, 101, 0), (240000, 512, 64, 0)])
def test_kmeans_plusplus_seeds_match_oracle(be, shape):
    n, d, k, seed = shape
    x = synth.gaussian_mixture(n, d, 400 if n == 240000 else k, seed)
    unit, _ = be.normalize_rows(be.to_device(x), want_f16=False)
    U = be.to_host(unit)
    differing = 0
    for rs in (0, 1, 2):
        first, uni, L = ko.draws(rs, n, k, 1)
        got = be.kmeans_plusplus(unit, k, int(first[0]), uni[0], L).cpu().numpy()
        exp, nt = ko.k_init(U, k, first[0], uni[0], L)
        diff = np.nonzero(got != exp)[0]
        if len(diff):     # allowed only at a step the oracle flags as a near tie
            assert diff[0] in nt, (rs, diff[:5], nt)
            differing += 1
    assert differing == 0


def _runs_tie(ref):
    """Two runs whose inertias agree to 1e-9: which one is kept depends on the last bits of float64 sums."""
    r = sorted(ref["run_inertias"])
    return len(r) > 1 and r[1] - r[0] <= 1e-9 * abs(r[0])


def _check_fit(est, x, k, init=None, n_init=3, random_state=0):
    ref = ko.spherical_kmeans(x, k, init=init, n_init=n_init, random_state=random_state)
    ref32 = ko.spherical_kmeans(x, k, init=init, n_init=n_init, random_state=random_state, accumulate="float32")
    if _runs_tie(ref):   # the same fit reached by two runs, possibly with other centre numbers: compare the inertia
        assert est.inertia_ == pytest.approx(ref["inertia"], rel=1e-6)
        return ref
    if sum(ref["ties"]) == 0:
        assert np.array_equal(est.labels_, ref["labels"])
        assert est.n_iter_ == ref["n_iter"]
    np.testing.assert_allclose(est.cluster_centers_, ref["centers"], rtol=1e-5, atol=1e-6)
    assert est.inertia_ == pytest.approx(ref["inertia"], rel=1e-6)
    if sum(ref32["ties"]) == 0 and not _runs_tie(ref32):
        assert np.array_equal(est.labels_, ref32["labels"])
    return ref


@pytest.mark.parametrize("name", list(FIT_CASES))
def test_fit_with_explicit_unit_init(be, name, path):
    n, d, k, seed = FIT_CASES[name]
    x = synth.gaussian_mixture(n, d, k, seed)
    centres = np.random.default_rng(seed).standard_normal((k, d))      # the mixture centres, drawn as synth draws them
    init = ko.normalize(centres.astype(np.float32))
    est = SphericalKMeans(n_clusters=k, init=init, n_init=1, backend=be).fit(x)
    _check_fit(est, x, k, init=init, n_init=1)


@pytest.mark.parametrize("name", list(FIT_CASES))
def test_fit_with_kmeans_plusplus(be, name, path):
    n, d, k, seed = FIT_CASES[name]
    x = synth.gaussian_mixture(n, d, k, seed)
    est = SphericalKMeans(n_clusters=k, n_init=3, random_state=5, backend=be).fit(torch.from_numpy(x).cuda())
    _check_fit(est, x, k, n_init=3, random_state=5)


def test_relocation_case(be, path):
    x = np.abs(synth.gaussian_mixture(400, 16, 3, 5))
    init = np.vstack([x[0], x[1], x[2], -np.ones(16)]).astype(np.float32)
    est = SphericalKMeans(n_clusters=4, init=init, n_init=1, backend=be).fit(x)
    ref = _check_fit(est, x, 4, init=init, n_init=1)
    assert ref["relocations"][0]


@pytest.mark.parametrize("k", [1, 2])
def test_small_k(be, k):
    x = make_input(CASES["gmm_1200x64"])
    est = SphericalKMeans(n_clusters=k, n_init=2, random_state=3, backend=be).fit(x)
    _check_fit(est, x, k, n_init=2, random_state=3)
    if k == 1:
        assert not est.labels_.any()


def test_k_equals_n(be, path):
    x = synth.gaussian_mixture(300, 32, 6, 8)
    est = SphericalKMeans(n_clusters=300, n_init=1, random_state=0, backend=be).fit(x)
    _check_fit(est, x, 300, n_init=1, random_state=0)


def test_zero_rows(be, path):
    x = make_input(CASES["zeros_500x32"])
    for n_init in (1, 2):    # run 0 draws zero row 499 as a seed: a zero centre
        est = SphericalKMeans(n_clusters=6, n_init=n_init, random_state=1, backend=be).fit(x)
        _check_fit(est, x, 6, n_init=n_init, random_state=1)
        assert np.all(est.labels_[[0, 7, 8, 250, 499]] == 0)


def test_n_less_than_k_raises(be):
    x = synth.gaussian_mixture(10, 8, 2, 0)
    with pytest.raises(ValueError):
        SphericalKMeans(n_clusters=11, backend=be).fit(x)
    with pytest.raises(_lib.SlicError):
        be.spherical_kmeans(be.to_device(x), 11, first_ids=np.zeros(1), uniforms=np.zeros((1, 40)), n_local_trials=4)


def test_full_size_c3_k1000(be):
    """240 000 x 512, k = 1000, n_init = 1: the C3 matrix, fitted on the device; only the checks run elsewhere."""
    n, d, kk, seed = synth.CONFIGS["C3"]
    x = be.to_device(synth.gaussian_mixture(n, d, kk, seed))
    k = 1000
    a = SphericalKMeans(n_clusters=k, n_init=1, random_state=0, backend=be).fit(x)
    b = SphericalKMeans(n_clusters=k, n_init=1, random_state=0, backend=be).fit(x)
    assert np.array_equal(a.labels_, b.labels_) and np.array_equal(a.cluster_centers_, b.cluster_centers_)
    assert a.inertia_ == b.inertia_ and a.n_iter_ == b.n_iter_
    unit, _ = be.normalize_rows(x, want_f16=False)
    C = torch.from_numpy(a.cluster_centers_).cuda()
    lab = torch.from_numpy(a.labels_).cuda().long()
    # labels: the exact first neighbour among the centres, wherever the top-1 / top-2 gap is outside the margin
    idx, _ = be.nn_exact_top1(unit, C)
    s = torch.cat([unit[i:i + 16384].double() @ C.double().T for i in range(0, n, 16384)])
    top2 = torch.topk(s, 2, dim=1).values
    clear = (2 * (top2[:, 0] - top2[:, 1])) >= ko.TIE_MARGIN
    assert torch.equal(idx.long()[clear], lab[clear])
    # inertia: float64 recomputation of sum(float32(|x|^2 + |c|^2 - 2 x.c))
    u64, c64 = unit.double(), C.double()
    dots = (u64 * c64[lab]).sum(1)
    mind = ((u64 * u64).sum(1) + (c64 * c64).sum(1)[lab] - 2 * dots).float().double()
    assert a.inertia_ == pytest.approx(mind.sum().item(), rel=1e-6)
    # centres: the normalised float64 means of their members (clusters whose members the final E-step kept)
    sums, counts, _ = be.cluster_sums(unit, lab.int(), k)
    means = sums / sums.norm(dim=1, keepdim=True)
    close = ((means - C.double()).abs().max(dim=1).values <= 1e-6)
    assert close.float().mean().item() >= 0.99
