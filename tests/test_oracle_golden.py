"""The oracle (oracle/finch_oracle.py) against the fixtures produced by the UNMODIFIED reference
(tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

from oracle import finch_oracle as fo
from tests.golden.make_golden import CASES, make_input

SMALL = [k for k in CASES if k != "c1_9537x512"]


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


def _run_oracle(case, g):
    x = make_input(case)
    kw = dict(ensure_early_exit=case.get("ensure_early_exit", True), req_clust=case.get("req_clust"),
              return_trace=True)
    if case.get("use_initial_rank"):
        kw["initial_rank"] = g["initial_rank"]
    thr = case.get("flann_threshold")
    saved = fo.FLANN_THRESHOLD
    try:
        if thr is not None:
            fo.FLANN_THRESHOLD = thr
        return fo.finch(x, **kw)
    finally:
        fo.FLANN_THRESHOLD = saved


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference_golden(golden_dir, name):
    case, g = CASES[name], _load(golden_dir, name)
    c, num_clust, req_c, trace = _run_oracle(case, g)
    assert num_clust == g["num_clust"].tolist()
    assert c.dtype == np.int32 and np.array_equal(c, g["c"])
    if g["req_c"].size:
        assert np.array_equal(req_c, g["req_c"])
    else:
        assert req_c is None
    if not np.isnan(g["min_sim"]):
        assert float(trace["min_sim"]) == float(g["min_sim"])
    else:
        assert trace["min_sim"] is None
    for lvl in range(int(g["n_levels_run"])):
        ref_nn = g["nn_level%d" % lvl]
        if ref_nn.size:
            assert np.array_equal(trace["nn"][lvl], ref_nn), "level %d" % lvl


def test_oracle_matches_reference_golden_c1(golden_dir):
    """BASELINE config 1 (N=9537, D=512): the reference's CPU-runnable case."""
    g = _load(golden_dir, "c1_9537x512")
    c, num_clust, _, trace = _run_oracle(CASES["c1_9537x512"], g)
    assert num_clust == [1170, 101, 25, 8, 5] == g["num_clust"].tolist()
    assert np.array_equal(c, g["c"])
    assert np.array_equal(trace["nn"][0], g["nn_level0"])
    assert float(trace["min_sim"]) == float(g["min_sim"])


def test_labels_are_numbered_by_smallest_member(golden_dir):
    """Structural invariant the CUDA relabel relies on (SURVEY.md 8 a4)."""
    g = _load(golden_dir, "gmm_3000x128")
    for col in g["c"].T:
        first = np.full(col.max() + 1, len(col))
        np.minimum.at(first, col, np.arange(len(col)))
        assert np.all(np.diff(first) > 0)


def test_blocked_first_neighbors_equal_dense():
    x = make_input(CASES["gmm_1200x64"])
    nn_d, _ = fo.first_neighbors_dense(x)
    nn_b, d1, gap = fo.first_neighbors_blocked(x, block=256)
    assert np.array_equal(nn_d, nn_b)
    assert np.all(gap >= 0) and np.all(d1 >= 0)
    rows = np.array([5, 17, 1199])
    nn_s, _, _ = fo.first_neighbors_blocked(x, rows=rows)
    assert np.array_equal(nn_s, nn_d[rows])


def test_cluster_means_is_fp64_segmented_mean():
    x = make_input(CASES["gmm_777x200_odd"])
    lab = np.random.default_rng(0).integers(0, 40, len(x))
    lab = np.unique(lab, return_inverse=True)[1]
    m = fo.cluster_means(x, lab)
    assert m.dtype == np.float64
    direct = np.stack([x[lab == c].astype(np.float64).mean(0) for c in range(lab.max() + 1)])
    np.testing.assert_allclose(m, direct, rtol=0, atol=1e-12)


@pytest.mark.parametrize("name", ["gmm_1200x64", "gmm_2500x96_flann"])
def test_oracle_plain_call_matches_stored_reference_output(golden_dir, name):
    """The oracle called the way a caller of the reference calls FINCH (defaults, no trace) against the partition the
    reference computed with the same defaults (stored by make_golden.py), the second case through the FLANN branch."""
    case, g = CASES[name], _load(golden_dir, name)
    x = make_input(case)
    thr = case.get("flann_threshold")
    saved = fo.FLANN_THRESHOLD
    try:
        if thr is not None:
            fo.FLANN_THRESHOLD = thr
        c, n, _ = fo.finch(x)
    finally:
        fo.FLANN_THRESHOLD = saved
    assert n == g["num_clust"].tolist() and np.array_equal(c, g["c"])
