"""Spherical k-means timing on the GPU (csrc/skmeans.cu) with a bounded CPU oracle arm.

usage: python scripts/bench_spherical_kmeans.py OUT_DIR [--skip-cpu]

Workloads: 240 000 x 512 with k = 1000 (the C3 matrix of synth.py), 240 000 x 128 with k = 1000, and 240 000 x 512
with k = 20 (below the screen threshold); each with n_init 1 and 10.  Per workload: CUDA-event times of one k-means++
seeding, of one Lloyd iteration (difference of two explicit-init fits, 8 and 2 iterations at tol 0, over 6) on the
assignment path the fit uses and on the other one (SLIC_SKMEANS_SCREEN_MIN_K), and of the whole fit; iterations and
the screen's counters; shares of peak from the shapes.  Writes OUT_DIR/spherical_kmeans.json.
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from oracle import kmeans_oracle as ko
from video_similarity_search_b200 import synth
from video_similarity_search_b200.backend import CudaBackend
from video_similarity_search_b200.clustering import spherical_kmeans as skm

HBM_BPS = 7.7e12          # HGX B200 data sheet, one GPU
F16_FLOPS = 2.25e15       # dense FP16, one GPU
SCREEN_MIN_K = 256        # SK_SCREEN_MIN_K_DEFAULT in csrc/skmeans.cu
WORKLOADS = [("C3_512_k1000", 512, 1000), ("C3_128_k1000", 128, 1000), ("C3_512_k20", 512, 20)]


def events_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 else None
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def lloyd_iteration_ms(be, x, k, init, screen_min_k):
    os.environ["SLIC_SKMEANS_SCREEN_MIN_K"] = str(screen_min_k)
    try:
        be.spherical_kmeans(x, k, init=init, max_iter=2, tol=0.0)        # warm-up
        t2, r2 = events_ms(lambda: be.spherical_kmeans(x, k, init=init, max_iter=2, tol=0.0))
        t8, r8 = events_ms(lambda: be.spherical_kmeans(x, k, init=init, max_iter=8, tol=0.0))
    finally:
        del os.environ["SLIC_SKMEANS_SCREEN_MIN_K"]
    iters = r8[3] - r2[3]
    return ((t8 - t2) / iters if iters > 0 else None), [int(v) for v in r8[4]]


def main():
    out_dir = sys.argv[1]
    skip_cpu = "--skip-cpu" in sys.argv
    os.makedirs(out_dir, exist_ok=True)
    be = CudaBackend()
    n, _, kk, seed = synth.CONFIGS["C3"]
    result = dict(device_info(), workloads=[], notes=(
        "times are CUDA events around blocking calls; one Lloyd iteration = (fit with 8 iterations - fit with 2) / 6 "
        "from an explicit init, so it includes assignment, epilogue, sums, update and bookkeeping; "
        "assignment share of peak divides 2*N*k*D flop by that whole-iteration time"))
    for name, d, k in WORKLOADS:
        xh = synth.gaussian_mixture(n, d, kk, seed)
        x = be.to_device(xh)
        unit, _ = be.normalize_rows(x, want_f16=False)
        L = skm.n_local_trials(k)
        first, uni, _ = ko.draws(0, n, k, 1)
        be.kmeans_plusplus(unit, k, int(first[0]), uni[0], L)
        seed_ms, seeds = events_ms(lambda: be.kmeans_plusplus(unit, k, int(first[0]), uni[0], L))
        init = unit[seeds.long()].contiguous()
        screened = k >= SCREEN_MIN_K
        it_ms, it_stats = lloyd_iteration_ms(be, x, k, init, SCREEN_MIN_K)
        other_ms, _ = lloyd_iteration_ms(be, x, k, init, k + 1 if screened else 2)
        w = dict(name=name, n=n, d=d, k=k, L=L, assignment="screen" if screened else "exact",
                 seeding_ms_per_init=seed_ms, lloyd_iteration_ms=it_ms,
                 lloyd_iteration_ms_other_path=other_ms, other_path="exact" if screened else "screen",
                 lloyd_iteration_stats_8_iterations=it_stats,
                 seeding_bytes=n * d * 4 * (k - 1), seeding_hbm_share=(n * d * 4 * (k - 1) / HBM_BPS) / (seed_ms / 1e3),
                 assignment_flop=2.0 * n * k * d, runs=[])
        if it_ms:
            w["assignment_f16_share_of_whole_iteration"] = (2.0 * n * k * d / F16_FLOPS) / (it_ms / 1e3)
        for n_init in (1, 10):
            est = skm.SphericalKMeans(n_clusters=k, n_init=n_init, random_state=0, backend=be)
            fit_ms, _ = events_ms(lambda: est.fit(x))
            w["runs"].append(dict(n_init=n_init, fit_ms=fit_ms, n_iter=est.n_iter_, inertia=est.inertia_,
                                  screen_stats=dict(zip(["candidates_reranked", "rows_finished_exactly",
                                                         "list_compactions", "screened_assignments"],
                                                        [int(v) for v in est.last_stats_]))))
        if not skip_cpu and name == "C3_512_k1000":
            U = ko.normalize(xh)
            C = be.to_host(init)
            t0 = time.perf_counter()
            lab, mind, _, _ = ko.labels_inertia(U, C)
            ko.centers_dense(U, lab, mind, k)
            cpu_iter = time.perf_counter() - t0
            ks = 20
            f2, u2, L2 = ko.draws(0, n, ks, 1)
            t0 = time.perf_counter()
            ko.k_init(U, ks, f2[0], u2[0], L2)
            cpu_seed_small = time.perf_counter() - t0
            w["cpu_oracle"] = dict(lloyd_iteration_s=cpu_iter, seeding_s_at_k20=cpu_seed_small,
                                   seeding_s_per_init_extrapolated_to_k1000=cpu_seed_small * (k - 1) / (ks - 1),
                                   note="numpy float64 restatement on this host's CPU; seeding extrapolated linearly in k")
        result["workloads"].append(w)
        print(json.dumps(w), flush=True)
        del x, unit, init
        torch.cuda.empty_cache()
    with open(os.path.join(out_dir, "spherical_kmeans.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
