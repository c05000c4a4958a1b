#!/usr/bin/env python
"""bench.py - the hot path of BASELINE.json measured on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload C3|C1|C5] [--dump-outputs DIR]
  (N > 1: launched by torch.distributed.run, one rank per GPU, NCCL)

--steps K is the number of timed calls in every timed loop (a loop with a stalled call is timed once more: see
`remeasured` below).  --dump-outputs DIR: after the timed steps, the outputs of the
last timed FINCH call are written as DIR/<name>.npy in float64 (see dump_outputs); the inputs are seeded, so two builds
run with the same arguments can be compared output for output.

Workload (config.workload), default BASELINE configs[2]/[3]: FINCH full hierarchy on N = 240 000 x D = 512 synthetic
Gaussian-mixture embeddings (Kinetics-400 train size), seed 0 (video_similarity_search_b200.synth).  A "step" is one
complete FINCH call on that batch (all levels: first neighbours, components, means).  --workload C5 is BASELINE
configs[4] (N = 1 000 000 x D = 1 024 FINCH + top-50 retrieval of 100 000 queries), meant for --gpus 8.

  value        embeddings/s through the whole hierarchy with the matrix already resident in HBM
               (= N / seconds per step; the BASELINE metric "FINCH full-hierarchy seconds" is `finch_seconds`)
  e2e          the same through the reference-facing call FINCH(host matrix): host->device copy of the embeddings
               (pinned source) and device->host copy of the label matrix inside the timed region;
               e2e_pageable: the same call on a plain numpy array, as clustering/cluster_masks.py:80 hands it over
  roofline     the dominant kernel (nn_screen_kernel, tcgen05, float16 operands / float32 accumulate): flop the tensor
               cores EXECUTED per launch over its CUDA-event duration on its own stream, against the measured dense
               peak of MEASURED_PEAKS.json.  (`algorithmic_tflops` counts the full 2 n^2 d of SURVEY.md 8(d); the
               self-search computes only the tiles on or right of the diagonal, `symmetry_gain` is the ratio.)
  retrieval    the second half of BASELINE.json's metric: top-50 retrieval through the same screen (configs[1] and
               the configs[4] retrieval shape), ms / queries per second / fraction of the tensor peak
  cpu_baseline the oracle port of the reference (numpy / scipy / sklearn) on this box's host cores, bounded sample
  step_host_ms_rank0   host clock of every timed call of the headline loop; `remeasured`: a timed loop in which one call took
               more than 2.5 x the median call (a host stall) is measured again ONCE - the first attempt stays in the line
At N > 1 the level-0 nearest-neighbour stage is shared by the ranks (strong scaling: total work fixed).

--impl reference: the reference's CPU implementation (oracle port; the reference itself is pure Python that needs
pyflann above 70 000 rows, see oracle/finch_oracle.py) on the same workload: a bounded sample per step, plus ONE
full pass of the level-0 stage that checks the sample's linear extrapolation (--no-full-nn skips it).
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "C3"          # N=240000, D=512, K=400, seed 0
METRIC = "finch_full_hierarchy_embeddings_per_s"
UNIT = "embeddings/s"
C5_QUERIES = 100000      # BASELINE configs[4] does not fix Q; SURVEY.md 8(d) chose 100 000 (seed 1), k = 50


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=WORKLOAD, help="C3 (default) | C1 | C5")
    ap.add_argument("--cpu-sample-rows", type=int, default=4096, help="query rows of the timed CPU sample")
    ap.add_argument("--parity-rows", type=int, default=16384, help="rows checked against the oracle's first neighbours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-nn", action="store_true", help="reference arm: skip the one full pass of the level-0 stage")
    ap.add_argument("--no-retrieval", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a sample of the work and has no step output to write")
    return args


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel from a committed `ncu --set full`
# capture; keyed by (workload, ranks).  A constant taken from that capture, not re-measured per run (a number taken under
# the profiler's replay is evidence of traffic, never of time) - the line says so in `traffic_source`.
NCU_TRAFFIC = {("C3", 1): (2.087769e9 + 82.432768e6, "profiles/r2_sym_screen_kernel_ncu_full.txt (round-2 kernel, float16 operands)")}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p.get("bf16_tflops_sustained"),
                    hbm_gbs=p["hbm_gbs"], source="measured")
    return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


# --------------------------------------------------------------------------------------------------
# CPU side: the oracle port of the reference, bounded sample
# --------------------------------------------------------------------------------------------------
def use_all_cores():
    """BLAS threads = all host cores, whatever OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1,
    which would time the reference's sgemm on one core).  Returns (limiter, threads in use)."""
    want = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        lim = threadpool_limits(limits=want)
        got = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
        return lim, got
    except Exception:
        return None, 1


def within_component_neighbors(x, lab):
    """First neighbours restricted to rows of the same mixture component - a cheap way to obtain a realistic
    level-0 neighbour array for TIMING the CPU levels >= 1 (equal to the global first neighbour on all but a
    handful of rows; never used for a parity claim)."""
    from oracle import finch_oracle as fo
    nn = np.empty(len(x), dtype=np.int64)
    order = np.argsort(lab, kind="stable")
    bounds = np.flatnonzero(np.diff(lab[order])) + 1
    for grp in np.split(order, bounds):
        if len(grp) == 1:
            nn[grp] = grp
            continue
        j, _, _ = fo.first_neighbors_blocked(x[grp])
        nn[grp] = grp[j]
    return nn


def cpu_reference_step(x, nn_for_rest, sample_rows, rest_runs):
    """One bounded CPU step of the reference algorithm on the workload:
      (a) level-0 first-neighbour stage (finch.py:22-29 arithmetic, exact blocked form used above 70 000 rows)
          on `sample_rows` query rows x ALL columns, scaled linearly to all rows - timed in EVERY step;
      (b) everything after it - components, means, all levels >= 1 - in full (oracle finch with initial_rank): ~15 s of
          deterministic work, timed in the first REST_RUNS steps of a run and their mean reused by the later ones, so
          that a --steps 20 run stays within minutes (`rest_runs` collects the measurements).
    Returns (estimated seconds for the whole hierarchy, detail dict)."""
    from oracle import finch_oracle as fo
    n = len(x)
    rows = np.linspace(0, n - 1, sample_rows).astype(np.int64)
    t0 = time.perf_counter()
    fo.first_neighbors_blocked(x, rows=rows)
    t_nn = time.perf_counter() - t0
    if len(rest_runs) < REST_RUNS:
        t0 = time.perf_counter()
        c, num_clust, _ = fo.finch(x, initial_rank=nn_for_rest)
        rest_runs.append((time.perf_counter() - t0, [int(v) for v in num_clust]))
    t_rest = statistics.mean(r[0] for r in rest_runs)
    est = t_nn * (n / float(sample_rows)) + t_rest
    return est, dict(nn_sample_s=t_nn, nn_stage_est_s=t_nn * n / float(sample_rows), rest_s=t_rest,
                     rest_runs_timed=len(rest_runs), num_clust=rest_runs[-1][1])


REST_RUNS = 3


def workload_string(n, d, k, seed):
    return "FINCH full hierarchy, N=%d x D=%d Gaussian mixture (K=%d, seed %d), cosine" % (n, d, k, seed)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import finch_oracle as fo
    from video_similarity_search_b200 import synth
    _lim, cores = use_all_cores()
    n, d, k, seed = synth.CONFIGS[args.workload]
    x, lab, _ = synth.gaussian_mixture(n, d, k, seed, return_labels=True)
    nn = within_component_neighbors(x, lab)
    sample = min(args.cpu_sample_rows, n)
    times, detail = [], None
    cpu_warmup = min(args.warmup, 1)     # (a CPU BLAS pass has nothing to warm beyond its first call; keeps the arm to minutes)
    rest_runs = []
    for i in range(cpu_warmup + args.steps):
        est, detail = cpu_reference_step(x, nn, sample, rest_runs)
        if i >= cpu_warmup:
            times.append(est)
    sec = statistics.mean(times)
    full = None
    if not args.no_full_nn and n * float(n) * d <= 7e13:
        # ONE complete pass of the level-0 stage (all rows x all columns): checks that scaling the sample is fair
        t0 = time.perf_counter()
        fo.first_neighbors_blocked(x)
        full = time.perf_counter() - t0
        detail["nn_stage_full_s"] = full
        detail["nn_stage_full_over_estimate"] = full / detail["nn_stage_est_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": n / sec, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "cpu_warmup_steps_run": cpu_warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(n, d, k, seed)},
        "finch_seconds": sec,
        "cpu_baseline": {"value": n / sec, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "level-0 NN stage on %d of %d query rows x all columns in every step, scaled linearly in "
                                   "rows; levels >= 1, components and means in full, timed in the first %d steps (their mean is "
                                   "reused by the later steps: deterministic work of ~15 s) - oracle port of finch.py with "
                                   "the exact-NN stand-in the reference needs above 70 000 rows; BLAS threads pinned to "
                                   "all %d host cores whatever OMP_NUM_THREADS says%s"
                                   % (sample, n, len(rest_runs), cores, "" if full is None else
                                      "; one full pass of the level-0 stage took %.1f s against %.1f s extrapolated"
                                      % (full, detail["nn_stage_est_s"])),
                         "detail": detail},
        "e2e": {"value": n / sec, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------
# GPU side
# --------------------------------------------------------------------------------------------------
_SAMPLER_SRC = r"""
import sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
         ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
         ("hw_power_brake_slowdown", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown)]
period, want_power = float(sys.argv[2]), sys.argv[3] == "1"
print("MAX", nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM), flush=True)
while True:
    try:
        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        print("S", time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
              nv.nvmlDeviceGetPowerUsage(h) / 1000.0 if want_power else -1.0, ",".join(n for n, b in names if mask & b), flush=True)
    except Exception:
        pass
    time.sleep(period)
"""


def has_stalled_call(host_ms_per_call, factor=2.5):
    """The re-measurement rule of the timed loops: one call took more than `factor` x the median call."""
    return len(host_ms_per_call) >= 3 and max(host_ms_per_call) > factor * statistics.median(host_ms_per_call)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, c, num_clust, max_bytes=DUMP_BYTES):
    """Write what FINCH returned to its caller as float64 .npy files (labels are integers, exact in float64):
    c.npy [N, P] and num_clust.npy [P].  When the label matrix would take the files over `max_bytes`, c.npy holds a
    fixed sample of its rows (seed 0, ascending) and c_rows.npy their indices."""
    os.makedirs(out_dir, exist_ok=True)
    c = np.asarray(c)
    arrays = {"num_clust": np.asarray(num_clust, dtype=np.float64)}
    room = max_bytes - arrays["num_clust"].nbytes
    if c.size * 8 <= room:
        arrays["c"] = c.astype(np.float64)
    else:
        rows = np.sort(np.random.default_rng(0).choice(c.shape[0], room // (8 * (c.shape[1] + 1)), replace=False))
        arrays["c"] = c[rows].astype(np.float64)
        arrays["c_rows"] = rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region by a SEPARATE process (NVML polled every
    ~5 ms; nvidia-smi -lms 100 as the fallback when pynvml cannot initialise).  A separate process keeps the polling off
    this process's GIL and driver locks; scripts/sampler_probe.py measured the step time at 8 GPUs with and without it
    (5 / 20 / 100 ms periods, with and without the power query): no difference beyond run-to-run noise (6.35-6.6 ms)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_s=None, power=None):
        self.gpu_index = gpu_index
        self.proc = None
        self.kind = None
        self.t0 = self.t1 = None
        # SLIC_BENCH_SAMPLER="<period in ms>[,nopower]" overrides (experiments: scripts/sampler_probe.py)
        env = os.environ.get("SLIC_BENCH_SAMPLER", "")
        self.period_s = period_s if period_s is not None else (float(env.split(",")[0]) * 1e-3 if env else 0.005)
        self.power = power if power is not None else ("nopower" not in env)

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.gpu_index < len(ids) and ids[self.gpu_index].isdigit():
                return int(ids[self.gpu_index])
        return self.gpu_index

    def launch(self):
        """Start the sampling process (call well before the timed region: the interpreter takes a moment to come up)."""
        env = dict(os.environ)
        env.pop("CUDA_VISIBLE_DEVICES", None)
        try:
            import pynvml  # noqa: F401  (only to know that the child can import it)
            self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, str(self._physical_index()), str(self.period_s),
                                          "1" if self.power else "0"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True, env=env)
            self.kind = "nvml"
            first = self.proc.stdout.readline()          # "MAX <mhz>": the child is up and polling
            if first.startswith("MAX"):
                self.max_mhz = float(first.split()[1])
                return
            self.proc.kill()                             # (NVML did not initialise in the child)
            self.proc = None
        except Exception:
            self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.kind = "smi"
        except Exception:
            self.proc = None

    def start(self):
        if self.proc is None:
            self.launch()
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no sampler (pynvml and nvidia-smi unavailable)"]}
        time.sleep(0.02)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        if self.kind == "nvml":
            sm, power, reasons = [], [], set()
            for ln in out.splitlines():
                f = ln.split()
                if len(f) < 4 or f[0] != "S":
                    continue
                t = float(f[1])
                if t < self.t0 or t > self.t1:
                    continue
                sm.append(float(f[2]))
                if float(f[3]) >= 0:
                    power.append(float(f[3]))
                if len(f) > 4:
                    reasons.update(v for v in f[4].split(",") if v)
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm),
                    "power_w_max": max(power) if power else None, "reasons": sorted(reasons),
                    "how": "NVML polled every %g ms by a separate process during the timed steps" % (self.period_s * 1e3)}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "how": "nvidia-smi -lms 100 during the timed steps"}


def device_mixture(torch, n, d, k, seed, device):
    """Gaussian mixture generated ON the device (same Philox stream on every rank): the C5 shapes (4 GB per matrix)
    would otherwise cost every rank minutes of numpy time and 8 GB of host memory."""
    g = torch.Generator(device=device).manual_seed(seed)
    centres = torch.randn(k, d, device=device, generator=g)
    out = torch.empty(n, d, device=device)
    for s in range(0, n, 65536):
        e = min(n, s + 65536)
        lab = torch.randint(0, k, (e - s,), device=device, generator=g)
        out[s:e] = centres[lab] + torch.randn(e - s, d, device=device, generator=g)
    return out, centres


def retrieval_record(torch, be, lib, peaks, q, x, k, steps, world, label, check_exact):
    """Top-k retrieval (iic_retrieve_clips.py:295-296 / evaluate.py:226-231 shape) through the tensor-core screen:
    CUDA-event time of the whole call (normalise + screen + exact re-rank + sort), the screen kernel alone, and the
    fraction of the tensor peak.  world > 1: query rows sharded over the ranks, ids all-gathered."""
    import torch.distributed as dist
    from video_similarity_search_b200 import _lib
    from video_similarity_search_b200.sharded import topk_neighbors_sharded

    def call():
        if world > 1:
            return topk_neighbors_sharded(q, x, k, backend=be)
        return be.topk_neighbors(q, x, k)

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    lib.slic_profile_screen(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    per_call = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = call()                 # (synchronises internally: the candidate counters are read back)
        per_call.append((time.perf_counter() - t0) * 1e3)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    kms, fl = ctypes.c_float(0), ctypes.c_double(0)
    _lib.check(lib.slic_last_screen_time(ctypes.byref(kms), ctypes.byref(fl)), "slic_last_screen_time")
    lib.slic_profile_screen(0)
    if world > 1:
        t = torch.tensor([ms, kms.value], dtype=torch.float64, device=be.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, kernel_ms = float(t[0]), float(t[1])
    else:
        kernel_ms = kms.value
    nq, n, d = q.shape[0], x.shape[0], x.shape[1]
    d_pad = (d + 63) // 64 * 64
    tf = fl.value / (kernel_ms * 1e-3) / 1e12          # this rank's share of 2 Q N d over its kernel time
    rec = {"shape": "%d queries x %d database x %d, k=%d" % (nq, n, d, k), "ms": ms, "queries_per_s": nq / (ms * 1e-3),
           "screen_kernel_ms": kernel_ms, "screen_tflops_per_gpu": tf, "frac_of_peak": tf / peaks["bf16_tflops"],
           "flop_per_launch": fl.value, "d_pad": d_pad, "n_gpus": world, "data": label,
           "host_ms_per_call_min_median_max": [min(per_call), statistics.median(per_call), max(per_call)]}
    if check_exact and world == 1:
        # identical indices from the exact float64-accumulating kernels (no screen): the parity of the top-k path
        ux, _ = be.normalize_rows(x, want_f16=False)
        uq, _ = be.normalize_rows(q, want_f16=False)
        ei, _ = be.topk_cosine(uq, ux, k)
        rec["indices_equal_exact_kernels"] = bool(torch.equal(ei, out[0]))
    return rec


def run_b200(args):
    import torch
    import torch.distributed as dist
    from video_similarity_search_b200 import _lib, synth
    from video_similarity_search_b200.backend import CudaBackend
    from video_similarity_search_b200.clustering.finch import FINCH
    from video_similarity_search_b200.sharded import FINCH_sharded, sharded_first_neighbors

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    be = CudaBackend()
    lib = _lib.load()

    n, d, k, seed = synth.CONFIGS[args.workload]
    big = args.workload == "C5"     # generated on the device; no host copy per rank (see device_mixture)
    if big:
        x_dev, centres_dev = device_mixture(torch, n, d, k, seed, be.device)
        x_host = x_pinned = None
    else:
        x_host, lab_host, _ = synth.gaussian_mixture(n, d, k, seed, return_labels=True)
        x_pinned = torch.from_numpy(x_host).pin_memory()
        x_dev = x_pinned.to(be.device, non_blocking=True)
    torch.cuda.synchronize()
    search = sharded_first_neighbors(be) if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=be.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps):
        """EXACTLY `steps` calls between barrier+synchronize, CUDA events on the current stream, max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        walls.clear()
        for _ in range(steps):
            t0 = time.perf_counter()
            out = fn()
            walls.append((time.perf_counter() - t0) * 1e3)     # (host clock per call: shows a single stalled step)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, out

    walls = []

    def step_resident():
        return FINCH(x_dev, verbose=False, backend=be, first_neighbors=search)

    def host_step(src):
        # the call a reference user makes: host matrix in, numpy out (H2D of the embeddings, D2H of the labels inside).
        # N > 1: FINCH_sharded - every rank uploads 1 / N of the rows and an all-gather over NVLink assembles the matrix
        if world > 1:
            return lambda: FINCH_sharded(src, verbose=False, backend=be)
        return lambda: FINCH(src, verbose=False, backend=be)

    def step_nn_only():
        return (search(x_dev) if search else be.first_neighbors(x_dev))

    def warm(fn, k):
        """k untimed calls with the holding pattern of timed(): the previous result stays alive while the next is computed.
        FINCH delivers its label matrix in page-locked buffers that are reused once the caller has dropped the result
        (backend.PinnedResultPool), so the steady state of such a loop needs two of them - a buffer allocated inside a
        timed region (cudaHostAlloc of 31 MB: 14 ms) would be start-up cost booked as step time."""
        out = None
        for _ in range(k):
            out = fn()
        barrier()      # (N > 1: the first barrier of a process has start-up work of its own - seen as a 55 ms first timed call
        return out     #  at 2 GPUs when timed() was the first to issue one)

    warmup = max(args.warmup, 3)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.launch()             # (separate process; comes up during the warm-up steps)
    warm(step_resident, warmup)      # (also builds the stream-ordered memory pool)
    # Multi-GPU: the first steps after start-up run slower than the steady state whatever is timed - measured at 8 GPUs
    # (scripts/sampler_probe.py): 7.75 ms per step for steps 4-8 of the process, 6.4-6.6 for the next 25, 6.35 from then on
    # (peer mappings, NVLink links and eight processes' allocator pools settling; the clock sampler was ruled out by the
    # same probe).  Extra UNTIMED settling steps at N > 1, reported in the line; the K timed steps are unchanged.
    settle = 12 if world > 1 else 0
    warm(step_resident, settle)
    if rank == 0:
        sampler.start()
    # One stalled call (a host hiccup: page reclaim under an allocation, a descheduled rank the peers then wait for - seen
    # in this harness as 0.1-0.9 s inside single calls of every one of the timed loops, before and after any change to
    # the library) turns K x 27 ms into a second.  Like the driver's own rule for clock anomalies such a measurement is
    # repeated ONCE and the first attempt stays in the line (`remeasured`); every rank takes the same decision.
    remeasured = {}

    def timed_checked(name, fn, steps, before=None):
        if before:
            before()
        ms, out = timed(fn, steps)
        stall = torch.tensor([1 if has_stalled_call(walls) else 0], dtype=torch.int32, device=be.device)
        if world > 1:
            dist.all_reduce(stall, op=dist.ReduceOp.MAX)
        if int(stall.item()):
            remeasured[name] = {"first_attempt_ms_per_step": ms, "first_attempt_host_ms_per_call_rank0": [round(v, 3) for v in walls],
                                "rule": "a call took more than 2.5 x the median call on some rank: measured again, once"}
            del out
            warm(fn, 2)
            if before:
                before()
            ms, out = timed(fn, steps)
        return ms, out

    mark = {}
    ms_step, result = timed_checked("resident", step_resident, args.steps,
                                    before=lambda: mark.__setitem__("launches0", lib.slic_launch_count()))
    launches0 = mark["launches0"]
    step_walls = [round(v, 3) for v in walls]
    launches = (lib.slic_launch_count() - launches0)
    clocks = sampler.stop() if rank == 0 else None
    c, num_clust, _ = result

    # dominant kernel: per-launch CUDA-event time of nn_screen_kernel at level 0 (events recorded around the kernel on its
    # stream; the level-0 call is the only screen launch in step_nn_only)
    lib.slic_profile_screen(1)
    screen_ms = []
    flop, exec_flop = ctypes.c_double(0), ctypes.c_double(0)
    for _ in range(args.steps):
        step_nn_only()
        ms = ctypes.c_float(0)
        _lib.check(lib.slic_last_screen_time(ctypes.byref(ms), ctypes.byref(flop)), "slic_last_screen_time")
        _lib.check(lib.slic_last_screen_exec_flop(ctypes.byref(exec_flop)), "slic_last_screen_exec_flop")
        screen_ms.append(ms.value)
    lib.slic_profile_screen(0)
    screen_ms_avg = max_over_ranks(statistics.mean(screen_ms))
    screen_ms_ranks = None
    if world > 1:      # every rank's own kernel time: the shares are equal in tiles, the slowest rank sets the stage's time
        mine = torch.tensor([statistics.mean(screen_ms)], dtype=torch.float64, device=be.device)
        every = torch.empty(world, dtype=torch.float64, device=be.device)
        dist.all_gather_into_tensor(every, mine)
        screen_ms_ranks = [round(v, 4) for v in every.cpu().tolist()]

    def nn_only_dropped():
        step_nn_only()     # (results dropped at once: keeping one alive while the next is computed makes the framework's
        return None        #  allocator grow by 0.7 GB of unit rows per call until its cache has settled)

    for _ in range(2):
        nn_only_dropped()
    ms_nn, _ = timed_checked("nn_stage", nn_only_dropped, args.steps)
    # everything after the level-0 search (components, means, all further levels, labels to the host): one FINCH call
    # with the level-0 neighbours handed in
    cached = step_nn_only()
    tail_step = lambda: FINCH(x_dev, verbose=False, backend=be, first_neighbors=lambda m: cached)   # noqa: E731
    warm(tail_step, 3)   # (with caller-supplied neighbours the driver sizes its buffers for n clusters - pool growth)
    ms_tail, _ = timed_checked("tail", tail_step, args.steps)
    del cached, _
    ms_e2e = ms_e2e_pageable = None
    if not big:
        warm(host_step(x_pinned), 3)
        ms_e2e, _ = timed_checked("e2e", host_step(x_pinned), args.steps)
        del _
        warm(host_step(x_host), 3)
        ms_e2e_pageable, _ = timed_checked("e2e_pageable", host_step(x_host), args.steps)
        del _

    sharded_equal = None
    if world > 1:
        # parity of the exchange step, outside the timed region: the merged multi-GPU first neighbours must equal the
        # single-GPU search of the same matrix on this rank, bit for bit (indices and float32 distances)
        nn_s, d_s, _ = search(x_dev)
        nn_1, d_1, _ = be.first_neighbors(x_dev)
        ok = torch.tensor([int(torch.equal(nn_s, nn_1) and torch.equal(d_s, d_1))], device=be.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        sharded_equal = bool(ok.item())

    peaks = load_peaks()
    retrieval = None
    if not args.no_retrieval:
        retrieval = {}
        if not big:
            tr, _, te, _ = synth.c2_retrieval()
            retrieval["C2_top50"] = retrieval_record(torch, be, lib, peaks, be.to_device(te), be.to_device(tr), 50,
                                                     args.steps, world, "BASELINE configs[1], host-generated", True)
        if big or (world == 1 and args.workload == "C3"):
            if big:
                xq = x_dev
                cen = centres_dev
            else:
                xq, cen = device_mixture(torch, 1000000, 1024, 1000, 0, be.device)
            g = torch.Generator(device=be.device).manual_seed(1)
            q5 = cen[torch.randint(0, cen.shape[0], (C5_QUERIES,), device=be.device, generator=g)] + \
                torch.randn(C5_QUERIES, cen.shape[1], device=be.device, generator=g)
            retrieval["C5_top50"] = retrieval_record(torch, be, lib, peaks, q5, xq, 50, args.steps, world,
                                                     "BASELINE configs[4] retrieval shape (Q not fixed by BASELINE: 100 000), "
                                                     "device-generated mixture", False)
            del q5
            if not big:
                del xq
                torch.cuda.empty_cache()

    if world > 1:
        from video_similarity_search_b200.sharded import close_peer_groups
        close_peer_groups()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    exec_tf = exec_flop.value / (screen_ms_avg * 1e-3) / 1e12
    algo_tf = flop.value / (screen_ms_avg * 1e-3) / 1e12
    d_pad = (d + 63) // 64 * 64
    traffic = NCU_TRAFFIC.get((args.workload, world))
    if world == 1:
        par = "1 GPU"
    else:
        par = ("level-0 NN: the %d ranks share the tiles of the symmetric screen's triangle through NVLink peer windows "
               "(csrc/comm.cu): ONE screen kernel per rank publishes its pre-pass row bests into every rank's memory (red.max) "
               "and ONE merge kernel reads the ranks' (distance, neighbour) keys in place - no collective call on the critical "
               "path of the resident step (two flag barriers in device memory); levels >= 1 replicated on every rank; e2e adds "
               "one NCCL all-gather of the rows each rank uploaded (1/%d of the matrix per rank over PCIe)" % (world, world))
    line = {
        "metric": METRIC, "value": n / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "settle_steps_untimed": settle, "ms_per_step": ms_step, "step_host_ms_rank0": step_walls,
        "remeasured": remeasured or None, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f16 screen (f32 accumulate) + f32/f64 exact re-rank", "data": "synthetic",
        "config": {"workload": workload_string(n, d, k, seed),
                   "l2": "inputs exceed L2 (%.0f MB fp32 + %.0f MB fp16 per step)" % (n * d * 4 / 1e6, n * d_pad * 2 / 1e6),
                   "partitions": [int(v) for v in num_clust],
                   "parallelism": par,
                   "data_source": "device-generated (torch Philox, same stream on every rank)" if big else "numpy, seeded"},
        "finch_seconds": ms_step * 1e-3,
        "nn_stage": {"ms": ms_nn, "queries_per_s": n / (ms_nn * 1e-3)},
        "tail_ms_given_level0_neighbours": ms_tail,
        "gpu_launches": int(launches), "gpu_launches_per_step": launches / float(args.steps),
        "clocks": clocks,
        "roofline": {"kernel": "nn_screen_kernel (level 0, %d x %d x %d%s)" % (n, n, d_pad, "" if world == 1 else
                                                                               ", this rank's 1/%d of the tiles" % world),
                     "bound": "tensor", "achieved": exec_tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": exec_tf / peaks["bf16_tflops"],
                     "peak_source": peaks["source"] + " burst dense bf16 (cuBLAS; float16 operands run at the same rate)",
                     "frac_of_sustained": (exec_tf / peaks["bf16_tflops_sustained"]) if peaks.get("bf16_tflops_sustained") else None,
                     "kernel_ms": screen_ms_avg, "kernel_ms_per_rank": screen_ms_ranks, "flop_per_launch": exec_flop.value,
                     # the ALGORITHMIC figure of SURVEY.md 8(d) (full square, no symmetry discount) - not a hardware rate
                     "algorithmic_flop_per_launch": flop.value, "algorithmic_tflops": algo_tf,
                     "symmetry_gain": flop.value / exec_flop.value if exec_flop.value else None,
                     "traffic": traffic[0] if traffic else None,
                     "traffic_source": (traffic[1] + "; constant from that capture, not re-measured per run") if traffic else
                                       "no ncu capture for this (workload, ranks)",
                     "traffic_unit": "bytes/launch (ncu dram read+write)"},
    }
    if ms_e2e is not None:
        h2d, d2h = int(n * d * 4), int(c.size * 4 * world)
        # whole job: every rank uploads its 1 / N share of the rows (the rest arrives over NVLink); labels back per rank
        line["e2e"] = {"value": n / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "source": "pinned host memory"}
        line["e2e_pageable"] = {"value": n / (ms_e2e_pageable * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e_pageable,
                                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                "source": "plain numpy array (pageable), as clustering/cluster_masks.py:80 hands it over"}
    else:
        line["e2e"] = None
        line["e2e_note"] = "C5 is generated on the device (8 x 4 GB of host staging avoided): no host-buffer leg"
    if retrieval is not None:
        line["retrieval"] = retrieval

    parity = {}
    if world == 1:
        from oracle import finch_oracle as fo
        # (1) EVERY row: the tensor-core path against the exact float64-accumulating kernel (no screen)
        nn_dev, dist_dev, unit = be.first_neighbors(x_dev)
        t0 = time.perf_counter()
        exact_rows = n if not big else 65536
        rows_t = None
        if exact_rows == n:
            nn_ex, _ = be.nn_exact_top1(unit, unit, self_offset=0)
            same = bool(torch.equal(nn_ex, nn_dev))
            mism = int((nn_ex != nn_dev).sum())
        else:
            rows_t = torch.linspace(0, n - 1, exact_rows, device=be.device).long().to(torch.int32)
            nn_ex, _ = be.nn_exact_top1(unit, unit, self_offset=0, q_rows=rows_t)
            mism = int((nn_ex != nn_dev[rows_t.long()]).sum())
            same = mism == 0
        torch.cuda.synchronize()
        parity["first_neighbors_tc_equals_exact_kernel"] = {"rows_checked": int(exact_rows), "of": n, "equal": same,
                                                            "mismatches": mism, "seconds": time.perf_counter() - t0}
        del nn_ex
        if x_host is None:
            x_host = x_dev.cpu().numpy()
        nn_host = nn_dev.cpu().numpy().astype(np.int64)
        if not args.no_cpu_baseline:
            _lim, cores = use_all_cores()
            # (2) oracle first neighbours (the reference's arithmetic, blocked) on a row sample; the first
            #     `cpu_sample_rows` of them are also the timed CPU sample
            prow = min(args.parity_rows if not big else 2048, n)
            sample = min(args.cpu_sample_rows, prow)
            rows = np.linspace(0, n - 1, prow).astype(np.int64)
            t0 = time.perf_counter()
            enn_a, _, gap_a = fo.first_neighbors_blocked(x_host, rows=rows[:sample])
            t_nn = time.perf_counter() - t0
            if prow > sample:
                enn_b, _, gap_b = fo.first_neighbors_blocked(x_host, rows=rows[sample:])
                enn, gap = np.concatenate([enn_a, enn_b]), np.concatenate([gap_a, gap_b])
            else:
                enn, gap = enn_a, gap_a
            clear = gap > 2e-6
            parity["first_neighbors_equal_oracle"] = {
                "rows_checked": int(prow), "tie_margin": 2e-6, "tie_rows": int((~clear).sum()),
                "equal_outside_ties": bool(np.array_equal(nn_host[rows][clear], enn[clear])),
                "mismatches_incl_ties": int((nn_host[rows] != enn).sum())}
            # (3) levels >= 1: the oracle run from the GPU's level-0 neighbours must give the GPU's partition
            t0 = time.perf_counter()
            if n <= fo.FLANN_THRESHOLD:
                co, no, _ = fo.finch(x_host, nn0_override=nn_host)
            else:
                co, no, _ = fo.finch(x_host, initial_rank=nn_host)
            t_rest = time.perf_counter() - t0
            parity["levels_ge1_equal_oracle_given_gpu_nn0"] = bool(no == num_clust and np.array_equal(co, c))
            est = t_nn * n / float(sample) + t_rest
            line["cpu_baseline"] = {
                "value": n / est, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "level-0 NN stage on %d of %d query rows x all columns (%.1f s), scaled linearly in rows; levels >= 1, "
                          "components and means timed in full (%.1f s) - oracle port of finch.py with the exact-NN stand-in the "
                          "reference needs above 70 000 rows; the reference arm (--impl reference) also runs the level-0 stage "
                          "once in full" % (sample, n, t_nn, t_rest),
                "finch_seconds_est": est}
    if sharded_equal is not None:
        parity["sharded_first_neighbors_equal_single_gpu_on_every_rank"] = sharded_equal
    line["parity"] = parity
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, c, num_clust)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
