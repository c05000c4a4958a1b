"""Device backend: thin torch-tensor wrappers over the C ABI (include/slic_b200.h).

torch supplies device memory and the current stream; every computation is a call into
libslic_b200.so.  There is no CPU implementation here - without a CUDA device `CudaBackend()`
raises.  (tests/fake_backend.py provides a numpy stand-in with the same method names so that the
host logic in clustering/finch.py can be exercised on a box without a GPU; it is test
infrastructure and is never selected by the product code.)
"""
import ctypes
import os
import sys
import threading
import time
import weakref

import numpy as np
import torch

from . import _lib

_DT = {torch.float32: _lib.SLIC_F32, torch.float64: _lib.SLIC_F64}

# below this many rows the tensor-core screen is pure launch overhead: use the exact kernel
SCREEN_MIN_ROWS = 2048
# the top-k screen keeps k running scores per row in shared memory (TC_TOPK_MAX in nn_screen_tc.cu)
TOPK_SCREEN_MAX_K = 64


def _p(t):
    return None if t is None else t.data_ptr()


def d_pad_of(d):
    return (d + 63) // 64 * 64


class PinnedResultPool:
    """Page-locked host buffers that results are DELIVERED in (no staging copy on the host side): take() hands out a
    numpy byte array backed by a pinned buffer; the buffer is reused only after that array - and every view of it,
    i.e. whatever the caller still holds of the result - has been garbage-collected (weak reference).  cudaHostAlloc
    costs 12-80 ms for the 31 MB of a 240 000-row hierarchy (measured), so buffers are kept: at most `keep` idle ones,
    and a caller who holds on to more than `keep` results gets ordinary right-sized copies from then on (deliver()),
    so that page-locked memory stays bounded.  `alloc` is injectable for tests without a GPU."""

    def __init__(self, keep=4, alloc=None):
        self._entries = []      # [buffer (uint8 tensor), weakref to the numpy array handed out | None]
        self._keep = keep
        self._lock = threading.Lock()   # (a backend may be called from several host threads)
        self._alloc = alloc or (lambda nbytes: torch.empty(nbytes, dtype=torch.uint8, pin_memory=True))

    def take(self, nbytes):
        """-> (numpy uint8 [nbytes] in page-locked memory, its address)."""
        with self._lock:
            return self._take(nbytes)

    def _take(self, nbytes):
        free = [e for e in self._entries if e[1] is None or e[1]() is None]
        fit = [e for e in free if e[0].numel() >= nbytes]
        if fit:
            entry = min(fit, key=lambda e: e[0].numel())
        else:
            drop = free[max(self._keep - 1, 0):]             # idle buffers that are too small: let them go
            self._entries = [e for e in self._entries if not any(e is x for x in drop)]
            t0 = time.perf_counter()
            entry = [self._alloc(max(int(nbytes), 1 << 22)), None]
            self._entries.append(entry)
            if os.environ.get("SLIC_POOL_TRACE"):
                print("[slic] result pool: new page-locked buffer of %.1f MB in %.2f ms (%d buffers, %d busy)"
                      % (entry[0].numel() / 1e6, (time.perf_counter() - t0) * 1e3, len(self._entries),
                         sum(1 for e in self._entries if e[1] is not None and e[1]() is not None)), file=sys.stderr, flush=True)
        arr = entry[0].numpy()
        entry[1] = weakref.ref(arr)
        return arr[:nbytes], entry[0].data_ptr()

    def deliver(self, view):
        """The result as the caller receives it: the view of the page-locked buffer itself, or - when more than `keep`
        buffers are out with callers - a copy in ordinary memory (the buffer is free again once `view` is dropped)."""
        busy = sum(1 for e in self._entries if e[1] is not None and e[1]() is not None)
        return view.copy() if busy > self._keep else view


class CudaBackend:
    name = "cuda"

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("video_similarity_search_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.lib = _lib.load()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.slic_require_device(), "slic_require_device")
        self.last_stats = None
        self._stage = None
        self._results = PinnedResultPool()
        self._multi = None

    # -- plumbing ------------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def to_device(self, array, dtype=None):
        t = torch.as_tensor(array)
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        if t.device.type == "cpu" and not t.is_pinned() and t.numel() * t.element_size() >= (8 << 20):
            # a large pageable host array (plain numpy): slic_copy_to_device stages it through pinned buffers with
            # several host threads - about 3x the rate of the driver's single-threaded staging behind tensor.to()
            t = t.contiguous()
            out = torch.empty(t.shape, dtype=t.dtype, device=self.device)
            self.copy_to_device(out, t)
            return out
        return t.to(self.device, non_blocking=True).contiguous()

    def copy_to_device(self, dst, src_host):
        """dst (device tensor, contiguous) <- src_host (CPU tensor, contiguous, same bytes), on the current stream."""
        nbytes = src_host.numel() * src_host.element_size()
        assert dst.is_contiguous() and src_host.is_contiguous() and dst.numel() * dst.element_size() == nbytes
        with torch.cuda.device(self.device):
            _lib.call("slic_copy_to_device", _p(dst), src_host.data_ptr(), nbytes, self._stream())

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def to_host(self, t):
        """Device -> numpy through a pinned staging buffer (a pageable D2H of the [N, P] label matrix costs
        milliseconds; pinned it is PCIe-bound)."""
        nbytes = t.numel() * t.element_size()
        if nbytes < (1 << 16):
            return t.cpu().numpy()
        t = t.contiguous()
        if self._stage is None or self._stage.numel() < nbytes:      # grow-only pinned staging (cudaHostAlloc is ~1 ms)
            self._stage = torch.empty(max(nbytes, 1 << 22), dtype=torch.uint8, pin_memory=True)
        stage = self._stage[:nbytes].view(t.dtype).view(t.shape)
        stage.copy_(t, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return stage.numpy().copy()

    # -- K1 --------------------------------------------------------------------------------------
    def normalize_rows(self, x, want_f16=True):
        """-> (unit [n,d] same dtype, unit_f16 [n,d_pad] or None)."""
        n, d = x.shape
        unit = torch.empty_like(x)
        dp = d_pad_of(d)
        ub = torch.empty((n, dp), dtype=torch.float16, device=x.device) if want_f16 else None
        _lib.call("slic_normalize_rows", _p(x), n, d, _DT[x.dtype], _p(unit), None, _p(ub), dp, self._stream())
        return unit, ub

    def center_columns(self, x):
        """x - x.mean(dim=0, keepdim=True) for a float32 matrix (slic_center_columns)."""
        out = torch.empty_like(x)
        _lib.call("slic_center_columns", _p(x), x.shape[0], x.shape[1], _p(out), None, self._stream())
        return out

    def nn_exact_top1(self, q_unit, x_unit, self_offset=-1, q_rows=None):
        nq = q_unit.shape[0] if q_rows is None else q_rows.shape[0]
        n, d = x_unit.shape
        idx = torch.empty(nq, dtype=torch.int32, device=x_unit.device)
        dist = torch.empty(nq, dtype=x_unit.dtype, device=x_unit.device)
        _lib.call("slic_nn_exact_top1", _p(q_unit), _p(q_rows), nq, _p(x_unit), n, d, _DT[x_unit.dtype],
                  self_offset, _p(idx), _p(dist), self._stream())
        return idx, dist

    def nn_top1(self, q_unit, q_f16, x_unit, x_f16, self_offset=-1, eps=0.0):
        """tcgen05 screen + exact re-rank (slic_nn_top1)."""
        nq = q_unit.shape[0]
        n, d = x_unit.shape
        idx = torch.empty(nq, dtype=torch.int32, device=x_unit.device)
        dist = torch.empty(nq, dtype=x_unit.dtype, device=x_unit.device)
        stats = torch.zeros(4, dtype=torch.int32, device=x_unit.device)
        _lib.call("slic_nn_top1", _p(q_unit), _p(q_f16), nq, _p(x_unit), _p(x_f16), n, d, x_f16.shape[1],
                  _DT[x_unit.dtype], self_offset, float(eps), _p(idx), _p(dist), _p(stats), self._stream())
        self.last_stats = stats
        return idx, dist

    def first_neighbors(self, x, row_range=None):
        """First neighbour of every row of x (or of rows [r0, r1)) among all rows of x, self excluded.
        -> (nn int32, dist x.dtype, unit).  Chooses the screen for large inputs, the exact kernel below."""
        n = x.shape[0]
        use_screen = n >= SCREEN_MIN_ROWS
        unit, ub = self.normalize_rows(x, want_f16=use_screen)
        r0, r1 = (0, n) if row_range is None else row_range
        if r1 <= r0:
            return (torch.empty(0, dtype=torch.int32, device=x.device), torch.empty(0, dtype=x.dtype, device=x.device),
                    unit)
        if use_screen:
            nn, dist = self.nn_top1(unit[r0:r1], ub[r0:r1], unit, ub, self_offset=r0)
        else:
            nn, dist = self.nn_exact_top1(unit[r0:r1], unit, self_offset=r0)
        return nn, dist, unit

    # rows from which the self-search runs on the symmetric screen (SYM_MIN_ROWS_FWD in csrc/nn_screen_tc.cu)
    SYM_MIN_ROWS = 16384

    def supports_triangle_parts(self, x):
        """True when the multi-process share of the symmetric self-search applies (level 0: float32, large n)."""
        return x.dtype == torch.float32 and x.shape[0] >= self.SYM_MIN_ROWS

    def first_neighbors_part(self, x, part, parts, reduce_max=None):
        """This process's share of the symmetric first-neighbour search of all rows of x.
        reduce_max: callable applying an element-wise MAX over the parts to an int32 device tensor in place (the
        all-reduce).  Given it, the search runs in two phases - slic_sym_row_bests on this part's rows, the exchange,
        then slic_nn_top1_sym_part seeded with every row's best - so that the candidate filter starts tight on every
        part; without it each part runs its own pre-pass over all rows (single-process use / tests).
        -> (keys int64 [n + 1], unit): keys[i] = (distance bits << 32) | neighbour for the best pair this part saw,
        keys[n] = completeness flag; an element-wise MIN over the parts merges them."""
        n, d = x.shape
        unit, ub = self.normalize_rows(x, want_f16=True)
        bests = None
        if reduce_max is not None and parts > 1:
            bests = torch.empty(n, dtype=torch.int32, device=x.device)
            _lib.call("slic_sym_row_bests", _p(unit), _p(ub), n, d, ub.shape[1], int(part), int(parts), _p(bests),
                      self._stream())
            reduce_max(bests)
        keys = torch.empty(n + 1, dtype=torch.int64, device=x.device)
        stats = torch.zeros(4, dtype=torch.int32, device=x.device)
        _lib.call("slic_nn_top1_sym_part", _p(unit), _p(ub), n, d, ub.shape[1], int(part), int(parts), _p(bests), 0.0,
                  _p(keys), _p(stats), self._stream())
        self.last_stats = stats
        return keys, unit

    # -- peer windows (csrc/comm.cu): one process per GPU -----------------------------------------------
    def comm_window_create(self, max_rows):
        """-> (comm handle, 64-byte IPC handle of this rank's window as bytes)."""
        comm = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        with torch.cuda.device(self.device):
            _lib.call("slic_comm_window_create", int(max_rows), ctypes.addressof(comm), ctypes.addressof(handle))
        return comm, bytes(handle)

    def comm_connect(self, comm, rank, world, all_handles):
        buf = (ctypes.c_ubyte * (64 * world)).from_buffer_copy(all_handles)
        with torch.cuda.device(self.device):
            _lib.call("slic_comm_connect", comm, int(rank), int(world), ctypes.addressof(buf))

    def comm_destroy(self, comm):
        _lib.call("slic_comm_destroy", comm)

    def comm_first_neighbors(self, comm, x):
        """Level-0 first neighbours of all rows of x, the O(N^2 D) stage shared by the ranks connected through `comm`
        (slic_comm_nn_top1: every rank calls it with the same matrix).  -> (nn, dist, unit, status) with status a
        device int32[2] = {rows without a neighbour, incomplete flag}; nothing here waits for the device."""
        n, d = x.shape
        unit, ub = self.normalize_rows(x, want_f16=True)
        nn = torch.empty(n, dtype=torch.int32, device=x.device)
        dist = torch.empty(n, dtype=torch.float32, device=x.device)
        status = torch.empty(2, dtype=torch.int32, device=x.device)
        _lib.call("slic_comm_nn_top1", comm, _p(unit), _p(ub), n, d, ub.shape[1], _p(nn), _p(dist), _p(status), self._stream())
        return nn, dist, unit, status

    def _labels_sink(self, n, cap, device, host_labels):
        """Destination of a hierarchy's [N, P] label matrix: device memory, or (host_labels) a page-locked host buffer
        that the last kernel of the hierarchy writes over PCIe - the labels are then on the host when the call returns.
        -> (address for the C ABI, finish(p) -> the [N, P] matrix, keep-alive)."""
        if host_labels:
            try:
                arr, addr = self._results.take(n * cap * 4)
                return addr, (lambda p: self._results.deliver(arr[: n * p * 4].view(np.int32).reshape(n, p))), arr
            except RuntimeError:      # no page-locked memory to be had: device buffer, then the staged copy of to_host()
                pass
        labels = torch.empty(n * cap, dtype=torch.int32, device=device)
        if host_labels:
            return _p(labels), (lambda p: self.to_host(labels[: n * p].view(n, p))), labels
        return _p(labels), (lambda p: labels[: n * p].view(n, p)), labels

    def finch_native_comm(self, comm, data, ensure_early_exit=True, host_labels=False):
        """slic_comm_finch: the whole hierarchy with the level-0 search shared by the ranks connected through `comm`
        (every rank calls it with the same device matrix).  -> as finch_native."""
        n, d = data.shape
        cap = self.FINCH_CAPACITY
        sink, finish, _keep = self._labels_sink(n, cap, data.device, host_labels)
        num = (ctypes.c_int32 * cap)()
        levels, has = ctypes.c_int32(0), ctypes.c_int32(0)
        ms = ctypes.c_float(0)
        _lib.call("slic_comm_finch", comm, _p(data), n, d, int(bool(ensure_early_exit)), cap, sink,
                  ctypes.addressof(num), ctypes.addressof(levels), ctypes.addressof(ms), ctypes.addressof(has), self._stream())
        p = levels.value
        return finish(p), [int(v) for v in num[:p]], (np.float32(ms.value) if has.value else None)

    # -- rank-0-driven multi-GPU FINCH (csrc/comm.cu): one process, all GPUs of the box -------------------
    def enable_multi_gpu(self, devices=None, max_rows=1 << 21):
        """From now on finch_host() - i.e. FINCH(host matrix) - shares the level-0 search among `devices` (default:
        every visible GPU) through slic_finch_multi; the first device of the list runs levels >= 1.  The call site
        (online_train.py:619-627: rank 0 clusters, the other ranks wait) stays as it is."""
        if devices is None:
            devices = list(range(torch.cuda.device_count()))
        devices = [int(torch.device(v).index) if not isinstance(v, int) else v for v in devices]
        self.disable_multi_gpu()
        if len(devices) < 2:
            return
        arr = (ctypes.c_int32 * len(devices))(*devices)
        comm = ctypes.c_void_p()
        _lib.call("slic_comm_create", ctypes.addressof(arr), len(devices), int(max_rows), ctypes.addressof(comm))
        self._multi = (comm, devices, int(max_rows))

    def disable_multi_gpu(self):
        multi = getattr(self, "_multi", None)
        if multi is not None:
            _lib.call("slic_comm_destroy", multi[0])
        self._multi = None

    def multi_gpu_timeline(self):
        """ms of the last multi-GPU finch_host call: (upload + forward, normalise + search, whole call)."""
        out = (ctypes.c_float * 3)()
        _lib.call("slic_comm_last_timeline", self._multi[0], ctypes.addressof(out))
        return tuple(out)

    def unpack_neighbor_keys(self, keys):
        """Merged keys [n + 1] -> (nn int32 [n], dist float32 [n], complete bool).  One host read-back."""
        n = keys.shape[0] - 1
        nn = torch.empty(n, dtype=torch.int32, device=keys.device)
        dist = torch.empty(n, dtype=torch.float32, device=keys.device)
        status = torch.empty(1, dtype=torch.int32, device=keys.device)
        _lib.call("slic_unpack_neighbor_keys", _p(keys), n, _p(nn), _p(dist), _p(status), self._stream())
        flags = torch.stack((keys[n], status[0].to(torch.int64))).tolist()
        return nn, dist, flags[0] == 1 and flags[1] == 0

    def screen_scores_debug(self, q_f16, x_f16):
        nq, n = q_f16.shape[0], x_f16.shape[0]
        out = torch.zeros((nq, n), dtype=torch.float32, device=x_f16.device)
        _lib.call("slic_screen_scores_debug", _p(q_f16), nq, _p(x_f16), n, x_f16.shape[1], _p(out), self._stream())
        return out

    def distance_matrix(self, q, x, metric="cosine", same=False):
        nq, d = q.shape
        n = x.shape[0]
        out = torch.empty((nq, n), dtype=x.dtype, device=x.device)
        m = _lib.SLIC_METRIC_COSINE if metric == "cosine" else _lib.SLIC_METRIC_EUCLIDEAN
        _lib.call("slic_distance_matrix", _p(q), nq, _p(x), n, d, _DT[x.dtype], m, int(same), _p(out), n, self._stream())
        return out

    def rows_topk(self, mat, k):
        nq, n = mat.shape
        idx = torch.empty((nq, k), dtype=torch.int32, device=mat.device)
        val = torch.empty((nq, k), dtype=mat.dtype, device=mat.device)
        _lib.call("slic_rows_topk", _p(mat), nq, n, mat.stride(0), _DT[mat.dtype], k, _p(idx), _p(val), self._stream())
        return idx, val

    def topk_cosine(self, q_unit, x_unit, k, self_offset=-1, q_f16=None, x_f16=None, eps=0.0):
        """Top-k cosine neighbours, ascending distance, ties -> lowest column.  With the f16 copies of both
        sides and k <= 64 on a large database: tcgen05 screen + exact re-rank (slic_topk_cosine_tc);
        otherwise the exact kernels (slic_topk_cosine)."""
        nq, d = q_unit.shape
        n = x_unit.shape[0]
        idx = torch.empty((nq, k), dtype=torch.int32, device=x_unit.device)
        val = torch.empty((nq, k), dtype=x_unit.dtype, device=x_unit.device)
        if q_f16 is not None and x_f16 is not None and k <= TOPK_SCREEN_MAX_K and n >= SCREEN_MIN_ROWS:
            stats = torch.zeros(4, dtype=torch.int32, device=x_unit.device)
            _lib.call("slic_topk_cosine_tc", _p(q_unit), _p(q_f16), nq, _p(x_unit), _p(x_f16), n, d, x_f16.shape[1],
                      _DT[x_unit.dtype], k, self_offset, float(eps), _p(idx), _p(val), _p(stats), self._stream())
            self.last_stats = stats
            return idx, val
        _lib.call("slic_topk_cosine", _p(q_unit), nq, _p(x_unit), n, d, _DT[x_unit.dtype], k, self_offset, _p(idx),
                  _p(val), self._stream())
        return idx, val

    def topk_neighbors(self, q, x, k, same=False):
        """Normalise both sides (sklearn's normalize) and return their top-k cosine neighbours; picks the
        tensor-core path when the shape allows it.  same=True: q is x, self excluded."""
        use_screen = x.shape[0] >= SCREEN_MIN_ROWS and k <= TOPK_SCREEN_MAX_K
        ux, xb = self.normalize_rows(x, want_f16=use_screen)
        uq, qb = (ux, xb) if same else self.normalize_rows(q, want_f16=use_screen)
        return self.topk_cosine(uq, ux, k, self_offset=0 if same else -1, q_f16=qb, x_f16=xb)

    def hit_at_k(self, topk_idx, q_labels, x_labels, ks):
        ks_t = torch.tensor(list(ks), dtype=torch.int32, device=topk_idx.device)
        hits = torch.empty(len(ks), dtype=torch.int32, device=topk_idx.device)
        _lib.call("slic_hit_at_k", _p(topk_idx), topk_idx.shape[0], topk_idx.stride(0), _p(q_labels), _p(x_labels),
                  _p(ks_t), len(ks), _p(hits), self._stream())
        return hits

    # -- K2 --------------------------------------------------------------------------------------
    def components(self, nn, min_sim=None, unit=None, dist=None):
        """-> (labels int32 [n], num_clust python int).  Synchronises to read the count."""
        n = nn.shape[0]
        labels = torch.empty(n, dtype=torch.int32, device=nn.device)
        count = torch.empty(1, dtype=torch.int32, device=nn.device)
        use_filter = min_sim is not None
        d = unit.shape[1] if use_filter else 0
        dt = _DT[unit.dtype] if use_filter else 0
        _lib.call("slic_finch_components", _p(nn), n, int(use_filter), float(min_sim) if use_filter else 0.0,
                  _p(unit) if use_filter else None, d, dt, _p(dist) if use_filter else None, _p(labels), _p(count),
                  self._stream())
        c = int(count.item())
        if c < 0:      # the reference's sparse-matrix constructor raises on such indices (finch.py:41-43)
            raise ValueError("components: %d first-neighbour indices lie outside [0, n)" % -c)
        return labels, c

    def min_sim(self, nn, unit, dist):
        out = torch.empty(1, dtype=torch.float32, device=nn.device)
        _lib.call("slic_finch_min_sim", _p(nn), nn.shape[0], _p(unit), unit.shape[1], _DT[unit.dtype], _p(dist), _p(out),
                  self._stream())
        return out.cpu().numpy()[0]          # np.float32 scalar, as the reference holds it

    def closest_link(self, nn, unit, dist):
        out = torch.empty(2, dtype=torch.int32, device=nn.device)
        _lib.call("slic_finch_closest_link", _p(nn), nn.shape[0], _p(unit), unit.shape[1], _DT[unit.dtype], _p(dist),
                  _p(out), self._stream())
        i, j = out.tolist()
        return i, j

    # -- K3 --------------------------------------------------------------------------------------
    def compose_labels(self, prev, u):
        n = u.shape[0] if prev is None else prev.shape[0]
        out = torch.empty(n, dtype=torch.int32, device=u.device)
        _lib.call("slic_compose_labels", _p(prev), _p(u), n, _p(out), self._stream())
        return out

    def segmented_mean(self, data, labels, num_clust):
        n, d = data.shape
        out = torch.empty((num_clust, d), dtype=torch.float64, device=data.device)
        _lib.call("slic_segmented_mean", _p(data), _p(labels), n, d, num_clust, _p(out), self._stream())
        return out

    def cluster_sums(self, data, labels, num_clust):
        """-> (sums f64 [C,d], counts int32 [C], means f64 [C,d]) of the float32 rows (slic_cluster_sums)."""
        n, d = data.shape
        sums = torch.empty((num_clust, d), dtype=torch.float64, device=data.device)
        means = torch.empty((num_clust, d), dtype=torch.float64, device=data.device)
        counts = torch.empty(num_clust, dtype=torch.int32, device=data.device)
        _lib.call("slic_cluster_sums", _p(data), _p(labels), n, d, num_clust, _p(sums), _p(counts), _p(means),
                  self._stream())
        return sums, counts, means

    def merge_cluster_sums(self, sums_prev, counts_prev, u, num_clust):
        """Sums / counts / means of the next level from those of this one (slic_merge_cluster_sums)."""
        n_prev, d = sums_prev.shape
        sums = torch.empty((num_clust, d), dtype=torch.float64, device=sums_prev.device)
        means = torch.empty((num_clust, d), dtype=torch.float64, device=sums_prev.device)
        counts = torch.empty(num_clust, dtype=torch.int32, device=sums_prev.device)
        _lib.call("slic_merge_cluster_sums", _p(sums_prev), _p(counts_prev), _p(u), n_prev, d, num_clust, _p(sums),
                  _p(counts), _p(means), self._stream())
        return sums, counts, means

    # -- K6 spherical k-means (csrc/skmeans.cu) -------------------------------------------------------
    def kmeans_plusplus(self, unit, k, first_id, uniforms, n_local_trials):
        """k-means++ seeds of the float32 unit rows (slic_kmeans_plusplus).  uniforms: float64 [(k - 1) * L] host draws.
        -> int32 device tensor [k] of row indices."""
        n, d = unit.shape
        u = np.ascontiguousarray(uniforms, dtype=np.float64).reshape(-1)
        if u.size != (k - 1) * n_local_trials:
            raise ValueError("kmeans_plusplus: need (k - 1) * L uniforms")
        seeds = torch.empty(k, dtype=torch.int32, device=unit.device)
        _lib.call("slic_kmeans_plusplus", _p(unit), n, d, int(k), int(first_id), u.ctypes.data if u.size else None,
                  int(n_local_trials), _p(seeds), self._stream())
        return seeds

    def spherical_kmeans(self, x, k, init=None, first_ids=None, uniforms=None, n_local_trials=1, n_init=1, max_iter=300,
                         tol=1e-4):
        """The whole fit on the device (slic_spherical_kmeans).  x: float32 device [n, d] (raw rows); init: float32 device
        [k, d] or None; first_ids int64 [n_init] and uniforms float64 [n_init, (k - 1) * L]: the host draws.
        -> (labels int32 [n], centres float32 [k, d] (device tensors), inertia float, n_iter int, stats int64 [4])."""
        n, d = x.shape
        labels = torch.empty(n, dtype=torch.int32, device=x.device)
        centres = torch.empty((k, d), dtype=torch.float32, device=x.device)
        inertia, n_iter = ctypes.c_double(0.0), ctypes.c_int32(0)
        stats = np.zeros(4, dtype=np.int64)
        fid = None if first_ids is None else np.ascontiguousarray(first_ids, dtype=np.int64)
        u = None if uniforms is None else np.ascontiguousarray(uniforms, dtype=np.float64)
        with torch.cuda.device(self.device):
            _lib.call("slic_spherical_kmeans", _p(x), n, d, int(k), _p(init), None if fid is None else fid.ctypes.data,
                      None if u is None or u.size == 0 else u.ctypes.data, int(n_local_trials), int(n_init), int(max_iter),
                      float(tol), _p(labels), _p(centres), ctypes.addressof(inertia), ctypes.addressof(n_iter),
                      stats.ctypes.data, self._stream())
        return labels, centres, inertia.value, n_iter.value, stats

    # -- whole hierarchy (csrc/finch_driver.cu) ------------------------------------------------------
    FINCH_CAPACITY = 32   # label columns provided to the native driver (a FINCH level at least halves the clusters
                          # unless the min_sim cut intervenes; more levels -> SlicError status -5, see FINCH())

    def finch_native(self, data, nn0=None, dist0=None, unit0=None, dense0=False, ensure_early_exit=True, host_labels=False):
        """slic_finch on a device-resident float32 matrix.  -> (c int32 [N, P], num_clust list, min_sim or None); c is a
        device tensor, or with host_labels a numpy array in page-locked memory written by the device (see _labels_sink)."""
        n, d = data.shape
        cap = self.FINCH_CAPACITY
        sink, finish, _keep = self._labels_sink(n, cap, data.device, host_labels)
        num = (ctypes.c_int32 * cap)()
        levels, has = ctypes.c_int32(0), ctypes.c_int32(0)
        ms = ctypes.c_float(0)
        _lib.call("slic_finch", _p(data), n, d, _p(nn0), _p(dist0), _p(unit0), int(bool(dense0)), int(bool(ensure_early_exit)),
                  cap, sink, ctypes.addressof(num), ctypes.addressof(levels), ctypes.addressof(ms),
                  ctypes.addressof(has), self._stream())
        p = levels.value
        return finish(p), [int(v) for v in num[:p]], (np.float32(ms.value) if has.value else None)

    def finch_host(self, x, initial_rank=None, ensure_early_exit=True):
        """slic_finch_host on a C-contiguous float32 numpy matrix (pageable or pinned): chunked upload hidden behind the
        level-0 screen.  -> (c int32 [N, P] numpy, num_clust list, min_sim or None)."""
        n, d = x.shape
        cap = self.FINCH_CAPACITY
        # the labels are delivered in a page-locked buffer of the result pool: the device writes the [N, P] matrix into it
        # directly and the caller receives a view of it - no staging copy on either side
        try:
            raw, _ = self._results.take(n * cap * 4)
            out = raw.view(np.int32)
        except RuntimeError:          # no page-locked memory to be had: pageable destination (device buffer + copy inside)
            out = np.empty(n * cap, dtype=np.int32)
        num = (ctypes.c_int32 * cap)()
        levels, has = ctypes.c_int32(0), ctypes.c_int32(0)
        ms = ctypes.c_float(0)
        rank = None
        if initial_rank is not None:
            rank = np.ascontiguousarray(np.asarray(initial_rank), dtype=np.int64)
            if rank.shape != (n,):
                raise ValueError("initial_rank must have one entry per row of data")
        multi = getattr(self, "_multi", None)
        with torch.cuda.device(self.device):
            if multi is not None:
                _lib.call("slic_finch_multi", multi[0], x.ctypes.data, n, d, None if rank is None else rank.ctypes.data,
                          int(bool(ensure_early_exit)), cap, out.ctypes.data, ctypes.addressof(num),
                          ctypes.addressof(levels), ctypes.addressof(ms), ctypes.addressof(has))
            else:
                _lib.call("slic_finch_host", x.ctypes.data, n, d, None if rank is None else rank.ctypes.data,
                          int(bool(ensure_early_exit)), cap, out.ctypes.data, ctypes.addressof(num), ctypes.addressof(levels),
                          ctypes.addressof(ms), ctypes.addressof(has))
        p = levels.value
        return (self._results.deliver(out[: n * p].reshape(n, p)), [int(v) for v in num[:p]],
                (np.float32(ms.value) if has.value else None))

    # -- K4 --------------------------------------------------------------------------------------
    def label_mask(self, a, b, prepend_ones=False, negate=False):
        na, nb = a.shape[0], b.shape[0]
        out = torch.empty((na, nb + int(prepend_ones)), dtype=torch.bool, device=a.device)
        _lib.call("slic_label_mask_u8", _p(a), na, _p(b), nb, int(prepend_ones), int(negate), _p(out), self._stream())
        return out

    def label_mask_bits(self, a, b, negate=False):
        na, nb = a.shape[0], b.shape[0]
        out = torch.zeros((na, (nb + 31) // 32), dtype=torch.int32, device=a.device)
        _lib.call("slic_label_mask_bits", _p(a), na, _p(b), nb, int(negate), _p(out), self._stream())
        return out

    def dense_labels(self, labels):
        """np.unique(labels, return_inverse=True) on the device for int32 labels (slic_dense_labels).
        -> (dense int32 [n], uniq int32 [count], count)."""
        n = labels.shape[0]
        dense = torch.empty(n, dtype=torch.int32, device=labels.device)
        uniq = torch.empty(n, dtype=torch.int32, device=labels.device)
        num = torch.empty(1, dtype=torch.int32, device=labels.device)
        _lib.call("slic_dense_labels", _p(labels), n, _p(dense), _p(uniq), _p(num), self._stream())
        count = int(num.item())
        return dense, uniq[:count], count

    def scatter_last_wins(self, values, positions, n_out, fill=-1):
        """out[positions[i]] = values[i] in order of i (slic_scatter_last_wins).  -> (out int32 [n_out], out_of_range int)."""
        out = torch.empty(n_out, dtype=torch.int32, device=values.device)
        bad = torch.empty(1, dtype=torch.int32, device=values.device)
        _lib.call("slic_scatter_last_wins", _p(values), _p(positions), values.shape[0], n_out, int(fill), _p(out), _p(bad),
                  self._stream())
        return out, int(bad.item())

    def cluster_metrics(self, labels_true, labels_pred, num_true, num_pred, want_emi=True):
        """-> [mi, h_true, h_pred, emi, classes, clusters] as Python floats (slic_cluster_metrics; one read-back)."""
        out = torch.empty(6, dtype=torch.float64, device=labels_true.device)
        _lib.call("slic_cluster_metrics", _p(labels_true), _p(labels_pred), labels_true.shape[0], int(num_true),
                  int(num_pred), int(bool(want_emi)), _p(out), self._stream())
        vals = out.tolist()
        if vals[0] != vals[0]:      # NaN: the kernel met labels outside [0, num) and refused to count them
            raise ValueError("cluster_metrics: %d labels lie outside [0, num_true) x [0, num_pred)" % int(-vals[4]))
        return vals

    def group_by_label(self, labels, num_labels):
        n = labels.shape[0]
        order = torch.empty(n, dtype=torch.int32, device=labels.device)
        offsets = torch.empty(num_labels + 1, dtype=torch.int32, device=labels.device)
        _lib.call("slic_group_by_label", _p(labels), n, num_labels, _p(order), _p(offsets), self._stream())
        return order, offsets


_default = None


def default_backend():
    """The process-wide CUDA backend (created on first use; raises without a GPU)."""
    global _default
    if _default is None:
        _default = CudaBackend()
    return _default


def set_default_backend(backend):
    """Tests only: install a stand-in backend."""
    global _default
    _default = backend
