// Shared host/device helpers for the slic_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/slic_b200.h"

namespace slic {

void set_error(const char* fmt, ...);
// nn_screen_tc.cu: post-mortem text of a timed-out wait in a gated screen launch ("" when there is none)
const char* timeout_record_text();

#define SLIC_CUDA_OK(expr)                                                                     \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            slic::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return SLIC_ERR_CUDA;                                                              \
        }                                                                                      \
    } while (0)

#define SLIC_REQUIRE(cond, msg)                                        \
    do {                                                               \
        if (!(cond)) {                                                 \
            slic::set_error("%s:%d %s", __FILE__, __LINE__, msg);      \
            return SLIC_ERR_INVALID_ARG;                               \
        }                                                              \
    } while (0)

#define SLIC_PROPAGATE(expr)              \
    do {                                  \
        int _s = (expr);                  \
        if (_s != SLIC_OK) return _s;     \
    } while (0)

// every kernel launch in the library goes through this: checks the launch and counts it
// (slic_launch_count(), read by bench.py for its gpu_launches claim)
void count_launch();
#define SLIC_LAUNCH_OK()                  \
    do {                                  \
        SLIC_CUDA_OK(cudaGetLastError()); \
        slic::count_launch();             \
    } while (0)

inline cudaStream_t as_stream(slic_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// Stream-ordered temporary: freed (stream-ordered) when it goes out of scope.
struct Scratch {
    void* ptr = nullptr;
    cudaStream_t stream = nullptr;
    cudaError_t alloc(size_t bytes, cudaStream_t s) {
        stream = s;
        if (bytes == 0) bytes = 16;
        return cudaMallocAsync(&ptr, bytes, s);
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
    ~Scratch() {
        if (ptr) cudaFreeAsync(ptr, stream);
    }
    Scratch() = default;
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
};

int num_sms();

// nn_exact.cu: exact top-k cosine neighbours (dense row blocks + radix select) of the listed query rows;
// the finisher for rows the tensor-core top-k screen could not settle.
int exact_topk_cosine_rows(const void* q, const int* q_rows, int64_t nq, const void* x, int64_t n, int d, int dtype, int k,
                           int64_t self_offset, int* idx_out, void* dist_out, cudaStream_t st);

// nn_screen_tc.cu: level-0 first-neighbour search whose database is still being uploaded (finch_driver.cu).
// gates[c] (device int32, zero-initialised) becomes non-zero once rows [c * chunk_rows, (c + 1) * chunk_rows) of the
// f16 matrix are in place; `after` runs on the host right after the screen kernel has been launched.
struct GateSpec {
    const int* gates;
    int num_chunks;
    int64_t chunk_rows;   // multiple of 256
};
typedef int (*AfterScreenFn)(void* ctx);
// Multi-GPU fused search: where this rank's screen kernel publishes pre-pass results (comm.cu owns the memory: every
// pointer lies in a peer-mapped window of one of the ranks of the box).
constexpr int SLIC_MAX_PEERS = 7;   // ranks of one box - 1
struct ScreenPeers {
    int num_peers;
    unsigned int* own_best;                    // [n] this rank's row bests (its window; the peers write into it)
    int* own_sync;                             // this rank's pre-pass arrival counter (its window)
    unsigned int* peer_best[SLIC_MAX_PEERS];   // the same two of every other rank
    int* peer_sync[SLIC_MAX_PEERS];
};
// can CTAs of the given shape co-reside with the persistent screen kernel of a gated self-search (see nn_screen_tc.cu)
bool screen_can_overlap_upload(int64_t n, int d_pad, int guest_threads, int guest_regs);
// prep.cu: CTA shape of the float32 normalise kernel (the guest of a gated launch)
int normalize_kernel_shape(int* threads, int* regs);
// true: a self-search of n rows runs the symmetric screen (upper-triangular tiles, row + column filters)
bool screen_self_search_is_symmetric(int64_t n);
// stats_ext (device, 8 ints, optional): asynchronous mode - the call never waits for the device and leaves
// {[1] rows still to be finished exactly, [4] pipeline error, [5] candidate-log overflow} there; any non-zero value
// means the result is incomplete and the search must be repeated through the synchronous path (slic_nn_top1).
int nn_top1_f32_gated(const float* q_unit, const uint16_t* q_f16, int64_t nq, const float* x_unit,
                      const uint16_t* x_f16, int64_t n, int d, int d_pad, int64_t self_offset, float eps, int* idx_out,
                      float* dist_out, int* stats_out, const GateSpec* gate, AfterScreenFn after, void* after_ctx,
                      cudaStream_t st, int* stats_ext = nullptr);
// self-search of all rows (first neighbour + distance in `dtype`), asynchronous as above
int nn_top1_self_async(const void* unit, const uint16_t* ub, int64_t n, int d, int d_pad, int dtype, int* idx_out,
                       void* dist_out, int* stats_ext, cudaStream_t st);

// This rank's part of the fused multi-GPU self-search (comm.cu): pre-pass over its 1 / parts of the row units, published
// to every rank from inside the kernel, then its 1 / parts of the symmetric screen's triangle and the exact re-rank.
// idx_out / dist_out [n]: the best pair this rank saw for EVERY row (idx 0x7fffffff: none).  Asynchronous: stats_dev
// (8 ints) receives {[1] rows without a record, [4] pipeline error, [5] log overflow}.
int nn_top1_sym_fused(const float* unit, const uint16_t* ub, int64_t n, int d, int d_pad, int part, int parts,
                      const ScreenPeers* peers, AfterScreenFn before_screen, void* before_ctx, int* idx_out,
                      float* dist_out, int* stats_dev, cudaStream_t st);
// finch_driver.cu: the hierarchy after a level-0 search done elsewhere (comm.cu), labels to the host; see there
int finch_tail_to_host(const float* data, int64_t n, int d, int* nn, float* dist, const float* unit, const uint16_t* ub,
                       int* blk16, bool ensure_early_exit, int capacity, int* labels_out_host, int* num_clust_host,
                       int* num_levels_host, float* min_sim_host, int* has_min_sim_host, cudaStream_t st);
// the same with the [n, capacity] label buffer on the device (every rank of a per-process group keeps its own copy)
int finch_tail_device(const float* data, int64_t n, int d, int* nn, float* dist, const float* unit, const uint16_t* ub,
                      int* blk16, bool ensure_early_exit, int capacity, int* labels_out_dev, int* num_clust_host,
                      int* num_levels_host, float* min_sim_host, int* has_min_sim_host, cudaStream_t st);
int finch_host_single(const float* x_host, int64_t n, int d, const int64_t* initial_rank_host, bool ensure_early_exit,
                      int capacity, int* labels_out_host, int* num_clust_host, int* num_levels_host, float* min_sim_host,
                      int* has_min_sim_host);
// per-row key of the multi-GPU merge: (float32 distance bits << 32) | neighbour; MIN over the ranks = np.argmin's rule
constexpr unsigned long long SYM_KEY_NONE = 0x7fffffff7fffffffull;

// host_entry.cu: host -> device copies of pageable memory through pinned staging buffers filled by several host threads
constexpr int STAGE_SLOTS = 3;
struct StagePool {
    void* buf[STAGE_SLOTS] = {nullptr, nullptr, nullptr};
    cudaEvent_t done[STAGE_SLOTS] = {nullptr, nullptr, nullptr};
    bool busy[STAGE_SLOTS] = {false, false, false};
    size_t cap = 0;
    int ensure(size_t bytes);   // three pinned buffers of at least `bytes` each
};
StagePool& stage_pool();        // the calling thread's pool
bool host_is_pageable(const void* p);
void stage_threads_shared();          // the calling thread shares the host with other uploading threads (comm.cu workers)
void* pinned_device_view(void* p);   // device-writable view of page-locked host memory, or nullptr
void parallel_host_copy(void* dst, const void* src, size_t bytes);
int copy_to_device_staged(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st);

__host__ __device__ static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- driver-internal forms of K2 / K3 (finch_driver.cu): counts stay on the device --------------------------------
// cc.cu: components of the first-neighbour graph; min_sim (when filtering) is read from device memory; csr_offsets
// [clusters + 1] / csr_counts [clusters] (optional) receive the CSR row pointers and row counts of the clusters.
int finch_components_csr(const int* nn, int64_t n, int use_filter, const float* min_sim_dev, const void* unit, int d,
                         int dtype, const void* dist_nn, int* labels, int* num_clust_dev, int* csr_offsets,
                         int* csr_counts, cudaStream_t st, int* bad_count_dev = nullptr /* += indices outside [0, n) */);
// segmean.cu: order = stable argsort(labels); num_labels_bound only sizes the radix passes
int order_rows_by_label(const int* labels, int64_t n, int64_t num_labels_bound, int* order, cudaStream_t st);
// segmean.cu: sums / counts / means of the clusters from their CSR grouping; num_clust_dev (optional) = actual count
// on the device, num_clust then being an upper bound that sizes temporaries and grids
template <typename T>
int cluster_sums_csr(const T* data, const int* weights, const int* order, const int* offsets, int64_t n, int d,
                     int num_clust, const int* num_clust_dev, double* sums_out, int* counts_out, double* means_out,
                     cudaStream_t st);

// finch_small.cu: all remaining levels of a hierarchy whose current level has <= SMALL_LEVEL_MAX_ROWS clusters, in one
// cooperative launch with the level loop and the exit rules of finch.py:151-163 on the device.
constexpr int SMALL_LEVEL_MAX_ROWS = 2048;
struct SmallLevelsArgs {
    int64_t n_rows;          // N: rows of the original matrix
    int d;
    int capacity;            // label columns available in `cols`
    int* cols;               // [capacity][N] composed labels, column l = partition l (columns < levels are filled)
    int* summary;            // [0] levels kept (in / out), [1] status out (0 ok, 1 more levels than capacity, 2 the
                             // entering level has more than SMALL_LEVEL_MAX_ROWS clusters), [2 + l] clusters of level l
    double* sums[2];         // [rows of the entering level, d] each; index 0 holds the entering level's state
    int* counts[2];
    double* means[2];
    double* unit;            // [rows, d]
    double* gram;            // small_levels_gram_elems(rows) doubles
    int* nn;                 // [rows]
    double* dist;            // [rows]
    int* parent;             // [rows]
    int use_filter;          // finch.py:51-52 applies (level 0 had dense distances and ensure_early_exit)
    const float* min_sim_dev;
    unsigned long long* trace;   // optional [SMALL_TRACE_STAMPS] globaltimer stamps at the phase boundaries (diagnostic)
};
constexpr int SMALL_TRACE_STAMPS = 96;
size_t small_levels_gram_elems(int64_t m);
int launch_small_levels(const SmallLevelsArgs& args, cudaStream_t st);

// ---- device helpers ---------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// (distance, index) ordering used everywhere a neighbour is chosen.  The reference takes np.argmin of
// distances held in the array dtype (finch.py:27-29): the smaller distance wins and equal distances -
// including float32 values that only tie after rounding - go to the lower index.  Callers therefore pass
// the distance ALREADY ROUNDED to the reference dtype (cosine_distance_from_sim<T>), widened to double.
__device__ __forceinline__ bool closer(double dd, int j, double db, int jb) {
    return (dd < db) || (dd == db && j < jb);
}

// distance in the reference dtype from a float64 similarity: sklearn cosine_distances does
// S *= -1; S += 1; clip(S, 0, 2) in the array dtype (sklearn/metrics/pairwise.py:1174-1177).
template <typename T>
__device__ __forceinline__ T cosine_distance_from_sim(double s) {
    T st = static_cast<T>(s);
    T dd = static_cast<T>(1) - st;
    dd = dd < static_cast<T>(0) ? static_cast<T>(0) : dd;
    dd = dd > static_cast<T>(2) ? static_cast<T>(2) : dd;
    return dd;
}

// exact <a, b> of two rows of unit vectors, float64 accumulation, one warp per pair.
template <typename T>
__device__ __forceinline__ double warp_dot(const T* __restrict__ a, const T* __restrict__ b, int d, int lane);

template <>
__device__ __forceinline__ double warp_dot<float>(const float* __restrict__ a, const float* __restrict__ b,
                                                  int d, int lane) {
    double acc = 0.0;
    if ((d & 3) == 0 && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0) {
        const float4* a4 = reinterpret_cast<const float4*>(a);
        const float4* b4 = reinterpret_cast<const float4*>(b);
        for (int k = lane; k < (d >> 2); k += 32) {
            float4 x = __ldg(a4 + k), y = __ldg(b4 + k);
            acc = fma((double)x.x, (double)y.x, acc);
            acc = fma((double)x.y, (double)y.y, acc);
            acc = fma((double)x.z, (double)y.z, acc);
            acc = fma((double)x.w, (double)y.w, acc);
        }
    } else {
        for (int k = lane; k < d; k += 32) acc = fma((double)__ldg(a + k), (double)__ldg(b + k), acc);
    }
    return warp_sum(acc);
}

template <>
__device__ __forceinline__ double warp_dot<double>(const double* __restrict__ a, const double* __restrict__ b,
                                                   int d, int lane) {
    double acc = 0.0;
    if ((d & 1) == 0 && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0) {
        const double2* a2 = reinterpret_cast<const double2*>(a);
        const double2* b2 = reinterpret_cast<const double2*>(b);
        for (int k = lane; k < (d >> 1); k += 32) {
            double2 x = __ldg(a2 + k), y = __ldg(b2 + k);
            acc = fma(x.x, y.x, acc);
            acc = fma(x.y, y.y, acc);
        }
    } else {
        for (int k = lane; k < d; k += 32) acc = fma(__ldg(a + k), __ldg(b + k), acc);
    }
    return warp_sum(acc);
}

}  // namespace slic
