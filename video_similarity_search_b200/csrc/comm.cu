// Multi-GPU level-0 search of one box over NVLink peer memory, and the rank-0-driven FINCH entry built on it.
//
// Reference call site: online_train.py:619-627, 660-662 - rank 0 clusters while the other ranks sit in a barrier.  Here
// the O(N^2 D) first-neighbour stage (clustering/finch.py:27-29) is shared by all GPUs of the box, every GPU holding the
// full matrix; the rest of the hierarchy (components, means, levels >= 1: milliseconds) runs on one GPU.
//
// Two ways to form the group, one data path:
//   * one PROCESS per GPU (torch.distributed jobs): slic_comm_window_create + slic_comm_connect - every rank allocates a
//     "window" with cudaMalloc, exports it as a CUDA IPC handle, the host side exchanges the 64-byte handles (any
//     transport; sharded.py uses the process group) and every rank maps the windows of its peers;
//   * one process for ALL GPUs (the unmodified reference call site): slic_comm_create(devices) enables peer access and
//     starts one worker thread per device; slic_finch_multi(comm, host matrix) is the drop-in for FINCH(data).
//
// Window of a rank: [header: barrier flags, pre-pass counter][row bests, uint32 x max_rows][keys, uint64 x (max_rows+1)].
//
// Data path per search (all on the rank's stream, no host synchronisation, NO collective library call):
//   1. init kernel resets the rank's own row bests / counter               (nn_screen_tc.cu, sym_init_kernel)
//   2. barrier A   flags written into every peer's window, spin on the own  (nobody publishes into a window before its reset)
//   3. ONE screen kernel per rank: pre-pass over its 1/G of the row blocks - the epilogue publishes every row's best with
//      red.max into ALL windows and counts its arrival on ALL counters - then its 1/G of the symmetric screen's triangle,
//      whose units wait for the arrivals of every rank's pre-pass.  (Round 1: two launches + an NCCL all-reduce MAX.)
//   4. exact re-rank of the rank's candidates, packed as (distance bits << 32 | neighbour) keys into its window
//   5. barrier B, then ONE merge kernel: every rank reads the G key arrays over NVLink and takes the element-wise MIN
//      (= np.argmin's rule: smallest distance, then lowest index) straight into nn / dist.  (Round 1: NCCL all-reduce MIN
//      + unpack kernel.)
// Bytes over NVLink per rank: 4 N (G-1)/G of published bests (+ one counter add per pre-pass warp) + 8 N (G-1) of keys read.
#include <stdlib.h>
#include <string.h>

#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

struct slic_comm {};   // opaque to C callers

namespace slic {

constexpr int COMM_MAX_RANKS = SLIC_MAX_PEERS + 1;
constexpr int COMM_PHASES = 4;
constexpr size_t WIN_HEADER_BYTES = 1024;
constexpr int COMM_UPLOAD_PIECES = 4;   // rank-0-driven upload: a worker's share crosses PCIe in pieces, forwarded as they land
struct WindowHeader {
    int flags[COMM_PHASES][COMM_MAX_RANKS];   // flags[phase][src] = epoch of the last barrier rank `src` has entered
    int sync_counter;                         // pre-pass arrivals of all ranks' screen kernels (this search)
};
static_assert(sizeof(WindowHeader) <= WIN_HEADER_BYTES, "window header");
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static size_t win_best_off() { return WIN_HEADER_BYTES; }
static size_t win_keys_off(int64_t max_rows) { return WIN_HEADER_BYTES + align_up((size_t)max_rows * 4, 256); }
static size_t win_bytes(int64_t max_rows) { return win_keys_off(max_rows) + align_up((size_t)(max_rows + 1) * 8, 256); }

struct WindowPtrs {
    unsigned char* w[COMM_MAX_RANKS];
};

// One thread per rank of the group: publish "this rank has reached barrier (phase, epoch)" into that rank's window, then
// wait until that rank has published the same into ours.  Everything this stream did before (kernel boundary + system
// fence) is visible to a peer that has seen the flag.  Bounded: a missing rank costs ~2 s and sets *err (the search is
// then reported incomplete and repeated on one GPU) - it never traps or hangs.
__global__ void comm_barrier_kernel(WindowPtrs wp, int rank, int world, int phase, int epoch, int* err) {
    const int g = threadIdx.x;
    if (g >= world) return;
    __threadfence_system();
    int* dst = &reinterpret_cast<WindowHeader*>(wp.w[g])->flags[phase][rank];
    asm volatile("st.release.sys.global.b32 [%0], %1;" ::"l"(dst), "r"(epoch) : "memory");
    const int* src = &reinterpret_cast<WindowHeader*>(wp.w[rank])->flags[phase][g];
    long long t0 = 0;
    unsigned polls = 0;
    while (true) {
        int v;
        asm volatile("ld.acquire.sys.global.b32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
        if (v - epoch >= 0) break;
        __nanosleep(64);
        if ((++polls & 0xff) == 0) {
            const long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) {
                if (err) atomicExch(err, 1);
                break;
            }
        }
    }
    __threadfence_system();
}

// keys[i] = (distance bits << 32) | neighbour of the best pair this rank saw for row i; keys[n] = 1 iff its search was
// complete (no pipeline error, no log overflow: stats[4], stats[5]).
__global__ void comm_pack_keys_kernel(const int* __restrict__ idx, const float* __restrict__ dist, int64_t n,
                                      const int* __restrict__ stats, unsigned long long* __restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int j = idx[i];
        keys[i] = j == 0x7fffffff ? SYM_KEY_NONE : (((unsigned long long)__float_as_uint(dist[i]) << 32) | (unsigned int)j);
    } else if (i == n) {
        keys[n] = (stats[4] == 0 && stats[5] == 0) ? 1ull : 0ull;
    }
}

// element-wise MIN over the ranks' key arrays (read in place over NVLink), unpacked: nn / dist of every row on this
// rank.  *unsettled += rows no rank had a record for, *incomplete = 1 when some rank's search was incomplete.
__global__ void comm_merge_keys_kernel(WindowPtrs wp, size_t keys_off, int world, int64_t n, int* __restrict__ idx,
                                       float* __restrict__ dist, int* __restrict__ unsettled, int* __restrict__ incomplete) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    unsigned long long k = ~0ull;
    for (int g = 0; g < world; ++g) {
        const unsigned long long v = reinterpret_cast<const unsigned long long*>(wp.w[g] + keys_off)[i];
        k = v < k ? v : k;
    }
    if (i == n) {
        if (k == 0ull) *incomplete = 1;
        return;
    }
    idx[i] = (int)(unsigned int)(k & 0xffffffffull);
    dist[i] = __uint_as_float((unsigned int)(k >> 32));
    if (k == SYM_KEY_NONE) atomicAdd(unsettled, 1);
}

class HostBarrier {
  public:
    explicit HostBarrier(int n) : n_(n) {}
    void wait() {
        std::unique_lock<std::mutex> lk(m_);
        const unsigned gen = gen_;
        if (++count_ == n_) {
            count_ = 0;
            ++gen_;
            cv_.notify_all();
        } else {
            cv_.wait(lk, [&] { return gen_ != gen; });
        }
    }

  private:
    std::mutex m_;
    std::condition_variable cv_;
    int n_, count_ = 0;
    unsigned gen_ = 0;
};

struct MultiJob {
    const float* x_host;
    int64_t n;
    int d;
    bool ensure_early_exit;
    int capacity;
    int* labels_out_host;
    int* num_clust_host;
    int* num_levels_host;
    float* min_sim_host;
    int* has_min_sim_host;
    float* data[COMM_MAX_RANKS];   // every worker's [n, d] matrix (published before the pushes start)
    int status[COMM_MAX_RANKS];
    char error[COMM_MAX_RANKS][512];
    float ms_upload, ms_search, ms_total;   // rank 0's CUDA-event timeline of the call (slic_comm_last_timeline)
};

struct Comm : slic_comm {
    bool single = false;
    int world = 0;
    int rank = -1;       // one process per GPU: this process's rank / device
    int device = -1;
    int64_t max_rows = 0;
    unsigned char* win[COMM_MAX_RANKS] = {};
    bool mapped[COMM_MAX_RANKS] = {};   // IPC mappings to close
    bool connected = false;
    int epoch = 0;
    // single process
    int devices[COMM_MAX_RANKS] = {};
    cudaStream_t streams[COMM_MAX_RANKS] = {};
    cudaStream_t forward[COMM_MAX_RANKS] = {};                     // device -> peers copies of the pieces already uploaded
    cudaEvent_t piece_up[COMM_MAX_RANKS][COMM_UPLOAD_PIECES] = {};   // piece p of worker r's share has reached its device
    cudaEvent_t uploaded[COMM_MAX_RANKS] = {};
    cudaEvent_t t0 = nullptr, t1 = nullptr, t2 = nullptr, t3 = nullptr;
    std::vector<std::thread> threads;
    std::unique_ptr<HostBarrier> bar;      // the workers among themselves
    std::mutex m;
    std::condition_variable cv;
    unsigned job_gen = 0, done_count = 0;
    bool quit = false;
    MultiJob* job = nullptr;
    std::mutex call_mutex;                 // one slic_finch_multi at a time
    float last_ms[3] = {0, 0, 0};
};

static WindowPtrs window_ptrs(const Comm* c) {
    WindowPtrs wp;
    for (int g = 0; g < COMM_MAX_RANKS; ++g) wp.w[g] = c->win[g];
    return wp;
}

struct BarrierCtx {
    const Comm* c;
    int rank, phase, epoch;
    int* err;
    cudaStream_t st;
};
static int enqueue_barrier(void* ctx) {
    const BarrierCtx* b = static_cast<const BarrierCtx*>(ctx);
    comm_barrier_kernel<<<1, 32, 0, b->st>>>(window_ptrs(b->c), b->rank, b->c->world, b->phase, b->epoch, b->err);
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

// This rank's share of the group's first-neighbour search of all rows (see the header of this file).  unit / ub: the
// normalised matrix on this rank's device; idx_out / dist_out [n]: the MERGED result, identical on every rank.
// Device ints, zeroed by the caller: *unsettled += rows left without a neighbour, *incomplete = 1 when some rank's search
// was incomplete or a rank did not show up at a barrier (the caller then repeats the search on one GPU).
static int comm_nn_top1_rank(const Comm* c, int rank, int epoch, const float* unit, const uint16_t* ub, int64_t n, int d,
                             int d_pad, int* idx_out, float* dist_out, int* unsettled, int* incomplete, cudaStream_t st) {
    SLIC_REQUIRE(n <= c->max_rows, "comm search: more rows than the windows were created for");
    ScreenPeers sp;
    memset(&sp, 0, sizeof(sp));
    sp.own_best = reinterpret_cast<unsigned int*>(c->win[rank] + win_best_off());
    sp.own_sync = &reinterpret_cast<WindowHeader*>(c->win[rank])->sync_counter;
    for (int g = 0; g < c->world; ++g) {
        if (g == rank) continue;
        sp.peer_best[sp.num_peers] = reinterpret_cast<unsigned int*>(c->win[g] + win_best_off());
        sp.peer_sync[sp.num_peers] = &reinterpret_cast<WindowHeader*>(c->win[g])->sync_counter;
        ++sp.num_peers;
    }
    Scratch lidx, ldist, lstats;
    SLIC_CUDA_OK(lidx.alloc((size_t)n * sizeof(int), st));
    SLIC_CUDA_OK(ldist.alloc((size_t)n * sizeof(float), st));
    SLIC_CUDA_OK(lstats.alloc(8 * sizeof(int), st));
    BarrierCtx a = {c, rank, 0, epoch, incomplete, st};
    SLIC_PROPAGATE(nn_top1_sym_fused(unit, ub, n, d, d_pad, rank, c->world, &sp, enqueue_barrier, &a, lidx.as<int>(),
                                     ldist.as<float>(), lstats.as<int>(), st));
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(c->win[rank] + win_keys_off(c->max_rows));
    comm_pack_keys_kernel<<<(unsigned)ceil_div(n + 1, 256), 256, 0, st>>>(lidx.as<int>(), ldist.as<float>(), n,
                                                                          lstats.as<int>(), keys);
    SLIC_LAUNCH_OK();
    BarrierCtx b = {c, rank, 1, epoch, incomplete, st};
    SLIC_PROPAGATE(enqueue_barrier(&b));
    comm_merge_keys_kernel<<<(unsigned)ceil_div(n + 1, 256), 256, 0, st>>>(window_ptrs(c), win_keys_off(c->max_rows), c->world,
                                                                           n, idx_out, dist_out, unsettled, incomplete);
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

// ---- single process, one worker thread per device -------------------------------------------------------------------
static int d_pad_of(int d) { return (d + 63) / 64 * 64; }

static int worker_call(Comm* c, int r, MultiJob* job, int epoch) {
    const int64_t n = job->n;
    const int d = job->d, dp = d_pad_of(d), world = c->world;
    cudaStream_t st = c->streams[r];
    int status = SLIC_OK;
    // every step is skipped once this worker has failed, but every host barrier is still entered: the other workers
    // must not wait for a rank that has gone
#define STEP(expr)                                \
    do {                                          \
        if (status == SLIC_OK) status = (expr);   \
    } while (0)
#define CUDA_STEP(expr)                                                                                   \
    do {                                                                                                  \
        if (status == SLIC_OK) {                                                                          \
            cudaError_t _e = (expr);                                                                      \
            if (_e != cudaSuccess) {                                                                      \
                set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));           \
                status = SLIC_ERR_CUDA;                                                                   \
            }                                                                                             \
        }                                                                                                 \
    } while (0)
    Scratch data, unit, ub, idx, dist, blk;
    CUDA_STEP(data.alloc((size_t)n * d * sizeof(float), st));
    CUDA_STEP(unit.alloc((size_t)n * d * sizeof(float), st));
    CUDA_STEP(ub.alloc((size_t)n * dp * 2, st));
    CUDA_STEP(idx.alloc((size_t)n * sizeof(int), st));
    CUDA_STEP(dist.alloc((size_t)n * sizeof(float), st));
    CUDA_STEP(blk.alloc(16 * sizeof(int), st));
    CUDA_STEP(cudaMemsetAsync(blk.ptr, 0, 16 * sizeof(int), st));
    CUDA_STEP(cudaStreamSynchronize(st));   // the buffer exists before a peer's stream copies into it
    job->data[r] = data.as<float>();
    c->bar->wait();
    // upload: this worker's 1/G of the rows host -> its device, then device -> every peer (copy engines over NVLink);
    // the G workers share the host's PCIe root, so G full uploads would cost G times the bytes over the same links
    const int64_t per = ceil_div(n, world);
    const int64_t r0 = per * r < n ? per * r : n, r1 = r0 + per < n ? r0 + per : n;
    if (r == 0) CUDA_STEP(cudaEventRecord(c->t0, st));
    if (r1 > r0) {
        // piece p + 1 crosses PCIe (host -> this device, stream st) while piece p travels on to the peers over NVLink
        // (copy engines, stream forward[r]): the forwards of all but the last piece are hidden behind the upload
        // (a pageable source is staged through pinned buffers by host threads, which is the slower leg anyway: one piece -
        // measured with pieces at 2 GPUs: upload + forward 12.8 -> 15 ms)
        const int pieces = ((size_t)(r1 - r0) * d * sizeof(float) >= ((size_t)32 << 20) && !host_is_pageable(job->x_host))
                               ? COMM_UPLOAD_PIECES
                               : 1;
        const int64_t step = ceil_div(r1 - r0, pieces);
        for (int p = 0; p < pieces; ++p) {
            const int64_t a = r0 + step * p < r1 ? r0 + step * p : r1, b = a + step < r1 ? a + step : r1;
            if (b <= a) continue;
            const size_t bytes = (size_t)(b - a) * d * sizeof(float);
            STEP(copy_to_device_staged(data.as<float>() + a * d, job->x_host + a * d, bytes, st));   // (pageable: staged by threads)
            CUDA_STEP(cudaEventRecord(c->piece_up[r][p], st));
            CUDA_STEP(cudaStreamWaitEvent(c->forward[r], c->piece_up[r][p], 0));
            for (int k = 1; k < world; ++k) {
                const int g = (r + k) % world;   // every worker starts with a different peer
                if (job->data[g])
                    CUDA_STEP(cudaMemcpyPeerAsync(job->data[g] + a * d, c->devices[g], data.as<float>() + a * d, c->devices[r],
                                                  bytes, c->forward[r]));
            }
        }
    }
    CUDA_STEP(cudaEventRecord(c->uploaded[r], c->forward[r]));   // (forward[r] has waited for the last piece: upload AND forwards)
    CUDA_STEP(cudaStreamWaitEvent(st, c->uploaded[r], 0));       // this worker's buffers are not reused before its forwards end
    c->bar->wait();
    for (int g = 0; g < world; ++g)
        if (g != r) CUDA_STEP(cudaStreamWaitEvent(st, c->uploaded[g], 0));
    if (r == 0) CUDA_STEP(cudaEventRecord(c->t1, st));
    STEP(slic_normalize_rows(data.ptr, n, d, SLIC_F32, unit.ptr, nullptr, ub.as<uint16_t>(), dp, (slic_stream_t)st));
    STEP(comm_nn_top1_rank(c, r, epoch, unit.as<float>(), ub.as<uint16_t>(), n, d, dp, idx.as<int>(), dist.as<float>(),
                           blk.as<int>() + 1, blk.as<int>() + 5, st));
    if (r == 0) {
        CUDA_STEP(cudaEventRecord(c->t2, st));
        STEP(finch_tail_to_host(data.as<float>(), n, d, idx.as<int>(), dist.as<float>(), unit.as<float>(), ub.as<uint16_t>(),
                                blk.as<int>(), job->ensure_early_exit, job->capacity, job->labels_out_host,
                                job->num_clust_host, job->num_levels_host, job->min_sim_host, job->has_min_sim_host, st));
        CUDA_STEP(cudaEventRecord(c->t3, st));
    }
    {   // drained whatever happened above: peers copy into this worker's buffers and read its window until they are done
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess && status == SLIC_OK) {
            set_error("comm worker %d: %s", r, cudaGetErrorString(e));
            status = SLIC_ERR_CUDA;
        }
    }
    c->bar->wait();
    if (r == 0 && status == SLIC_OK) {
        cudaEventElapsedTime(&job->ms_upload, c->t0, c->t1);
        cudaEventElapsedTime(&job->ms_search, c->t1, c->t2);
        cudaEventElapsedTime(&job->ms_total, c->t0, c->t3);
    }
#undef STEP
#undef CUDA_STEP
    return status;
}

static void worker_main(Comm* c, int r) {
    cudaSetDevice(c->devices[r]);
    stage_threads_shared();
    unsigned seen = 0;
    int epoch = 0;
    while (true) {
        MultiJob* job;
        {
            std::unique_lock<std::mutex> lk(c->m);
            c->cv.wait(lk, [&] { return c->quit || c->job_gen != seen; });
            if (c->quit) return;
            seen = c->job_gen;
            job = c->job;
        }
        const int s = worker_call(c, r, job, ++epoch);
        job->status[r] = s;
        if (s != SLIC_OK) {
            strncpy(job->error[r], slic_last_error(), sizeof(job->error[r]) - 1);
            job->error[r][sizeof(job->error[r]) - 1] = 0;
        }
        {
            std::lock_guard<std::mutex> lk(c->m);
            ++c->done_count;
        }
        c->cv.notify_all();
    }
}

static void destroy_comm(Comm* c) {
    if (!c) return;
    if (c->single) {
        {
            std::lock_guard<std::mutex> lk(c->m);
            c->quit = true;
        }
        c->cv.notify_all();
        for (std::thread& t : c->threads) t.join();
        int prev = 0;
        cudaGetDevice(&prev);
        for (int g = 0; g < c->world; ++g) {
            cudaSetDevice(c->devices[g]);
            if (c->streams[g]) cudaStreamDestroy(c->streams[g]);
            if (c->forward[g]) cudaStreamDestroy(c->forward[g]);
            for (int p = 0; p < COMM_UPLOAD_PIECES; ++p)
                if (c->piece_up[g][p]) cudaEventDestroy(c->piece_up[g][p]);
            if (c->uploaded[g]) cudaEventDestroy(c->uploaded[g]);
            if (c->win[g]) cudaFree(c->win[g]);
        }
        if (c->world > 0) {
            cudaSetDevice(c->devices[0]);
            for (cudaEvent_t e : {c->t0, c->t1, c->t2, c->t3})
                if (e) cudaEventDestroy(e);
        }
        cudaSetDevice(prev);
    } else {
        for (int g = 0; g < COMM_MAX_RANKS; ++g)
            if (c->mapped[g]) cudaIpcCloseMemHandle(c->win[g]);
        if (c->rank >= 0 && c->win[c->rank]) cudaFree(c->win[c->rank]);
        else if (c->rank < 0 && c->win[0]) cudaFree(c->win[0]);
    }
    cudaGetLastError();
    delete c;
}

}  // namespace slic

extern "C" {

int slic_comm_window_create(int64_t max_rows, slic_comm_t** comm_out, void* ipc_handle_out) {
    using namespace slic;
    SLIC_REQUIRE(max_rows > 0 && max_rows < ((int64_t)1 << 31) && comm_out && ipc_handle_out, "comm_window_create: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == SLIC_COMM_HANDLE_BYTES, "IPC handle size");
    SLIC_PROPAGATE(slic_require_device());
    std::unique_ptr<Comm> c(new Comm());
    c->max_rows = max_rows;
    SLIC_CUDA_OK(cudaGetDevice(&c->device));
    void* w = nullptr;
    SLIC_CUDA_OK(cudaMalloc(&w, win_bytes(max_rows)));
    c->win[0] = static_cast<unsigned char*>(w);   // moved to win[rank] by slic_comm_connect
    SLIC_CUDA_OK(cudaMemset(w, 0, win_bytes(max_rows)));
    cudaIpcMemHandle_t h;
    SLIC_CUDA_OK(cudaIpcGetMemHandle(&h, w));
    memcpy(ipc_handle_out, &h, sizeof(h));
    *comm_out = c.release();
    return SLIC_OK;
}

int slic_comm_connect(slic_comm_t* comm, int32_t rank, int32_t world, const void* all_handles) {
    using namespace slic;
    Comm* c = static_cast<Comm*>(comm);
    SLIC_REQUIRE(c && !c->single && !c->connected, "comm_connect: not an unconnected window");
    SLIC_REQUIRE(world >= 1 && world <= COMM_MAX_RANKS && rank >= 0 && rank < world && all_handles,
                 "comm_connect: world must be in [1, 8] and rank in [0, world)");
    unsigned char* own = c->win[0];
    c->win[0] = nullptr;
    c->win[rank] = own;
    c->rank = rank;
    c->world = world;
    for (int g = 0; g < world; ++g) {
        if (g == rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const unsigned char*>(all_handles) + (size_t)g * SLIC_COMM_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        SLIC_CUDA_OK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        c->win[g] = static_cast<unsigned char*>(p);
        c->mapped[g] = true;
    }
    c->connected = true;
    return SLIC_OK;
}

int slic_comm_nn_top1(slic_comm_t* comm, const float* unit_dev, const uint16_t* f16_dev, int64_t n, int32_t d, int32_t d_pad,
                      int32_t* idx_out_dev, float* dist_out_dev, int32_t* status_out_dev, slic_stream_t stream) {
    using namespace slic;
    Comm* c = static_cast<Comm*>(comm);
    SLIC_REQUIRE(c && !c->single && c->connected, "comm_nn_top1: the group is not connected (slic_comm_connect)");
    SLIC_REQUIRE(n > 1 && d > 0 && d_pad >= d && d_pad % 64 == 0, "comm_nn_top1: bad shape");
    SLIC_REQUIRE(unit_dev && f16_dev && idx_out_dev && dist_out_dev && status_out_dev, "comm_nn_top1: null pointer");
    SLIC_REQUIRE((reinterpret_cast<uintptr_t>(f16_dev) & 15) == 0, "comm_nn_top1: f16 matrix must be 16-byte aligned");
    SLIC_PROPAGATE(slic_require_device());
    int dev = -1;
    SLIC_CUDA_OK(cudaGetDevice(&dev));
    SLIC_REQUIRE(dev == c->device, "comm_nn_top1: called on another device than the window lives on");
    cudaStream_t st = as_stream(stream);
    // status_out_dev[0] = rows left without a neighbour, [1] = 1 when some rank's search was incomplete
    SLIC_CUDA_OK(cudaMemsetAsync(status_out_dev, 0, 2 * sizeof(int), st));
    return comm_nn_top1_rank(c, c->rank, ++c->epoch, unit_dev, f16_dev, n, d, d_pad, idx_out_dev, dist_out_dev, status_out_dev,
                             status_out_dev + 1, st);
}

int slic_comm_finch(slic_comm_t* comm, const float* data_dev, int64_t n, int32_t d, int32_t ensure_early_exit,
                    int32_t capacity, int32_t* labels_out_dev, int32_t* num_clust_out_host, int32_t* num_levels_out_host,
                    float* min_sim_out_host, int32_t* has_min_sim_out_host, slic_stream_t stream) {
    using namespace slic;
    Comm* c = static_cast<Comm*>(comm);
    SLIC_REQUIRE(c && !c->single && c->connected, "comm_finch: the group is not connected (slic_comm_connect)");
    SLIC_REQUIRE(n > 1 && n < ((int64_t)1 << 31) && d > 0, "comm_finch: bad shape");
    SLIC_REQUIRE(data_dev && labels_out_dev && num_clust_out_host && num_levels_out_host, "comm_finch: null pointer");
    SLIC_REQUIRE(capacity >= 1, "comm_finch: the label buffer needs at least one column");
    SLIC_PROPAGATE(slic_require_device());
    int dev = -1;
    SLIC_CUDA_OK(cudaGetDevice(&dev));
    SLIC_REQUIRE(dev == c->device, "comm_finch: called on another device than the window lives on");
    if (!screen_self_search_is_symmetric(n) || n > c->max_rows) {
        set_error("comm_finch: the shared search takes 16384 <= n <= max_rows (%lld) rows", (long long)c->max_rows);
        return SLIC_ERR_UNSUPPORTED;
    }
    cudaStream_t st = as_stream(stream);
    const int dp = d_pad_of(d);
    Scratch unit, ub, nn, dist, blk;
    SLIC_CUDA_OK(unit.alloc((size_t)n * d * sizeof(float), st));
    SLIC_CUDA_OK(ub.alloc((size_t)n * dp * 2, st));
    SLIC_CUDA_OK(nn.alloc((size_t)n * sizeof(int), st));
    SLIC_CUDA_OK(dist.alloc((size_t)n * sizeof(float), st));
    SLIC_CUDA_OK(blk.alloc(16 * sizeof(int), st));
    SLIC_CUDA_OK(cudaMemsetAsync(blk.ptr, 0, 16 * sizeof(int), st));
    SLIC_PROPAGATE(slic_normalize_rows(data_dev, n, d, SLIC_F32, unit.ptr, nullptr, ub.as<uint16_t>(), dp, stream));
    SLIC_PROPAGATE(comm_nn_top1_rank(c, c->rank, ++c->epoch, unit.as<float>(), ub.as<uint16_t>(), n, d, dp, nn.as<int>(),
                                     dist.as<float>(), blk.as<int>() + 1, blk.as<int>() + 5, st));
    // levels >= 1, components and means: replicated on every rank (milliseconds), so that every rank holds the labels
    return finch_tail_device(data_dev, n, d, nn.as<int>(), dist.as<float>(), unit.as<float>(), ub.as<uint16_t>(),
                             blk.as<int>(), ensure_early_exit != 0, capacity, labels_out_dev, num_clust_out_host,
                             num_levels_out_host, min_sim_out_host, has_min_sim_out_host, st);
}

int slic_comm_create(const int32_t* devices, int32_t num_devices, int64_t max_rows, slic_comm_t** comm_out) {
    using namespace slic;
    SLIC_REQUIRE(devices && comm_out && num_devices >= 1 && num_devices <= COMM_MAX_RANKS,
                 "comm_create: between 1 and 8 devices of one box");
    SLIC_REQUIRE(max_rows > 0 && max_rows < ((int64_t)1 << 31), "comm_create: bad max_rows");
    SLIC_PROPAGATE(slic_require_device());
    int count = 0, prev = 0;
    SLIC_CUDA_OK(cudaGetDeviceCount(&count));
    SLIC_CUDA_OK(cudaGetDevice(&prev));
    for (int g = 0; g < num_devices; ++g) {
        SLIC_REQUIRE(devices[g] >= 0 && devices[g] < count, "comm_create: device index out of range");
        for (int h = 0; h < g; ++h) SLIC_REQUIRE(devices[h] != devices[g], "comm_create: a device is listed twice");
    }
    Comm* c = new Comm();
    c->single = true;
    c->world = num_devices;
    c->max_rows = max_rows;
    int status = SLIC_OK;
    for (int g = 0; g < num_devices && status == SLIC_OK; ++g) {
        c->devices[g] = devices[g];
        status = [&]() -> int {
            SLIC_CUDA_OK(cudaSetDevice(devices[g]));
            SLIC_PROPAGATE(slic_require_device());
            for (int h = 0; h < num_devices; ++h) {
                if (h == g) continue;
                int can = 0;
                SLIC_CUDA_OK(cudaDeviceCanAccessPeer(&can, devices[g], devices[h]));
                if (!can) {
                    set_error("comm_create: device %d cannot access device %d (no NVLink / P2P path)", devices[g], devices[h]);
                    return SLIC_ERR_UNSUPPORTED;
                }
                const cudaError_t e = cudaDeviceEnablePeerAccess(devices[h], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) SLIC_CUDA_OK(e);
                cudaGetLastError();
            }
            {
                // The [n, d] matrices the workers forward to each other live in the stream-ordered pool (Scratch), which
                // cudaDeviceEnablePeerAccess does not cover: without this grant cudaMemcpyPeerAsync quietly stages every
                // forward through host memory (measured at 2 GPUs, C3: upload + forward 14.5 ms for 246 MB per device,
                // three PCIe crossings instead of one PCIe crossing and one NVLink hop).
                cudaMemPool_t pool;
                SLIC_CUDA_OK(cudaDeviceGetDefaultMemPool(&pool, devices[g]));
                std::vector<cudaMemAccessDesc> grant;
                for (int h = 0; h < num_devices; ++h) {
                    if (h == g) continue;
                    cudaMemAccessDesc a;
                    memset(&a, 0, sizeof(a));
                    a.location.type = cudaMemLocationTypeDevice;
                    a.location.id = devices[h];
                    a.flags = cudaMemAccessFlagsProtReadWrite;
                    grant.push_back(a);
                }
                if (!grant.empty()) SLIC_CUDA_OK(cudaMemPoolSetAccess(pool, grant.data(), grant.size()));
            }
            void* w = nullptr;
            SLIC_CUDA_OK(cudaMalloc(&w, win_bytes(max_rows)));
            c->win[g] = static_cast<unsigned char*>(w);
            SLIC_CUDA_OK(cudaMemset(w, 0, win_bytes(max_rows)));
            SLIC_CUDA_OK(cudaStreamCreateWithFlags(&c->streams[g], cudaStreamNonBlocking));
            SLIC_CUDA_OK(cudaStreamCreateWithFlags(&c->forward[g], cudaStreamNonBlocking));
            for (int p = 0; p < COMM_UPLOAD_PIECES; ++p)
                SLIC_CUDA_OK(cudaEventCreateWithFlags(&c->piece_up[g][p], cudaEventDisableTiming));
            SLIC_CUDA_OK(cudaEventCreateWithFlags(&c->uploaded[g], cudaEventDisableTiming));
            if (g == 0) {
                SLIC_CUDA_OK(cudaEventCreate(&c->t0));
                SLIC_CUDA_OK(cudaEventCreate(&c->t1));
                SLIC_CUDA_OK(cudaEventCreate(&c->t2));
                SLIC_CUDA_OK(cudaEventCreate(&c->t3));
            }
            SLIC_CUDA_OK(cudaDeviceSynchronize());
            return SLIC_OK;
        }();
    }
    cudaSetDevice(prev);
    if (status != SLIC_OK) {
        destroy_comm(c);
        return status;
    }
    c->bar.reset(new HostBarrier(num_devices));
    for (int g = 0; g < num_devices; ++g) c->threads.emplace_back(worker_main, c, g);
    *comm_out = c;
    return SLIC_OK;
}

int slic_finch_multi(slic_comm_t* comm, const float* x_host, int64_t n, int32_t d, const int64_t* initial_rank_host,
                     int32_t ensure_early_exit, int32_t capacity, int32_t* labels_out_host, int32_t* num_clust_out_host,
                     int32_t* num_levels_out_host, float* min_sim_out_host, int32_t* has_min_sim_out_host) {
    using namespace slic;
    Comm* c = static_cast<Comm*>(comm);
    SLIC_REQUIRE(c && c->single, "finch_multi: needs a group made by slic_comm_create");
    SLIC_REQUIRE(n >= 1 && n < ((int64_t)1 << 31) && d > 0, "finch_multi: bad shape");
    SLIC_REQUIRE(x_host && labels_out_host && num_clust_out_host && num_levels_out_host, "finch_multi: null pointer");
    SLIC_REQUIRE(capacity >= 1 && capacity <= 64, "finch_multi: capacity must be in [1, 64]");
    std::lock_guard<std::mutex> call_lock(c->call_mutex);
    if (c->world == 1 || initial_rank_host || !screen_self_search_is_symmetric(n) || n > c->max_rows) {
        // nothing to share (caller-supplied neighbours, a small matrix) or more rows than the windows hold: one GPU
        int prev = 0;
        SLIC_CUDA_OK(cudaGetDevice(&prev));
        SLIC_CUDA_OK(cudaSetDevice(c->devices[0]));
        const int s = finch_host_single(x_host, n, d, initial_rank_host, ensure_early_exit != 0, capacity, labels_out_host,
                                        num_clust_out_host, num_levels_out_host, min_sim_out_host, has_min_sim_out_host);
        cudaSetDevice(prev);
        return s;
    }
    MultiJob job;
    memset(&job, 0, sizeof(job));
    job.x_host = x_host;
    job.n = n;
    job.d = d;
    job.ensure_early_exit = ensure_early_exit != 0;
    job.capacity = capacity;
    job.labels_out_host = labels_out_host;
    job.num_clust_host = num_clust_out_host;
    job.num_levels_host = num_levels_out_host;
    job.min_sim_host = min_sim_out_host;
    job.has_min_sim_host = has_min_sim_out_host;
    {
        std::unique_lock<std::mutex> lk(c->m);
        c->job = &job;
        c->done_count = 0;
        ++c->job_gen;
        c->cv.notify_all();
        c->cv.wait(lk, [&] { return c->done_count == (unsigned)c->world; });
        c->job = nullptr;
    }
    for (int g = 0; g < c->world; ++g) {
        if (job.status[g] != SLIC_OK) {
            set_error("finch_multi: device %d: %s", c->devices[g], job.error[g]);
            return job.status[g];
        }
    }
    c->last_ms[0] = job.ms_upload;
    c->last_ms[1] = job.ms_search;
    c->last_ms[2] = job.ms_total;
    return SLIC_OK;
}

int slic_comm_last_timeline(slic_comm_t* comm, float* ms_out_host) {
    using namespace slic;
    Comm* c = static_cast<Comm*>(comm);
    SLIC_REQUIRE(c && c->single && ms_out_host, "comm_last_timeline: bad arguments");
    for (int i = 0; i < 3; ++i) ms_out_host[i] = c->last_ms[i];
    return SLIC_OK;
}

int slic_comm_destroy(slic_comm_t* comm) {
    slic::destroy_comm(static_cast<slic::Comm*>(comm));
    return SLIC_OK;
}

}  // extern "C"
