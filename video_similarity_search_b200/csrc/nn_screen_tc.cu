// K1-tc: first-neighbour / top-k screen on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), with the per-row
// candidate filter fused into the epilogue so the nq x n score matrix never reaches HBM.
// Replaces the O(n^2 D) sgemm/dgemm + three n^2 elementwise passes + argmin behind
// clustering/finch.py:27-29 (sklearn pairwise_distances -> OpenBLAS).
//
// Work decomposition
//   tile  = 256 x 256 scores, K = d_pad in 64-wide slabs (f16, 128-byte swizzled rows), computed by a CTA PAIR (cluster
//           of 2, tcgen05 cta_group::2): each CTA stages its own 128 query rows of A and half of the B slab, and the
//           leader issues tcgen05.mma M256 N256 K16 that read both halves.  Two 256-column accumulators in TMEM, so the
//           filter of tile t overlaps the MMAs of tile t + 1.
//   unit  = a pair's 256 query rows x a run of column tiles (a column split, or an entry of an explicit unit list).
//   CTA   = persistent, one per SM.  The leader's producer thread draws unit ids from a global counter (dynamic
//           queue) and hands them to every role of both CTAs through the unit ring (TC_UQ_DEPTH slots in shared
//           memory, cluster-scope barriers).  10 warps, 11 for the symmetric kernels:
//           warp 0     TMA producer: A and B slabs into the operand ring (A once per unit when it is resident)
//           warp 1     MMA issuer (the leader's lane 0): commits to the stage's "empty" and the accumulator's "full" barrier
//           warps 2-9  epilogue: tcgen05.ld 32 columns at a time out of TMEM; warp w reads TMEM lanes 32 * (w % 4) and
//                      the 128-column half (w - 2) / 4 of every tile, one thread = one (query row, column half) stream
//           warp 10    SYM only: publishes the column thresholds of the coming tiles
//   Concurrent pairs work on different row blocks of the SAME column range, so every B slab is fetched from HBM once per
//   wave and served to the other SMs from L2.
//
// Template axes of nn_screen_kernel (six instantiations):
//   TOPK  first neighbour, or the k best (per-row score histograms in shared memory)
//   ARES  d_pad <= 512: the unit's A rows stay resident in shared memory and only B streams; wider rows stream both
//   SYM   self-search over the upper triangle of tiles, off-diagonal tiles filtered along rows and columns (top-1 only)
//
// Fused filter (per query row = one epilogue thread, state in registers)
//   best = running maximum of the screened scores seen so far; a column is appended to the row's
//   candidate list iff score >= best - eps at the time it is seen.  Because best only grows, the list
//   is a superset of {j : score_j >= final best - eps}; with eps >= 2 * (max screening error) that set
//   contains the exact first neighbour.  The common case costs one FMNMX3 per two scores plus one
//   compare per 32; appends are rare (O(log n) per row).  A full list is first compacted against the
//   current threshold; only if it is still full is the row flagged and later finished by the exact
//   kernel - the result never depends on f16 precision.
//
// Bound: tensor pipe.  Algorithmic work 2 * nq * n * d_pad flop; HBM traffic ~ (nq + n) * d_pad * 2 bytes.
//
// Variants measured and removed (records under profiles/):
//   128-column tiles with four accumulators: 31.6 against 22.2 ms at C3 (r2_screen_pipeline_trace.txt)
//   L2 prefetch of the B slabs ahead of the ring: 23.3 -> 24.3 ms at C3 (r2_screen_pipeline_trace.txt)
//   static unit striding instead of the dynamic queue: round 1 row of r2_screen_pipeline_trace.txt
//   one box-wide unit queue for a multi-GPU search: slower than fixed shares (r2_runs/exp_sq8.log)
//   single-CTA 128 x 256 tiles: a third more L2 -> SM operand traffic per flop than a pair (r2_ptxas_table.txt lists them)
//   column-chunk width of the symmetric plan: 64 tiles is the fastest (r2_runs/exp_chunk.log)
#include <cuda.h>
#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <math_constants.h>

#include <algorithm>
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace slic {

constexpr int TC_BM = 128, TC_BK = 64, TC_UMMA_K = 16;
// Column-tile width: two 256-column accumulators in TMEM, every epilogue warp filters one 128-column half of EVERY tile.
constexpr int TC_BN = 256;
// K slabs per ring stage of the A-resident kernels.  2 = three 32 KB stages, 8 MMAs per barrier round trip.  (1 = six 16 KB
// stages was measured in round 2 at C3: operand wait of the MMA issuer 15 % -> 25 %, kernel 22.6 -> 24.1 ms: the finer
// hand-over costs more in round trips than it gains in ring occupancy.)
constexpr int TC_ARES_SPS = 2;
constexpr int TC_ROW_UNIT = 256;   // rows of a CTA pair's unit (the symmetric planner counts row units and column tiles)
static_assert(TC_ROW_UNIT == TC_BN, "a row unit's diagonal block is one column tile");
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 2;   // 16 KB
// Each CTA of a pair stages its own 128 query rows of A and HALF of the B slab (16 KB); the tensor cores of both SMs read
// both halves.
// ARES (d_pad <= 512): the unit's A rows (128 x d_pad f16 <= 128 KB) are loaded ONCE per unit and stay resident; only B
//           slabs stream through the ring.  A is the one operand no other SM shares, so this removes most of the
//           L2 -> SM traffic that bounds the streaming variants.
constexpr int TC_ARES_MAX_SLABS = 8;
// barrier block behind the operands: 38 eight-byte slots (pipeline barriers, TMEM slot, log counters, unit ring)
constexpr uint32_t TC_BAR_BYTES = 384;
constexpr int TC_UQ_DEPTH = 4;   // unit ring: ids of the units the scheduler has handed out, consumed in order by every role
constexpr int TC_TMEM_COLS = 512;
constexpr int TC_ACCS = TC_TMEM_COLS / TC_BN;   // accumulators in TMEM
template <bool ARES, bool TOPK> struct TcCfg {
    static constexpr uint32_t B_ROWS = TC_BN / 2;
    static constexpr uint32_t B_BYTES = B_ROWS * TC_BK * 2;
    static constexpr uint32_t A_RES_BYTES = ARES ? TC_ARES_MAX_SLABS * TC_A_BYTES : 0;      // 128 KB
    // K slabs per ring stage: the A-resident top-1 kernel moves two (32 KB of B per CTA and barrier round trip,
    // 8 MMAs per wait / commit); the top-k variant has 32 KB less shared memory and keeps four single-slab stages
    static constexpr int SPS = ARES ? TC_ARES_SPS : 2;
    static constexpr uint32_t SLAB_BYTES = ARES ? B_BYTES : TC_A_BYTES + B_BYTES;   // one K slab of a stage
    static constexpr uint32_t STAGE_BYTES = SPS * SLAB_BYTES;
    // A-resident: 96 KB (64 KB with the top-k histograms) of ring behind the 128 KB of A rows
    static constexpr int STAGES = ARES ? (TOPK ? 64 : 96) * 1024 / (int)STAGE_BYTES : 3;
    static_assert(STAGES >= 2 && STAGES <= 6, "ring depth");
    static constexpr uint32_t OPERAND_BYTES = A_RES_BYTES + STAGES * STAGE_BYTES;            // 192 KB, ARES: 192 / 224 KB
    static constexpr uint32_t SMEM_BYTES = OPERAND_BYTES + TC_BAR_BYTES /*barriers, unit ring*/ + 960 /*alignment slack*/ +
                                           (TOPK ? 32768u : 0u) /*histograms*/;
    // symmetric variant: + 1 KB of column thresholds (float16, rounded down); the A-resident layout then leaves 640
    // bytes of alignment slack.  An SM has 228 KB of shared memory and every resident CTA reserves 1 KB of it: a
    // window above 226 KB would own the SM outright, and the kernels that feed a gated launch from another stream
    // (normalise, gate memset) could never become resident next to it - the launch would wait for itself.
    static constexpr uint32_t SYM_THR_BYTES = 2 * 2 * 128 * 2;   // [2 parities][2 halves][128 columns] float16
    static constexpr uint32_t SYM_SMEM_BYTES = OPERAND_BYTES + TC_BAR_BYTES + SYM_THR_BYTES + (ARES ? 640u : 960u);
    static constexpr uint32_t CORESIDENT_MAX_BYTES = 233472 - 2 * 1024;
    static_assert(TOPK || SYM_SMEM_BYTES <= CORESIDENT_MAX_BYTES,
                  "symmetric variant leaves no shared memory for a co-resident CTA of the upload stream");
    static_assert(TOPK || SMEM_BYTES <= CORESIDENT_MAX_BYTES,
                  "top-1 variant (gated launches) leaves no shared memory for a co-resident CTA of the upload stream");
    static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of shared memory a CTA may use");
};
constexpr int TC_MAX_STAGES = 6;
constexpr int TC_EPI_WARPS = 8;   // two per TMEM lane quadrant: each takes one 128-column half of every tile
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;
// Symmetric kernels: an eleventh warp does nothing but publish the column thresholds of the coming tiles (two tiles
// ahead, double-buffered, mbarrier hand-shake), so that no epilogue warp ever waits for another one at a tile boundary.
// (Before: the first epilogue warp of each 128-column half wrote them and the half met at a named barrier per tile -
// measured at 22 % of the epilogue's stall samples, profiles/r1_sym_screen_kernel_ncu_full.txt.)
constexpr int TC_THREADS_SYM = TC_THREADS + 32;
// Screen operands are IEEE half precision (float16: 11 significant bits; kind::f16 runs float16 and bfloat16 at the same
// rate, and unit-vector components never leave float16's range).  Error allowance for unit rows: a component >= 2^-14
// carries relative rounding error <= 2^-11, a product of two <= 2^-10 (+ 2^-22), so the sum over k is off by
// <= 2^-10 * sum|a_k b_k| <= 2^-10; components in the subnormal range add <= 2^-25 each, <= 2^-18 in total for
// d <= 4096; the tensor core's float32 accumulation (products exact, additions possibly truncated) adds <= d * 2^-23
// <= 2^-11.  eps must be >= twice the worst-case |screened - exact|: 2 * (2^-10 + 2^-11 + 2^-18) < 2^-9 + 2^-10 + 2^-16.
// (The first version screened in bfloat16 with eps = 2^-7 + 2^-11: 2.8 x as wide a band, several times the candidates.)
constexpr float TC_DEFAULT_EPS = 0.001953125f + 0.0009765625f + 0.0000152587890625f;
// Wider rows (d_pad > 4096).  For any width the worst case is, term by term:
//   rounding of the normal components      (2^-10 + 2^-22) * sum|a_k b_k| <= 2^-10 + 2^-22
//   subnormal components                   2^-25 * (sum|a_k| + sum|b_k|) <= 2^-24 * sqrt(d_pad)   (Cauchy-Schwarz)
//   float32 accumulation                   d_pad * 2^-23 * max|partial sum| <= d_pad * 2^-23 * (1 + 2^-9)
// Twice that is 2^-9 + d_pad * 2^-22 + (2^-21 + 2^-23 * sqrt(d_pad) + d_pad * 2^-31), and the bracket is <= d_pad * 2^-28
// for every d_pad >= 4096 (at 4096: 1.00e-5 <= 1.53e-5, and the right side grows faster).  So
//   eps(d_pad) = 2^-9 + d_pad * (2^-22 + 2^-28)
// covers the bound at every width above 4096, grows with the accumulation term and equals TC_DEFAULT_EPS at 4096, where
// the two rules meet.  Up to 4096 the constant is kept as it is.
static float screen_default_eps(int d_pad) {
    if (d_pad <= 4096) return TC_DEFAULT_EPS;
    return (float)(0.001953125 + (double)d_pad * (0x1p-22 + 0x1p-28));
}
constexpr int TC_TOPK_MAX = 64;  // the top-k variant's per-row score histogram has saturating 8-bit counts: k must stay well below 255
constexpr int TC_HIST_BINS = 128;
constexpr int TC_HIST_STRIDE = 2 * TC_BM;   // one histogram per (row, column half)
constexpr uint32_t TC_TOPK_SMEM = TC_HIST_BINS * TC_HIST_STRIDE;  // 128 bins x 256 epilogue threads x uint8 = 32 KB
static_assert(TC_TOPK_SMEM == 32768, "TcCfg::SMEM_BYTES assumes 32 KB of histograms");

struct ScreenParams {
    int64_t nq, n;
    int num_k_slabs;       // d_pad / 64
    int64_t self_offset;   // query row r is database row r + self_offset (excluded); < 0: no exclusion
    float eps;
    int cap;               // candidate slots per (split, row)
    int splits;
    int tiles_per_split;   // 256-column tiles per split
    int64_t num_units;     // row blocks * splits
    int* cand_idx;         // [2 * splits][nq][cap]   (stream = split * 2 + column half of the tiles)
    float* cand_score;     // [2 * splits][nq][cap]
    int* cand_cnt;         // [2 * splits][nq]
    int* cand_flags;       // [2 * splits][nq]  bit0 = overflow, bit1 = compacted
    int topk;              // TOPK kernel: k (<= TC_TOPK_MAX); the candidate rule is "within eps of the k-th best"
    float* cand_kth;       // TOPK kernel: [splits][nq] lower bound of the split's k-th best screened score
    // TOPK kernel: [2 * splits][nq] the same bound as a histogram bin, ZEROED before the launch.  A stream (row, split,
    // half) publishes its final bin here and every stream STARTS from the highest bin any other stream of its row has
    // published: the k-th best over a subset of the columns is a lower bound of the k-th best over all of them, so the
    // seeded threshold is as valid as the stream's own - and with split-major units the streams of split s - 1 have
    // finished when those of split s start, which spares them the listing of their first tile and the whole threshold
    // ramp (~k ln(columns / 128) listings per stream).
    int* cand_tb;
    float* dump;           // debug: raw scores [nq][n] or nullptr
    int* error_flag;       // set when a barrier wait times out
    unsigned long long* trace;  // optional [8] cycle counters summed over CTAs (diagnostic, see slic_screen_trace)
    // Optional explicit unit list (gated and symmetric launches): entry u = {row unit, first column tile,
    // tile count | tile stride << 16, (gate + 1) | stream << 12 | column-direction flag << 28}.
    // A unit with gate g may only start once gates[g] != 0 - the rows of database chunk g (and of every earlier
    // chunk) have landed in HBM and been normalised by another stream while this kernel is already running.
    const int4* unit_table;
    const int* gates;
    // Symmetric self-search (SYM kernels): best_enc[r] = order-preserving encoding of the best screened score any CTA
    // has seen so far for row r.  Candidates go to a log: cand_idx = neighbour, cand_score = score, log_q = query row,
    // one region of log_region records per epilogue warp; cand_cnt[region] = records written, cand_flags[0] = overflow.
    unsigned int* best_enc;
    int* log_q;
    int log_region;
    // pre-pass -> triangle hand-over: every epilogue warp adds 1 to sync_counter when it finishes a pre-pass unit; a
    // triangle unit with gate g starts once the counter has reached sync_targets[g + 1] (all pre-pass units of the
    // chunks it touches), so that the column thresholds it reads are in place.  Affects speed only, never results.
    int* sync_counter;
    const int* sync_targets;
    // Dynamic scheduling: units are handed out in list order from this global counter (zeroed before the launch) to
    // whichever CTA pair becomes free - no pair idles while another still holds a queue of long units.
    int* queue;
    // Multi-GPU fused search (comm.cu): the pre-pass units of this rank publish their rows' bests into the best arrays
    // of the OTHER ranks as well (red.max over NVLink peer mappings) and count their arrivals on every rank's
    // sync_counter, so the triangle units of every rank start from thresholds for ALL rows - the exchange that used to
    // be a separate launch + all-reduce happens inside the one kernel.
    int num_peers;
    unsigned int* peer_best[SLIC_MAX_PEERS];
    int* peer_sync[SLIC_MAX_PEERS];
};

struct UnitInfo {
    int64_t row_unit;   // index of the unit's row-block pair
    int64_t ct0;        // first column tile
    int count, stride;  // tiles ct0 + k * stride, k < count
    int gate;           // -1: none
    int stream;         // candidate stream (column split) of the non-symmetric kernels
    bool coldir;        // SYM: tiles right of the diagonal also serve their columns as queries
};
__device__ __forceinline__ UnitInfo unit_info(const ScreenParams& p, int64_t u, int64_t n_col_tiles) {
    UnitInfo ui;
    if (p.unit_table) {
        const int4 e = __ldg(p.unit_table + u);
        ui.row_unit = e.x;
        ui.ct0 = e.y;
        ui.count = e.z & 0xffff;
        ui.stride = (int)((unsigned)e.z >> 16);
        ui.gate = (e.w & 0xfff) - 1;
        ui.stream = (e.w >> 12) & 0xffff;
        ui.coldir = ((e.w >> 28) & 1) != 0;
    } else {
        // Split-major: all row units of column split 0 first, then split 1, ...  The CTA pairs that run concurrently then
        // stream ONE column range and serve each other through L2 whatever their phases (with 74 pairs spread over a range,
        // every pair follows another within a few tiles).  Round 1 dealt the splits round-robin: three concurrent streams of
        // ~25 pairs each, gaps of ~50 tiles against an L2 window of ~27 - measured on the top-50 search of 100 000 x
        // 1 000 000 x 1 024 (ncu): 600 GB of DRAM reads per launch for 2 GB of operands, L2 hit rate 62 %, and the SM clock
        // pushed down to 1.0 GHz by the power the HBM drew.
        const int64_t row_units = p.num_units / p.splits;
        const int split = (int)(u / row_units);
        ui.row_unit = u % row_units;
        ui.ct0 = (int64_t)split * p.tiles_per_split;
        const int64_t left = n_col_tiles - ui.ct0;
        ui.count = (int)(left < p.tiles_per_split ? (left > 0 ? left : 0) : p.tiles_per_split);
        ui.stride = 1;
        ui.gate = -1;
        ui.stream = split;
        ui.coldir = false;
    }
    return ui;
}

// order-preserving map float -> uint32 (atomicMax / warp-reduce on scores of either sign); enc(-inf) = 0x007fffff
__device__ __forceinline__ unsigned enc_score(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_score(unsigned e) {
    return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e);
}
constexpr unsigned ENC_NEG_INF = 0x007fffffu;

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Post-mortem of a timed-out wait: a trap kills the context, so the record goes to MAPPED HOST memory (readable after
// the failure): {site, block, thread, a, b}.  site 1 = mbarrier (a = smem address, b = parity), 2 = upload gate
// (a = gate address low bits), 3 = pre-pass counter (a = value seen, b = target).  First writer wins.
__device__ int* g_timeout_record = nullptr;
__device__ int g_timeout_lock = 0;
__device__ __noinline__ void record_timeout(int site, int a, int b) {
    int* r = g_timeout_record;
    if (r && atomicCAS(&g_timeout_lock, 0, 1) == 0) {
        volatile int* v = r;
        v[1] = (int)blockIdx.x;
        v[2] = (int)threadIdx.x;
        v[3] = a;
        v[4] = b;
        v[0] = site;
        __threadfence_system();
    }
}

// Bounded wait: a protocol bug must not hang the GPU - after ~4 s the kernel flags the error and traps.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* error_flag) {
    uint32_t done = 0;
    long long t0 = 0;
    uint32_t polls = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
        if ((++polls & 0x3ff) == 0) {
            long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 8000000000ll) {
                if (error_flag) atomicExch(error_flag, 1);
                record_timeout(1, (int)bar, (int)parity);
                __trap();
            }
        }
    }
}
// wait + add the stall cycles to a trace slot (only when tracing)
__device__ __forceinline__ void mbar_wait_traced(uint32_t bar, uint32_t parity, int* error_flag, unsigned long long& acc,
                                                 bool tracing) {
    if (!tracing) {
        mbar_wait(bar, parity, error_flag);
        return;
    }
    const long long t0 = clock64();
    mbar_wait(bar, parity, error_flag);
    acc += (unsigned long long)(clock64() - t0);
}
// non-blocking probe of a barrier phase (one poll)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done != 0;
}
// Block until another stream has published database chunk `g` (a 32-bit flag written after the chunk's normalise
// kernel completed).  The acquire orders the flag read before this thread's later operations in the generic proxy;
// the proxy fence extends that to the TMA (async proxy) reads of the chunk that follow.
// The wait is bounded and NEVER traps: whether the upload's kernels become resident next to this persistent kernel is
// the scheduler's decision (CUDA_LAUNCH_BLOCKING, a tool that serialises kernels, MPS time slicing or a slow host can
// all keep the gate shut).  After ~2 s the kernel sets *error_flag = SCREEN_ERR_GATE and carries on with whatever the
// buffers hold - allocated memory, so nothing faults and the pipeline protocol is untouched; every later gate wait
// returns at once.  The host sees the flag, discards the result and repeats the search after the upload (finch_driver.cu).
constexpr int SCREEN_ERR_GATE = 3;
__device__ __forceinline__ void gate_wait(const int* gate, int* error_flag) {
    long long t0 = 0;
    uint32_t polls = 0;
    while (true) {
        int v;
        asm volatile("ld.acquire.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(gate) : "memory");
        if (v != 0) break;
        __nanosleep(256);
        if ((++polls & 0xff) == 0) {
            if (error_flag && *reinterpret_cast<volatile int*>(error_flag) == SCREEN_ERR_GATE) break;   // given up already
            long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) {   // ~2 s (well inside the 8e9-cycle bound of the mbarrier waits behind it)
                if (error_flag) atomicCAS(error_flag, 0, SCREEN_ERR_GATE);
                record_timeout(2, (int)(reinterpret_cast<uintptr_t>(gate) & 0xffff), v);
                break;
            }
        }
    }
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
// Pre-pass hand-over.  In a multi-GPU fused search the counter also collects the arrivals of the OTHER ranks' kernels,
// so - like a gate - it depends on work this kernel does not control: bounded, never traps.  (Thresholds read too early
// only cost speed, never results; the flag makes the host repeat the search anyway, since a rank may be missing.)
__device__ __forceinline__ void counter_wait(const int* counter, int target, int* error_flag) {
    long long t0 = 0;
    uint32_t polls = 0;
    while (true) {
        int v;
        asm volatile("ld.acquire.sys.global.b32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");   // (peers add over NVLink)
        if (v >= target) break;
        __nanosleep(128);
        if ((++polls & 0xff) == 0) {
            if (error_flag && *reinterpret_cast<volatile int*>(error_flag) == SCREEN_ERR_GATE) break;
            long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) {
                if (error_flag) atomicCAS(error_flag, 0, SCREEN_ERR_GATE);
                record_timeout(3, v, target);
                break;
            }
        }
    }
}
// shared::cluster address of the same smem offset in the pair's leader CTA (rank 0): clear the peer bit
constexpr uint32_t TC_PEER_BIT_MASK = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint32_t dst, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(leader_bar & TC_PEER_BIT_MASK)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & TC_PEER_BIT_MASK) : "memory");
}
// cluster-scope forms for the unit ring: the scheduler writes the peer CTA's ring slot, then arrives on the peer's barrier
__device__ __forceinline__ uint32_t peer_smem_addr(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_u32(uint32_t cluster_addr, uint32_t v) {
    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
__device__ __forceinline__ void mbar_arrive_release_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity, int* error_flag) {
    uint32_t done = 0;
    long long t0 = 0;
    uint32_t polls = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
        if ((++polls & 0x3ff) == 0) {
            long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 40000000000ll) {   // (a waiting role may legitimately sit behind a gated upload)
                if (error_flag) atomicExch(error_flag, 1);
                record_timeout(4, (int)bar, (int)parity);
                __trap();
            }
        }
    }
}
// Unit ring, consumer side.  Every role of a CTA pair (producers, MMA issuer, epilogue warps, threshold warp) walks the
// SAME sequence of unit ids: the scheduler (the leader CTA's producer thread) draws them from the global queue and
// writes them into slot k % TC_UQ_DEPTH of both CTAs' rings; a slot is reused once every reader of the pair has
// arrived on the leader's "empty" barrier.  Called by one thread, or by all lanes of a warp together.
struct UnitRing {
    uint32_t full, val;        // own CTA's barriers / values
    uint32_t empty_leader;     // shared::cluster address of the leader's "empty" barriers
    int slot;
    uint32_t phase;
};
__device__ __forceinline__ int ring_take(UnitRing& r, bool whole_warp, int* error_flag) {
    mbar_wait_cluster(r.full + 8u * r.slot, r.phase, error_flag);
    int u;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(u) : "r"(r.val + 4u * r.slot) : "memory");
    if (whole_warp) __syncwarp();   // every lane holds the id before the slot is released
    if (!whole_warp || (threadIdx.x & 31) == 0) mbar_arrive_release_cluster(r.empty_leader + 8u * r.slot);
    if (++r.slot == TC_UQ_DEPTH) {
        r.slot = 0;
        r.phase ^= 1u;
    }
    return u;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once the MMAs issued so far retire) on the barrier at this smem offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"((uint16_t)3)
        : "memory");
}
// TMEM -> registers, 32 lanes x 32 columns per warp.  Issue and wait are separate so that the load of the next
// 32-column chunk is in flight while the current one is filtered; the wait names the registers as in/out operands
// so that no use of them can be scheduled above it.
#define SLIC_V32_OUT(v)                                                                                              \
    "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),     \
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),      \
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),     \
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
#define SLIC_V32_INOUT(v)                                                                                            \
    "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),     \
        "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]),      \
        "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]),     \
        "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
__device__ __forceinline__ void tmem_ld_issue(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
        "%29,%30,%31}, [%32];"
        : SLIC_V32_OUT(v)
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" : SLIC_V32_INOUT(v)::"memory");
}

// K-major, 128-byte-swizzled operand tile (rows of 64 f16 = 128 B, 8-row groups 1024 B apart):
//   bits [0,14) start address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major, 1),
//   [32,46) stride byte offset >> 4 (1024 B), [46,48) descriptor version 1 (sm_100), [61,64) layout 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::f16 instruction descriptor: D=f32 (bits 4-5 = 1), A=B=float16 (format fields at bits 7-9 and 10-12 = 0; 1 would
// be bfloat16), both K-major, N >> 3 at bits 17-22, M >> 4 at bits 24-28.
// cta_group::2: the instruction spans both CTAs, M = 256
constexpr uint32_t TC_IDESC = (1u << 4) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)((2 * TC_BM) >> 4) << 24);

// ---- candidate list maintenance (slow path, rare) -------------------------------------------
struct RowState {
    float best, thr;
    int cnt, flags;
};

__device__ __noinline__ RowState push_candidate(RowState st, float s, int col, float eps, int cap,
                                                int* __restrict__ li, float* __restrict__ ls) {
    if (s > st.best) {
        st.best = s;
        st.thr = s - eps;
    }
    if (st.cnt == cap) {
        // compact against the current threshold (entries appended under an older, lower threshold)
        int w = 0;
        for (int r = 0; r < st.cnt; ++r) {
            const float sc = ls[r];
            if (sc >= st.thr) {
                ls[w] = sc;
                li[w] = li[r];
                ++w;
            }
        }
        st.cnt = w;
        st.flags |= 2;
    }
    if (st.cnt < cap) {
        ls[st.cnt] = s;
        li[st.cnt] = col;
        ++st.cnt;
    } else {
        st.flags |= 1;  // genuinely more than cap columns within eps of the best: exact kernel finishes the row
    }
    return st;
}

// ---- symmetric self-search: candidate log ---------------------------------------------------------------
// A row is met by many CTAs (as a row of its own units, as a column of every row unit left of it), so its candidates
// cannot live in one thread's private list.  Every epilogue warp instead appends (query, neighbour, score) records to
// its own region of a global log with plain stores - the slot comes from a shared-memory counter, nothing waits for
// HBM - and publishes improved row bests with a fire-and-forget atomic max.  The re-rank kernels then keep the records
// within eps of the row's final best.  A full region raises a flag and the caller repeats the search on the full square.
struct LogCtx {
    int* q;            // this warp's region of the log
    int* nb;
    float* s;
    unsigned int* cnt; // shared-memory record counter of this warp
    int region;        // records per region
    int* overflow;
};
// (arguments by value: a reference would force the caller's whole epilogue context into local memory)
__device__ __noinline__ void log_append_raw(int* lq, int* lnb, float* ls, unsigned int* cnt, int region, int* overflow,
                                            unsigned int* best_enc, int q, int nb, float s) {
    const unsigned pos = atomicAdd(cnt, 1u);
    if (pos < (unsigned)region) {
        lq[pos] = q;
        lnb[pos] = nb;
        ls[pos] = s;
    } else {
        *overflow = 1;
    }
    if (best_enc) atomicMax(best_enc + q, enc_score(s));   // result unused: compiles to RED, no round trip
}
__device__ __forceinline__ void log_append(const LogCtx& lg, unsigned int* best_enc, int q, int nb, float s) {
    log_append_raw(lg.q, lg.nb, lg.s, lg.cnt, lg.region, lg.overflow, best_enc, q, nb, s);
}
// Top-k variant of the row state.  Instead of the k running best scores themselves the row keeps a 128-bin
// histogram of the scores it has seen or listed (shared memory, uint8, h[bin * TC_HIST_STRIDE]; bin b >= 1 covers
// [b / 128, (b + 1) / 128), bin 0 everything below 2^-7).  tb is the highest bin with at least k listed scores at or
// above its lower edge, so edge(tb) <= (k-th best screened score so far); cge counts the listed scores in bins
// >= tb and ctb those in bin tb itself (registers).  Bins above tb hold < k <= 64 entries, so the 8-bit counts
// cannot wrap where they are read.  A column is a candidate iff score >= edge(tb) - eps when it is seen: edge(tb)
// only grows, so the list is a superset of {j : score_j >= final k-th best - eps}, which (|screen error| <= eps / 2)
// contains the exact top-k.  (A row whose k-th best similarity is not positive keeps edge = -1, lists every
// column, overflows and is finished by the exact kernel.)
struct RowStateK {
    float thr;
    int tb, cge, ctb, cnt, flags;
};

__device__ __forceinline__ int score_bin(float s) {
    const int b = __float2int_rd(s * (float)TC_HIST_BINS);
    return min(max(b, 0), TC_HIST_BINS - 1);
}
__device__ __forceinline__ float bin_edge(int b) { return b == 0 ? -1.0f : (float)b * (1.0f / (float)TC_HIST_BINS); }

// count one listed score; returns true when tb may have to advance
__device__ __forceinline__ bool hist_insert(RowStateK& st, uint8_t* __restrict__ h, float s, int k) {
    const int b = score_bin(s);
    if (b > st.tb) {
        h[b * TC_HIST_STRIDE] = (uint8_t)(h[b * TC_HIST_STRIDE] + 1);
        ++st.cge;
        return st.cge - st.ctb >= k;
    }
    if (b == st.tb) {
        ++st.cge;
        ++st.ctb;
    }
    return false;
}
__device__ __forceinline__ void hist_advance(RowStateK& st, const uint8_t* __restrict__ h, int k, float eps) {
    while (st.cge - st.ctb >= k) {   // at the last bin: cge == ctb
        st.cge -= st.ctb;
        ++st.tb;
        st.ctb = h[st.tb * TC_HIST_STRIDE];
    }
    st.thr = bin_edge(st.tb) - eps;
}

// `count`: also enter the score into the histogram (false while the unit's first tile is being listed - the
// bootstrap pass has already counted every column of that tile).
__device__ __noinline__ RowStateK push_candidate_topk(RowStateK st, float s, int col, float eps, int cap, int k,
                                                      bool count, uint8_t* __restrict__ h, int* __restrict__ li,
                                                      float* __restrict__ ls) {
    if (st.cnt == cap) {
        int w = 0;
        for (int r = 0; r < st.cnt; ++r) {
            const float sc = ls[r];
            if (sc >= st.thr) {
                ls[w] = sc;
                li[w] = li[r];
                ++w;
            }
        }
        st.cnt = w;
        st.flags |= 2;
    }
    if (st.cnt < cap) {
        ls[st.cnt] = s;
        li[st.cnt] = col;
        ++st.cnt;
    } else {
        st.flags |= 1;
    }
    if (count && hist_insert(st, h, s, k)) hist_advance(st, h, k, eps);
    return st;
}

// Listing a column is ~45 dependent instructions executed by ONE lane of a lone warp (each lane owns a different
// row), i.e. ~250 cycles per listed column if done on the spot.  Triggered columns are therefore parked in four
// registers per lane and listed in batches when some lane's buffer fills: all lanes with parked columns then run
// the listing code together.  The threshold is stale for parked columns, which only makes the list a superset.
struct Pending {
    float s0, s1, s2, s3;
    int c0, c1, c2, c3;
    int n;
};
__device__ __forceinline__ void pend_put(Pending& pd, float s, int col) {
    if (pd.n == 0) {
        pd.s0 = s;
        pd.c0 = col;
    } else if (pd.n == 1) {
        pd.s1 = s;
        pd.c1 = col;
    } else if (pd.n == 2) {
        pd.s2 = s;
        pd.c2 = col;
    } else {
        pd.s3 = s;
        pd.c3 = col;
    }
    ++pd.n;
}
__device__ __forceinline__ void pend_flush(Pending& pd, RowStateK& st, float eps, int cap, int k, bool count,
                                           uint8_t* __restrict__ h, int* __restrict__ li, float* __restrict__ ls) {
    if (pd.n > 0) st = push_candidate_topk(st, pd.s0, pd.c0, eps, cap, k, count, h, li, ls);
    if (pd.n > 1) st = push_candidate_topk(st, pd.s1, pd.c1, eps, cap, k, count, h, li, ls);
    if (pd.n > 2) st = push_candidate_topk(st, pd.s2, pd.c2, eps, cap, k, count, h, li, ls);
    if (pd.n > 3) st = push_candidate_topk(st, pd.s3, pd.c3, eps, cap, k, count, h, li, ls);
    pd.n = 0;
}

// float16 threshold (low / high half of w) minus a float32 score in ONE instruction (FHADD, sm_100 mixed precision);
// the difference of two nearby floats is exact, so (t - s <= 0) <=> (s >= t)
__device__ __forceinline__ float thr_lo_minus(uint32_t w, float s) {
    float d;
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tsub.rn.f32.f16 %0, lo, %2;\n\t}" : "=f"(d) : "r"(w), "f"(s));
    return d;
}
__device__ __forceinline__ float thr_hi_minus(uint32_t w, float s) {
    float d;
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tsub.rn.f32.f16 %0, hi, %2;\n\t}" : "=f"(d) : "r"(w), "f"(s));
    return d;
}

// ---- per-thread epilogue context and the filter of one 32-column chunk ----------------------------
template <bool TOPK>
struct EpiCtx {
    const ScreenParams* p;
    typename std::conditional<TOPK, RowStateK, RowState>::type st;
    Pending pd;          // TOPK only
    uint8_t* hist;       // TOPK only
    int* li;
    float* ls;
    int64_t row, self_col;
    bool row_ok, count, tracing;
    unsigned long long n_trig, n_chunks;
    LogCtx lg;           // SYM only
};

template <bool TOPK, bool SYM>
__device__ __forceinline__ void epi_chunk(EpiCtx<TOPK>& cx, uint32_t (&v)[32], int64_t col_base, bool plain,
                                          bool cdir = false, uint32_t thr_s = 0u /* shared-memory address */) {
    const ScreenParams& p = *cx.p;
    if (!plain) {   // warp-uniform: the tile touches the end of the database, holds the rows' own columns, or is dumped
        if (col_base >= p.n) return;  // whole chunk is padding
        if (col_base + 32 > p.n || (cx.self_col >= col_base && cx.self_col < col_base + 32)) {
#pragma unroll
            for (int t = 0; t < 32; ++t)
                if (col_base + t >= p.n || col_base + t == cx.self_col) v[t] = __float_as_uint(-CUDART_INF_F);
        }
        if (p.dump && cx.row_ok) {
#pragma unroll
            for (int t = 0; t < 32; ++t)
                if (col_base + t < p.n) p.dump[cx.row * p.n + col_base + t] = __uint_as_float(v[t]);
        }
    }
    if constexpr (TOPK) {
        float g[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            g[q] = __uint_as_float(v[8 * q]);
#pragma unroll
            for (int t = 1; t < 8; ++t) g[q] = fmaxf(g[q], __uint_as_float(v[8 * q + t]));
        }
        const float m = fmaxf(fmaxf(g[0], g[1]), fmaxf(g[2], g[3]));
        if (cx.tracing) {
            ++cx.n_chunks;
            cx.n_trig += __any_sync(0xffffffffu, cx.row_ok && m >= cx.st.thr) ? 1 : 0;
        }
        if (cx.row_ok && m >= cx.st.thr) {
            // rare path, kept small (the whole epilogue must stay inside the instruction cache): per group of 8
            // columns take the maximum while it qualifies, park it, blank it, repeat
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float gm = g[q];
                while (gm >= cx.st.thr && gm > -CUDART_INF_F) {
                    int ga = 0;
                    float best = __uint_as_float(v[8 * q]);
#pragma unroll
                    for (int t = 1; t < 8; ++t) {
                        const float s = __uint_as_float(v[8 * q + t]);
                        if (s > best) {
                            best = s;
                            ga = t;
                        }
                    }
                    const int col = (int)(col_base + 8 * q + ga);
                    if (cx.pd.n < 4)
                        pend_put(cx.pd, best, col);
                    else
                        cx.st = push_candidate_topk(cx.st, best, col, p.eps, p.cap, p.topk, cx.count, cx.hist, cx.li,
                                                    cx.ls);
                    gm = -CUDART_INF_F;
#pragma unroll
                    for (int t = 0; t < 8; ++t) {
                        if (t == ga) v[8 * q + t] = __float_as_uint(-CUDART_INF_F);
                        gm = fmaxf(gm, __uint_as_float(v[8 * q + t]));
                    }
                }
            }
        }
        if (__any_sync(0xffffffffu, cx.pd.n >= 3))
            pend_flush(cx.pd, cx.st, p.eps, p.cap, p.topk, cx.count, cx.hist, cx.li, cx.ls);
    } else {
        // group maxima (8 columns each) first: the rare paths below only look inside groups that qualify
        float g[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            g[q] = __uint_as_float(v[8 * q]);
#pragma unroll
            for (int t = 1; t < 8; ++t) g[q] = fmaxf(g[q], __uint_as_float(v[8 * q + t]));
        }
        const float m = fmaxf(fmaxf(g[0], g[1]), fmaxf(g[2], g[3]));
        if (cx.row_ok && m >= cx.st.thr) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (g[q] < cx.st.thr) continue;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    const float s = __uint_as_float(v[8 * q + t]);
                    if (s >= cx.st.thr && s > -CUDART_INF_F) {
                        if constexpr (SYM) {
                            if (s > cx.st.best) {
                                cx.st.best = s;
                                cx.st.thr = s - p.eps;
                            }
                            log_append(cx.lg, nullptr, (int)cx.row, (int)(col_base + 8 * q + t), s);   // best published at unit end
                        } else {
                            cx.st = push_candidate(cx.st, s, (int)(col_base + 8 * q + t), p.eps, p.cap, cx.li, cx.ls);
                        }
                    }
                }
            }
        }
        if constexpr (SYM) {
            if (cdir) {
                // column role.  thr[t] (shared memory, float16, written once per tile) = threshold of column col_base + t.
                // Every thread takes the minimum of (column threshold - score) over its row's 32 columns - the exact test, so
                // that the per-column spread of the thresholds cancels (block-level tests against the lowest threshold of a
                // group of columns were measured: they fire for 40-56 % of the blocks) - and only a row with a
                // non-positive margin looks closer.
                float mc = CUDART_INF_F;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t w0, w1, w2, w3;   // 8 thresholds (explicit ld.shared: a generic load would go the slow way round)
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3)
                                 : "r"(thr_s + 16u * j));
                    mc = fminf(mc, fminf(thr_lo_minus(w0, __uint_as_float(v[8 * j])), thr_hi_minus(w0, __uint_as_float(v[8 * j + 1]))));
                    mc = fminf(mc, fminf(thr_lo_minus(w1, __uint_as_float(v[8 * j + 2])), thr_hi_minus(w1, __uint_as_float(v[8 * j + 3]))));
                    mc = fminf(mc, fminf(thr_lo_minus(w2, __uint_as_float(v[8 * j + 4])), thr_hi_minus(w2, __uint_as_float(v[8 * j + 5]))));
                    mc = fminf(mc, fminf(thr_lo_minus(w3, __uint_as_float(v[8 * j + 6])), thr_hi_minus(w3, __uint_as_float(v[8 * j + 7]))));
                }
                const bool hit = cx.row_ok && mc <= 0.f;
                if (cx.tracing) {
                    ++cx.n_chunks;
                    cx.n_trig += __any_sync(0xffffffffu, hit) ? 1 : 0;
                }
                if (hit) {
#pragma unroll
                    for (int t = 0; t < 32; t += 2) {
                        uint32_t w;
                        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(thr_s + 2u * t));
                        const float s0 = __uint_as_float(v[t]), s1 = __uint_as_float(v[t + 1]);
                        if (thr_lo_minus(w, s0) <= 0.f) log_append(cx.lg, p.best_enc, (int)(col_base + t), (int)cx.row, s0);
                        if (thr_hi_minus(w, s1) <= 0.f) log_append(cx.lg, p.best_enc, (int)(col_base + t + 1), (int)cx.row, s1);
                    }
                }
            }
        }
    }
}

// ---- the kernel ------------------------------------------------------------------------------
// Register cap of the top-1 kernels.  A gated launch runs while another stream normalises the arriving chunks: those
// CTAs must become resident NEXT TO this persistent kernel or the launch waits for itself.  Registers are allocated
// per SM sub-partition (16 384 each); the 10 warps of a screen CTA put 3 on two of the four, so
// 3 * 32 * 152 = 14 592 leaves 1 792 registers there - one warp of a 128-thread guest CTA (<= 56 registers/thread).
// (slic_screen_can_overlap_upload checks the built kernels against this arithmetic before a gated launch.)
constexpr int TC_TOP1_MAX_REGS = 152;
template <bool TOPK, bool ARES, bool SYM = false>
__global__ void __maxnreg__(TOPK ? 168 : TC_TOP1_MAX_REGS) nn_screen_kernel(const __grid_constant__ CUtensorMap tmap_q,
                                                                  const __grid_constant__ CUtensorMap tmap_x,
                                                                  const ScreenParams p) {
    typedef TcCfg<ARES, TOPK> Cfg;
    constexpr int STAGES = Cfg::STAGES;
    static_assert(!SYM || !TOPK, "the symmetric variant exists for the top-1 kernels only");
    extern __shared__ uint8_t smem_raw[];
    // (the dynamic smem window starts at the same offset in both CTAs of a pair, so the aligned offsets agree)
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    {
        // the layout needs OPERAND + barrier block (+ thresholds / histograms) behind the 1 KB-aligned base; the window
        // is sized with less than 1 KB of slack, so check (uniform across the grid) instead of assuming
        uint32_t dyn_bytes;
        asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_bytes));
        const uint32_t need = Cfg::OPERAND_BYTES + TC_BAR_BYTES + (SYM ? Cfg::SYM_THR_BYTES : 0u) + (TOPK ? TC_TOPK_SMEM : 0u);
        if ((uint32_t)(smem - smem_raw) + need > dyn_bytes) {
            if (threadIdx.x == 0 && p.error_flag) atomicExch(p.error_flag, 2);
            return;
        }
    }
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OPERAND_BYTES);
    const uint32_t bar_full = smem_u32(bars);                              // [STAGES]  (the leader's are used)
    const uint32_t bar_empty = smem_u32(bars + TC_MAX_STAGES);             // [STAGES]
    const uint32_t bar_acc_full = smem_u32(bars + 12);    // [TC_ACCS]
    const uint32_t bar_acc_empty = smem_u32(bars + 16);   // [TC_ACCS]  (the leader's are used)
    const uint32_t bar_a_full = smem_u32(bars + 20);      // ARES: resident A landed (leader's used)
    const uint32_t bar_a_empty = smem_u32(bars + 21);     // ARES: the unit's MMAs retired
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);
    // (slots 24-27: the epilogue warps' log counters, see s_logcnt)
    const uint32_t bar_thr_full = smem_u32(bars + 28);    // SYM [2]: thresholds of a tile are in place (threshold warp)
    const uint32_t bar_thr_empty = smem_u32(bars + 32);   // SYM [2]: the tile's epilogue warps of this CTA are done with them
    const uint32_t bar_uq_full = smem_u32(bars + 36);     // [TC_UQ_DEPTH]: ring slot holds a unit id (own CTA's copy)
    const uint32_t bar_uq_empty = smem_u32(bars + 40);    // [TC_UQ_DEPTH]: every role of the pair has read it (leader's used)
    const uint32_t uq_val = smem_u32(bars + 44);          // [TC_UQ_DEPTH] int32 unit ids, -1 = no more units
    static_assert(46 * 8 <= TC_BAR_BYTES && 2 * TC_MAX_STAGES <= 12, "barrier block layout");
    const uint32_t smem_base = smem_u32(smem);                 // ARES: resident A, slab ks at + ks * 16 KB
    const uint32_t ring_base = smem_base + Cfg::A_RES_BYTES;   // operand ring

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool tracing = p.trace != nullptr;
    const uint32_t cta_rank = cluster_ctarank();   // 0 = leader: issues the MMAs of the pair

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_q) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);    // the (leader's) producer's arrive.expect_tx
            mbar_init(bar_empty + 8 * s, 1);   // one tcgen05.commit
        }
        for (int a = 0; a < TC_ACCS; ++a) {
            mbar_init(bar_acc_full + 8 * a, 1);
            mbar_init(bar_acc_empty + 8 * a, 2 * TC_EPI_WARPS);  // one arrive per epilogue warp of the pair
        }
        mbar_init(bar_a_full, 1);
        mbar_init(bar_a_empty, 1);
        for (int s = 0; s < TC_UQ_DEPTH; ++s) {
            mbar_init(bar_uq_full + 8 * s, 1);   // the scheduler's arrive
            // readers of a slot, pair-wide: 8 epilogue warps (+ threshold warp) per CTA, the leader's MMA issuer, the peer's producer
            mbar_init(bar_uq_empty + 8 * s, 2 * (TC_EPI_WARPS + (SYM ? 1 : 0)) + 2);
        }
        if constexpr (SYM) {
            for (int b = 0; b < 2; ++b) {
                mbar_init(bar_thr_full + 8 * b, 1);
                mbar_init(bar_thr_empty + 8 * b, TC_EPI_WARPS);
            }
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(TC_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // the peer's barriers are initialised before anything remote touches them
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

    const int64_t n_col_tiles = (p.n + TC_BN - 1) / TC_BN;
    UnitRing ring;
    ring.full = bar_uq_full;
    ring.val = uq_val;
    ring.empty_leader = peer_smem_addr(bar_uq_empty, 0u);
    ring.slot = 0;
    ring.phase = 0u;

    if (warp == 0) {
        // ===================== TMA producer (every CTA: its own A rows, its share of the B slab) =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, a_phase = 0;
            unsigned long long t_wait = 0;
            const bool scheduler = cta_rank == 0;
            int u_next = scheduler ? atomicAdd(p.queue, 1) : 0;
            while (true) {
                int u;
                if (scheduler) {
                    // hand the next unit to every role of the pair (-1: the queue is exhausted)
                    u = u_next < p.num_units ? u_next : -1;
                    mbar_wait_cluster(bar_uq_empty + 8u * ring.slot, ring.phase ^ 1u, p.error_flag);
#pragma unroll
                    for (uint32_t r = 0; r < 2u; ++r) {
                        st_cluster_u32(peer_smem_addr(uq_val + 4u * ring.slot, r), (uint32_t)u);
                        mbar_arrive_release_cluster(peer_smem_addr(bar_uq_full + 8u * ring.slot, r));
                    }
                    if (++ring.slot == TC_UQ_DEPTH) {
                        ring.slot = 0;
                        ring.phase ^= 1u;
                    }
                    if (u >= 0) u_next = atomicAdd(p.queue, 1);   // (the round trip overlaps this unit's loads)
                } else {
                    u = ring_take(ring, false, p.error_flag);
                }
                if (u < 0) break;
                const UnitInfo ui = unit_info(p, u, n_col_tiles);
                const int64_t row_block = ui.row_unit * 2 + cta_rank;
                if (ui.gate >= 0) gate_wait(p.gates + ui.gate, p.error_flag);
                if constexpr (SYM) {
                    if (ui.coldir && p.sync_counter)
                        counter_wait(p.sync_counter, __ldg(p.sync_targets + ui.gate + 1), p.error_flag);
                }
                if constexpr (ARES) {
                    // the previous unit's MMAs have retired -> replace the resident A rows (all K slabs, one barrier)
                    mbar_wait_traced(bar_a_empty, a_phase ^ 1, p.error_flag, t_wait, tracing);
                    if (cta_rank == 0) mbar_expect_tx(bar_a_full, 2 * (uint32_t)p.num_k_slabs * TC_A_BYTES);
                    for (int ks = 0; ks < p.num_k_slabs; ++ks)
                        tma_load_2d_pair(&tmap_q, smem_base + ks * TC_A_BYTES, bar_a_full, ks * TC_BK,
                                         (int)(row_block * TC_BM));
                    a_phase ^= 1;
                }
                for (int kt = 0; kt < ui.count; ++kt) {
                    const int64_t ct = ui.ct0 + (int64_t)kt * ui.stride;
                    for (int ks = 0; ks < p.num_k_slabs; ks += Cfg::SPS) {
                        mbar_wait_traced(bar_empty + 8 * stage, phase ^ 1, p.error_flag, t_wait, tracing);
                        const uint32_t a_dst = ring_base + stage * Cfg::STAGE_BYTES;
                        const uint32_t b_dst = ARES ? a_dst : a_dst + TC_A_BYTES;
                        // both CTAs' bytes complete on the LEADER's full barrier
                        if constexpr (ARES) {
                            const int nsl = min(Cfg::SPS, p.num_k_slabs - ks);
                            if (cta_rank == 0) mbar_expect_tx(bar_full + 8 * stage, 2 * (uint32_t)nsl * Cfg::B_BYTES);
                            for (int j = 0; j < nsl; ++j)
                                tma_load_2d_pair(&tmap_x, b_dst + j * Cfg::SLAB_BYTES, bar_full + 8 * stage, (ks + j) * TC_BK,
                                                 (int)(ct * TC_BN + cta_rank * Cfg::B_ROWS));
                        } else {
                            const int nsl = min(Cfg::SPS, p.num_k_slabs - ks);
                            if (cta_rank == 0) mbar_expect_tx(bar_full + 8 * stage, 2 * (uint32_t)nsl * Cfg::SLAB_BYTES);
                            for (int j = 0; j < nsl; ++j) {
                                tma_load_2d_pair(&tmap_q, a_dst + j * Cfg::SLAB_BYTES, bar_full + 8 * stage, (ks + j) * TC_BK,
                                                 (int)(row_block * TC_BM));
                                tma_load_2d_pair(&tmap_x, b_dst + j * Cfg::SLAB_BYTES, bar_full + 8 * stage, (ks + j) * TC_BK,
                                                 (int)(ct * TC_BN + cta_rank * Cfg::B_ROWS));
                            }
                        }
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
            if (tracing) atomicAdd(p.trace + 0, t_wait);   // producer stalled on a free smem stage
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (one thread; in a pair only the leader's) =====================
        if (lane == 0 && cta_rank == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0, a_phase = 0;
            unsigned long long t_acc = 0, t_smem = 0;
            const long long t_begin = tracing ? clock64() : 0;
            unsigned long long t_ring = 0, n_units = 0;
            while (true) {
                const long long tr0 = tracing ? clock64() : 0;
                const int u = ring_take(ring, false, p.error_flag);
                if (tracing) t_ring += (unsigned long long)(clock64() - tr0);
                if (u < 0) break;
                ++n_units;
                const int n_tiles = unit_info(p, u, n_col_tiles).count;
                if constexpr (ARES) {
                    mbar_wait_traced(bar_a_full, a_phase, p.error_flag, t_smem, tracing);
                    tc_fence_after();
                    a_phase ^= 1;
                }
                for (int kt = 0; kt < n_tiles; ++kt) {
                    mbar_wait_traced(bar_acc_empty + 8 * acc, acc_phase ^ 1, p.error_flag, t_acc, tracing);
                    tc_fence_after();
                    const uint32_t tmem_d = tmem_base + (uint32_t)(acc * TC_BN);
                    for (int ks = 0; ks < p.num_k_slabs; ks += Cfg::SPS) {
                        mbar_wait_traced(bar_full + 8 * stage, phase, p.error_flag, t_smem, tracing);
                        tc_fence_after();
                        const uint32_t st_addr = ring_base + stage * Cfg::STAGE_BYTES;
#pragma unroll
                        for (int j = 0; j < Cfg::SPS; ++j) {
                            if (ks + j < p.num_k_slabs) {
                                const uint32_t sl_addr = st_addr + j * Cfg::SLAB_BYTES;
                                const uint64_t da = umma_smem_desc(ARES ? smem_base + (ks + j) * TC_A_BYTES : sl_addr);
                                const uint64_t db = umma_smem_desc(ARES ? sl_addr : sl_addr + TC_A_BYTES);
#pragma unroll
                                for (int k = 0; k < TC_BK / TC_UMMA_K; ++k) {
                                    // advancing 16 f16 = 32 bytes along K inside the swizzle atom: +2 in the address field
                                    umma_f16_pair(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), TC_IDESC,
                                                  (uint32_t)((ks | j | k) != 0));
                                }
                            }
                        }
                        // frees the smem stage (in both CTAs) once these MMAs retire
                        umma_commit_pair(bar_empty + 8 * stage);
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                    // accumulator complete -> epilogue (of both CTAs)
                    umma_commit_pair(bar_acc_full + 8 * acc);
                    if (++acc == TC_ACCS) {
                        acc = 0;
                        acc_phase ^= 1;
                    }
                }
                if constexpr (ARES) umma_commit_pair(bar_a_empty);   // the resident A rows may be replaced (both CTAs)
            }
            if (tracing) {
                atomicAdd(p.trace + 1, t_acc);    // MMA issuer stalled on a free accumulator (epilogue too slow)
                atomicAdd(p.trace + 2, t_smem);   // MMA issuer stalled on operands (TMA / L2 too slow)
                atomicAdd(p.trace + 3, (unsigned long long)(clock64() - t_begin));   // MMA issuer total
                atomicAdd(p.trace + 8, t_ring);    // MMA issuer waited for the next unit id (scheduler / pre-pass hand-over)
                atomicAdd(p.trace + 10, n_units);
            }
        }
    } else if (SYM && warp == 2 + TC_EPI_WARPS) {
        // ===================== SYM: column-threshold publisher =====================
        // For every tile strictly right of the diagonal (the epilogue's "column role"): threshold of column c =
        // best score published for row c so far - eps, as float16 rounded DOWN (a lower threshold only adds candidates;
        // 2^-11 against eps = 2^-7), with a finite lower bound (threshold - masked score = +inf, never NaN).
        // Buffers (1 KB in all): 2 x [256 columns], consumed by all eight epilogue warps of the CTA; `cseq` counts the
        // column-role tiles.
        uint16_t* thr_buf = reinterpret_cast<uint16_t*>(smem + Cfg::OPERAND_BYTES + TC_BAR_BYTES);
        constexpr unsigned ENC_POS_INF = 0xff800000u;
        constexpr int PER_LANE = TC_BN / 32;
        unsigned cseq = 0u;
        for (int u; (u = ring_take(ring, true, p.error_flag)) >= 0;) {
            const UnitInfo ui = unit_info(p, u, n_col_tiles);
            if (!ui.coldir) continue;
            if (p.sync_counter) {   // published bests of the pre-pass are in place (speed only, as for the epilogue)
                if (lane == 0) counter_wait(p.sync_counter, __ldg(p.sync_targets + ui.gate + 1), p.error_flag);
                __syncwarp();
            }
            for (int kt = 0; kt < ui.count; ++kt) {
                const int64_t ct = ui.ct0 + (int64_t)kt * ui.stride;
                if (ct == ui.row_unit) continue;   // the diagonal tile (TC_ROW_UNIT == TC_BN)
                const uint32_t buf = cseq & 1u, ph = (cseq >> 1) & 1u;
                unsigned e[PER_LANE];   // fetched first: the L2 round trip overlaps the wait for the buffer
#pragma unroll
                for (int j = 0; j < PER_LANE; ++j) {
                    const int64_t c = ct * TC_BN + lane + 32 * j;
                    e[j] = c < p.n ? __ldcg(p.best_enc + c) : ENC_POS_INF;
                }
                mbar_wait(bar_thr_empty + 8 * buf, ph ^ 1u, p.error_flag);
                const uint32_t ta = smem_u32(thr_buf + buf * 256u) + 2u * lane;
#pragma unroll
                for (int j = 0; j < PER_LANE; ++j) {
                    const unsigned short t = __half_as_ushort(__float2half_rd(fmaxf(dec_score(e[j]) - p.eps, -60000.f)));
                    asm volatile("st.shared.b16 [%0], %1;" ::"r"(ta + 64u * j), "h"(t) : "memory");
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_thr_full + 8 * buf);
                ++cseq;
            }
        }
    } else {
        // ===================== epilogue: fused candidate filter =====================
        // Warp w reads TMEM lanes [32 * (w % 4), +32) (the hardware's lane window of that warp) and the 128-column
        // half (w - 2) / 4 of every tile: one thread = one (query row, column half) stream with its own list.
        const int quad = warp & 3;
        const int half = (warp - 2) >> 2;
        const int row_in_tile = quad * 32 + lane;
        unsigned seq_all = 0;   // tiles the pair has been through; accumulator of tile s: s % TC_ACCS, barrier phase (s / TC_ACCS) & 1
        unsigned long long t_full = 0;
        const long long t_begin = tracing ? clock64() : 0;
        EpiCtx<TOPK> cx;
        cx.p = &p;
        cx.tracing = tracing;
        cx.n_trig = 0;
        cx.n_chunks = 0;
        if constexpr (TOPK) cx.hist = smem + Cfg::OPERAND_BYTES + TC_BAR_BYTES + half * TC_BM + row_in_tile;
        unsigned int* s_logcnt = reinterpret_cast<unsigned int*>(bars + 24) + (warp - 2);   // slots 24-27 of the barrier block
        uint16_t* thr_buf = reinterpret_cast<uint16_t*>(smem + Cfg::OPERAND_BYTES + TC_BAR_BYTES);   // SYM: float16 column thresholds
        unsigned tile_seq = 0;   // SYM: column-role tiles this warp has taken
        const int64_t log_region_id = (int64_t)blockIdx.x * TC_EPI_WARPS + (warp - 2);
        if constexpr (SYM) {
            if (lane == 0) *s_logcnt = 0u;
            __syncwarp();
            cx.lg.q = p.log_q + log_region_id * p.log_region;
            cx.lg.nb = p.cand_idx + log_region_id * p.log_region;
            cx.lg.s = p.cand_score + log_region_id * p.log_region;
            cx.lg.cnt = s_logcnt;
            cx.lg.region = p.log_region;
            cx.lg.overflow = p.cand_flags;
        }
        unsigned long long t_unit = 0;
        while (true) {
            const long long tr0 = tracing ? clock64() : 0;
            const int u = ring_take(ring, true, p.error_flag);
            if (u < 0) break;
            const UnitInfo ui = unit_info(p, u, n_col_tiles);
            if constexpr (SYM) {
                // a triangle unit reads published thresholds: not before every pre-pass unit it depends on has finished
                // (the producer waits for the same counter, but this warp runs ahead of the first accumulator)
                if (ui.coldir && p.sync_counter) {
                    if (lane == 0) counter_wait(p.sync_counter, __ldg(p.sync_targets + ui.gate + 1), p.error_flag);
                    __syncwarp();
                }
            }
            if (tracing) t_unit += (unsigned long long)(clock64() - tr0);
            const int64_t row_block = ui.row_unit * 2 + cta_rank;
            cx.row = row_block * TC_BM + row_in_tile;
            cx.row_ok = cx.row < p.nq;
            cx.self_col = (p.self_offset >= 0 && cx.row_ok) ? cx.row + p.self_offset : -1;
            const int64_t slot = SYM ? 0 : (int64_t)(ui.stream * 2 + half) * p.nq + (cx.row_ok ? cx.row : 0);
            cx.li = p.cand_idx + slot * p.cap;
            cx.ls = p.cand_score + slot * p.cap;
            if constexpr (TOPK) {
                for (int i = 0; i < TC_HIST_BINS; ++i) cx.hist[i * TC_HIST_STRIDE] = 0;
                int seed = 0;
                if (p.cand_tb && cx.row_ok)
                    for (int s2 = 0; s2 < 2 * p.splits; ++s2) seed = max(seed, __ldcg(p.cand_tb + (int64_t)s2 * p.nq + cx.row));
                cx.st.tb = seed;
                cx.st.cge = 0;
                cx.st.ctb = 0;
                cx.st.thr = bin_edge(seed) - p.eps;
                cx.pd.n = 0;
            } else if constexpr (SYM) {
                // start from the best score any CTA has published for this row (pre-pass, earlier units, column roles)
                cx.st.best = cx.row_ok ? dec_score(__ldcg(p.best_enc + cx.row)) : -CUDART_INF_F;
                cx.st.thr = cx.st.best - p.eps;
            } else {
                cx.st.best = -CUDART_INF_F;
                cx.st.thr = -CUDART_INF_F;
            }
            cx.st.cnt = 0;
            cx.st.flags = 0;
            uint32_t va[32], vb[32];
            bool prefetched = false;   // va holds an in-flight load of the coming tile's first chunk
            bool first = true;         // no tile of this unit taken yet
            for (int kt = 0; kt < ui.count; ++kt, ++seq_all) {
                const int acc = (int)(seq_all % (unsigned)TC_ACCS);
                const uint32_t acc_phase = (seq_all / (unsigned)TC_ACCS) & 1u;
                const int64_t ct = ui.ct0 + (int64_t)kt * ui.stride;
                const int64_t col0 = ct * TC_BN + half * 128;
                // SYM: tiles strictly right of the diagonal also serve their columns as queries; their thresholds come from
                // the threshold warp through shared memory
                bool cdir = false;
                uint32_t thr_tile = 0u;   // shared-memory address of this tile's 128 column thresholds
                uint32_t thr_done_bar = 0u;
                if constexpr (SYM) {
                    cdir = ui.coldir && ct != ui.row_unit;
                    if (cdir) {   // the threshold warp runs two tiles ahead: this wait is normally a single poll
                        const uint32_t buf = tile_seq & 1u, ph = (tile_seq >> 1) & 1u;
                        thr_tile = smem_u32(thr_buf + (buf * 2 + half) * 128);
                        thr_done_bar = bar_thr_empty + 8 * buf;
                        mbar_wait(bar_thr_full + 8 * buf, ph, p.error_flag);
                        ++tile_seq;
                    }
                }
                // (top-1 variants: the first chunk of this tile may already be in flight - issued at the end of the previous
                //  tile, see below)
                if (TOPK || !prefetched) {
                    mbar_wait_traced(bar_acc_full + 8 * acc, acc_phase, p.error_flag, t_full, tracing);
                    tc_fence_after();
                }
                const uint32_t tbase = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * TC_BN + half * 128);
                if constexpr (TOPK) {
                    cx.count = !first;
                    if (first) {
                        // bootstrap: count every column of the stream's first 128 (uniform control flow, nothing is
                        // listed), which yields the first threshold; the columns are then read again below
#pragma unroll 1
                        for (int c = 0; c < 4; ++c) {
                            tmem_ld_issue(tbase + (uint32_t)(c * 32), va);
                            tmem_ld_wait(va);
                            const int64_t col_base = col0 + c * 32;
                            if (col_base >= p.n || !cx.row_ok) continue;
#pragma unroll
                            for (int t = 0; t < 32; ++t) {
                                if (col_base + t < p.n && col_base + t != cx.self_col)
                                    hist_insert(cx.st, cx.hist, __uint_as_float(va[t]), p.topk);
                            }
                            hist_advance(cx.st, cx.hist, p.topk, p.eps);   // per chunk: bins above tb stay below 96 entries
                        }
                    }
                }
                // warp-uniform: no column of this 128-column half needs masking (inside the database, not the rows' own
                // columns, no debug dump) - the filter then skips all per-column checks
                const bool plain = col0 + 128 <= p.n && !p.dump &&
                                   (p.self_offset < 0 || row_block * TC_BM + p.self_offset + TC_BM <= col0 ||
                                    row_block * TC_BM + p.self_offset >= col0 + 128);
                if constexpr (TOPK) {
                    // software pipeline over the 4 chunks of this half: chunk c + 1 is in flight while chunk c is filtered
                    tmem_ld_issue(tbase, vb);
#pragma unroll 1
                    for (int c = 0; c < 4; ++c) {
                        tmem_ld_wait(vb);
#pragma unroll
                        for (int t = 0; t < 32; ++t) va[t] = vb[t];
                        if (c < 3) {
                            tmem_ld_issue(tbase + (uint32_t)(32 * (c + 1)), vb);
                        } else {
                            // every TMEM read of this accumulator is complete: hand it back before the last filter
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive_leader(bar_acc_empty + 8 * acc);
                        }
                        epi_chunk<TOPK, false>(cx, va, col0 + 32 * c, plain);
                    }
                } else {
                    // the same pipeline with the two register buffers swapping roles (no copies): two chunks per trip
                    if (!prefetched) tmem_ld_issue(tbase, va);
                    prefetched = false;
#pragma unroll 1
                    for (int h = 0; h < 2; ++h) {
                        tmem_ld_wait(va);
                        tmem_ld_issue(tbase + (uint32_t)(64 * h + 32), vb);
                        epi_chunk<false, SYM>(cx, va, col0 + 64 * h, plain, cdir, thr_tile + 128u * h);
                        tmem_ld_wait(vb);
                        if (h == 0) {
                            tmem_ld_issue(tbase + 64u, va);
                        } else {
                            // every TMEM read of this accumulator is complete: hand it back before the last filter
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive_leader(bar_acc_empty + 8 * acc);
                            // Cross-tile prefetch: if this warp's NEXT tile of the unit is already complete in its accumulator,
                            // start reading its first chunk now, so that the load's latency (queueing behind the other warps on
                            // the TMEM read port) hides behind the filter of this tile's last chunk instead of being exposed at
                            // every tile boundary.  One poll, warp-uniform decision; a miss falls back to the blocking wait.
                            if (kt + 1 < ui.count) {
                                const unsigned nxt = seq_all + 1;
                                const int acc_n = (int)(nxt % (unsigned)TC_ACCS);
                                const bool ready = __all_sync(0xffffffffu, mbar_test(bar_acc_full + 8 * acc_n, (nxt / (unsigned)TC_ACCS) & 1u));
                                if (ready) {
                                    tc_fence_after();
                                    tmem_ld_issue(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc_n * TC_BN + half * 128),
                                                  va);
                                    prefetched = true;
                                }
                            }
                        }
                        epi_chunk<false, SYM>(cx, vb, col0 + 64 * h + 32, plain, cdir, thr_tile + 128u * h + 64u);
                    }
                    if constexpr (SYM) {
                        if (cdir) {   // this warp no longer reads the tile's thresholds
                            __syncwarp();
                            if (lane == 0) mbar_arrive(thr_done_bar);
                        }
                    }
                }
                if constexpr (TOPK) {
                    // parked columns of the first tile must be listed before columns start being counted
                    if (first) pend_flush(cx.pd, cx.st, p.eps, p.cap, p.topk, false, cx.hist, cx.li, cx.ls);
                }
                first = false;
            }
            if constexpr (TOPK) pend_flush(cx.pd, cx.st, p.eps, p.cap, p.topk, true, cx.hist, cx.li, cx.ls);
            if constexpr (SYM) {
                // publish this unit's best for the row; the shared list is already in place
                if (cx.row_ok && cx.st.best > -CUDART_INF_F) {
                    const unsigned e = enc_score(cx.st.best);
                    atomicMax(p.best_enc + cx.row, e);
                    if (!ui.coldir)   // pre-pass: every other rank learns this row's first threshold too
                        for (int g = 0; g < p.num_peers; ++g) atomicMax(p.peer_best[g] + cx.row, e);
                }
                if (!ui.coldir && p.sync_counter) {   // pre-pass unit done: its rows' thresholds are published
                    if (p.num_peers) __threadfence_system();
                    else __threadfence();
                    __syncwarp();
                    if (lane == 0) {
                        atomicAdd(p.sync_counter, 1);
                        for (int g = 0; g < p.num_peers; ++g) atomicAdd(p.peer_sync[g], 1);
                    }
                }
            } else if (cx.row_ok) {
                p.cand_cnt[slot] = cx.st.cnt;
                p.cand_flags[slot] = cx.st.flags;
                if constexpr (TOPK) {
                    p.cand_kth[slot] = bin_edge(cx.st.tb);
                    if (p.cand_tb) p.cand_tb[slot] = cx.st.tb;
                }
            }
        }
        if constexpr (SYM) {
            __syncwarp();
            if (lane == 0) p.cand_cnt[log_region_id] = (int)min(*s_logcnt, (unsigned)p.log_region);
        }
        if (tracing && lane == 0 && warp == 2) {
            atomicAdd(p.trace + 4, t_full);    // epilogue warp 0 stalled on a complete accumulator (MMA slower)
            atomicAdd(p.trace + 5, (unsigned long long)(clock64() - t_begin));   // epilogue warp 0 total
            atomicAdd(p.trace + 6, cx.n_trig);    // 32-column chunks in which some row had a candidate
            atomicAdd(p.trace + 7, cx.n_chunks);
            atomicAdd(p.trace + 9, t_unit);    // epilogue warp 0 waited for a unit id / the pre-pass hand-over
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();   // the peer no longer reads this CTA's smem or signals its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
    }
}

// ---- exact re-rank of the surviving candidates (one warp per query row) ------------------------
template <typename T>
__global__ void __launch_bounds__(256) rerank_top1_kernel(const T* __restrict__ q_unit, const T* __restrict__ x_unit,
                                                          int64_t nq, int d, float eps, int cap, int splits,
                                                          const int* __restrict__ cand_idx,
                                                          const float* __restrict__ cand_score,
                                                          const int* __restrict__ cand_cnt,
                                                          const int* __restrict__ cand_flags, int* __restrict__ idx_out,
                                                          T* __restrict__ dist_out, int* __restrict__ overflow_rows,
                                                          int* __restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= nq) return;
    float gbest = -CUDART_INF_F;
    int flags = 0;
    for (int sp = 0; sp < splits; ++sp) {
        const int64_t slot = (int64_t)sp * nq + r;
        const int c = min(cand_cnt[slot], cap);   // (the symmetric kernel counts appends past the end)
        flags |= cand_flags[slot];
        for (int e = lane; e < c; e += 32) gbest = fmaxf(gbest, cand_score[slot * cap + e]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gbest = fmaxf(gbest, __shfl_xor_sync(0xffffffffu, gbest, o));
    const float thr = gbest - eps;
    const T* qr = q_unit + r * d;
    double best_d = CUDART_INF;  // best distance, rounded to T as the reference holds it
    int best_j = 0x7fffffff, reranked = 0;
    for (int sp = 0; sp < splits; ++sp) {
        const int64_t slot = (int64_t)sp * nq + r;
        const int c = min(cand_cnt[slot], cap);
        for (int e = 0; e < c; ++e) {
            if (cand_score[slot * cap + e] < thr) continue;  // warp-uniform
            const int j = cand_idx[slot * cap + e];
            const double s = warp_dot<T>(qr, x_unit + (int64_t)j * d, d, lane);
            ++reranked;
            const double dist = (double)cosine_distance_from_sim<T>(s);
            if (closer(dist, j, best_d, best_j)) {
                best_d = dist;
                best_j = j;
            }
        }
    }
    if (lane == 0) {
        idx_out[r] = best_j == 0x7fffffff ? -1 : best_j;
        if (dist_out) dist_out[r] = (T)best_d;
        atomicAdd(&stats[0], reranked);
        if (flags & 2) atomicAdd(&stats[2], 1);
        if ((flags & 1) || best_j == 0x7fffffff) {
            const int pos = atomicAdd(&stats[1], 1);
            overflow_rows[pos] = (int)r;
        }
    }
}

template <typename T>
__global__ void scatter_rows_kernel(const int* __restrict__ rows, int count, const int* __restrict__ idx_src,
                                    const T* __restrict__ dist_src, int* __restrict__ idx_out, T* __restrict__ dist_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    idx_out[rows[i]] = idx_src[i];
    if (dist_out) dist_out[rows[i]] = dist_src[i];
}

// ---- exact re-rank for the top-k variant (one CTA per query row) -------------------------------
// Gathers the columns whose screened score is within eps of the best available lower bound of the row's
// k-th best screened score (the largest per-split k-th best), evaluates them exactly in T, sorts them by
// (distance, column) and emits the first k.  Rows that overflowed a list, gathered more than RK_MAX
// columns or fewer than k go to the exact kernel.
constexpr int RK_THREADS = 128, RK_MAX = 1024, RK_BINS = 1024;

template <typename T>
__global__ void __launch_bounds__(RK_THREADS) rerank_topk_kernel(const T* __restrict__ q_unit, const T* __restrict__ x_unit,
                                                                 int64_t nq, int d, float eps, int cap, int splits, int k,
                                                                 const int* __restrict__ cand_idx,
                                                                 const float* __restrict__ cand_score,
                                                                 const int* __restrict__ cand_cnt,
                                                                 const int* __restrict__ cand_flags,
                                                                 const float* __restrict__ cand_kth,
                                                                 int* __restrict__ idx_out, T* __restrict__ dist_out,
                                                                 int* __restrict__ overflow_rows, int* __restrict__ stats) {
    __shared__ int s_idx[RK_MAX];
    __shared__ T s_dist[RK_MAX];
    __shared__ int s_hist[RK_BINS];
    __shared__ int s_part[RK_THREADS];
    __shared__ int s_m, s_flags;
    __shared__ float s_thr;
    const int64_t r = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        float kth = -CUDART_INF_F;
        int fl = 0, listed = 0;
        for (int sp = 0; sp < splits; ++sp) {
            kth = fmaxf(kth, cand_kth[(int64_t)sp * nq + r]);
            fl |= cand_flags[(int64_t)sp * nq + r];
            listed += cand_cnt[(int64_t)sp * nq + r];
        }
        atomicAdd(&stats[3], listed >> 4);   // columns listed by the screen, in units of 16
        s_thr = kth - eps;
        s_flags = fl;
        s_m = 0;
    }
    __syncthreads();
    // Tighten the threshold: the streams' own bounds are k-th bests of a FRACTION of the columns.  A 1024-bin
    // histogram (bin width 2^-10) of every listed score above the coarse threshold gives the merged k-th best to
    // within one bin: edge(bin holding the k-th largest) <= k-th best screened score of the whole row.
    for (int b = tid; b < RK_BINS; b += RK_THREADS) s_hist[b] = 0;
    __syncthreads();
    const float thr0 = s_thr;
    for (int sp = 0; sp < splits; ++sp) {
        const int64_t slot = (int64_t)sp * nq + r;
        const int c = cand_cnt[slot];
        for (int e = tid; e < c; e += RK_THREADS) {
            const float sc = cand_score[slot * cap + e];
            if (sc >= thr0) atomicAdd(&s_hist[min(max(__float2int_rd(sc * (float)RK_BINS), 0), RK_BINS - 1)], 1);
        }
    }
    __syncthreads();
    {
        constexpr int PER = RK_BINS / RK_THREADS;   // bins per thread
        int local = 0;
#pragma unroll
        for (int i = 0; i < PER; ++i) local += s_hist[tid * PER + i];
        s_part[tid] = local;
        __syncthreads();
        for (int off = 1; off < RK_THREADS; off <<= 1) {   // inclusive suffix sums over threads
            const int add = tid + off < RK_THREADS ? s_part[tid + off] : 0;
            __syncthreads();
            s_part[tid] += add;
            __syncthreads();
        }
        const int above = tid + 1 < RK_THREADS ? s_part[tid + 1] : 0;   // listed scores in bins owned by later threads
        if (above < k && s_part[tid] >= k) {   // exactly one thread: the k-th largest lies in one of its bins
            int cum = above, b = tid * PER + PER - 1;
            for (; b > tid * PER; --b) {
                cum += s_hist[b];
                if (cum >= k) break;
            }
            const float edge = b == 0 ? -1.0f : (float)b * (1.0f / (float)RK_BINS);
            s_thr = fmaxf(thr0, edge - eps);
        }
    }
    __syncthreads();
    const float thr = s_thr;
    for (int sp = 0; sp < splits; ++sp) {
        const int64_t slot = (int64_t)sp * nq + r;
        const int c = cand_cnt[slot];
        for (int e = tid; e < c; e += RK_THREADS) {
            if (cand_score[slot * cap + e] >= thr) {
                const int pos = atomicAdd(&s_m, 1);
                if (pos < RK_MAX) s_idx[pos] = cand_idx[slot * cap + e];
            }
        }
    }
    __syncthreads();
    const int m = s_m;
    if ((s_flags & 1) || m > RK_MAX || m < k) {
        if (tid == 0) overflow_rows[atomicAdd(&stats[1], 1)] = (int)r;
        return;
    }
    const T* qr = q_unit + r * d;
    for (int e = warp; e < m; e += RK_THREADS / 32) {
        const double s = warp_dot<T>(qr, x_unit + (int64_t)s_idx[e] * d, d, lane);
        if (lane == 0) s_dist[e] = cosine_distance_from_sim<T>(s);
    }
    int m2 = 2;
    while (m2 < m) m2 <<= 1;
    for (int e = m + tid; e < m2; e += RK_THREADS) {
        s_dist[e] = (T)CUDART_INF;
        s_idx[e] = 0x7fffffff;
    }
    __syncthreads();
    for (int size = 2; size <= m2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < (m2 >> 1); t += RK_THREADS) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const T da = s_dist[lo], db = s_dist[hi];
                const int ia = s_idx[lo], ib = s_idx[hi];
                const bool a_after_b = (da > db) || (da == db && ia > ib);
                if (a_after_b == up) {
                    s_dist[lo] = db; s_dist[hi] = da;
                    s_idx[lo] = ib; s_idx[hi] = ia;
                }
            }
            __syncthreads();
        }
    }
    for (int j = tid; j < k; j += RK_THREADS) {
        idx_out[r * k + j] = s_idx[j];
        if (dist_out) dist_out[r * k + j] = s_dist[j];
    }
    if (tid == 0) {
        atomicAdd(&stats[0], m);
        if (s_flags & 2) atomicAdd(&stats[2], 1);
    }
}

template <typename T>
__global__ void scatter_topk_rows_kernel(const int* __restrict__ rows, int count, int k, const int* __restrict__ idx_src,
                                         const T* __restrict__ dist_src, int* __restrict__ idx_out,
                                         T* __restrict__ dist_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)count * k) return;
    const int64_t dst = (int64_t)rows[i / k] * k + (i % k);
    idx_out[dst] = idx_src[i];
    if (dist_out) dist_out[dst] = dist_src[i];
}

// ---- host side ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int get_encode_fn(EncodeTiledFn* out) {
    static EncodeTiledFn cached = nullptr;
    if (!cached) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        SLIC_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) {
            set_error("cuTensorMapEncodeTiled is not available from the driver");
            return SLIC_ERR_UNSUPPORTED;
        }
        cached = reinterpret_cast<EncodeTiledFn>(fn);
    }
    *out = cached;
    return SLIC_OK;
}

// rows x d_pad f16, row-major; box = 64 (K) x box_rows, 128-byte swizzle, out-of-bounds rows read as zero
static int make_tmap(CUtensorMap* map, const uint16_t* base, int64_t rows, int d_pad, int box_rows) {
    EncodeTiledFn enc;
    SLIC_PROPAGATE(get_encode_fn(&enc));
    cuuint64_t gdim[2] = {(cuuint64_t)d_pad, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)d_pad * 2};
    cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<uint16_t*>(base), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld d_pad=%d)", (int)r, (long long)rows, d_pad);
        return SLIC_ERR_CUDA;
    }
    return SLIC_OK;
}

// optional CUDA-event timing of the screen kernel on its own stream (bench.py's roofline leg)
static bool g_profile = false, g_have_sample = false;
static unsigned long long* g_trace = nullptr;   // device [12], allocated by slic_screen_trace(1)
static cudaEvent_t g_ev_start = nullptr, g_ev_stop = nullptr;
static double g_last_flop = 0.0, g_last_exec_flop = 0.0;

struct ScreenPlan {
    int splits, tiles_per_split;
    int64_t units;
};

static ScreenPlan plan_screen(int64_t nq, int64_t n) {
    const int64_t row_blocks = ceil_div(nq, TC_ROW_UNIT), col_tiles = ceil_div(n, TC_BN);
    const int64_t sms = num_sms() / 2;
    // enough units for >= ~6 waves when the problem allows it, but keep >= 2048 columns (8 tiles) per unit
    int64_t want = ceil_div(6 * sms, row_blocks);
    const int64_t min_tiles = 8;
    int64_t max_splits = col_tiles / min_tiles > 0 ? col_tiles / min_tiles : 1;
    int64_t splits = want < 1 ? 1 : (want > max_splits ? max_splits : want);
    ScreenPlan pl;
    pl.tiles_per_split = (int)ceil_div(col_tiles, splits);
    pl.splits = (int)ceil_div(col_tiles, pl.tiles_per_split);
    pl.units = row_blocks * pl.splits;
    return pl;
}

// Top-k variant: every unit restarts with an empty threshold (its first tile is listed in full and the
// threshold then tightens like k / columns seen), so units should be as long as the wave structure allows:
// minimise waves x (tiles per unit + start-up cost in tile times).
static ScreenPlan plan_screen_topk(int64_t nq, int64_t n, int k) {
    const int64_t row_blocks = ceil_div(nq, TC_ROW_UNIT), col_tiles = ceil_div(n, TC_BN);
    const int64_t sms = num_sms() / 2;
    const int64_t startup = 6;   // bootstrap pass + threshold ramp of a unit, in tile times
    int64_t best_s = 1, best_cost = INT64_MAX;
    // a stream (half of a unit's tiles) should see >= ~32 k columns, or its own k-th best says little about the row's
    const int64_t min_tps = ceil_div((int64_t)32 * k, TC_BN / 2);
    // (two passes: the cheapest plan, then the FEWEST splits within 2 % of it - every split is one more pair of candidate
    //  streams per row, each restarting from an empty threshold: measured on 100 000 x 1 000 000 x 1 024, k = 50, 7 splits
    //  of 559 tiles against 3 of 1 303 - equal in this model - run the screen at 0.56 against 0.70 of the tensor peak)
    for (int pass = 0; pass < 2; ++pass) {
        for (int64_t sp = 1; sp <= col_tiles && sp <= 64; ++sp) {
            const int64_t tps = ceil_div(col_tiles, sp);
            if (sp > 1 && tps < min_tps) break;
            const int64_t real = ceil_div(col_tiles, tps);
            const int64_t waves = ceil_div(row_blocks * real, sms);
            const int64_t cost = waves * (tps + startup);
            if (pass == 0) {
                if (cost < best_cost) {
                    best_cost = cost;
                    best_s = real;
                }
            } else if (cost * 100 <= best_cost * 102) {
                best_s = real;
                break;
            }
        }
    }
    ScreenPlan pl;
    pl.tiles_per_split = (int)ceil_div(col_tiles, best_s);
    pl.splits = (int)ceil_div(col_tiles, pl.tiles_per_split);
    pl.units = row_blocks * pl.splits;
    return pl;
}

// candidate slots per (split, row) of the top-k variant: the first tile (256) + ~k ln(columns / 256) later
// listings + the eps band, with a factor 3 of head room; rows that still overflow are compacted, then finished exactly
static int topk_cap(int k, int64_t cols_per_split) {
    double later = cols_per_split > 128 ? (double)k * log((double)cols_per_split / 128.0) : 0.0;
    int64_t want = 128 + (int64_t)(3.0 * later) + 128;
    int cap = 512;
    while (cap < want && cap < 4096) cap <<= 1;
    return cap;
}

typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const ScreenParams);
// A rows resident in shared memory when they fit, streamed with B otherwise
static bool screen_ares(int d_pad) { return d_pad / TC_BK <= TC_ARES_MAX_SLABS; }
static void pick_screen_kernel(bool sym, bool ares, bool is_topk, KernelFn* fn, size_t* smem_bytes) {
    if (sym) {
        *fn = ares ? (KernelFn)nn_screen_kernel<false, true, true> : (KernelFn)nn_screen_kernel<false, false, true>;
        *smem_bytes = ares ? TcCfg<true, false>::SYM_SMEM_BYTES : TcCfg<false, false>::SYM_SMEM_BYTES;
    } else if (ares) {
        *fn = is_topk ? (KernelFn)nn_screen_kernel<true, true> : (KernelFn)nn_screen_kernel<false, true>;
        *smem_bytes = is_topk ? TcCfg<true, true>::SMEM_BYTES : TcCfg<true, false>::SMEM_BYTES;
    } else {
        *fn = is_topk ? (KernelFn)nn_screen_kernel<true, false> : (KernelFn)nn_screen_kernel<false, false>;
        *smem_bytes = is_topk ? TcCfg<false, true>::SMEM_BYTES : TcCfg<false, false>::SMEM_BYTES;
    }
}

static int* g_timeout_record_host = nullptr;   // mapped pinned memory, [8]
static int arm_timeout_record() {
    if (!g_timeout_record_host) {
        SLIC_CUDA_OK(cudaHostAlloc(&g_timeout_record_host, 8 * sizeof(int), cudaHostAllocMapped));
        int* dev_view = nullptr;
        SLIC_CUDA_OK(cudaHostGetDevicePointer(&dev_view, g_timeout_record_host, 0));
        SLIC_CUDA_OK(cudaMemcpyToSymbol(g_timeout_record, &dev_view, sizeof(dev_view)));
    }
    for (int i = 0; i < 8; ++i) g_timeout_record_host[i] = 0;
    return SLIC_OK;
}
// appended to the error text of a failed screen launch
const char* timeout_record_text() {
    static thread_local char buf[160];
    const int* r = g_timeout_record_host;
    if (!r || r[0] == 0) return "";
    snprintf(buf, sizeof(buf), " [timed-out wait: site %d (1 mbarrier, 2 upload gate, 3 pre-pass counter) block %d thread %d a=%d b=%d]",
             r[0], r[1], r[2], r[3], r[4]);
    return buf;
}

static int launch_screen(const uint16_t* q_f16, int64_t nq, const uint16_t* x_f16, int64_t n, int d_pad,
                         int64_t self_offset, float eps, int cap, const ScreenPlan& pl, int* cand_idx, float* cand_score,
                         int* cand_cnt, int* cand_flags, float* dump, int* error_flag, cudaStream_t st, int topk = 0,
                         float* cand_kth = nullptr, const int4* unit_table = nullptr, const int* gates = nullptr,
                         unsigned int* best_enc = nullptr, int64_t exec_tiles = 0, int* log_q = nullptr,
                         int log_region = 0, int* sync_counter = nullptr, const int* sync_targets = nullptr,
                         const ScreenPeers* peers = nullptr, int* cand_tb = nullptr) {
    if (gates) SLIC_PROPAGATE(arm_timeout_record());
    CUtensorMap tq, tx;
    SLIC_PROPAGATE(make_tmap(&tq, q_f16, nq, d_pad, TC_BM));
    SLIC_PROPAGATE(make_tmap(&tx, x_f16, n, d_pad, TC_BN / 2));
    ScreenParams p;
    p.nq = nq;
    p.n = n;
    p.num_k_slabs = d_pad / TC_BK;
    p.self_offset = self_offset;
    p.eps = eps;
    p.cap = cap;
    p.splits = pl.splits;
    p.tiles_per_split = pl.tiles_per_split;
    p.num_units = pl.units;
    p.cand_idx = cand_idx;
    p.cand_score = cand_score;
    p.cand_cnt = cand_cnt;
    p.cand_flags = cand_flags;
    p.topk = topk;
    p.cand_kth = cand_kth;
    p.cand_tb = cand_tb;
    p.dump = dump;
    p.error_flag = error_flag;
    p.trace = g_trace;
    p.unit_table = unit_table;
    p.gates = gates;
    p.best_enc = best_enc;
    p.log_q = log_q;
    p.log_region = log_region;
    p.sync_counter = sync_counter;
    p.sync_targets = sync_targets;
    p.num_peers = 0;
    for (int g = 0; g < SLIC_MAX_PEERS; ++g) {
        p.peer_best[g] = nullptr;
        p.peer_sync[g] = nullptr;
    }
    if (peers) {
        p.num_peers = peers->num_peers;
        for (int g = 0; g < peers->num_peers; ++g) {
            p.peer_best[g] = peers->peer_best[g];
            p.peer_sync[g] = peers->peer_sync[g];
        }
    }
    Scratch queue;   // (freed in stream order, i.e. after the kernel)
    SLIC_CUDA_OK(queue.alloc(sizeof(int), st));
    SLIC_CUDA_OK(cudaMemsetAsync(queue.ptr, 0, sizeof(int), st));
    p.queue = queue.as<int>();
    const bool sym = best_enc != nullptr;
    const bool is_topk = topk > 0;
    const bool ares = screen_ares(d_pad);
    if (sym && (is_topk || !unit_table)) {
        set_error("symmetric screen: needs the top-1 kernel and a unit list");
        return SLIC_ERR_UNSUPPORTED;
    }
    KernelFn fn;
    size_t smem_bytes;
    pick_screen_kernel(sym, ares, is_topk, &fn, &smem_bytes);
    static bool attr_done[64][8] = {{false}};
    int dev = 0;
    SLIC_CUDA_OK(cudaGetDevice(&dev));
    bool& attr_set = attr_done[dev & 63][(sym ? 4 : 0) + (ares ? 2 : 0) + (is_topk ? 1 : 0)];
    if (!attr_set) {
        SLIC_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        attr_set = true;
    }
    const int64_t pairs = num_sms() / 2;
    const int64_t grid = (pl.units < pairs ? pl.units : pairs) * 2;
    if (g_profile) {
        if (!g_ev_start) {
            SLIC_CUDA_OK(cudaEventCreate(&g_ev_start));
            SLIC_CUDA_OK(cudaEventCreate(&g_ev_stop));
        }
        SLIC_CUDA_OK(cudaEventRecord(g_ev_start, st));
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(sym ? TC_THREADS_SYM : TC_THREADS);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SLIC_CUDA_OK(cudaLaunchKernelEx(&cfg, fn, tq, tx, p));
    SLIC_LAUNCH_OK();
    if (g_profile) {
        SLIC_CUDA_OK(cudaEventRecord(g_ev_stop, st));
        g_last_flop = 2.0 * (double)nq * (double)n * (double)d_pad;
        g_last_exec_flop = exec_tiles > 0 ? 2.0 * (double)exec_tiles * TC_ROW_UNIT * TC_BN * (double)d_pad : g_last_flop;
        g_have_sample = true;
    }
    return SLIC_OK;
}

// Small host -> device transfers of launch metadata (unit tables, barrier targets) go through a ring of pinned
// buffers: a cudaMemcpyAsync from pageable memory may wait for the stream's earlier work before it returns, which
// would stall the host in the middle of an otherwise asynchronous level.  An entry is reused only after the copy
// that last read it has completed (event).
struct PinnedSlot {
    void* host = nullptr;
    size_t cap = 0;
    cudaEvent_t done = nullptr;
    bool used = false;
};
static int stage_to_device(void* dst_dev, const void* src, size_t bytes, cudaStream_t st) {
    constexpr int SLOTS = 8;
    static thread_local PinnedSlot ring[SLOTS];
    static thread_local int next = 0;
    if (bytes == 0) return SLIC_OK;
    PinnedSlot& s = ring[next];
    next = (next + 1) % SLOTS;
    if (s.used) SLIC_CUDA_OK(cudaEventSynchronize(s.done));
    if (s.cap < bytes) {
        // (rare: a slot starts at 1 MB - the unit table of a 240 000-row search is 140 KB - because cudaFreeHost /
        // cudaHostAlloc synchronise the device and take milliseconds)
        if (s.host) SLIC_CUDA_OK(cudaFreeHost(s.host));
        s.cap = bytes < ((size_t)1 << 20) ? ((size_t)1 << 20) : bytes + bytes / 2;
        SLIC_CUDA_OK(cudaHostAlloc(&s.host, s.cap, cudaHostAllocDefault));
    }
    if (!s.done) SLIC_CUDA_OK(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    memcpy(s.host, src, bytes);
    SLIC_CUDA_OK(cudaMemcpyAsync(dst_dev, s.host, bytes, cudaMemcpyHostToDevice, st));
    SLIC_CUDA_OK(cudaEventRecord(s.done, st));
    s.used = true;
    return SLIC_OK;
}

constexpr int TC_CAP = 32;

// Gated launch: the database arrives in `num_chunks` row chunks (host -> device copy + normalise on another stream).
// Column split s = chunk s; the unit (row unit r, split s) needs chunk max(chunk of r's last row, s), and units are
// ordered by that gate so that the persistent CTAs consume the triangle of chunk pairs as it fills:
//   gate 0: rows of chunk 0 x columns of chunk 0;  gate g: (rows of chunks <= g) x chunk g  and  chunk g x (chunks < g).
// Inside a gate the units of one column range are adjacent, so concurrent CTAs still share their B slabs through L2.
static int4 unit_entry(int64_t row_unit, int64_t ct0, int count, int stride, int gate, int stream, bool coldir) {
    int4 e;
    e.x = (int)row_unit;
    e.y = (int)ct0;
    e.z = (count & 0xffff) | (stride << 16);
    e.w = ((gate + 1) & 0xfff) | ((stream & 0xffff) << 12) | (coldir ? (1 << 28) : 0);
    return e;
}

// Symmetric self-search (Q == X): S = X X^T is symmetric, so only tiles on or right of the diagonal are computed
// (T (T + 1) / 2 of T^2 256 x 256 tiles) and every off-diagonal tile is filtered twice: along its rows for the row
// block's queries and along its columns for the column block's.
//   pre-pass  every row unit x SYM_SAMPLE_TILES column tiles spread over the (already available) database, rows only:
//             gives every row a first threshold before it is met as a column.  ~2 * SAMPLE / T of extra work.
//   triangle  column chunks of SYM_CHUNK_TILES tiles, chunk-major: the units of one chunk are adjacent in the list,
//             so the ~74 concurrently running CTA pairs stream the same 16 MB of B tiles and share them through L2
//             (row-major orders were measured: each pair then streams its own column range from HBM and the kernel
//             becomes DRAM-bound).
// part / parts: this process takes one contiguous 1 / parts share of the triangle (multi-GPU); the pre-pass is done by everyone.
constexpr int SYM_CHUNK_TILES = 64;
constexpr int SYM_SAMPLE_TILES = 16;
// mode: SYM_FULL      pre-pass over all row units + this part's share of the triangle
//       SYM_BESTS     ONLY a pre-pass, over this part's 1 / parts of the row units (multi-GPU phase 1: the parts then
//                     exchange the row bests, so that every part starts the triangle with thresholds for ALL rows)
//       SYM_TRIANGLE  ONLY this part's share of the triangle (row bests were seeded by the caller)
//       SYM_FUSED     SYM_BESTS followed by SYM_TRIANGLE in ONE unit list (multi-GPU, comm.cu): the pre-pass units publish
//                     to every rank's best array from inside the kernel and the triangle units wait for the pre-pass
//                     arrivals of ALL ranks (*prepass_units_all = their number over all parts)
enum SymMode { SYM_FULL = 0, SYM_BESTS = 1, SYM_TRIANGLE = 2, SYM_FUSED = 3 };
constexpr int SYM_FUSED_PRE_TILES = 16;   // fused pre-pass: a row unit's sample is cut into units of this many tiles (balance)
static int plan_screen_sym(int64_t n, int part, int parts, const GateSpec* g, ScreenPlan* pl, std::vector<int4>* table,
                           SymMode mode = SYM_FULL, int64_t* prepass_units_all = nullptr) {
    const bool own_rows_prepass = mode == SYM_BESTS || mode == SYM_FUSED;
    // R row units of 256 rows (a CTA pair's rows), T column tiles of 256 columns: the diagonal block of row unit r is
    // column tile r and is filtered along rows only
    const int64_t R = ceil_div(n, TC_ROW_UNIT), T = ceil_div(n, TC_BN);
    SLIC_REQUIRE(T < 65536, "symmetric screen: too many column tiles");
    SLIC_REQUIRE(parts >= 1 && part >= 0 && part < parts, "symmetric screen: bad partition");
    int64_t chunk_tiles_gate = 0, chunk_units_gate = 0;
    if (g) {
        SLIC_REQUIRE(g->gates && g->num_chunks >= 1 && g->num_chunks < 4095 && g->chunk_rows > 0 &&
                         g->chunk_rows % TC_ROW_UNIT == 0,
                     "gated screen: chunk_rows must be a positive multiple of 256");
        SLIC_REQUIRE(ceil_div(n, g->chunk_rows) == g->num_chunks, "gated screen: chunks do not tile the database");
        chunk_tiles_gate = g->chunk_rows / TC_BN;
        chunk_units_gate = g->chunk_rows / TC_ROW_UNIT;
    }
    table->clear();
    // pre-pass sample: tiles spread over the whole matrix, or over the first upload chunk when the rest is in flight
    const int64_t span = g ? (chunk_tiles_gate < T ? chunk_tiles_gate : T) : T;
    // SYM_BESTS / SYM_FUSED: every part pays a warm-up of loose thresholds at the start of its (short) share of the
    // triangle, so a stronger sample pays off from 4 parts on.  Round 1 (bfloat16 screen, eps 2^-7), 8 parts, C3: 16 / 32 /
    // 64 blocks -> 3.96 / 3.64 / 3.30 ms for the triangle share against +0.1 ms per 16 blocks here: 64.  Round 2 (float16,
    // eps 2^-9 + 2^-10: a loose threshold admits far fewer candidates), 4 parts, whole level-0 stage: 7.35 / 7.17 / 7.37 ms:
    // flat, 32.
    int samples = own_rows_prepass ? (parts >= 4 ? 2 * SYM_SAMPLE_TILES : SYM_SAMPLE_TILES) : SYM_SAMPLE_TILES / parts;
    if (own_rows_prepass && samples > span / 4) samples = (int)(span / 4);   // small inputs: a sample, not the whole square
    // small inputs (a hierarchy's level 1): the pre-pass must stay a sample - measured at 21 436 x 512 float64 centroids:
    // 16 / 10 / 4 sample blocks -> 0.88 / 0.79 / 0.72 ms for the whole search
    if (mode == SYM_FULL && R < 128 && samples > R / 16) samples = (int)(R / 16);
    if (samples < 4) samples = 4;
    if (samples > span) samples = (int)span;
    const int stride = (int)(span / samples);
    const int64_t pre0 = own_rows_prepass ? R * part / parts : 0;
    const int64_t pre1 = own_rows_prepass ? R * (part + 1) / parts : R;
    const int pre_len = mode == SYM_FUSED ? SYM_FUSED_PRE_TILES : samples;
    if (prepass_units_all) *prepass_units_all = R * ceil_div(samples, pre_len);
    for (int64_t r = pre0; r < pre1 && mode != SYM_TRIANGLE; ++r) {
        const int gate = g ? (int)(r / chunk_units_gate) : -1;
        for (int s0 = 0; s0 < samples; s0 += pre_len)
            table->push_back(unit_entry(r, (int64_t)s0 * stride, samples - s0 < pre_len ? samples - s0 : pre_len, stride, gate, 0,
                                        false));
    }
    // part / parts: a CONTIGUOUS range of the chunk-major unit list holding 1 / parts of the triangle's tiles.  (Dealing
    // the units round-robin was measured at 8 ranks: a rank's 74 concurrent CTA pairs then span ~9 column chunks, the B
    // tiles are no longer shared through L2 and the kernel runs at half speed.)
    const int64_t chunk_tiles = SYM_CHUNK_TILES;   // 16 384 columns = 16 MB of f16 B rows at d_pad 512
    int64_t total_tiles = 0;
    for (int64_t c0 = 0; c0 < T; c0 += chunk_tiles) {
        const int64_t c1 = c0 + chunk_tiles < T ? c0 + chunk_tiles : T;
        for (int64_t r = 0; r < c1; ++r) total_tiles += c1 - (r > c0 ? r : c0);
    }
    // Unit length: units are handed out dynamically (p.queue), so the last ones to finish leave at most one unit of
    // idle time per CTA pair - keep a unit well below a pair's share of the work (level 1 of a hierarchy has ~60 blocks per
    // pair in total), but long enough to amortise the reload of the resident A rows (one block's worth of traffic).
    const int64_t pairs = num_sms() / 2 > 0 ? num_sms() / 2 : 1;
    int64_t unit_len = total_tiles / parts / (pairs * 12);
    unit_len = unit_len < 8 ? 8 : (unit_len > chunk_tiles ? chunk_tiles : unit_len);
    int64_t seen_tiles = 0;
    for (int64_t c0 = 0; c0 < T && mode != SYM_BESTS; c0 += chunk_tiles) {
        const int64_t c1 = c0 + chunk_tiles < T ? c0 + chunk_tiles : T;
        for (int64_t r = 0; r < c1; ++r) {
            const int gate = g ? (int)((c1 - 1) / chunk_tiles_gate) : -1;   // column chunk >= row chunk
            for (int64_t ct0 = r > c0 ? r : c0; ct0 < c1; ct0 += unit_len) {
                const int64_t cnt = c1 - ct0 < unit_len ? c1 - ct0 : unit_len;
                const int64_t owner = seen_tiles * parts / total_tiles;   // < parts: seen_tiles < total_tiles here
                seen_tiles += cnt;
                if (owner != part) continue;
                table->push_back(unit_entry(r, ct0, (int)cnt, 1, gate, 0, true));
            }
        }
    }
    if (g)   // consume the upload in arrival order: (pre-pass, triangle) of gate 0, then of gate 1, ...
        std::stable_sort(table->begin(), table->end(), [](const int4& a, const int4& b) { return (a.w & 0xfff) < (b.w & 0xfff); });
    pl->splits = 1;
    pl->tiles_per_split = (int)T;
    pl->units = (int64_t)table->size();
    return SLIC_OK;
}

static int plan_screen_gated(int64_t nq, int64_t n, int64_t self_offset, const GateSpec& g, ScreenPlan* pl,
                             std::vector<int4>* table) {
    const int64_t rows_per_unit = TC_ROW_UNIT;
    SLIC_REQUIRE(g.gates && g.num_chunks >= 1 && g.num_chunks < 32768 && g.chunk_rows > 0 && g.chunk_rows % TC_ROW_UNIT == 0,
                 "gated screen: chunk_rows must be a positive multiple of 256");
    SLIC_REQUIRE(ceil_div(n, g.chunk_rows) == g.num_chunks, "gated screen: chunks do not tile the database");
    SLIC_REQUIRE(self_offset >= 0 && self_offset + nq <= n, "gated screen: queries must be database rows");
    const int64_t row_units = ceil_div(nq, rows_per_unit);
    pl->tiles_per_split = (int)(g.chunk_rows / TC_BN);
    pl->splits = g.num_chunks;
    pl->units = row_units * pl->splits;
    table->clear();
    table->reserve((size_t)pl->units);
    for (int gate = 0; gate < g.num_chunks; ++gate)
        for (int s = 0; s <= gate; ++s)
            for (int64_t r = 0; r < row_units; ++r) {
                int64_t last = (r + 1) * rows_per_unit - 1;
                if (last > nq - 1) last = nq - 1;
                const int rc = (int)((last + self_offset) / g.chunk_rows);
                const int need = rc > s ? rc : s;
                if (need != gate) continue;
                const int64_t ct0 = (int64_t)s * pl->tiles_per_split;
                int64_t cnt = ceil_div(n, TC_BN) - ct0;
                if (cnt > pl->tiles_per_split) cnt = pl->tiles_per_split;
                table->push_back(unit_entry(r, ct0, (int)cnt, 1, gate, s, false));
            }
    SLIC_REQUIRE((int64_t)table->size() == pl->units, "gated screen: internal unit count mismatch");
    return SLIC_OK;
}

template <typename T>
static int nn_top1_sym_impl(const T* unit, const uint16_t* ub, int64_t n, int d, int d_pad, float eps, int* idx_out,
                            T* dist_out, int* stats_out, cudaStream_t st, int part, int parts, const GateSpec* gate,
                            AfterScreenFn after, void* after_ctx, bool* overflowed, int mode = 0,
                            const int* bests_in = nullptr, int* bests_out = nullptr, int* stats_ext = nullptr,
                            const ScreenPeers* peers = nullptr, AfterScreenFn before_screen = nullptr,
                            void* before_ctx = nullptr);
static bool screen_sym_allowed();
constexpr int64_t SYM_MIN_ROWS_FWD = 16384;   // below: too few tiles to fill the machine with half of them

template <typename T>
static int nn_top1_impl(const T* q_unit, const uint16_t* q_f16, int64_t nq, const T* x_unit, const uint16_t* x_f16,
                        int64_t n, int d, int d_pad, int64_t self_offset, float eps, int* idx_out, T* dist_out,
                        int* stats_out, cudaStream_t st, const GateSpec* gate = nullptr, AfterScreenFn after = nullptr,
                        void* after_ctx = nullptr, int* stats_ext = nullptr) {
    // stats_ext: asynchronous mode, see nn_top1_sym_impl ([1] rows to finish exactly, [4] pipeline error, [5] log overflow)
    if (q_f16 == x_f16 && q_unit == x_unit && nq == n && self_offset == 0 && n >= SYM_MIN_ROWS_FWD && screen_sym_allowed()) {
        bool overflowed = false;
        SLIC_PROPAGATE(nn_top1_sym_impl<T>(x_unit, x_f16, n, d, d_pad, eps, idx_out, dist_out, stats_out, st, 0, 1, gate,
                                           after, after_ctx, &overflowed, 0, nullptr, nullptr, stats_ext));
        if (stats_ext || !overflowed) return SLIC_OK;
        // (degenerate input: almost every pair within eps of the best) - the full square with per-row lists and the
        // exact finisher handles it; the upload, if any, has been enqueued and joined already
        gate = nullptr;
        after = nullptr;
    }
    ScreenPlan pl = plan_screen(nq, n);
    std::vector<int4> table;
    Scratch table_dev;
    if (gate) {
        SLIC_PROPAGATE(plan_screen_gated(nq, n, self_offset, *gate, &pl, &table));
        SLIC_CUDA_OK(table_dev.alloc(table.size() * sizeof(int4), st));
        SLIC_PROPAGATE(stage_to_device(table_dev.ptr, table.data(), table.size() * sizeof(int4), st));
    }
    const int64_t slots = (int64_t)pl.splits * 2 * nq;   // one list per (split, 128-column half of the tiles, row)
    Scratch ci, cs, cc, cf, ovr, stats;
    SLIC_CUDA_OK(ci.alloc(slots * TC_CAP * sizeof(int), st));
    SLIC_CUDA_OK(cs.alloc(slots * TC_CAP * sizeof(float), st));
    SLIC_CUDA_OK(cc.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(cf.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(ovr.alloc(nq * sizeof(int), st));
    int* stats_dev = stats_ext;
    if (!stats_dev) {
        SLIC_CUDA_OK(stats.alloc(8 * sizeof(int), st));
        stats_dev = stats.as<int>();
    }
    SLIC_CUDA_OK(cudaMemsetAsync(stats_dev, 0, 8 * sizeof(int), st));
    SLIC_PROPAGATE(launch_screen(q_f16, nq, x_f16, n, d_pad, self_offset, eps, TC_CAP, pl, ci.as<int>(), cs.as<float>(),
                                 cc.as<int>(), cf.as<int>(), nullptr, stats_dev + 4, st, 0, nullptr,
                                 gate ? table_dev.as<int4>() : nullptr, gate ? gate->gates : nullptr));
    // gated: the caller now enqueues the upload that feeds the running kernel and makes `st` wait for its end
    if (after) SLIC_PROPAGATE(after(after_ctx));
    rerank_top1_kernel<T><<<(unsigned)ceil_div(nq, 8), 256, 0, st>>>(q_unit, x_unit, nq, d, eps, TC_CAP, 2 * pl.splits,
                                                                     ci.as<int>(), cs.as<float>(), cc.as<int>(),
                                                                     cf.as<int>(), idx_out, dist_out, ovr.as<int>(),
                                                                     stats_dev);
    SLIC_LAUNCH_OK();
    if (stats_ext) return SLIC_OK;   // asynchronous mode: rows flagged in stats_ext[1] are finished by the caller's retry
    int host_stats[8];
    SLIC_CUDA_OK(cudaMemcpyAsync(host_stats, stats_dev, sizeof(host_stats), cudaMemcpyDeviceToHost, st));
    SLIC_CUDA_OK(cudaStreamSynchronize(st));
    if (host_stats[4] != 0) {
        set_error("nn_screen_kernel: pipeline barrier timed out");
        return SLIC_ERR_CUDA;
    }
    const int n_over = host_stats[1];
    if (n_over > 0) {
        Scratch oi, od;
        SLIC_CUDA_OK(oi.alloc((int64_t)n_over * sizeof(int), st));
        SLIC_CUDA_OK(od.alloc((int64_t)n_over * sizeof(T), st));
        SLIC_PROPAGATE(slic_nn_exact_top1(q_unit, ovr.as<int>(), n_over, x_unit, n, d,
                                          sizeof(T) == 4 ? SLIC_F32 : SLIC_F64, self_offset, oi.as<int>(), od.ptr, st));
        scatter_rows_kernel<T><<<(unsigned)ceil_div(n_over, 256), 256, 0, st>>>(ovr.as<int>(), n_over, oi.as<int>(),
                                                                                od.as<T>(), idx_out, dist_out);
        SLIC_LAUNCH_OK();
    }
    if (stats_out) SLIC_CUDA_OK(cudaMemcpyAsync(stats_out, stats_dev, 4 * sizeof(int), cudaMemcpyDeviceToDevice, st));
    return SLIC_OK;
}

template <typename T>
static int topk_tc_impl(const T* q_unit, const uint16_t* q_f16, int64_t nq, const T* x_unit, const uint16_t* x_f16,
                        int64_t n, int d, int d_pad, int k, int64_t self_offset, float eps, int* idx_out, T* dist_out,
                        int* stats_out, cudaStream_t st) {
    const ScreenPlan pl = plan_screen_topk(nq, n, k);
    const int TC_CAP_TOPK = topk_cap(k, (int64_t)pl.tiles_per_split * (TC_BN / 2));
    const int64_t slots = (int64_t)pl.splits * 2 * nq;   // one list per (split, 128-column half of the tiles, row)
    Scratch ci, cs, cc, cf, ck, ctb, ovr, stats;
    SLIC_CUDA_OK(ctb.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(cudaMemsetAsync(ctb.ptr, 0, slots * sizeof(int), st));
    SLIC_CUDA_OK(ci.alloc(slots * TC_CAP_TOPK * sizeof(int), st));
    SLIC_CUDA_OK(cs.alloc(slots * TC_CAP_TOPK * sizeof(float), st));
    SLIC_CUDA_OK(cc.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(cf.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(ck.alloc(slots * sizeof(float), st));
    SLIC_CUDA_OK(ovr.alloc(nq * sizeof(int), st));
    SLIC_CUDA_OK(stats.alloc(8 * sizeof(int), st));
    SLIC_CUDA_OK(cudaMemsetAsync(stats.ptr, 0, 8 * sizeof(int), st));
    SLIC_PROPAGATE(launch_screen(q_f16, nq, x_f16, n, d_pad, self_offset, eps, TC_CAP_TOPK, pl, ci.as<int>(),
                                 cs.as<float>(), cc.as<int>(), cf.as<int>(), nullptr, stats.as<int>() + 4, st, k,
                                 ck.as<float>(), nullptr, nullptr, nullptr, 0, nullptr, 0, nullptr, nullptr, nullptr,
                                 ctb.as<int>()));
    rerank_topk_kernel<T><<<(unsigned)nq, RK_THREADS, 0, st>>>(q_unit, x_unit, nq, d, eps, TC_CAP_TOPK, 2 * pl.splits, k,
                                                               ci.as<int>(), cs.as<float>(), cc.as<int>(), cf.as<int>(),
                                                               ck.as<float>(), idx_out, dist_out, ovr.as<int>(),
                                                               stats.as<int>());
    SLIC_LAUNCH_OK();
    int host_stats[8];
    SLIC_CUDA_OK(cudaMemcpyAsync(host_stats, stats.ptr, sizeof(host_stats), cudaMemcpyDeviceToHost, st));
    SLIC_CUDA_OK(cudaStreamSynchronize(st));
    if (host_stats[4] != 0) {
        set_error("nn_screen_kernel: pipeline barrier timed out");
        return SLIC_ERR_CUDA;
    }
    const int n_over = host_stats[1];
    if (n_over > 0) {
        Scratch oi, od;
        SLIC_CUDA_OK(oi.alloc((int64_t)n_over * k * sizeof(int), st));
        SLIC_CUDA_OK(od.alloc((int64_t)n_over * k * sizeof(T), st));
        SLIC_PROPAGATE(exact_topk_cosine_rows(q_unit, ovr.as<int>(), n_over, x_unit, n, d,
                                              sizeof(T) == 4 ? SLIC_F32 : SLIC_F64, k, self_offset, oi.as<int>(), od.ptr,
                                              st));
        scatter_topk_rows_kernel<T><<<(unsigned)ceil_div((int64_t)n_over * k, 256), 256, 0, st>>>(
            ovr.as<int>(), n_over, k, oi.as<int>(), od.as<T>(), idx_out, dist_out);
        SLIC_LAUNCH_OK();
    }
    if (stats_out) SLIC_CUDA_OK(cudaMemcpyAsync(stats_out, stats.ptr, 4 * sizeof(int), cudaMemcpyDeviceToDevice, st));
    return SLIC_OK;
}

// ---- symmetric self-search ------------------------------------------------------------------------
constexpr int SYM_LOG_PER_ROW = 96;       // log capacity in records per database row (12 bytes + sizeof(T) each)
constexpr int64_t SYM_LOG_MIN = (int64_t)1 << 23;

// SLIC_SCREEN_SYM=0 keeps the full-square screen for self-searches (experiments / fallback)
static bool screen_sym_allowed();
bool screen_self_search_is_symmetric(int64_t n) { return n >= SYM_MIN_ROWS_FWD && screen_sym_allowed(); }
static bool screen_sym_allowed() {
    static int cached = -1;
    if (cached < 0) {
        const char* e = getenv("SLIC_SCREEN_SYM");
        cached = (e && atoi(e) == 0) ? 0 : 1;
    }
    return cached != 0;
}

// order-preserving score encoding <-> the same order as SIGNED int32 (what an all-reduce MAX over int32 compares)
__global__ void flip_sign_bit_kernel(const unsigned int* __restrict__ in, int64_t n, unsigned int* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] ^ 0x80000000u;
}

// all the per-launch state of a symmetric search in ONE launch: counters, log counts, row minima, row bests, outputs
__global__ void sym_init_kernel(int* __restrict__ stats8, int* __restrict__ lcnt, int64_t regions,
                                unsigned char* __restrict__ rmin_bytes, int64_t rmin_n_bytes, int* __restrict__ sync_counter,
                                unsigned int* __restrict__ best, const unsigned int* __restrict__ bests_in, int64_t n,
                                unsigned int* __restrict__ idx_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 8) stats8[i] = 0;
    if (i == 0) *sync_counter = 0;
    if (i < regions) lcnt[i] = 0;
    if (i < n) {
        best[i] = bests_in ? (bests_in[i] ^ 0x80000000u) : ENC_NEG_INF;   // exchanged bests arrive in signed-comparable form
        if (idx_out) idx_out[i] = 0x7fffffffu;
    }
    // row minima: all-ones (above every distance's bit pattern), 16 bytes per thread
    const int64_t b = i * 16;
    if (b + 16 <= rmin_n_bytes) *reinterpret_cast<uint4*>(rmin_bytes + b) = make_uint4(~0u, ~0u, ~0u, ~0u);
    else
        for (int64_t k = b; k < rmin_n_bytes; ++k) rmin_bytes[k] = 0xff;
}

__global__ void fill_u32_kernel(unsigned int* out, int64_t n, unsigned int v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = v;
}

template <typename T> struct DistBits;
template <> struct DistBits<float> {
    typedef unsigned int type;
    static __device__ __forceinline__ type of(float d) { return __float_as_uint(d); }        // d >= 0: monotone
    static __device__ __forceinline__ float back(type b) { return __uint_as_float(b); }
};
template <> struct DistBits<double> {
    typedef unsigned long long type;
    static __device__ __forceinline__ type of(double d) { return (type)__double_as_longlong(d); }
    static __device__ __forceinline__ double back(type b) { return __longlong_as_double((long long)b); }
};

// Re-rank, pass 1: one CTA per log region.  A record survives iff its screened score is within eps of its row's FINAL
// best; survivors are evaluated exactly (one warp per record, float64 accumulation) and the row keeps the smallest
// distance (rounded to T as the reference holds it).  edist[record] = that distance, or -1 for a dropped record.
template <typename T>
__global__ void __launch_bounds__(256) sym_rerank_dist_kernel(const T* __restrict__ unit, int d, float eps, int region,
                                                              const int* __restrict__ log_q, const int* __restrict__ log_nb,
                                                              const float* __restrict__ log_s,
                                                              const int* __restrict__ log_cnt,
                                                              const unsigned int* __restrict__ best_enc,
                                                              typename DistBits<T>::type* __restrict__ row_min,
                                                              T* __restrict__ edist, int* __restrict__ stats) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * region;
    const int cnt = log_cnt[blockIdx.x];
    if (threadIdx.x == 0) {
        atomicAdd(&stats[3], cnt >> 4);   // records logged by the screen, in units of 16
        atomicMax(&stats[6], cnt);        // fullest region
    }
    int reranked = 0;
    for (int e0 = warp * 32; e0 < cnt; e0 += nwarps * 32) {
        const int e = e0 + lane;
        int q = 0, nb = 0;
        bool keep = false;
        if (e < cnt) {
            q = log_q[base + e];
            nb = log_nb[base + e];
            keep = log_s[base + e] >= dec_score(best_enc[q]) - eps;
            if (!keep) edist[base + e] = (T)-1;
        }
        unsigned mask = __ballot_sync(0xffffffffu, keep);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            const int qq = __shfl_sync(0xffffffffu, q, src), nn = __shfl_sync(0xffffffffu, nb, src);
            const double sim = warp_dot<T>(unit + (int64_t)qq * d, unit + (int64_t)nn * d, d, lane);
            if (lane == 0) {
                const T dist = cosine_distance_from_sim<T>(sim);
                edist[base + e0 + src] = dist;
                atomicMin(row_min + qq, DistBits<T>::of(dist));
            }
            ++reranked;
        }
    }
    if (lane == 0 && reranked) atomicAdd(&stats[0], reranked);
}

// pass 2: among the records that attain the row's smallest distance the lowest neighbour index wins (np.argmin)
template <typename T>
__global__ void __launch_bounds__(256) sym_rerank_pick_kernel(int region, const int* __restrict__ log_q,
                                                              const int* __restrict__ log_nb,
                                                              const int* __restrict__ log_cnt,
                                                              const typename DistBits<T>::type* __restrict__ row_min,
                                                              const T* __restrict__ edist, int* __restrict__ idx_out,
                                                              T* __restrict__ dist_out) {
    const int64_t base = (int64_t)blockIdx.x * region;
    const int cnt = log_cnt[blockIdx.x];
    for (int e = threadIdx.x; e < cnt; e += blockDim.x) {
        const T dist = edist[base + e];
        if (dist < (T)0) continue;
        const int q = log_q[base + e];
        if (DistBits<T>::of(dist) == row_min[q]) {
            atomicMin(idx_out + q, log_nb[base + e]);
            if (dist_out) dist_out[q] = dist;
        }
    }
}

// rows that received no record at all (cannot happen unless the log overflowed) are reported for the exact kernel
__global__ void sym_unsettled_rows_kernel(int* __restrict__ idx_out, int64_t n, int* __restrict__ rows, int* __restrict__ stats) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && idx_out[i] == 0x7fffffff) rows[atomicAdd(&stats[1], 1)] = (int)i;
}

template <typename T>
static int nn_top1_sym_impl(const T* unit, const uint16_t* ub, int64_t n, int d, int d_pad, float eps, int* idx_out,
                            T* dist_out, int* stats_out, cudaStream_t st, int part, int parts, const GateSpec* gate,
                            AfterScreenFn after, void* after_ctx, bool* overflowed, int mode, const int* bests_in,
                            int* bests_out, int* stats_ext, const ScreenPeers* peers, AfterScreenFn before_screen,
                            void* before_ctx) {
    // peers (SYM_FUSED only): the row bests and the pre-pass counter live in this rank's peer-mapped window; before_screen
    // runs on the host between the initialisation kernel and the screen launch (comm.cu enqueues the cross-rank barrier
    // there: no rank may publish into a window that has not been reset yet).
    // stats_ext (device, 8 ints, optional): ASYNCHRONOUS mode - nothing here waits for the device.  The counters
    // {[1] rows without a neighbour, [4] pipeline error, [5] log overflow} land in stats_ext; if any is non-zero the
    // result is incomplete and the caller repeats the search through the synchronous path (which has the fallbacks).
    typedef typename DistBits<T>::type Bits;
    *overflowed = false;
    ScreenPlan pl;
    std::vector<int4> table;
    int64_t prepass_units_all = 0;
    SLIC_PROPAGATE(plan_screen_sym(n, part, parts, gate, &pl, &table, (SymMode)mode, &prepass_units_all));
    SLIC_REQUIRE((mode == SYM_FUSED) == (peers != nullptr), "symmetric screen: the fused mode needs peer windows (and only it)");
    SLIC_REQUIRE(mode != SYM_FUSED || (stats_ext && !gate), "symmetric screen: the fused mode is asynchronous and ungated");
    int64_t exec_tiles = 0;
    for (const int4& e : table) exec_tiles += e.z & 0xffff;
    // sync_targets[g + 1] = epilogue-warp arrivals of all pre-pass units with gate <= g (index 0: ungated)
    const int num_gates = gate ? gate->num_chunks : 0;
    std::vector<int> targets(num_gates + 1, 0);
    for (const int4& e : table) {
        if ((e.w >> 28) & 1) continue;          // triangle unit
        const int g = (e.w & 0xfff) - 1;
        for (int k = g + 1; k <= num_gates; ++k) targets[k] += 2 * TC_EPI_WARPS;   // g = -1 (ungated): index 0
    }
    if (mode == SYM_FUSED) targets[0] = (int)(prepass_units_all * 2 * TC_EPI_WARPS);   // the pre-pass units of ALL ranks
    const int64_t groups = num_sms() / 2;
    const int64_t grid = (pl.units < groups ? pl.units : groups) * 2;
    const int64_t regions = grid * TC_EPI_WARPS;
    // (small inputs log more per row - every row starts from scratch in the pre-pass - and spread it less evenly)
    int64_t capacity = (int64_t)SYM_LOG_PER_ROW * n > SYM_LOG_MIN ? (int64_t)SYM_LOG_PER_ROW * n : SYM_LOG_MIN;
    if (mode == SYM_BESTS) capacity = SYM_LOG_MIN;   // the records of phase 1 are discarded (an overflow is harmless)
    const int64_t region = ceil_div(capacity, regions);
    SLIC_REQUIRE(region < ((int64_t)1 << 31), "symmetric screen: log region too large");
    Scratch table_dev, lq, lnb, ls, lcnt, best, rmin, edist, ovr, stats;
    // unit table followed by the barrier targets: one transfer.  sync: [0] counter, then the targets (device view)
    const size_t table_bytes = table.size() * sizeof(int4);
    SLIC_CUDA_OK(table_dev.alloc(table_bytes + (targets.size() + 4) * sizeof(int), st));
    {
        std::vector<unsigned char> blob(table_bytes + (targets.size() + 1) * sizeof(int));
        memcpy(blob.data(), table.data(), table_bytes);
        const int zero = 0;
        memcpy(blob.data() + table_bytes, &zero, sizeof(int));
        memcpy(blob.data() + table_bytes + sizeof(int), targets.data(), targets.size() * sizeof(int));
        SLIC_PROPAGATE(stage_to_device(table_dev.ptr, blob.data(), blob.size(), st));
    }
    int* sync_dev = reinterpret_cast<int*>(static_cast<unsigned char*>(table_dev.ptr) + table_bytes);
    SLIC_CUDA_OK(lq.alloc(regions * region * sizeof(int), st));
    SLIC_CUDA_OK(lnb.alloc(regions * region * sizeof(int), st));
    SLIC_CUDA_OK(ls.alloc(regions * region * sizeof(float), st));
    SLIC_CUDA_OK(edist.alloc(regions * region * sizeof(T), st));
    SLIC_CUDA_OK(lcnt.alloc(regions * sizeof(int), st));
    if (!peers) SLIC_CUDA_OK(best.alloc(n * sizeof(unsigned int), st));
    unsigned int* best_dev = peers ? peers->own_best : best.as<unsigned int>();
    int* sync_counter_dev = peers ? peers->own_sync : sync_dev;
    SLIC_CUDA_OK(rmin.alloc(n * sizeof(Bits), st));
    SLIC_CUDA_OK(ovr.alloc(n * sizeof(int), st));
    int* stats_dev = stats_ext;
    if (!stats_dev) {
        SLIC_CUDA_OK(stats.alloc(8 * sizeof(int), st));
        stats_dev = stats.as<int>();
    }
    int* flag_dev = stats_dev + 5;   // the log-overflow flag lives in the same block: one read-back fetches everything
    {
        const int64_t rmin_bytes = n * (int64_t)sizeof(Bits);
        int64_t threads = n > regions ? n : regions;
        if (ceil_div(rmin_bytes, 16) > threads) threads = ceil_div(rmin_bytes, 16);
        if (threads < 8) threads = 8;
        sym_init_kernel<<<(unsigned)ceil_div(threads, 256), 256, 0, st>>>(stats_dev, lcnt.as<int>(), regions,
                                                                         static_cast<unsigned char*>(rmin.ptr), rmin_bytes,
                                                                         sync_counter_dev, best_dev,
                                                                         (const unsigned int*)bests_in, n, (unsigned int*)idx_out);
        SLIC_LAUNCH_OK();
    }
    if (before_screen) SLIC_PROPAGATE(before_screen(before_ctx));
    SLIC_PROPAGATE(launch_screen(ub, n, ub, n, d_pad, 0, eps, 0, pl, lnb.as<int>(), ls.as<float>(), lcnt.as<int>(),
                                 flag_dev, nullptr, stats_dev + 4, st, 0, nullptr, table_dev.as<int4>(),
                                 gate ? gate->gates : nullptr, best_dev, exec_tiles, lq.as<int>(),
                                 (int)region, sync_counter_dev, sync_dev + 1, peers));
    if (g_profile && parts > 1) g_last_flop /= (double)parts;   // this process's share of the algorithmic 2 n^2 d
    if (after) SLIC_PROPAGATE(after(after_ctx));
    if (mode == SYM_BESTS) {   // phase 1 of the multi-GPU search: the row bests are the result, the log is discarded
        flip_sign_bit_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(best_dev, n, (unsigned int*)bests_out);
        SLIC_LAUNCH_OK();
        int host_err = 0;
        SLIC_CUDA_OK(cudaMemcpyAsync(&host_err, stats_dev + 4, sizeof(int), cudaMemcpyDeviceToHost, st));
        SLIC_CUDA_OK(cudaStreamSynchronize(st));
        if (host_err != 0) {
            set_error(host_err == 2 ? "nn_screen_kernel: shared-memory window is not aligned as the symmetric layout assumes"
                                    : "nn_screen_kernel: pipeline barrier timed out");
            return SLIC_ERR_CUDA;
        }
        return SLIC_OK;
    }
    sym_rerank_dist_kernel<T><<<(unsigned)regions, 256, 0, st>>>(unit, d, eps, (int)region, lq.as<int>(), lnb.as<int>(),
                                                                 ls.as<float>(), lcnt.as<int>(), best_dev,
                                                                 rmin.as<Bits>(), edist.as<T>(), stats_dev);
    SLIC_LAUNCH_OK();
    sym_rerank_pick_kernel<T><<<(unsigned)regions, 256, 0, st>>>((int)region, lq.as<int>(), lnb.as<int>(), lcnt.as<int>(),
                                                                 rmin.as<Bits>(), edist.as<T>(), idx_out, dist_out);
    SLIC_LAUNCH_OK();
    sym_unsettled_rows_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(idx_out, n, ovr.as<int>(), stats_dev);
    SLIC_LAUNCH_OK();
    if (stats_ext) return SLIC_OK;   // asynchronous mode: the caller reads stats_ext with its own read-back
    int host_stats[8];
    SLIC_CUDA_OK(cudaMemcpyAsync(host_stats, stats_dev, sizeof(host_stats), cudaMemcpyDeviceToHost, st));
    SLIC_CUDA_OK(cudaStreamSynchronize(st));
    if (host_stats[4] == 2) {
        set_error("nn_screen_kernel: shared-memory window is not aligned as the symmetric layout assumes (set SLIC_SCREEN_SYM=0)");
        return SLIC_ERR_UNSUPPORTED;
    }
    if (host_stats[4] != 0) {
        set_error("nn_screen_kernel: pipeline barrier timed out");
        return SLIC_ERR_CUDA;
    }
    if (const char* dbg = getenv("SLIC_SYM_DEBUG")) {
        if (atoi(dbg) == 2) {   // dump the candidate log for offline analysis (scripts/sym_log_stats.py)
            std::vector<int> hq((size_t)(regions * region)), hnb((size_t)(regions * region)), hc((size_t)regions);
            std::vector<float> hs((size_t)(regions * region));
            cudaMemcpy(hq.data(), lq.ptr, hq.size() * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(hnb.data(), lnb.ptr, hnb.size() * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(hs.data(), ls.ptr, hs.size() * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(hc.data(), lcnt.ptr, hc.size() * 4, cudaMemcpyDeviceToHost);
            FILE* f = fopen("/tmp/slic_sym_log.bin", "wb");
            if (f) {
                long long hdr[3] = {(long long)n, (long long)regions, (long long)region};
                fwrite(hdr, sizeof(hdr), 1, f);
                fwrite(hc.data(), 4, hc.size(), f);
                fwrite(hq.data(), 4, hq.size(), f);
                fwrite(hnb.data(), 4, hnb.size(), f);
                fwrite(hs.data(), 4, hs.size(), f);
                fclose(f);
            }
        }
    }
    if (host_stats[5] != 0) {   // a log region filled up: records are missing, the caller repeats on the full square
        if (getenv("SLIC_SYM_DEBUG"))
            fprintf(stderr, "[slic] symmetric screen: log overflow, n=%lld regions=%lld region=%lld records=%d fullest=%d\n",
                    (long long)n, (long long)regions, (long long)region, host_stats[3] * 16, host_stats[6]);
        *overflowed = true;
        return SLIC_OK;
    }
    if (getenv("SLIC_SYM_DEBUG"))
        fprintf(stderr, "[slic] symmetric screen: n=%lld regions=%lld region=%lld records=%d fullest=%d\n", (long long)n,
                (long long)regions, (long long)region, host_stats[3] * 16, host_stats[6]);
    const int n_over = host_stats[1];
    if (n_over > 0 && parts == 1) {   // (parts > 1: the caller merges the parts first and finishes what is left)
        Scratch oi, od;
        SLIC_CUDA_OK(oi.alloc((int64_t)n_over * sizeof(int), st));
        SLIC_CUDA_OK(od.alloc((int64_t)n_over * sizeof(T), st));
        SLIC_PROPAGATE(slic_nn_exact_top1(unit, ovr.as<int>(), n_over, unit, n, d, sizeof(T) == 4 ? SLIC_F32 : SLIC_F64, 0,
                                          oi.as<int>(), od.ptr, st));
        scatter_rows_kernel<T><<<(unsigned)ceil_div(n_over, 256), 256, 0, st>>>(ovr.as<int>(), n_over, oi.as<int>(),
                                                                                od.as<T>(), idx_out, dist_out);
        SLIC_LAUNCH_OK();
    }
    if (stats_out) SLIC_CUDA_OK(cudaMemcpyAsync(stats_out, stats_dev, 4 * sizeof(int), cudaMemcpyDeviceToDevice, st));
    return SLIC_OK;
}

// ---- multi-GPU symmetric self-search: every process screens a contiguous 1 / parts share of the triangle ----------------
// key = (float32 distance bits << 32) | neighbour: distances are >= 0, so their bit patterns order like the values and
// an element-wise MIN over the processes' key arrays (one all-reduce) picks the smallest distance and, among equal
// distances, the lowest neighbour index - np.argmin's rule.  A row without a record keeps the largest key.
__global__ void sym_pack_keys_kernel(const int* __restrict__ idx, const float* __restrict__ dist, int64_t n,
                                     unsigned long long* __restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = idx[i];
    keys[i] = j == 0x7fffffff ? SYM_KEY_NONE : (((unsigned long long)__float_as_uint(dist[i]) << 32) | (unsigned int)j);
}

__global__ void sym_unpack_keys_kernel(const unsigned long long* __restrict__ keys, int64_t n, int* __restrict__ idx,
                                       float* __restrict__ dist, int* __restrict__ unsettled) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys[i];
    idx[i] = (int)(unsigned int)(k & 0xffffffffull);
    dist[i] = __uint_as_float((unsigned int)(k >> 32));
    if (k == SYM_KEY_NONE) atomicAdd(unsettled, 1);
}

// Can CTAs of `guest_threads` threads x `guest_regs` registers (no shared memory of their own) become resident next to
// the persistent top-1 screen kernel that a gated self-search of n rows x d_pad would launch?  Resources per SM:
// 228 KB of shared memory with 1 KB reserved per resident CTA; 4 sub-partitions of 16 384 registers, warps dealt
// round-robin, registers allocated per warp in units of 8 per thread.  false -> the caller uploads first, then searches.
bool screen_can_overlap_upload(int64_t n, int d_pad, int guest_threads, int guest_regs) {
    const bool sym = screen_self_search_is_symmetric(n);
    KernelFn fn;
    size_t smem_bytes;
    pick_screen_kernel(sym, screen_ares(d_pad), false, &fn, &smem_bytes);
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, fn) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    const int host_regs = (fa.numRegs + 7) / 8 * 8, gr = (guest_regs + 7) / 8 * 8;
    const int host_threads = sym ? TC_THREADS_SYM : TC_THREADS;
    const int host_warps = (host_threads / 32 + 3) / 4, guest_warps = (guest_threads / 32 + 3) / 4;   // on the fullest sub-partition
    const bool regs_ok = 32 * (host_warps * host_regs + guest_warps * gr) <= 16384;
    const bool smem_ok = smem_bytes + 2 * 1024 <= 233472;
    const bool threads_ok = host_threads + guest_threads <= 2048;
    if (getenv("SLIC_SYM_DEBUG"))
        fprintf(stderr, "[slic] overlap check: screen %d regs, %zu B smem; guest %d threads x %d regs -> regs %d smem %d\n",
                fa.numRegs, smem_bytes, guest_threads, guest_regs, (int)regs_ok, (int)smem_ok);
    return regs_ok && smem_ok && threads_ok;
}

int nn_top1_f32_gated(const float* q_unit, const uint16_t* q_f16, int64_t nq, const float* x_unit,
                      const uint16_t* x_f16, int64_t n, int d, int d_pad, int64_t self_offset, float eps, int* idx_out,
                      float* dist_out, int* stats_out, const GateSpec* gate, AfterScreenFn after, void* after_ctx,
                      cudaStream_t st, int* stats_ext) {
    if (eps <= 0.f) eps = screen_default_eps(d_pad);
    return nn_top1_impl<float>(q_unit, q_f16, nq, x_unit, x_f16, n, d, d_pad, self_offset, eps, idx_out, dist_out,
                               stats_out, st, gate, after, after_ctx, stats_ext);
}

int nn_top1_self_async(const void* unit, const uint16_t* ub, int64_t n, int d, int d_pad, int dtype, int* idx_out,
                       void* dist_out, int* stats_ext, cudaStream_t st) {
    const float eps = screen_default_eps(d_pad);
    if (dtype == SLIC_F32)
        return nn_top1_impl<float>((const float*)unit, ub, n, (const float*)unit, ub, n, d, d_pad, 0, eps, idx_out,
                                   (float*)dist_out, nullptr, st, nullptr, nullptr, nullptr, stats_ext);
    return nn_top1_impl<double>((const double*)unit, ub, n, (const double*)unit, ub, n, d, d_pad, 0, eps, idx_out,
                                (double*)dist_out, nullptr, st, nullptr, nullptr, nullptr, stats_ext);
}

int nn_top1_sym_fused(const float* unit, const uint16_t* ub, int64_t n, int d, int d_pad, int part, int parts,
                      const ScreenPeers* peers, AfterScreenFn before_screen, void* before_ctx, int* idx_out,
                      float* dist_out, int* stats_dev, cudaStream_t st) {
    if (!screen_self_search_is_symmetric(n)) {
        set_error("fused multi-GPU search: the symmetric screen needs n >= %lld rows", (long long)SYM_MIN_ROWS_FWD);
        return SLIC_ERR_UNSUPPORTED;
    }
    bool overflowed = false;
    return nn_top1_sym_impl<float>(unit, ub, n, d, d_pad, screen_default_eps(d_pad), idx_out, dist_out, nullptr, st, part,
                                   parts, nullptr, nullptr, nullptr, &overflowed, SYM_FUSED, nullptr, nullptr, stats_dev, peers,
                                   before_screen, before_ctx);
}

}  // namespace slic

extern "C" {

int slic_nn_top1(const void* q_unit_dev, const uint16_t* q_f16_dev, int64_t nq, const void* x_unit_dev,
                 const uint16_t* x_f16_dev, int64_t n, int32_t d, int32_t d_pad, int32_t dtype, int64_t self_offset,
                 float eps, int32_t* idx_out_dev, void* dist_out_dev, int32_t* stats_out_dev, slic_stream_t stream) {
    SLIC_REQUIRE(nq > 0 && n > 1 && n < ((int64_t)1 << 31) && nq < ((int64_t)1 << 31), "nn_top1: bad shape");
    SLIC_REQUIRE(d > 0 && d_pad >= d && d_pad % 64 == 0, "nn_top1: d_pad must be a multiple of 64 >= d");
    SLIC_REQUIRE(q_unit_dev && q_f16_dev && x_unit_dev && x_f16_dev && idx_out_dev, "nn_top1: null pointer");
    SLIC_REQUIRE(dtype == SLIC_F32 || dtype == SLIC_F64, "nn_top1: bad dtype");
    SLIC_REQUIRE((reinterpret_cast<uintptr_t>(q_f16_dev) & 15) == 0 && (reinterpret_cast<uintptr_t>(x_f16_dev) & 15) == 0,
                 "nn_top1: f16 matrices must be 16-byte aligned");
    SLIC_PROPAGATE(slic_require_device());
    if (eps <= 0.f) eps = slic::screen_default_eps(d_pad);
    cudaStream_t st = slic::as_stream(stream);
    if (dtype == SLIC_F32)
        return slic::nn_top1_impl<float>((const float*)q_unit_dev, q_f16_dev, nq, (const float*)x_unit_dev, x_f16_dev,
                                         n, d, d_pad, self_offset, eps, idx_out_dev, (float*)dist_out_dev,
                                         stats_out_dev, st);
    return slic::nn_top1_impl<double>((const double*)q_unit_dev, q_f16_dev, nq, (const double*)x_unit_dev, x_f16_dev, n,
                                      d, d_pad, self_offset, eps, idx_out_dev, (double*)dist_out_dev, stats_out_dev,
                                      st);
}

int slic_sym_row_bests(const float* unit_dev, const uint16_t* f16_dev, int64_t n, int32_t d, int32_t d_pad, int32_t part,
                       int32_t parts, int32_t* bests_out_dev, slic_stream_t stream) {
    using namespace slic;
    SLIC_REQUIRE(n > 1 && n < ((int64_t)1 << 31), "sym_row_bests: bad shape");
    SLIC_REQUIRE(d > 0 && d_pad >= d && d_pad % 64 == 0, "sym_row_bests: d_pad must be a multiple of 64 >= d");
    SLIC_REQUIRE(unit_dev && f16_dev && bests_out_dev, "sym_row_bests: null pointer");
    SLIC_REQUIRE(parts >= 1 && part >= 0 && part < parts, "sym_row_bests: part must be in [0, parts)");
    SLIC_REQUIRE((reinterpret_cast<uintptr_t>(f16_dev) & 15) == 0, "sym_row_bests: f16 matrix must be 16-byte aligned");
    SLIC_PROPAGATE(slic_require_device());
    if (!screen_self_search_is_symmetric(n)) {
        set_error("sym_row_bests: the symmetric screen needs n >= %lld rows (and SLIC_SCREEN_SYM != 0)", (long long)SYM_MIN_ROWS_FWD);
        return SLIC_ERR_UNSUPPORTED;
    }
    bool overflowed = false;
    return nn_top1_sym_impl<float>(unit_dev, f16_dev, n, d, d_pad, screen_default_eps(d_pad), nullptr, nullptr, nullptr,
                                   as_stream(stream), part, parts, nullptr, nullptr, nullptr, &overflowed, SYM_BESTS, nullptr,
                                   bests_out_dev);
}

int slic_nn_top1_sym_part(const float* unit_dev, const uint16_t* f16_dev, int64_t n, int32_t d, int32_t d_pad,
                          int32_t part, int32_t parts, const int32_t* row_bests_dev, float eps, uint64_t* keys_out_dev,
                          int32_t* stats_out_dev, slic_stream_t stream) {
    using namespace slic;
    SLIC_REQUIRE(n > 1 && n < ((int64_t)1 << 31), "nn_top1_sym_part: bad shape");
    SLIC_REQUIRE(d > 0 && d_pad >= d && d_pad % 64 == 0, "nn_top1_sym_part: d_pad must be a multiple of 64 >= d");
    SLIC_REQUIRE(unit_dev && f16_dev && keys_out_dev, "nn_top1_sym_part: null pointer");
    SLIC_REQUIRE(parts >= 1 && part >= 0 && part < parts, "nn_top1_sym_part: part must be in [0, parts)");
    SLIC_REQUIRE((reinterpret_cast<uintptr_t>(f16_dev) & 15) == 0, "nn_top1_sym_part: f16 matrix must be 16-byte aligned");
    SLIC_PROPAGATE(slic_require_device());
    if (!screen_self_search_is_symmetric(n)) {
        set_error("nn_top1_sym_part: the symmetric screen needs n >= %lld rows (and SLIC_SCREEN_SYM != 0)",
                  (long long)SYM_MIN_ROWS_FWD);
        return SLIC_ERR_UNSUPPORTED;
    }
    if (eps <= 0.f) eps = screen_default_eps(d_pad);
    cudaStream_t st = as_stream(stream);
    Scratch idx, dist;
    SLIC_CUDA_OK(idx.alloc((size_t)n * sizeof(int), st));
    SLIC_CUDA_OK(dist.alloc((size_t)n * sizeof(float), st));
    bool overflowed = false;
    SLIC_PROPAGATE(nn_top1_sym_impl<float>(unit_dev, f16_dev, n, d, d_pad, eps, idx.as<int>(), dist.as<float>(),
                                           stats_out_dev, st, part, parts, nullptr, nullptr, nullptr, &overflowed,
                                           row_bests_dev ? SYM_TRIANGLE : SYM_FULL, row_bests_dev, nullptr));
    sym_pack_keys_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(idx.as<int>(), dist.as<float>(), n,
                                                                     (unsigned long long*)keys_out_dev);
    SLIC_LAUNCH_OK();
    // keys[n] = 1, or 0 when this part's candidate log overflowed (records are missing): MIN over the parts tells
    // every process whether the merged result is complete
    const unsigned long long flag = overflowed ? 0ull : 1ull;
    SLIC_CUDA_OK(cudaMemcpyAsync(keys_out_dev + n, &flag, sizeof(flag), cudaMemcpyHostToDevice, st));
    SLIC_CUDA_OK(cudaStreamSynchronize(st));   // `flag` lives on this frame
    return SLIC_OK;
}

int slic_debug_sym_plan(int64_t n, int32_t part, int32_t parts, int32_t mode, int32_t gated_chunks, int32_t* units_out_host,
                        int64_t capacity, int64_t* num_units_out_host) {
    using namespace slic;
    SLIC_REQUIRE(n > 1 && n < ((int64_t)1 << 31) && num_units_out_host, "debug_sym_plan: bad arguments");
    SLIC_REQUIRE(mode >= 0 && mode <= 3, "debug_sym_plan: mode must be 0 (full), 1 (row bests), 2 (triangle) or 3 (fused)");
    SLIC_REQUIRE(gated_chunks >= 0 && gated_chunks < 4095, "debug_sym_plan: bad chunk count");
    GateSpec gs = {reinterpret_cast<const int*>(num_units_out_host) /* never dereferenced by the planner */, 0, 0};
    if (gated_chunks > 0) {
        gs.chunk_rows = ceil_div(ceil_div(n, gated_chunks), 256) * 256;
        gs.num_chunks = (int)ceil_div(n, gs.chunk_rows);
    }
    ScreenPlan pl;
    std::vector<int4> table;
    SLIC_PROPAGATE(plan_screen_sym(n, part, parts, gated_chunks > 0 ? &gs : nullptr, &pl, &table, (SymMode)mode));
    *num_units_out_host = (int64_t)table.size();
    if (units_out_host) {
        SLIC_REQUIRE(capacity >= (int64_t)table.size(), "debug_sym_plan: unit buffer too small");
        for (size_t u = 0; u < table.size(); ++u) {
            const int4 e = table[u];
            int32_t* o = units_out_host + 6 * u;
            o[0] = e.x;                                  // row unit (256 rows)
            o[1] = e.y;                                  // first column tile
            o[2] = e.z & 0xffff;                         // tile count
            o[3] = (int)((unsigned)e.z >> 16);           // tile stride
            o[4] = (e.w & 0xfff) - 1;                    // gate (-1: none)
            o[5] = (e.w >> 28) & 1;                      // column direction (triangle unit)
        }
    }
    return SLIC_OK;
}

int slic_unpack_neighbor_keys(const uint64_t* keys_dev, int64_t n, int32_t* idx_out_dev, float* dist_out_dev,
                              int32_t* status_out_dev, slic_stream_t stream) {
    using namespace slic;
    SLIC_REQUIRE(n > 0 && keys_dev && idx_out_dev && dist_out_dev && status_out_dev, "unpack_neighbor_keys: bad argument");
    SLIC_PROPAGATE(slic_require_device());
    cudaStream_t st = as_stream(stream);
    SLIC_CUDA_OK(cudaMemsetAsync(status_out_dev, 0, sizeof(int), st));
    sym_unpack_keys_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>((const unsigned long long*)keys_dev, n, idx_out_dev,
                                                                       dist_out_dev, status_out_dev);
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

int slic_topk_cosine_tc(const void* q_unit_dev, const uint16_t* q_f16_dev, int64_t nq, const void* x_unit_dev,
                        const uint16_t* x_f16_dev, int64_t n, int32_t d, int32_t d_pad, int32_t dtype, int32_t k,
                        int64_t self_offset, float eps, int32_t* idx_out_dev, void* dist_out_dev, int32_t* stats_out_dev,
                        slic_stream_t stream) {
    SLIC_REQUIRE(nq >= 0 && n > 0 && n < ((int64_t)1 << 31) && nq < ((int64_t)1 << 31), "topk_cosine_tc: bad shape");
    SLIC_REQUIRE(d > 0 && d_pad >= d && d_pad % 64 == 0, "topk_cosine_tc: d_pad must be a multiple of 64 >= d");
    SLIC_REQUIRE(k > 0 && k <= slic::TC_TOPK_MAX && k <= n - (self_offset >= 0 ? 1 : 0),
                 "topk_cosine_tc: k must satisfy 1 <= k <= min(64, columns available)");
    SLIC_REQUIRE(q_unit_dev && q_f16_dev && x_unit_dev && x_f16_dev && idx_out_dev, "topk_cosine_tc: null pointer");
    SLIC_REQUIRE(dtype == SLIC_F32 || dtype == SLIC_F64, "topk_cosine_tc: bad dtype");
    SLIC_REQUIRE((reinterpret_cast<uintptr_t>(q_f16_dev) & 15) == 0 && (reinterpret_cast<uintptr_t>(x_f16_dev) & 15) == 0,
                 "topk_cosine_tc: f16 matrices must be 16-byte aligned");
    if (nq == 0) return SLIC_OK;
    SLIC_PROPAGATE(slic_require_device());
    if (eps <= 0.f) eps = slic::screen_default_eps(d_pad);
    cudaStream_t st = slic::as_stream(stream);
    if (dtype == SLIC_F32)
        return slic::topk_tc_impl<float>((const float*)q_unit_dev, q_f16_dev, nq, (const float*)x_unit_dev, x_f16_dev,
                                         n, d, d_pad, k, self_offset, eps, idx_out_dev, (float*)dist_out_dev,
                                         stats_out_dev, st);
    return slic::topk_tc_impl<double>((const double*)q_unit_dev, q_f16_dev, nq, (const double*)x_unit_dev, x_f16_dev, n,
                                      d, d_pad, k, self_offset, eps, idx_out_dev, (double*)dist_out_dev, stats_out_dev,
                                      st);
}

int slic_profile_screen(int32_t enable) {
    slic::g_profile = enable != 0;
    slic::g_have_sample = false;
    return SLIC_OK;
}

int slic_screen_trace(int32_t enable, uint64_t* counters_out_host) {
    using namespace slic;
    if (counters_out_host && g_trace) {
        SLIC_CUDA_OK(cudaDeviceSynchronize());
        SLIC_CUDA_OK(cudaMemcpy(counters_out_host, g_trace, 12 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    }
    if (enable && !g_trace) {
        SLIC_CUDA_OK(cudaMalloc(&g_trace, 12 * sizeof(uint64_t)));
    } else if (!enable && g_trace) {
        SLIC_CUDA_OK(cudaDeviceSynchronize());
        SLIC_CUDA_OK(cudaFree(g_trace));
        g_trace = nullptr;
    }
    if (g_trace) SLIC_CUDA_OK(cudaMemset(g_trace, 0, 12 * sizeof(uint64_t)));
    return SLIC_OK;
}

int slic_last_screen_time(float* ms_out, double* flop_out) {
    SLIC_REQUIRE(ms_out && flop_out, "last_screen_time: null pointer");
    if (!slic::g_have_sample) {
        slic::set_error("last_screen_time: no profiled launch (call slic_profile_screen(1) first)");
        return SLIC_ERR_INVALID_ARG;
    }
    SLIC_CUDA_OK(cudaEventSynchronize(slic::g_ev_stop));
    SLIC_CUDA_OK(cudaEventElapsedTime(ms_out, slic::g_ev_start, slic::g_ev_stop));
    *flop_out = slic::g_last_flop;
    return SLIC_OK;
}

int slic_last_screen_exec_flop(double* flop_out) {
    SLIC_REQUIRE(flop_out, "last_screen_exec_flop: null pointer");
    *flop_out = slic::g_have_sample ? slic::g_last_exec_flop : 0.0;
    return SLIC_OK;
}

int slic_screen_scores_debug(const uint16_t* q_f16_dev, int64_t nq, const uint16_t* x_f16_dev, int64_t n,
                             int32_t d_pad, float* out_dev, slic_stream_t stream) {
    using namespace slic;
    SLIC_REQUIRE(nq > 0 && n > 0 && d_pad > 0 && d_pad % 64 == 0, "screen_scores_debug: bad shape");
    SLIC_REQUIRE(q_f16_dev && x_f16_dev && out_dev, "screen_scores_debug: null pointer");
    SLIC_PROPAGATE(slic_require_device());
    cudaStream_t st = as_stream(stream);
    const ScreenPlan pl = plan_screen(nq, n);
    const int64_t slots = (int64_t)pl.splits * 2 * nq;   // one list per (split, 128-column half of the tiles, row)
    Scratch ci, cs, cc, cf, err;
    SLIC_CUDA_OK(ci.alloc(slots * TC_CAP * sizeof(int), st));
    SLIC_CUDA_OK(cs.alloc(slots * TC_CAP * sizeof(float), st));
    SLIC_CUDA_OK(cc.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(cf.alloc(slots * sizeof(int), st));
    SLIC_CUDA_OK(err.alloc(sizeof(int), st));
    SLIC_CUDA_OK(cudaMemsetAsync(err.ptr, 0, sizeof(int), st));
    SLIC_PROPAGATE(launch_screen(q_f16_dev, nq, x_f16_dev, n, d_pad, -1, screen_default_eps(d_pad), TC_CAP, pl, ci.as<int>(),
                                 cs.as<float>(), cc.as<int>(), cf.as<int>(), out_dev, err.as<int>(), st));
    int host_err = 0;
    SLIC_CUDA_OK(cudaMemcpyAsync(&host_err, err.ptr, sizeof(int), cudaMemcpyDeviceToHost, st));
    SLIC_CUDA_OK(cudaStreamSynchronize(st));
    if (host_err) {
        set_error("nn_screen_kernel: pipeline barrier timed out");
        return SLIC_ERR_CUDA;
    }
    return SLIC_OK;
}

}  // extern "C"
