// Spherical k-means (spherecluster 0.1 SphericalKMeans.fit over scikit-learn 0.22 helpers; the method
// clustering/cluster_masks.py:38-98 selects with method='spherical_kmeans'), the whole fit on the device.
//
// One run of n_init:
//   seeding   k-means++ on the unit rows (_k_init): per step one pass over X evaluates all L candidates
//             (sk_pp_candidates_kernel: candidate distances, running minimum, per-block float64 potentials), a one-CTA
//             kernel adds the block potentials in a fixed order and picks the candidate, a third keeps the winner's
//             minimum and scans it (block-local inclusive float64 prefix + a one-CTA scan of the block totals); the
//             next step's searchsorted reads those two arrays.  HBM bound: N * D * 4 bytes per step.
//   Lloyd     assignment (tcgen05 screen + exact re-rank for k >= the screen threshold, the exact kernel below, a fill
//             for k = 1), a float64 epilogue for mindist and the inertia, slic_cluster_sums' float64 sums, empty-cluster
//             relocation (no-op when nothing is empty), float64 normalisation of the centres with their f16 copy, the
//             float64 shift and the best-so-far bookkeeping.  Every kernel after the assignment reads a device status
//             block and does nothing once the run has converged; the host enqueues SK_BATCH iterations and reads the
//             status once per batch.  The screen runs in its asynchronous mode: when it reports rows it could not
//             settle, the iteration is marked and skipped on the device, and the host repeats it through the
//             synchronous search (which finishes those rows with the exact kernel) before it resumes batching.
//   final     if the last shift was above zero, labels and inertia are recomputed against the best centres.
// Across runs the one with the smallest inertia (strict) is kept, on the device.
//
// Every floating-point reduction is float64 over a fixed partition (SK_ROWS rows per block, warps in order, block
// partials added in index order by one CTA): no atomics on floating-point results, bit-identical from run to run.
#include <cuda_fp16.h>
#include <math.h>
#include <math_constants.h>
#include <stdlib.h>

#include <initializer_list>
#include <utility>
#include <vector>

#include "common.cuh"

namespace slic {

constexpr int SK_THREADS = 256;
constexpr int SK_WARPS = SK_THREADS / 32;
constexpr int SK_ROWS = 256;   // rows per block of every row reduction (8 warps x 32 consecutive rows)
constexpr int SK_MAX_L = 32;   // k-means++ candidates per step: 2 + int(log(k)) <= 23 for any int32 k
constexpr int SK_BATCH = 4;    // Lloyd iterations enqueued per status read-back
constexpr int SK_RED = 1024;   // threads of the one-CTA reductions
// below this many centres the assignment runs on the exact kernel (a 256-column screen tile would be mostly padding)
constexpr int SK_SCREEN_MIN_K_DEFAULT = 256;

struct SkState {
    double tol_abs;            // mean(var(unit, axis=0)) * tol
    double pot;                // k-means++ potential of the current seed set
    double inertia;            // of the latest E-step
    double best_inertia;       // of this run
    double shift;              // of the latest update
    double fit_inertia;        // of the best run so far
    long long stats[4];        // candidates re-ranked, rows finished exactly, list compactions, screened assignments
    int best_l;                // winning candidate of the latest seed step
    int done;                  // this run has converged
    int dirty;                 // an asynchronous assignment left rows unsettled: the rest of the batch is skipped
    int dirty_iter;
    int n_iter;
    int improve;               // the latest iteration improved the inertia: copy labels and centres
    int redo;                  // the final E-step replaces the best labels (last shift > 0)
    int take;                  // this run is the best so far
    int fit_n_iter;
};

__device__ __forceinline__ bool sk_active(const SkState* s) { return !s->done && !s->dirty; }

// ---- one-CTA fixed-order float64 sum of v[0..m) (every thread receives the result) ----------------------------------
template <int THREADS>
__device__ double block_sum_fixed(const double* __restrict__ v, int64_t m) {
    __shared__ double red[THREADS];
    double a = 0.0;
    for (int64_t i = threadIdx.x; i < m; i += THREADS) a += v[i];
    red[threadIdx.x] = a;
    __syncthreads();
    for (int s = THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

// |x_i|^2 in float64 (one warp per row)
__global__ void __launch_bounds__(SK_THREADS) sk_sqnorm_kernel(const float* __restrict__ unit, int64_t n, int d,
                                                               double* __restrict__ sqnorm) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * SK_WARPS + (threadIdx.x >> 5);
    if (i >= n) return;
    const double s = warp_dot<float>(unit + i * d, unit + i * d, d, lane);
    if (lane == 0) sqnorm[i] = s;
}

// ---- tolerance: column sums and sums of squares over fixed row slabs, then one CTA ------------------------------------
__global__ void __launch_bounds__(256) sk_col_partial_kernel(const float* __restrict__ unit, int64_t n, int d,
                                                             double* __restrict__ part /* [slabs][d][2] */) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= d) return;
    const int64_t r0 = (int64_t)blockIdx.y * SK_ROWS, r1 = r0 + SK_ROWS < n ? r0 + SK_ROWS : n;
    double s = 0.0, q = 0.0;
    for (int64_t r = r0; r < r1; ++r) {
        const double v = unit[r * d + col];
        s += v;
        q = fma(v, v, q);
    }
    part[((int64_t)blockIdx.y * d + col) * 2] = s;
    part[((int64_t)blockIdx.y * d + col) * 2 + 1] = q;
}

__global__ void __launch_bounds__(SK_RED) sk_tol_kernel(const double* __restrict__ part, int64_t slabs, int64_t n, int d,
                                                        double tol, SkState* st) {
    __shared__ double red[SK_RED];
    double acc = 0.0;
    for (int col = threadIdx.x; col < d; col += SK_RED) {
        double s = 0.0, q = 0.0;
        for (int64_t b = 0; b < slabs; ++b) {
            s += part[(b * d + col) * 2];
            q += part[(b * d + col) * 2 + 1];
        }
        const double mean = s / (double)n;
        const double var = q / (double)n - mean * mean;
        acc += var > 0.0 ? var : 0.0;
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = SK_RED / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) st->tol_abs = red[0] / (double)d * tol;
}

__global__ void sk_fit_init_kernel(SkState* st) {
    st->fit_inertia = CUDART_INF;
    st->fit_n_iter = 0;
    for (int j = 0; j < 4; ++j) st->stats[j] = 0;
}

__global__ void sk_run_init_kernel(SkState* st) {
    st->best_inertia = CUDART_INF;
    st->shift = 0.0;
    st->done = 0;
    st->dirty = 0;
    st->dirty_iter = -1;
    st->n_iter = 0;
    st->improve = 0;
    st->redo = 0;
    st->take = 0;
}

// ---- k-means++ ----------------------------------------------------------------------------------------------------
// ids[l] = clip(searchsorted(cumsum(closest), u[l] * pot, 'left'), n - 1).  The inclusive prefix of row i is
// boff[i / SK_ROWS] + local[i]: non-decreasing in i, because the last local value of a block is its total.
// first >= 0: the first seed, ids[0] = first.
__global__ void sk_pp_draw_kernel(const double* __restrict__ local, const double* __restrict__ boff, int64_t n,
                                  const double* __restrict__ u, int L, const SkState* st, int first, int* __restrict__ ids) {
    const int l = threadIdx.x;
    if (l >= L) return;
    if (first >= 0) {
        ids[l] = first;
        return;
    }
    const double val = u[l] * st->pot;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const double v = boff[mid / SK_ROWS] + local[mid];
        if (v < val) lo = mid + 1;
        else hi = mid;
    }
    ids[l] = (int)(lo < n ? lo : n - 1);
}

// One pass over X for all L candidates: m_l[i] = min(closest[i], sqdist(X[ids[l]], X[i])) with sqdist = max(|a|^2 + |b|^2
// - 2 a.b, 0) in float64 rounded to float32; cand[l][i] = m_l[i], part[l][block] = float64 sum of the block's m_l.
// closest == nullptr: the first seed (no running minimum yet).
template <int LMAX>
__global__ void __launch_bounds__(SK_THREADS) sk_pp_candidates_kernel(const float* __restrict__ unit,
                                                                      const double* __restrict__ sqnorm, int64_t n, int d,
                                                                      const int* __restrict__ ids, int L,
                                                                      const float* __restrict__ closest,
                                                                      float* __restrict__ cand, double* __restrict__ part,
                                                                      int64_t nb) {
    __shared__ double s_pot[SK_WARPS][LMAX];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* crow[LMAX];
    double cn[LMAX], pot[LMAX];
#pragma unroll
    for (int l = 0; l < LMAX; ++l) {
        const int id = l < L ? ids[l] : ids[0];
        crow[l] = unit + (int64_t)id * d;
        cn[l] = sqnorm[id];
        pot[l] = 0.0;
    }
    const int64_t r0 = (int64_t)blockIdx.x * SK_ROWS + warp * 32;
    for (int j = 0; j < 32; ++j) {
        const int64_t i = r0 + j;
        if (i >= n) break;
        const float* xr = unit + i * d;
        double acc[LMAX];
#pragma unroll
        for (int l = 0; l < LMAX; ++l) acc[l] = 0.0;
        for (int k = lane; k < d; k += 32) {
            const double x = (double)xr[k];
#pragma unroll
            for (int l = 0; l < LMAX; ++l)
                if (l < L) acc[l] = fma(x, (double)__ldg(crow[l] + k), acc[l]);
        }
        const double xn = sqnorm[i];
        const float cl = closest ? closest[i] : CUDART_INF_F;
#pragma unroll
        for (int l = 0; l < LMAX; ++l) {
            if (l < L) {
                const double s = warp_sum(acc[l]);
                double q = (cn[l] + xn) - 2.0 * s;
                if (q < 0.0) q = 0.0;
                const float m = fminf(cl, (float)q);
                if (lane == 0) cand[(int64_t)l * n + i] = m;
                pot[l] += (double)m;
            }
        }
    }
    if (lane == 0)
#pragma unroll
        for (int l = 0; l < LMAX; ++l) s_pot[warp][l] = pot[l];
    __syncthreads();
    if ((int)threadIdx.x < L) {
        double a = 0.0;
        for (int w = 0; w < SK_WARPS; ++w) a += s_pot[w][threadIdx.x];
        part[(int64_t)threadIdx.x * nb + blockIdx.x] = a;
    }
}

// pot_l = fixed-order sum of the block potentials; the smallest wins (ties: first candidate), seeds[c] = its row
__global__ void __launch_bounds__(SK_RED) sk_pp_pick_kernel(const double* __restrict__ part, int64_t nb, int L,
                                                            const int* __restrict__ ids, SkState* st, int* __restrict__ seeds,
                                                            int c) {
    __shared__ double pots[SK_MAX_L];
    for (int l = 0; l < L; ++l) {
        const double p = block_sum_fixed<SK_RED>(part + (int64_t)l * nb, nb);
        if (threadIdx.x == 0) pots[l] = p;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int best = 0;
        for (int l = 1; l < L; ++l)
            if (pots[l] < pots[best]) best = l;
        st->best_l = best;
        st->pot = pots[best];
        seeds[c] = ids[best];
    }
}

// closest = m_best; local = block-local inclusive float64 prefix of it, bsum[block] = its last value
__global__ void __launch_bounds__(SK_ROWS) sk_pp_commit_kernel(const float* __restrict__ cand, int64_t n, const SkState* st,
                                                               float* __restrict__ closest, double* __restrict__ local,
                                                               double* __restrict__ bsum) {
    __shared__ double s_warp[SK_ROWS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * SK_ROWS + threadIdx.x;
    float m = 0.f;
    if (i < n) {
        m = cand[(int64_t)st->best_l * n + i];
        closest[i] = m;
    }
    double v = (double)m;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = 0.0;
        for (int w = 0; w < SK_ROWS / 32; ++w) {
            const double t = s_warp[w];
            s_warp[w] = run;
            run += t;
        }
    }
    __syncthreads();
    v += s_warp[warp];
    if (i < n) local[i] = v;
    if (threadIdx.x == SK_ROWS - 1) bsum[blockIdx.x] = v;
}

// exclusive prefix of the block totals (contiguous chunks per thread, chunk totals scanned by one thread)
__global__ void __launch_bounds__(SK_RED) sk_scan_blocks_kernel(const double* __restrict__ bsum, int64_t nb,
                                                                double* __restrict__ boff) {
    __shared__ double s[SK_RED];
    const int64_t chunk = (nb + SK_RED - 1) / SK_RED;
    const int64_t b0 = threadIdx.x * chunk, b1 = b0 + chunk < nb ? b0 + chunk : nb;
    double a = 0.0;
    for (int64_t b = b0; b < b1; ++b) a += bsum[b];
    s[threadIdx.x] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = 0.0;
        for (int t = 0; t < SK_RED; ++t) {
            const double x = s[t];
            s[t] = run;
            run += x;
        }
    }
    __syncthreads();
    double run = s[threadIdx.x];
    for (int64_t b = b0; b < b1; ++b) {
        boff[b] = run;
        run += bsum[b];
    }
}

// centres = X[seeds] (no renormalisation), their f16 copy and |c|^2 (one warp per centre)
__global__ void __launch_bounds__(SK_THREADS) sk_gather_kernel(const float* __restrict__ unit, const int* __restrict__ seeds,
                                                               int k, int d, int d_pad, float* __restrict__ centres,
                                                               __half* __restrict__ f16, double* __restrict__ cnorm2) {
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * SK_WARPS + (threadIdx.x >> 5);
    if (c >= k) return;
    const float* src = unit + (int64_t)seeds[c] * d;
    double cn = 0.0;
    for (int j = lane; j < d_pad; j += 32) {
        float v = 0.f;
        if (j < d) {
            v = src[j];
            centres[(int64_t)c * d + j] = v;
            cn = fma((double)v, (double)v, cn);
        }
        f16[(int64_t)c * d_pad + j] = __float2half_rn(v);
    }
    cn = warp_sum(cn);
    if (lane == 0) cnorm2[c] = cn;
}

// ---- Lloyd ---------------------------------------------------------------------------------------------------------
__global__ void sk_fill_kernel(int* __restrict__ labels, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) labels[i] = 0;
}

// an asynchronous screen leaves -1 for a row without candidates (such an iteration is dirty and repeated): keep every
// label a valid cluster id so that the grouping enqueued behind it stays in bounds
__global__ void sk_clamp_labels_kernel(int* __restrict__ labels, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && labels[i] < 0) labels[i] = 0;
}

// after the screen: asynchronous mode - rows left unsettled or a pipeline error make the iteration dirty (skipped here,
// repeated by the host through the synchronous search); otherwise (and always in synchronous mode) count the statistics
__global__ void sk_check_kernel(const int* __restrict__ stats, int async_mode, int force, int iter, SkState* st) {
    if (!force && !sk_active(st)) return;
    if (async_mode && (stats[1] != 0 || stats[4] != 0)) {
        st->dirty = 1;
        st->dirty_iter = iter;
        return;
    }
    st->stats[0] += stats[0];
    st->stats[1] += stats[1];
    st->stats[2] += stats[2];
    st->stats[3] += 1;
}

// mindist_i = |x_i|^2 + |c|^2 - 2 x_i.c in float64, rounded to float32; part[block] = float64 sum of the block's mindist
__global__ void __launch_bounds__(SK_THREADS) sk_estep_kernel(const float* __restrict__ unit, const double* __restrict__ sqnorm,
                                                              int64_t n, int d, const float* __restrict__ centres,
                                                              const double* __restrict__ cnorm2,
                                                              const int* __restrict__ labels, const SkState* st, int force,
                                                              float* __restrict__ mindist, double* __restrict__ part) {
    if (!force && !sk_active(st)) return;
    __shared__ double s_w[SK_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * SK_ROWS + warp * 32;
    double acc = 0.0;
    for (int j = 0; j < 32; ++j) {
        const int64_t i = r0 + j;
        if (i >= n) break;
        const int c = labels[i];
        const double s = warp_dot<float>(unit + i * d, centres + (int64_t)c * d, d, lane);
        const float m = (float)((sqnorm[i] + cnorm2[c]) - 2.0 * s);
        if (lane == 0) mindist[i] = m;
        acc += (double)m;
    }
    if (lane == 0) s_w[warp] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0;
        for (int w = 0; w < SK_WARPS; ++w) a += s_w[w];
        part[blockIdx.x] = a;
    }
}

// order-preserving key of a float (larger float -> larger key)
__device__ __forceinline__ unsigned int float_order_key(float f) {
    const unsigned int b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// inertia, then _centers_dense's relocation: the i-th empty cluster (ascending id) takes the i-th farthest row (mindist
// descending, ties: higher row first) as its sum with count 1.  E rounds of a block-wide arg-max below the previous key.
__global__ void __launch_bounds__(SK_RED) sk_update_kernel(const double* __restrict__ part, int64_t nb,
                                                           const float* __restrict__ mindist, int64_t n,
                                                           const float* __restrict__ unit, int d, double* __restrict__ sums,
                                                           int* __restrict__ counts, int k, SkState* st) {
    __shared__ int s_active, s_empty, s_c;
    __shared__ unsigned long long s_key[SK_RED / 32];
    if (threadIdx.x == 0) {
        s_active = sk_active(st);
        s_empty = 0;
    }
    __syncthreads();
    if (!s_active) return;
    const double inertia = block_sum_fixed<SK_RED>(part, nb);
    if (threadIdx.x == 0) st->inertia = inertia;
    int e = 0;
    for (int c = threadIdx.x; c < k; c += SK_RED) e += counts[c] == 0;
    if (e) atomicAdd(&s_empty, e);
    __syncthreads();
    const int empties = s_empty;
    if (empties == 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long prev = ~0ull;
    int next_c = 0;
    for (int r = 0; r < empties; ++r) {
        unsigned long long best = 0ull;
        for (int64_t i = threadIdx.x; i < n; i += SK_RED) {
            const unsigned long long key = ((unsigned long long)float_order_key(mindist[i]) << 32) | (unsigned long long)i;
            if (key < prev && key > best) best = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o);
            best = t > best ? t : best;
        }
        if (lane == 0) s_key[warp] = best;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long b = 0ull;
            for (int w = 0; w < SK_RED / 32; ++w) b = s_key[w] > b ? s_key[w] : b;
            s_key[0] = b;
            while (counts[next_c] != 0) ++next_c;
            s_c = next_c;
            counts[next_c] = 1;
        }
        __syncthreads();
        prev = s_key[0];
        const int64_t row = (int64_t)(prev & 0xffffffffull);
        const int c = s_c;
        for (int j = threadIdx.x; j < d; j += SK_RED) sums[(int64_t)c * d + j] = (double)unit[row * d + j];
        __syncthreads();
    }
}

// centres = normalize(sums / counts) in float64, rounded to float32, with their f16 copy, |c|^2 and the per-centre shift
// sum((old - new)^2) in float64.  S = float: explicit init rows (counts == nullptr).  One warp per centre.
template <typename S>
__global__ void __launch_bounds__(SK_THREADS) sk_normalize_kernel(const S* __restrict__ sums, const int* __restrict__ counts,
                                                                  int k, int d, int d_pad, const SkState* st, int force,
                                                                  const float* __restrict__ old, float* __restrict__ centres,
                                                                  __half* __restrict__ f16, double* __restrict__ cnorm2,
                                                                  double* __restrict__ shift_part) {
    if (!force && !sk_active(st)) return;
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * SK_WARPS + (threadIdx.x >> 5);
    if (c >= k) return;
    const double cnt = counts ? (double)counts[c] : 1.0;
    const S* src = sums + (int64_t)c * d;
    double nrm2 = 0.0;
    for (int j = lane; j < d; j += 32) {
        const double m = (double)src[j] / cnt;
        nrm2 = fma(m, m, nrm2);
    }
    double nrm = sqrt(warp_sum(nrm2));
    if (nrm == 0.0) nrm = 1.0;
    double cn = 0.0, sh = 0.0;
    for (int j = lane; j < d_pad; j += 32) {
        float v = 0.f;
        if (j < d) {
            v = (float)(((double)src[j] / cnt) / nrm);
            centres[(int64_t)c * d + j] = v;
            cn = fma((double)v, (double)v, cn);
            if (old) {
                const double df = (double)old[(int64_t)c * d + j] - (double)v;
                sh = fma(df, df, sh);
            }
        }
        f16[(int64_t)c * d_pad + j] = __float2half_rn(v);
    }
    cn = warp_sum(cn);
    sh = warp_sum(sh);
    if (lane == 0) {
        cnorm2[c] = cn;
        if (shift_part) shift_part[c] = sh;
    }
}

// shift, best-so-far decision (strict), convergence; n_iter = iter + 1
__global__ void __launch_bounds__(SK_RED) sk_iter_end_kernel(const double* __restrict__ shift_part, int k, SkState* st,
                                                             int iter) {
    __shared__ int s_active;
    if (threadIdx.x == 0) s_active = sk_active(st);
    __syncthreads();
    if (!s_active) {
        if (threadIdx.x == 0) st->improve = 0;
        return;
    }
    const double shift = block_sum_fixed<SK_RED>(shift_part, k);
    if (threadIdx.x == 0) {
        st->shift = shift;
        const int imp = st->inertia < st->best_inertia;
        if (imp) st->best_inertia = st->inertia;
        st->improve = imp;
        st->n_iter = iter + 1;
        if (shift <= st->tol_abs) st->done = 1;
    }
}

// after the final E-step: redo = (last shift > 0) replaces the best labels and inertia; then the run-level comparison
__global__ void __launch_bounds__(SK_RED) sk_run_end_kernel(const double* __restrict__ part, int64_t nb, SkState* st) {
    const double inertia = block_sum_fixed<SK_RED>(part, nb);
    if (threadIdx.x == 0) {
        st->redo = st->shift > 0.0;
        if (st->redo) st->best_inertia = inertia;
        st->take = st->best_inertia < st->fit_inertia;
        if (st->take) {
            st->fit_inertia = st->best_inertia;
            st->fit_n_iter = st->n_iter;
        }
    }
}

struct CopySegs {
    const unsigned int* src[4];
    unsigned int* dst[4];
    int64_t words[4];
};
// copies the segments iff *flag != 0 (a flag set on the device by the kernel before)
__global__ void sk_cond_copy_kernel(const int* flag, CopySegs s) {
    if (!*flag) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int g = 0; g < 4; ++g)
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < s.words[g]; i += stride) s.dst[g][i] = s.src[g][i];
}

// ---- host side -------------------------------------------------------------------------------------------------------
static int screen_min_k() {
    const char* e = getenv("SLIC_SKMEANS_SCREEN_MIN_K");   // measurement switch (DESIGN section 8)
    if (e && atoi(e) >= 2) return atoi(e);
    return SK_SCREEN_MIN_K_DEFAULT;
}

static unsigned blocks_for(int64_t items, int per_block) { return (unsigned)ceil_div(items > 0 ? items : 1, per_block); }

struct SkWork {
    int64_t n = 0, nb = 0;
    int d = 0, d_pad = 0, k = 0, L = 0;
    const float* unit = nullptr;
    const uint16_t* unit_f16 = nullptr;
    Scratch sqnorm, state;
    // seeding
    Scratch ids, closest, cand, ppart, local, bsum, boff, u;
    // Lloyd
    Scratch labels, best_labels, mindist, epart, dist_tmp, sums, counts, shift_part, stats;
    Scratch cen[2], f16[2], cn2[2], best_cen, best_f16, best_cn2, seeds;
    SkState* st() const { return state.as<SkState>(); }
};

static int sk_alloc_common(SkWork& w, const float* unit, int64_t n, int d, int k, int L, cudaStream_t s) {
    w.unit = unit;
    w.n = n;
    w.d = d;
    w.k = k;
    w.L = L;
    w.d_pad = (d + 63) / 64 * 64;
    w.nb = ceil_div(n, SK_ROWS);
    SLIC_CUDA_OK(w.sqnorm.alloc(n * sizeof(double), s));
    SLIC_CUDA_OK(w.state.alloc(sizeof(SkState), s));
    SLIC_CUDA_OK(cudaMemsetAsync(w.state.ptr, 0, sizeof(SkState), s));
    SLIC_CUDA_OK(w.seeds.alloc((size_t)k * sizeof(int), s));
    sk_sqnorm_kernel<<<blocks_for(n, SK_WARPS), SK_THREADS, 0, s>>>(unit, n, d, w.sqnorm.as<double>());
    SLIC_LAUNCH_OK();
    if (L > 0) {   // k-means++ buffers
        const int lc = L > 1 ? L : 1;
        SLIC_CUDA_OK(w.ids.alloc(SK_MAX_L * sizeof(int), s));
        SLIC_CUDA_OK(w.closest.alloc(n * sizeof(float), s));
        SLIC_CUDA_OK(w.cand.alloc((size_t)lc * n * sizeof(float), s));
        SLIC_CUDA_OK(w.ppart.alloc((size_t)lc * w.nb * sizeof(double), s));
        SLIC_CUDA_OK(w.local.alloc(n * sizeof(double), s));
        SLIC_CUDA_OK(w.bsum.alloc(w.nb * sizeof(double), s));
        SLIC_CUDA_OK(w.boff.alloc(w.nb * sizeof(double), s));
    }
    return SLIC_OK;
}

static int launch_candidates(SkWork& w, int L, bool first, cudaStream_t s) {
    const unsigned grid = (unsigned)w.nb;
    const float* closest = first ? nullptr : w.closest.as<float>();
#define SK_CAND(LM)                                                                                                   \
    sk_pp_candidates_kernel<LM><<<grid, SK_THREADS, 0, s>>>(w.unit, w.sqnorm.as<double>(), w.n, w.d, w.ids.as<int>(), L, \
                                                             closest, w.cand.as<float>(), w.ppart.as<double>(), w.nb)
    if (L <= 8) SK_CAND(8);
    else if (L <= 16) SK_CAND(16);
    else SK_CAND(32);
#undef SK_CAND
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

// k-means++ of _k_init on the unit rows; u_dev [(k - 1) * L] uniforms of this run; seeds -> w.seeds
static int sk_seed(SkWork& w, int first, const double* u_dev, cudaStream_t s) {
    const int k = w.k, L = w.L;
    for (int c = 0; c < k; ++c) {
        const int lc = c == 0 ? 1 : L;
        sk_pp_draw_kernel<<<1, 32, 0, s>>>(w.local.as<double>(), w.boff.as<double>(), w.n,
                                           c == 0 ? nullptr : u_dev + (int64_t)(c - 1) * L, lc, w.st(), c == 0 ? first : -1,
                                           w.ids.as<int>());
        SLIC_LAUNCH_OK();
        SLIC_PROPAGATE(launch_candidates(w, lc, c == 0, s));
        sk_pp_pick_kernel<<<1, SK_RED, 0, s>>>(w.ppart.as<double>(), w.nb, lc, w.ids.as<int>(), w.st(), w.seeds.as<int>(), c);
        SLIC_LAUNCH_OK();
        if (c + 1 < k) {
            sk_pp_commit_kernel<<<(unsigned)w.nb, SK_ROWS, 0, s>>>(w.cand.as<float>(), w.n, w.st(), w.closest.as<float>(),
                                                                   w.local.as<double>(), w.bsum.as<double>());
            SLIC_LAUNCH_OK();
            sk_scan_blocks_kernel<<<1, SK_RED, 0, s>>>(w.bsum.as<double>(), w.nb, w.boff.as<double>());
            SLIC_LAUNCH_OK();
        }
    }
    return SLIC_OK;
}

// labels of every row against centres cen/f16 (asynchronous screen: dirty marking; synchronous: exact finisher)
static int sk_assign(SkWork& w, const float* cen, const uint16_t* f16, bool sync, int force, int iter, cudaStream_t s) {
    int* labels = w.labels.as<int>();
    if (w.k == 1) {
        sk_fill_kernel<<<blocks_for(w.n, 256), 256, 0, s>>>(labels, w.n);
        SLIC_LAUNCH_OK();
        return SLIC_OK;
    }
    if (w.k < screen_min_k())
        return slic_nn_exact_top1(w.unit, nullptr, w.n, cen, w.k, w.d, SLIC_F32, -1, labels, w.dist_tmp.ptr, s);
    int* stats = w.stats.as<int>();
    if (sync) {
        SLIC_CUDA_OK(cudaMemsetAsync(stats, 0, 8 * sizeof(int), s));
        SLIC_PROPAGATE(nn_top1_f32_gated(w.unit, w.unit_f16, w.n, cen, f16, w.k, w.d, w.d_pad, -1, 0.f, labels,
                                         w.dist_tmp.as<float>(), stats, nullptr, nullptr, nullptr, s));
    } else {
        SLIC_PROPAGATE(nn_top1_f32_gated(w.unit, w.unit_f16, w.n, cen, f16, w.k, w.d, w.d_pad, -1, 0.f, labels,
                                         w.dist_tmp.as<float>(), nullptr, nullptr, nullptr, nullptr, s, stats));
        sk_clamp_labels_kernel<<<blocks_for(w.n, 256), 256, 0, s>>>(labels, w.n);
        SLIC_LAUNCH_OK();
    }
    sk_check_kernel<<<1, 1, 0, s>>>(stats, sync ? 0 : 1, force, iter, w.st());
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

static int sk_estep(SkWork& w, const float* cen, const double* cn2, int force, cudaStream_t s) {
    sk_estep_kernel<<<(unsigned)w.nb, SK_THREADS, 0, s>>>(w.unit, w.sqnorm.as<double>(), w.n, w.d, cen, cn2,
                                                          w.labels.as<int>(), w.st(), force, w.mindist.as<float>(),
                                                          w.epart.as<double>());
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

static int sk_cond_copy(const int* flag, std::initializer_list<std::pair<const void*, std::pair<void*, size_t>>> segs,
                        cudaStream_t s) {
    CopySegs cs = {};
    int g = 0;
    for (const auto& e : segs) {
        cs.src[g] = static_cast<const unsigned int*>(e.first);
        cs.dst[g] = static_cast<unsigned int*>(e.second.first);
        cs.words[g] = (int64_t)(e.second.second / 4);
        ++g;
    }
    sk_cond_copy_kernel<<<(unsigned)num_sms() * 2, 256, 0, s>>>(flag, cs);
    SLIC_LAUNCH_OK();
    return SLIC_OK;
}

// one Lloyd iteration; centres cen[it % 2] -> cen[(it + 1) % 2]
static int sk_iteration(SkWork& w, int it, bool sync_assign, cudaStream_t s) {
    const int a = it & 1, b = a ^ 1;
    const int k = w.k, d = w.d;
    SLIC_PROPAGATE(sk_assign(w, w.cen[a].as<float>(), w.f16[a].as<uint16_t>(), sync_assign, 0, it, s));
    SLIC_PROPAGATE(sk_estep(w, w.cen[a].as<float>(), w.cn2[a].as<double>(), 0, s));
    SLIC_PROPAGATE(slic_cluster_sums(w.unit, w.labels.as<int>(), w.n, d, k, w.sums.as<double>(), w.counts.as<int>(),
                                     nullptr, s));
    sk_update_kernel<<<1, SK_RED, 0, s>>>(w.epart.as<double>(), w.nb, w.mindist.as<float>(), w.n, w.unit, d,
                                          w.sums.as<double>(), w.counts.as<int>(), k, w.st());
    SLIC_LAUNCH_OK();
    sk_normalize_kernel<double><<<blocks_for(k, SK_WARPS), SK_THREADS, 0, s>>>(
        w.sums.as<double>(), w.counts.as<int>(), k, d, w.d_pad, w.st(), 0, w.cen[a].as<float>(), w.cen[b].as<float>(),
        w.f16[b].as<__half>(), w.cn2[b].as<double>(), w.shift_part.as<double>());
    SLIC_LAUNCH_OK();
    sk_iter_end_kernel<<<1, SK_RED, 0, s>>>(w.shift_part.as<double>(), k, w.st(), it);
    SLIC_LAUNCH_OK();
    return sk_cond_copy(&w.st()->improve,
                        {{w.labels.ptr, {w.best_labels.ptr, (size_t)w.n * 4}},
                         {w.cen[b].ptr, {w.best_cen.ptr, (size_t)k * d * 4}},
                         {w.f16[b].ptr, {w.best_f16.ptr, (size_t)k * w.d_pad * 2}},
                         {w.cn2[b].ptr, {w.best_cn2.ptr, (size_t)k * 8}}},
                        s);
}

static int sk_read_state(const SkWork& w, SkState* h, cudaStream_t s) {
    SLIC_CUDA_OK(cudaMemcpyAsync(h, w.state.ptr, sizeof(SkState), cudaMemcpyDeviceToHost, s));
    SLIC_CUDA_OK(cudaStreamSynchronize(s));
    return SLIC_OK;
}

static int sk_fit(const float* x, int64_t n, int d, int k, const float* init, const int* first_ids, const double* uniforms,
                  int L, int n_init, int max_iter, double tol, int* labels_out, float* centers_out, double* inertia_out,
                  int* n_iter_out, int64_t* stats_out, cudaStream_t s) {
    SkWork w;
    // unit rows (sklearn normalize) and their f16 copy for the screen
    Scratch unit, unit_f16;
    const int d_pad = (d + 63) / 64 * 64;
    const bool screen = k >= 2 && k >= screen_min_k();
    SLIC_CUDA_OK(unit.alloc((size_t)n * d * sizeof(float), s));
    if (screen) SLIC_CUDA_OK(unit_f16.alloc((size_t)n * d_pad * sizeof(uint16_t), s));
    SLIC_PROPAGATE(slic_normalize_rows(x, n, d, SLIC_F32, unit.ptr, nullptr, screen ? unit_f16.as<uint16_t>() : nullptr,
                                       d_pad, s));
    SLIC_PROPAGATE(sk_alloc_common(w, unit.as<float>(), n, d, k, init ? 0 : L, s));
    w.unit_f16 = unit_f16.as<uint16_t>();
    SLIC_CUDA_OK(w.labels.alloc(n * sizeof(int), s));
    SLIC_CUDA_OK(w.best_labels.alloc(n * sizeof(int), s));
    SLIC_CUDA_OK(w.mindist.alloc(n * sizeof(float), s));
    SLIC_CUDA_OK(w.epart.alloc(w.nb * sizeof(double), s));
    SLIC_CUDA_OK(w.dist_tmp.alloc(n * sizeof(float), s));
    SLIC_CUDA_OK(w.sums.alloc((size_t)k * d * sizeof(double), s));
    SLIC_CUDA_OK(w.counts.alloc((size_t)k * sizeof(int), s));
    SLIC_CUDA_OK(w.shift_part.alloc((size_t)k * sizeof(double), s));
    SLIC_CUDA_OK(w.stats.alloc(8 * sizeof(int), s));
    for (int i = 0; i < 2; ++i) {
        SLIC_CUDA_OK(w.cen[i].alloc((size_t)k * d * sizeof(float), s));
        SLIC_CUDA_OK(w.f16[i].alloc((size_t)k * d_pad * sizeof(uint16_t), s));
        SLIC_CUDA_OK(w.cn2[i].alloc((size_t)k * sizeof(double), s));
    }
    SLIC_CUDA_OK(w.best_cen.alloc((size_t)k * d * sizeof(float), s));
    SLIC_CUDA_OK(w.best_f16.alloc((size_t)k * d_pad * sizeof(uint16_t), s));
    SLIC_CUDA_OK(w.best_cn2.alloc((size_t)k * sizeof(double), s));
    const int64_t per_run = (int64_t)(k - 1) * L;
    if (!init && per_run > 0) {
        SLIC_CUDA_OK(w.u.alloc((size_t)n_init * per_run * sizeof(double), s));
        SLIC_CUDA_OK(cudaMemcpyAsync(w.u.ptr, uniforms, (size_t)n_init * per_run * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    {   // tolerance on the unit rows
        Scratch cpart;
        SLIC_CUDA_OK(cpart.alloc((size_t)w.nb * d * 2 * sizeof(double), s));
        sk_col_partial_kernel<<<dim3(blocks_for(d, 256), (unsigned)w.nb), 256, 0, s>>>(w.unit, n, d, cpart.as<double>());
        SLIC_LAUNCH_OK();
        sk_tol_kernel<<<1, SK_RED, 0, s>>>(cpart.as<double>(), w.nb, n, d, tol, w.st());
        SLIC_LAUNCH_OK();
    }
    sk_fit_init_kernel<<<1, 1, 0, s>>>(w.st());
    SLIC_LAUNCH_OK();
    SkState h;
    for (int run = 0; run < n_init; ++run) {
        sk_run_init_kernel<<<1, 1, 0, s>>>(w.st());
        SLIC_LAUNCH_OK();
        if (init) {
            sk_normalize_kernel<float><<<blocks_for(k, SK_WARPS), SK_THREADS, 0, s>>>(
                init, nullptr, k, d, d_pad, w.st(), 1, nullptr, w.cen[0].as<float>(), w.f16[0].as<__half>(),
                w.cn2[0].as<double>(), nullptr);
            SLIC_LAUNCH_OK();
        } else {
            SLIC_PROPAGATE(sk_seed(w, first_ids[run], per_run > 0 ? w.u.as<double>() + run * per_run : nullptr, s));
            sk_gather_kernel<<<blocks_for(k, SK_WARPS), SK_THREADS, 0, s>>>(w.unit, w.seeds.as<int>(), k, d, d_pad,
                                                                            w.cen[0].as<float>(), w.f16[0].as<__half>(),
                                                                            w.cn2[0].as<double>());
            SLIC_LAUNCH_OK();
        }
        int it = 0;
        while (it < max_iter) {
            const int batch = max_iter - it < SK_BATCH ? max_iter - it : SK_BATCH;
            for (int j = 0; j < batch; ++j) SLIC_PROPAGATE(sk_iteration(w, it + j, false, s));
            SLIC_PROPAGATE(sk_read_state(w, &h, s));
            if (h.dirty) {   // repeat that iteration with the synchronous search, then resume after it
                const int j = h.dirty_iter;
                SLIC_CUDA_OK(cudaMemsetAsync(&w.st()->dirty, 0, sizeof(int), s));
                SLIC_PROPAGATE(sk_iteration(w, j, true, s));
                it = j + 1;
                SLIC_PROPAGATE(sk_read_state(w, &h, s));
            } else {
                it += batch;
            }
            if (h.done) break;
        }
        // final E-step against the best centres (its labels and inertia replace the best ones iff the last shift > 0)
        SLIC_PROPAGATE(sk_assign(w, w.best_cen.as<float>(), w.best_f16.as<uint16_t>(), true, 1, -1, s));
        SLIC_PROPAGATE(sk_estep(w, w.best_cen.as<float>(), w.best_cn2.as<double>(), 1, s));
        sk_run_end_kernel<<<1, SK_RED, 0, s>>>(w.epart.as<double>(), w.nb, w.st());
        SLIC_LAUNCH_OK();
        SLIC_PROPAGATE(sk_cond_copy(&w.st()->redo, {{w.labels.ptr, {w.best_labels.ptr, (size_t)n * 4}}}, s));
        SLIC_PROPAGATE(sk_cond_copy(&w.st()->take,
                                    {{w.best_labels.ptr, {labels_out, (size_t)n * 4}},
                                     {w.best_cen.ptr, {centers_out, (size_t)k * d * 4}}},
                                    s));
    }
    SLIC_PROPAGATE(sk_read_state(w, &h, s));
    *inertia_out = h.fit_inertia;
    *n_iter_out = h.fit_n_iter;
    if (stats_out)
        for (int j = 0; j < 4; ++j) stats_out[j] = h.stats[j];
    return SLIC_OK;
}

}  // namespace slic

extern "C" int slic_kmeans_plusplus(const float* unit_dev, int64_t n, int32_t d, int32_t k, int64_t first_id,
                                    const double* uniforms_host, int32_t L, int32_t* seeds_out_dev, slic_stream_t stream) {
    using namespace slic;
    SLIC_REQUIRE(n >= 1 && n < ((int64_t)1 << 31) && d > 0, "kmeans_plusplus: bad shape");
    SLIC_REQUIRE(k >= 1 && k <= n, "kmeans_plusplus: need 1 <= k <= n");
    SLIC_REQUIRE(L >= 1 && L <= SK_MAX_L, "kmeans_plusplus: need 1 <= L <= 32 candidates per step");
    SLIC_REQUIRE(first_id >= 0 && first_id < n, "kmeans_plusplus: first_id must be a row index");
    SLIC_REQUIRE(unit_dev && seeds_out_dev && (k == 1 || uniforms_host), "kmeans_plusplus: null pointer");
    SLIC_PROPAGATE(slic_require_device());
    cudaStream_t s = as_stream(stream);
    SkWork w;
    SLIC_PROPAGATE(sk_alloc_common(w, unit_dev, n, d, k, L, s));
    if (k > 1) {
        SLIC_CUDA_OK(w.u.alloc((size_t)(k - 1) * L * sizeof(double), s));
        SLIC_CUDA_OK(cudaMemcpyAsync(w.u.ptr, uniforms_host, (size_t)(k - 1) * L * sizeof(double), cudaMemcpyHostToDevice, s));
    }
    SLIC_PROPAGATE(sk_seed(w, (int)first_id, w.u.as<double>(), s));
    SLIC_CUDA_OK(cudaMemcpyAsync(seeds_out_dev, w.seeds.ptr, (size_t)k * sizeof(int), cudaMemcpyDeviceToDevice, s));
    return SLIC_OK;
}

extern "C" int slic_spherical_kmeans(const float* x_dev, int64_t n, int32_t d, int32_t k, const float* init_dev,
                                     const int64_t* first_ids_host, const double* uniforms_host, int32_t L, int32_t n_init,
                                     int32_t max_iter, double tol, int32_t* labels_out_dev, float* centers_out_dev,
                                     double* inertia_out_host, int32_t* n_iter_out_host, int64_t* stats_out_host,
                                     slic_stream_t stream) {
    using namespace slic;
    SLIC_REQUIRE(n >= 1 && n < ((int64_t)1 << 31) && d > 0, "spherical_kmeans: bad shape");
    SLIC_REQUIRE(k >= 1, "spherical_kmeans: need k >= 1");
    SLIC_REQUIRE(n >= k, "spherical_kmeans: need n >= k (n_samples should be >= n_clusters)");
    SLIC_REQUIRE(n_init >= 1, "spherical_kmeans: need n_init >= 1");
    SLIC_REQUIRE(max_iter >= 1, "spherical_kmeans: need max_iter >= 1");
    SLIC_REQUIRE(tol >= 0.0, "spherical_kmeans: need tol >= 0");
    SLIC_REQUIRE(!init_dev || n_init == 1, "spherical_kmeans: an explicit init runs once (n_init must be 1)");
    SLIC_REQUIRE(init_dev || (L >= 1 && L <= SK_MAX_L), "spherical_kmeans: need 1 <= L <= 32 candidates per step");
    SLIC_REQUIRE(x_dev && labels_out_dev && centers_out_dev && inertia_out_host && n_iter_out_host,
                 "spherical_kmeans: null pointer");
    SLIC_REQUIRE(init_dev || (first_ids_host && (k == 1 || uniforms_host)), "spherical_kmeans: null pointer (draws)");
    if (!init_dev)
        for (int r = 0; r < n_init; ++r)
            SLIC_REQUIRE(first_ids_host[r] >= 0 && first_ids_host[r] < n, "spherical_kmeans: first seed outside [0, n)");
    SLIC_PROPAGATE(slic_require_device());
    std::vector<int> first(init_dev ? 0 : n_init);
    for (size_t r = 0; r < first.size(); ++r) first[r] = (int)first_ids_host[r];
    return sk_fit(x_dev, n, d, k, init_dev, first.data(), uniforms_host, init_dev ? 0 : L, n_init, max_iter, tol,
                  labels_out_dev, centers_out_dev, inertia_out_host, n_iter_out_host, stats_out_host, as_stream(stream));
}
