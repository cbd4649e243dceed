// agglomerate.cu -- complete and average linkage on the device (kernel-5 form of gkd_*_agglomerate).
//
// The cluster distances of the current clusters live in an n x n matrix in HBM (AggState, gkd_internal.cuh); slot x
// holds the cluster whose smallest id is x.  Both methods are reducible under the strict key (v, min label, max label):
// v(A u B, C) >= min(v(A, C), v(B, C)), and on a tie the merged label is the smaller one.  So every reciprocal pair of
// nearest neighbours is a merge of the sequential agglomeration, and the pairs of a round can merge at once.  A round:
//   scan:     each stale row (one CTA per row, a grid-stride over the stale list) finds its nearest active slot by the
//             exact key; every other row's neighbour is still valid by reducibility;
//   pair:     x and y = nn[x] merge when nn[y] = x and v <= max_dist; the smaller slot survives and appends the merge;
//   update:   one CTA per survivor i (partner j) rewrites row i: e(i, k) = e(i, k) (+) e(j, k) for a slot k that does not
//             merge (and the mirror entry e(k, i)), e(i, i') = the four entries of two merging pairs combined for a
//             survivor i'.  It reads rows i and j and writes row i and column i: the entries it reads are written by no
//             other CTA.  (+) is a max (complete) or a 128-bit integer add (average), so any order gives the same bits;
//   finalize: the partner slots go inactive; the survivors and the rows whose neighbour merged are the next stale rows;
//             a round that merged nothing sets AGG_DONE, and every later kernel exits at once.
// The host queues rounds in batches without reading anything between them.
#include <cuda_runtime.h>

#include "gkd_internal.cuh"

namespace gkd {

namespace {

constexpr int AGG_THREADS = 256;

__device__ __forceinline__ bool agg_within(const AggThreshold &t, uint64_t lo, uint64_t hi, uint64_t N) {
    if (t.all) return true;
    const unsigned __int128 S = (unsigned __int128)hi << 64 | lo, X = (unsigned __int128)t.m * N;
    unsigned __int128 rhs;
    if (t.shift >= 0) rhs = X << t.shift;  // max_dist < 2: shift <= 1, X < 2^117
    else rhs = -t.shift >= 128 ? 0 : X >> -t.shift;  // S is an integer: S <= X / 2^k  <=>  S <= floor(X / 2^k)
    return S <= rhs;
}

struct Best {
    uint64_t lo, hi, N;
    uint32_t k;
};

// x before y in the strict key (AGG_NONE is last); i's key ties break by the smaller other slot
__device__ __forceinline__ bool agg_before(const Best &x, const Best &y) {
    if (x.k == AGG_NONE) return false;
    if (y.k == AGG_NONE) return true;
    const int c = agg_cmp(x.lo, x.hi, x.N, y.lo, y.hi, y.N);
    return c < 0 || (c == 0 && x.k < y.k);
}

__device__ __forceinline__ Best shfl_best(const Best &b, int off) {
    return Best{__shfl_down_sync(0xffffffffu, b.lo, off), __shfl_down_sync(0xffffffffu, b.hi, off),
                __shfl_down_sync(0xffffffffu, b.N, off), __shfl_down_sync(0xffffffffu, b.k, off)};
}

__global__ void __launch_bounds__(AGG_THREADS) k_agg_init(AggState st) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < st.n) {
        st.size[x] = 1;
        st.nn[x] = st.mate[x] = AGG_NONE;
        st.stale[x] = x;
    }
    if (x < AGG_COUNTERS) {
        unsigned long long v = 0;
        if (x == AGG_N_STALE) v = st.n;
        if (x == AGG_DONE) v = st.n < 2 ? 1 : 0;
        if (x == AGG_BAD) v = ~0ull;
        st.ctr[x] = v;
    }
}

__global__ void __launch_bounds__(AGG_THREADS) k_agg_scatter(AggState st, const double *__restrict__ src, uint64_t first,
                                                             uint64_t count, const uint32_t *join_err) {
    if (join_err && *join_err) return;  // the chunk is redone and rewrites these entries
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    uint32_t i, j;
    upper_pair(first + t, st.n, i, j);
    const double d = src[t];
    const double w = d * 9007199254740992.0;  // d 2^53, exact
    if (!(d >= 0.0 && d <= 2.0 && w == floor(w))) {
        atomicMin(st.ctr + AGG_BAD, (unsigned long long)(first + t));
        return;
    }
    const uint64_t ij = (uint64_t)i * st.n + j, ji = (uint64_t)j * st.n + i;
    st.lo[ij] = st.lo[ji] = (uint64_t)w;
    if (st.average) st.hi[ij] = st.hi[ji] = 0;
}

__global__ void __launch_bounds__(AGG_THREADS) k_agg_scan(AggState st) {
    if (st.ctr[AGG_DONE]) return;
    __shared__ Best part[AGG_THREADS / 32];
    const uint32_t n_stale = (uint32_t)st.ctr[AGG_N_STALE], n = st.n;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t r = blockIdx.x; r < n_stale; r += gridDim.x) {
        const uint32_t i = st.stale[r];
        const uint64_t row = (uint64_t)i * n, si = st.size[i];
        Best b{0, 0, 1, AGG_NONE};
        for (uint32_t k = threadIdx.x; k < n; k += AGG_THREADS) {
            const uint32_t sk = st.size[k];
            if (!sk || k == i) continue;
            const Best c{st.lo[row + k], st.average ? st.hi[row + k] : 0, st.average ? si * sk : 1, k};
            if (agg_before(c, b)) b = c;
        }
        for (int off = 16; off; off >>= 1) {
            const Best o = shfl_best(b, off);
            if (agg_before(o, b)) b = o;
        }
        if (lane == 0) part[warp] = b;
        __syncthreads();
        if (warp == 0) {
            b = lane < AGG_THREADS / 32 ? part[lane] : Best{0, 0, 1, AGG_NONE};
            for (int off = 16; off; off >>= 1) {
                const Best o = shfl_best(b, off);
                if (agg_before(o, b)) b = o;
            }
            if (lane == 0) {
                st.nn[i] = b.k;
                st.nn_lo[i] = b.lo;
                st.nn_hi[i] = b.hi;
            }
        }
        __syncthreads();  // part[] is reused by the next row
    }
}

__global__ void __launch_bounds__(AGG_THREADS) k_agg_pair(AggState st, AggThreshold thr) {
    if (st.ctr[AGG_DONE]) return;
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x == 0) st.ctr[AGG_N_STALE] = 0;  // the scan has consumed the list; finalize refills it
    if (x >= st.n) return;
    const uint32_t sx = st.size[x], y = st.nn[x];
    uint32_t m = AGG_NONE, sy = 0;
    if (sx && y != AGG_NONE && st.nn[y] == x) {
        sy = st.size[y];
        if (agg_within(thr, st.nn_lo[x], st.nn_hi[x], st.average ? (uint64_t)sx * sy : 1)) m = y;
    }
    st.mate[x] = m;
    if (m == AGG_NONE || m < x) return;
    const uint32_t at = (uint32_t)atomicAdd(st.ctr + AGG_N_MERGES, 1ull);
    st.merges[at] = AggMerge{x, m, sx, sy, st.nn_lo[x], st.nn_hi[x]};
    st.surv[atomicAdd(st.ctr + AGG_N_SURV, 1ull)] = x;
    atomicAdd(st.ctr + AGG_ROUND_MERGES, 1ull);
}

__global__ void __launch_bounds__(AGG_THREADS) k_agg_update(AggState st) {
    if (st.ctr[AGG_DONE]) return;
    const uint32_t n_surv = (uint32_t)st.ctr[AGG_N_SURV], n = st.n;
    for (uint32_t r = blockIdx.x; r < n_surv; r += gridDim.x) {
        const uint32_t i = st.surv[r], j = st.mate[i];
        const uint64_t ri = (uint64_t)i * n, rj = (uint64_t)j * n;
        for (uint32_t k = threadIdx.x; k < n; k += AGG_THREADS) {
            if (k == i || k == j || !st.size[k]) continue;
            const uint32_t mk = st.mate[k];
            if (mk != AGG_NONE && mk < k) continue;  // the partner of a merge: its entries are dropped
            // entries (i, k) and (j, k); for a survivor k also (i, mk) and (j, mk)
            uint64_t lo = st.lo[ri + k], hi = st.average ? st.hi[ri + k] : 0;
            auto add = [&](uint64_t at) {
                const uint64_t l = st.lo[at];
                if (!st.average) {
                    lo = l > lo ? l : lo;
                    return;
                }
                const uint64_t s = lo + l;
                hi += st.hi[at] + (s < lo ? 1 : 0);
                lo = s;
            };
            add(rj + k);
            if (mk != AGG_NONE) {
                add(ri + mk);
                add(rj + mk);
            }
            st.lo[ri + k] = lo;
            if (st.average) st.hi[ri + k] = hi;
            if (mk == AGG_NONE) {  // the mirror entry; a survivor k writes its own row
                const uint64_t ki = (uint64_t)k * n + i;
                st.lo[ki] = lo;
                if (st.average) st.hi[ki] = hi;
            }
        }
        // other CTAs only test these two sizes for zero, and the outcome is the same before and after
        if (threadIdx.x == 0) {
            st.size[i] += st.size[j];
            st.size[j] = 0;
        }
    }
}

__global__ void __launch_bounds__(AGG_THREADS) k_agg_finalize(AggState st) {
    if (st.ctr[AGG_DONE]) return;
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x == 0) {
        if (st.ctr[AGG_ROUND_MERGES] == 0) st.ctr[AGG_DONE] = 1;
        else st.ctr[AGG_ROUNDS]++;
        st.ctr[AGG_ROUND_MERGES] = 0;
        st.ctr[AGG_N_SURV] = 0;
    }
    if (x >= st.n || !st.size[x]) return;
    const uint32_t y = st.nn[x];
    // a survivor, or a row whose nearest slot merged: its key may have grown
    if (st.mate[x] != AGG_NONE || (y != AGG_NONE && st.mate[y] != AGG_NONE))
        st.stale[atomicAdd(st.ctr + AGG_N_STALE, 1ull)] = x;
}

}  // namespace

uint64_t agg_state_bytes(uint32_t n, int average) {
    const uint64_t N = n;
    return N * N * 8 * (average ? 2 : 1) + N * (5 * 4 + 2 * 8) + N * sizeof(AggMerge) + AGG_COUNTERS * 8 + 256;
}

AggState agg_state_at(void *base, uint32_t n, int average) {
    AggState st{};
    const uint64_t N = n;
    st.n = n;
    st.average = average;
    st.lo = (uint64_t *)base;
    st.hi = average ? st.lo + N * N : nullptr;
    uint64_t *w = st.lo + N * N * (average ? 2 : 1);
    st.nn_lo = w;
    st.nn_hi = w + N;
    st.ctr = (unsigned long long *)(w + 2 * N);
    st.merges = (AggMerge *)(st.ctr + AGG_COUNTERS);
    st.size = (uint32_t *)(st.merges + N);
    st.nn = st.size + N;
    st.mate = st.nn + N;
    st.stale = st.mate + N;
    st.surv = st.stale + N;
    return st;
}

cudaError_t launch_agg_init(const AggState &st, cudaStream_t s) {
    const uint64_t m = std::max<uint64_t>(st.n, AGG_COUNTERS);
    k_agg_init<<<(unsigned)((m + AGG_THREADS - 1) / AGG_THREADS), AGG_THREADS, 0, s>>>(st);
    return cudaGetLastError();
}

cudaError_t launch_agg_scatter(const AggState &st, const double *src, uint64_t first, uint64_t count, const uint32_t *join_err,
                               cudaStream_t s) {
    if (count == 0) return cudaSuccess;
    k_agg_scatter<<<(unsigned)((count + AGG_THREADS - 1) / AGG_THREADS), AGG_THREADS, 0, s>>>(st, src, first, count, join_err);
    return cudaGetLastError();
}

cudaError_t launch_agg_rounds(const AggState &st, AggThreshold thr, uint32_t rounds, int n_sms, cudaStream_t s) {
    const unsigned node_blocks = (unsigned)(((uint64_t)st.n + AGG_THREADS - 1) / AGG_THREADS);
    const unsigned row_blocks = (unsigned)std::min<uint64_t>(st.n, (uint64_t)n_sms * 4);
    for (uint32_t r = 0; r < rounds; r++) {
        k_agg_scan<<<row_blocks, AGG_THREADS, 0, s>>>(st);
        k_agg_pair<<<node_blocks, AGG_THREADS, 0, s>>>(st, thr);
        k_agg_update<<<row_blocks, AGG_THREADS, 0, s>>>(st);
        k_agg_finalize<<<node_blocks, AGG_THREADS, 0, s>>>(st);
    }
    return cudaGetLastError();
}

}  // namespace gkd
