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

#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>

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

// the CTA's best candidate of row i (b: this thread's) to nn[i], nn_lo[i], nn_hi[i]; part: AGG_THREADS / 32 entries of
// shared memory, free again on return
__device__ __forceinline__ void row_best(const AggState &st, uint32_t i, Best b, Best *part, uint32_t lane, uint32_t warp) {
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

// the entry a distance is stored as: d 2^53 (agglomeration; false unless a multiple of 2^-53 in [0, 2]) or d itself
// (neighbour joining; false unless finite and in [0, 2])
__device__ __forceinline__ bool square_word(double d, uint64_t &w) {
    const double x = d * 9007199254740992.0;  // d 2^53, exact
    if (!(d >= 0.0 && d <= 2.0 && x == floor(x))) return false;
    w = (uint64_t)x;
    return true;
}
__device__ __forceinline__ bool square_word(double d, double &w) {
    w = d;
    return d >= 0.0 && d <= 2.0;
}

template <typename T>
__global__ void __launch_bounds__(AGG_THREADS) k_square_scatter(Square<T> sq, const double *__restrict__ src, uint64_t first,
                                                                uint64_t count, const uint32_t *join_err) {
    if (join_err && *join_err) return;  // the chunk is redone and rewrites these entries
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    uint32_t i, j;
    upper_pair(first + t, sq.n, i, j);
    T w;
    if (!square_word(src[t], w)) {
        atomicMin(sq.bad, (unsigned long long)(first + t));
        return;
    }
    const uint64_t ij = (uint64_t)i * sq.n + j, ji = (uint64_t)j * sq.n + i;
    sq.w[ij] = sq.w[ji] = w;
    if (sq.hi) sq.hi[ij] = sq.hi[ji] = 0;
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
        row_best(st, i, b, part, lane, warp);
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

// ---- complete linkage from the pairs within max_dist (CsRows) ----------------------------------------------------
// The rounds above with the matrix replaced by one sorted row per slot.  A pair beyond max_dist is +inf, and so is a
// tombstone; complete linkage is a max, so the merges up to max_dist are the same.  The update keeps the dense rule
// that a CTA reads only its own row, its partner's row and the neighbour words of other rows (never written), and that
// no two CTAs write one word.

__global__ void __launch_bounds__(AGG_THREADS) k_cs_append(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                                                           const double *__restrict__ dist, uint64_t count, uint32_t n,
                                                           CsList dst, uint64_t at, unsigned long long *bad) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const uint32_t x = a[t], y = b[t];
    const double d = dist[t];
    const double w = d * 9007199254740992.0;  // d 2^53, exact
    dst.a[at + t] = min(x, y);
    dst.b[at + t] = max(x, y);
    if (x >= n || y >= n || x == y || !(d >= 0.0 && d <= 2.0 && w == floor(w))) {
        dst.w[at + t] = CS_TOMB;
        atomicMin(bad, (unsigned long long)(at + t));
        return;
    }
    dst.w[at + t] = (uint64_t)w;
}

// both directions of every pair: key row << 32 | neighbour, value w
__global__ void __launch_bounds__(AGG_THREADS) k_cs_directed(CsList l, uint64_t count, uint64_t *__restrict__ keys,
                                                             uint64_t *__restrict__ vals) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const uint64_t a = l.a[t], b = l.b[t], w = l.w[t];
    keys[2 * t] = a << 32 | b;
    keys[2 * t + 1] = b << 32 | a;
    vals[2 * t] = vals[2 * t + 1] = w;
}

// off[r] = the first sorted key of row r (r <= n); nbr = the low words; the smallest repeated key to *dup
__global__ void __launch_bounds__(AGG_THREADS) k_cs_rows(const uint64_t *__restrict__ keys, uint64_t items, uint32_t n,
                                                         uint64_t *off, uint32_t *nbr, unsigned long long *dup) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t <= n) {
        const uint64_t want = t << 32;
        uint64_t lo = 0, hi = items;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (keys[mid] < want) lo = mid + 1;
            else hi = mid;
        }
        off[t] = lo;
    }
    if (t < items) {
        nbr[t] = (uint32_t)keys[t];
        if (t && keys[t] == keys[t - 1]) atomicMin(dup, (unsigned long long)keys[t]);
    }
}

constexpr uint64_t CS_NOWHERE = ~0ull;

// position of neighbour k in row x, or CS_NOWHERE
__device__ __forceinline__ uint64_t cs_find(const CsRows &r, uint32_t x, uint32_t k) {
    uint64_t lo = r.off[x], hi = r.off[x + 1];
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (r.nbr[mid] < k) lo = mid + 1;
        else hi = mid;
    }
    return lo < r.off[x + 1] && r.nbr[lo] == k ? lo : CS_NOWHERE;
}

// e(x, k), CS_TOMB when the pair is absent
__device__ __forceinline__ uint64_t cs_word(const CsRows &r, uint32_t x, uint32_t k) {
    const uint64_t p = cs_find(r, x, k);
    return p == CS_NOWHERE ? CS_TOMB : r.w[p];
}

__global__ void __launch_bounds__(AGG_THREADS) k_cs_scan(AggState st, CsRows r) {
    if (st.ctr[AGG_DONE]) return;
    __shared__ Best part[AGG_THREADS / 32];
    const uint32_t n_stale = (uint32_t)st.ctr[AGG_N_STALE];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t s = blockIdx.x; s < n_stale; s += gridDim.x) {
        const uint32_t i = st.stale[s];
        Best b{0, 0, 1, AGG_NONE};
        for (uint64_t e = r.off[i] + threadIdx.x; e < r.off[i + 1]; e += AGG_THREADS) {
            const uint64_t w = r.w[e];
            if (w == CS_TOMB) continue;
            const uint32_t k = r.nbr[e];
            if (!st.size[k]) continue;  // a partner of an earlier round whose entry in this row was left as it was
            const Best c{w, 0, 1, k};
            if (agg_before(c, b)) b = c;
        }
        row_best(st, i, b, part, lane, warp);
    }
}

// One CTA per survivor i with partner j.  Row i's entries: j and the other partners go; another survivor k (partner
// k') gets the max of e(i, k), e(j, k), e(i, k'), e(j, k'), or a tombstone when one is absent (its own CTA writes the
// same into row k); a slot k that does not merge gets max(e(i, k), e(j, k)) in row i and in row k, where e(k, j)
// becomes a tombstone.  A slot that does not merge and is a neighbour of j only loses e(k, j).  The partners' own rows
// are never read again.
__global__ void __launch_bounds__(AGG_THREADS) k_cs_update(AggState st, CsRows r) {
    if (st.ctr[AGG_DONE]) return;
    const uint32_t n_surv = (uint32_t)st.ctr[AGG_N_SURV];
    for (uint32_t s = blockIdx.x; s < n_surv; s += gridDim.x) {
        const uint32_t i = st.surv[s], j = st.mate[i];
        for (uint64_t e = r.off[j] + threadIdx.x; e < r.off[j + 1]; e += AGG_THREADS) {
            if (r.w[e] == CS_TOMB) continue;
            const uint32_t k = r.nbr[e];
            if (k == i || st.mate[k] != AGG_NONE || !st.size[k]) continue;
            if (cs_word(r, i, k) == CS_TOMB) r.w[cs_find(r, k, j)] = CS_TOMB;
        }
        __syncthreads();  // row i is read above and written below
        for (uint64_t e = r.off[i] + threadIdx.x; e < r.off[i + 1]; e += AGG_THREADS) {
            uint64_t v = r.w[e];
            if (v == CS_TOMB) continue;
            const uint32_t k = r.nbr[e];
            if (k == j) {
                r.w[e] = CS_TOMB;
                continue;
            }
            const uint32_t mk = st.mate[k];
            if (mk != AGG_NONE) {
                if (mk < k) continue;  // a partner: the scan skips it by its size from now on, and no thread writes it
                // CS_TOMB is the largest word, so an absent entry makes the max a tombstone
                v = max(max(v, cs_word(r, j, k)), max(cs_word(r, i, mk), cs_word(r, j, mk)));
                r.w[e] = v;
                continue;
            }
            if (!st.size[k]) continue;
            v = max(v, cs_word(r, j, k));
            r.w[e] = v;
            r.w[cs_find(r, k, i)] = v;
            const uint64_t p = cs_find(r, k, j);
            if (p != CS_NOWHERE) r.w[p] = CS_TOMB;
        }
        // other CTAs test the sizes of merging slots only after their mate, and the outcome is the same before and after
        if (threadIdx.x == 0) {
            st.size[i] += st.size[j];
            st.size[j] = 0;
        }
        __syncthreads();
    }
}

}  // namespace

uint64_t agg_nodes_bytes(uint32_t n) {
    const uint64_t N = n;
    return N * (5 * 4 + 2 * 8) + N * sizeof(AggMerge) + AGG_COUNTERS * 8 + 256;
}

uint64_t agg_state_bytes(uint32_t n, int average) { return (uint64_t)n * n * 8 * (average ? 2 : 1) + agg_nodes_bytes(n); }

AggState agg_state_at(void *base, uint32_t n, int average) {
    const uint64_t N = n;
    uint64_t *lo = (uint64_t *)base;
    AggState st = agg_nodes_at(lo + N * N * (average ? 2 : 1), n);
    st.average = average;
    st.lo = lo;
    st.hi = average ? lo + N * N : nullptr;
    return st;
}

AggState agg_nodes_at(void *base, uint32_t n) {
    AggState st{};
    const uint64_t N = n;
    st.n = n;
    uint64_t *w = (uint64_t *)base;
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

template <typename T>
cudaError_t launch_square_scatter(const Square<T> &sq, const double *src, uint64_t first, uint64_t count, const uint32_t *join_err,
                                  cudaStream_t s) {
    if (count == 0) return cudaSuccess;
    k_square_scatter<T><<<(unsigned)((count + AGG_THREADS - 1) / AGG_THREADS), AGG_THREADS, 0, s>>>(sq, src, first, count, join_err);
    return cudaGetLastError();
}
template cudaError_t launch_square_scatter<uint64_t>(const Square<uint64_t> &, const double *, uint64_t, uint64_t,
                                                     const uint32_t *, cudaStream_t);
template cudaError_t launch_square_scatter<double>(const Square<double> &, const double *, uint64_t, uint64_t,
                                                   const uint32_t *, cudaStream_t);

Square<uint64_t> agg_square(const AggState &st) { return {st.lo, st.average ? st.hi : nullptr, st.n, st.ctr + AGG_BAD}; }

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

uint64_t agg_dense_room() {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    uint64_t room = free_b;
    if (const char *e = getenv("GKD_AGG_MAX_BYTES")) room = std::min<uint64_t>(room, strtoull(e, nullptr, 10));
    return room;
}

cudaError_t launch_cs_append(const uint32_t *a, const uint32_t *b, const double *dist, uint64_t count, uint32_t n, CsList dst,
                             uint64_t at, unsigned long long *bad, cudaStream_t s) {
    if (count == 0) return cudaSuccess;
    k_cs_append<<<(unsigned)((count + AGG_THREADS - 1) / AGG_THREADS), AGG_THREADS, 0, s>>>(a, b, dist, count, n, dst, at, bad);
    return cudaGetLastError();
}

static int cs_end_bit(uint32_t n) {  // keys are below n << 32
    int bits = 1;
    while (bits < 32 && ((uint64_t)1 << bits) < n) bits++;
    return 32 + bits;
}

cudaError_t cs_sort_temp_bytes(uint64_t pairs, uint32_t n, size_t &bytes) {
    cub::DoubleBuffer<uint64_t> k(nullptr, nullptr), v(nullptr, nullptr);
    bytes = 0;
    return cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, v, (int64_t)(2 * pairs), 0, cs_end_bit(n));
}

cudaError_t launch_cs_rows(CsList l, uint64_t pairs, uint32_t n, uint64_t *keys[2], uint64_t *vals[2], void *temp,
                           size_t temp_bytes, uint64_t *off, uint32_t *nbr, unsigned long long *dup, int &current,
                           cudaStream_t s) {
    if (pairs) k_cs_directed<<<(unsigned)((pairs + AGG_THREADS - 1) / AGG_THREADS), AGG_THREADS, 0, s>>>(l, pairs, keys[0], vals[0]);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    cub::DoubleBuffer<uint64_t> k(keys[0], keys[1]), v(vals[0], vals[1]);
    if (pairs && (e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, k, v, (int64_t)(2 * pairs), 0, cs_end_bit(n), s)) != cudaSuccess)
        return e;
    current = k.selector;  // the values follow the keys
    const uint64_t m = std::max<uint64_t>(2 * pairs, (uint64_t)n + 1);
    k_cs_rows<<<(unsigned)((m + AGG_THREADS - 1) / AGG_THREADS), AGG_THREADS, 0, s>>>(k.Current(), 2 * pairs, n, off, nbr, dup);
    return cudaGetLastError();
}

cudaError_t launch_cs_rounds(const AggState &st, CsRows r, AggThreshold thr, uint32_t rounds, int n_sms, cudaStream_t s) {
    const unsigned node_blocks = (unsigned)(((uint64_t)st.n + AGG_THREADS - 1) / AGG_THREADS);
    const unsigned row_blocks = (unsigned)std::min<uint64_t>(st.n, (uint64_t)n_sms * 4);
    for (uint32_t k = 0; k < rounds; k++) {
        k_cs_scan<<<row_blocks, AGG_THREADS, 0, s>>>(st, r);
        k_agg_pair<<<node_blocks, AGG_THREADS, 0, s>>>(st, thr);
        k_cs_update<<<row_blocks, AGG_THREADS, 0, s>>>(st, r);
        k_agg_finalize<<<node_blocks, AGG_THREADS, 0, s>>>(st);
    }
    return cudaGetLastError();
}

}  // namespace gkd
