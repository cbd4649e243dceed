// nj.cu -- neighbour joining and BIONJ on the device (kernel-5 forms of gkd_*_nj and gkd_*_bionj).
//
// The distances live in an n x n matrix of doubles in HBM (NjState, gkd_internal.cuh), filled by launch_square_scatter.
// The r active clusters of a round hold slots 0 .. r - 1.  Every operation of the definition in gkd.h is one IEEE double
// operation rounded to nearest, in the order written there, so the arithmetic below uses the __d*_rn intrinsics: they
// are never contracted into an FMA.
//   start:   R[i] = the sum of column i (equal to row i), ascending, one thread per i; label[i] = i;
//   scan:    a grid-stride over the rows; row i offers the pairs (i, j), j in (i, r), so each pair of the r x r corner is
//            read once.  Q uses the pair's labels a < b, not its slots.  Each CTA writes its best (Q, a, b) to part[];
//            the last CTA to finish reduces part[] (the minimum of a total order, so the result does not depend on
//            which CTA was last) and appends the round's row; at r = 2 it appends the last row;
//   update:  one thread per active k: d(u, k) into row and column f, R[k]; the thread of f writes R[u];
//   move:    slot r - 1 moves into g's slot (row, column, sum, label) unless g held it.
// BIONJ keeps d in the upper triangle and V in the lower one (gkd_internal.cuh).  The fill, the start and the scan body are
// NJ's: the fill writes d to both triangles, so the start's column sums are R and S alike, and the scan reads row i from
// column i + 1 on, which is d.  The pick also fixes lambda from S[f], S[g] and V(f, g); its own update and move then read
// and write d and V each in its triangle.  No thread of the update reads S[f] or S[g], which the thread of f writes.
// The host queues every round without reading anything between them.
#include <cuda_runtime.h>

#include "gkd_internal.cuh"

namespace gkd {

namespace {

constexpr int NJ_THREADS = 256;
constexpr int NJ_UNROLL = 4;  // row entries in flight per thread
constexpr uint32_t NJ_NONE = 0xFFFFFFFFu;

// x before y: Q as doubles (-0.0 == +0.0), then the labels
__device__ __forceinline__ bool nj_before(const NjCand &x, const NjCand &y) {
    return x.q < y.q || (x.q == y.q && (x.a < y.a || (x.a == y.a && x.b < y.b)));
}

__device__ __forceinline__ NjCand shfl_cand(const NjCand &c, int off) {
    return NjCand{__shfl_down_sync(0xffffffffu, c.q, off), __shfl_down_sync(0xffffffffu, c.a, off),
                  __shfl_down_sync(0xffffffffu, c.b, off), __shfl_down_sync(0xffffffffu, c.sa, off),
                  __shfl_down_sync(0xffffffffu, c.sb, off)};
}

__device__ __forceinline__ NjCand nj_none() { return NjCand{__longlong_as_double(0x7FF0000000000000ll), NJ_NONE, NJ_NONE, 0, 0}; }

// the CTA's best of every thread's c, valid in thread 0; part: NJ_THREADS / 32 entries of shared memory
__device__ __forceinline__ NjCand cta_best(NjCand c, NjCand *part) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int off = 16; off; off >>= 1) {
        const NjCand o = shfl_cand(c, off);
        if (nj_before(o, c)) c = o;
    }
    if (lane == 0) part[warp] = c;
    __syncthreads();
    if (warp == 0) {
        c = lane < NJ_THREADS / 32 ? part[lane] : nj_none();
        for (int off = 16; off; off >>= 1) {
            const NjCand o = shfl_cand(c, off);
            if (nj_before(o, c)) c = o;
        }
    }
    return c;
}

__global__ void __launch_bounds__(NJ_THREADS) k_nj_start(NjState st) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.n) return;
    const uint32_t n = st.n;
    double s = 0.0;
    // column i: a warp reads 32 consecutive entries of one row per step.  d(i, i) = 0 is skipped: s is never -0.0, so
    // s + 0.0 == s
#pragma unroll 8
    for (uint32_t k = 0; k < n; k++) {
        const double v = st.d[(uint64_t)k * n + i];
        if (k != i) s = __dadd_rn(s, v);
    }
    st.R[i] = s;
    if (st.S) st.S[i] = s;  // V starts equal to d
    st.label[i] = i;
}

// Q(a, b) = ((r - 2) d - R_a) - R_b with a < b the labels
__device__ __forceinline__ NjCand nj_q(double rm2, double d, double Ri, uint32_t li, double Rj, uint32_t lj, uint32_t i, uint32_t j) {
    const double x = __dmul_rn(rm2, d);
    return li < lj ? NjCand{__dsub_rn(__dsub_rn(x, Ri), Rj), li, lj, i, j} : NjCand{__dsub_rn(__dsub_rn(x, Rj), Ri), lj, li, j, i};
}

template <bool BIONJ>
__global__ void __launch_bounds__(NJ_THREADS) k_nj_scan(NjState st, uint32_t r, uint32_t row) {
    const uint64_t n = st.n;
    if (r == 2) {  // the last row: the midpoint of the last edge
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            const double h = __dmul_rn(0.5, st.d[1]);
            const uint32_t l0 = st.label[0], l1 = st.label[1];
            st.ra[row] = min(l0, l1);
            st.rb[row] = max(l0, l1);
            st.la[row] = st.lb[row] = h;
        }
        return;
    }
    __shared__ NjCand part[NJ_THREADS / 32];
    __shared__ bool last;
    const double rm2 = (double)(r - 2);
    NjCand best = nj_none();
    for (uint32_t i = blockIdx.x; i + 1 < r; i += gridDim.x) {
        const double *__restrict__ di = st.d + i * n;
        const double Ri = __ldg(st.R + i);
        const uint32_t li = __ldg(st.label + i);
        for (uint32_t j0 = i + 1 + threadIdx.x; j0 < r; j0 += NJ_THREADS * NJ_UNROLL) {
            double v[NJ_UNROLL];
#pragma unroll
            for (int u = 0; u < NJ_UNROLL; u++) {
                const uint32_t j = j0 + u * NJ_THREADS;
                v[u] = j < r ? di[j] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < NJ_UNROLL; u++) {
                const uint32_t j = j0 + u * NJ_THREADS;
                if (j >= r) break;
                const NjCand c = nj_q(rm2, v[u], Ri, li, __ldg(st.R + j), __ldg(st.label + j), i, j);
                if (nj_before(c, best)) best = c;
            }
        }
    }
    best = cta_best(best, part);
    if (threadIdx.x == 0) {
        st.part[blockIdx.x] = best;
        __threadfence();
        last = atomicAdd(st.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    // the pick: every CTA's best is visible (each fenced before its ticket)
    __threadfence();
    best = nj_none();
    for (uint32_t p = threadIdx.x; p < gridDim.x; p += NJ_THREADS) {
        const NjCand c{__ldcg(&st.part[p].q), __ldcg(&st.part[p].a), __ldcg(&st.part[p].b), __ldcg(&st.part[p].sa),
                       __ldcg(&st.part[p].sb)};
        if (nj_before(c, best)) best = c;
    }
    best = cta_best(best, part);
    if (threadIdx.x == 0) {
        const uint32_t sf = best.sa, sg = best.sb;
        const uint64_t lo = min(sf, sg), hi = max(sf, sg);
        const double dfg = st.d[lo * n + hi];
        const double t = __ddiv_rn(__dsub_rn(st.R[sf], st.R[sg]), (double)(2 * (r - 2)));
        const double df = __dadd_rn(__dmul_rn(0.5, dfg), t);
        st.ra[row] = best.a;
        st.rb[row] = best.b;
        st.la[row] = df;
        st.lb[row] = __dsub_rn(dfg, df);
        if (BIONJ) {  // lambda = clamp(0.5 + (S_g - S_f) / (2 (r - 2) V(f, g)), 0, 1), or 0.5 when V(f, g) == 0
            const double vfg = st.d[hi * n + lo];
            double lam = 0.5;
            if (vfg != 0.0) {
                const double x = __dadd_rn(0.5, __ddiv_rn(__dsub_rn(st.S[sg], st.S[sf]), __dmul_rn((double)(2 * (r - 2)), vfg)));
                lam = x < 0.0 ? 0.0 : x > 1.0 ? 1.0 : x;
            }
            *st.lambda = lam;
        }
        st.pick[0] = sf;
        st.pick[1] = sg;
        *st.ticket = 0;
    }
}

// Thread k reads rows f and g and writes row f and column f: no entry one thread writes is read by another
__global__ void __launch_bounds__(NJ_THREADS) k_nj_update(NjState st, uint32_t r) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= r) return;
    const uint64_t n = st.n;
    const uint32_t sf = st.pick[0], sg = st.pick[1];
    if (k == sg) return;
    const double *df = st.d + sf * n, *dg = st.d + sg * n;
    const double dfg = df[sg];
    if (k == sf) {  // R_u = 0.5 ((R_f + R_g) - r d(f, g)); no other thread touches R[f] or R[g]
        st.R[sf] = __dmul_rn(0.5, __dsub_rn(__dadd_rn(st.R[sf], st.R[sg]), __dmul_rn((double)r, dfg)));
        return;
    }
    const double dfk = df[k], dgk = dg[k];
    const double duk = __dmul_rn(0.5, __dsub_rn(__dadd_rn(dfk, dgk), dfg));
    st.R[k] = __dadd_rn(__dsub_rn(__dsub_rn(st.R[k], dfk), dgk), duk);
    st.d[sf * n + k] = duk;
    st.d[k * n + sf] = duk;
}

// slot r - 1 into g's slot: thread k copies (r - 1, k) and (k, r - 1); neither is in row or column g
__global__ void __launch_bounds__(NJ_THREADS) k_nj_move(NjState st, uint32_t r) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t sg = st.pick[1], last = r - 1;
    if (sg == last || k >= last || k == sg) return;
    const uint64_t n = st.n;
    st.d[sg * n + k] = st.d[last * n + k];
    st.d[k * n + sg] = st.d[k * n + last];
    if (k == (sg == 0 ? 1u : 0u)) {
        st.R[sg] = st.R[last];
        st.label[sg] = st.label[last];
    }
}

// BIONJ.  Thread k reads d(f, k), d(g, k), V(f, k), V(g, k) and writes d(u, k), V(u, k) into f's entries, R[k] and S[k];
// the thread of f writes R[u] and S[u].  lambda was fixed by the pick, so no entry one thread writes is read by another.
__global__ void __launch_bounds__(NJ_THREADS) k_bionj_update(NjState st, uint32_t r, uint32_t row) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= r) return;
    const uint64_t n = st.n;
    const uint32_t sf = st.pick[0], sg = st.pick[1];
    if (k == sg) return;
    const double lam = *st.lambda, mu = __dsub_rn(1.0, lam), w = __dmul_rn(lam, mu);
    const double dfg = st.d[min(sf, sg) * n + max(sf, sg)], vfg = st.d[max(sf, sg) * n + min(sf, sg)];
    const double la = st.la[row], lb = st.lb[row];
    if (k == sf) {
        const double rm2 = (double)(r - 2);
        st.R[sf] = __dadd_rn(__dmul_rn(lam, __dsub_rn(__dsub_rn(st.R[sf], dfg), __dmul_rn(rm2, la))),
                             __dmul_rn(mu, __dsub_rn(__dsub_rn(st.R[sg], dfg), __dmul_rn(rm2, lb))));
        st.S[sf] = __dsub_rn(__dadd_rn(__dmul_rn(lam, __dsub_rn(st.S[sf], vfg)), __dmul_rn(mu, __dsub_rn(st.S[sg], vfg))),
                             __dmul_rn(rm2, __dmul_rn(w, vfg)));
        return;
    }
    const uint64_t fk = min(sf, k) * n + max(sf, k), kf = max(sf, k) * n + min(sf, k);
    const uint64_t gk = min(sg, k) * n + max(sg, k), kg = max(sg, k) * n + min(sg, k);
    const double dfk = st.d[fk], dgk = st.d[gk], vfk = st.d[kf], vgk = st.d[kg];
    const double duk = __dadd_rn(__dmul_rn(lam, __dsub_rn(dfk, la)), __dmul_rn(mu, __dsub_rn(dgk, lb)));
    const double vuk = __dsub_rn(__dadd_rn(__dmul_rn(lam, vfk), __dmul_rn(mu, vgk)), __dmul_rn(w, vfg));
    st.R[k] = __dadd_rn(__dsub_rn(__dsub_rn(st.R[k], dfk), dgk), duk);
    st.S[k] = __dadd_rn(__dsub_rn(__dsub_rn(st.S[k], vfk), vgk), vuk);
    st.d[fk] = duk;
    st.d[kf] = vuk;
}

// BIONJ: slot r - 1 into g's slot.  Thread k (k < r - 1) copies d(r - 1, k) from [k n + r - 1] into g's upper entry and
// V(r - 1, k) from [(r - 1) n + k] into g's lower entry; for k < g these are not NJ's row and column
__global__ void __launch_bounds__(NJ_THREADS) k_bionj_move(NjState st, uint32_t r) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t sg = st.pick[1], last = r - 1;
    if (sg == last || k >= last || k == sg) return;
    const uint64_t n = st.n, lo = min(sg, k), hi = max(sg, k);
    const double d = st.d[k * n + last], v = st.d[last * n + k];
    st.d[lo * n + hi] = d;
    st.d[hi * n + lo] = v;
    if (k == (sg == 0 ? 1u : 0u)) {
        st.R[sg] = st.R[last];
        st.S[sg] = st.S[last];
        st.label[sg] = st.label[last];
    }
}

template <bool BIONJ>
void queue_rounds(const NjState &st, uint32_t max_ctas, cudaStream_t s) {
    for (uint32_t r = st.n, row = 0; r >= 3; r--, row++) {
        const unsigned nodes = (r + NJ_THREADS - 1) / NJ_THREADS;
        k_nj_scan<BIONJ><<<std::min(r - 1, max_ctas), NJ_THREADS, 0, s>>>(st, r, row);
        if (BIONJ) {
            k_bionj_update<<<nodes, NJ_THREADS, 0, s>>>(st, r, row);
            k_bionj_move<<<nodes, NJ_THREADS, 0, s>>>(st, r);
        } else {
            k_nj_update<<<nodes, NJ_THREADS, 0, s>>>(st, r);
            k_nj_move<<<nodes, NJ_THREADS, 0, s>>>(st, r);
        }
    }
    k_nj_scan<BIONJ><<<1, NJ_THREADS, 0, s>>>(st, 2, st.n - 2);
}

}  // namespace

uint64_t nj_state_bytes(uint32_t n) {
    const uint64_t N = n;
    return N * N * 8 + N * (8 + 4) + N * 24 + NJ_MAX_CTAS * sizeof(NjCand) + 256;
}

uint64_t bionj_state_bytes(uint32_t n) { return nj_state_bytes(n) + (uint64_t)n * 8 + 8; }

NjState nj_state_at(void *base, uint32_t n, bool bionj) {
    NjState st{};
    const uint64_t N = n;
    st.n = n;
    st.d = (double *)base;
    st.R = st.d + N * N;
    st.la = st.R + N;
    if (bionj) {
        st.S = st.la;
        st.la = st.S + N;
    }
    st.lb = st.la + N;
    st.part = (NjCand *)(st.lb + N);
    st.bad = (unsigned long long *)(st.part + NJ_MAX_CTAS);
    if (bionj) {
        st.lambda = (double *)st.bad;
        st.bad = (unsigned long long *)(st.lambda + 1);
    }
    st.ticket = (unsigned int *)(st.bad + 1);
    st.pick = (uint32_t *)(st.ticket + 1);
    st.label = st.pick + 2;
    st.ra = st.label + N;
    st.rb = st.ra + N;
    return st;
}

cudaError_t launch_nj_rounds(const NjState &st, int n_sms, cudaStream_t s) {
    const uint32_t n = st.n;
    if (n < 2) return cudaSuccess;
    k_nj_start<<<(n + NJ_THREADS - 1) / NJ_THREADS, NJ_THREADS, 0, s>>>(st);
    const uint32_t max_ctas = std::min<uint32_t>(NJ_MAX_CTAS, (uint32_t)n_sms * 4);
    if (st.S)
        queue_rounds<true>(st, max_ctas, s);
    else
        queue_rounds<false>(st, max_ctas, s);
    return cudaGetLastError();
}

}  // namespace gkd
