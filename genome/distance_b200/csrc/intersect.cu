// intersect.cu -- kernel 4 (pairwise set intersection count) and kernel 5 (distance epilogue) of
// libgkd.so.  sm_100a only; no tensor cores (this is merge work, not a contraction).
//
// Reference semantics restated:
//   SequenceKmers.similarity(other): number of members of one HashSet<String> found in the other
//   SequenceKmers.distance(other):   I == 0 ? 1.0 : 1.0 - I / ((|A| + |B|) - I), |A|+|B| a Java int sum
//   (called at FastaDistanceProcessor.java:186, GenomeProcessor.java:140, DistanceRepsProcessor.java:101,190,
//    FastaDistanceRepsProcessor.java:128).
//   Pair order: strict upper triangle in list order (FastaDistanceProcessor.java:177) or every
//   (query, base) pair (GenomeProcessor.java:140-146).
//
// Kernel 4 design (B200), round 2: warp-cooperative merge over VALUE-partitioned runs.
//   Sets are sorted by a bijective mix of the key and carry a table of bucket offsets (gkd_internal.cuh),
//   so the merge partition is a table lookup: bucket f of A and bucket f of B cover the same key range.
//   * a warp owns a work item = (pair, run of 32-bucket groups); items come from one global counter and
//     are enumerated pair-major, so the warps resident at one time share a few row sets (served from the
//     126 MB L2) and walk a pair's two key streams front to back;
//   * per group, lane t reads its bucket bounds from both tables (two coalesced loads per set), lane 0
//     requests the group's two contiguous key ranges with TMA bulk copies (cp.async.bulk, SASS UBLKCP)
//     into the warp's own shared-memory stage guarded by an mbarrier (expect_tx / try_wait.parity); the
//     offsets of the group after next and the copies of the next group are in flight while the current
//     group is merged;
//   * every lane then merges its two runs (<= tmax keys each on average) from shared memory with a
//     branch-light two-pointer loop on the 32-bit low words (64-bit for keys wider than 42 bits): ~10
//     SASS instructions per step for 32 lanes, against ~100 per 58 keys for the round-1 ballot kernel;
//   * sets of different size meet at the level of the larger one: the lanes partition the larger set
//     exactly and several lanes share one (coarser) bucket of the smaller set, so a pair never costs
//     more than ~2x the keys of its larger set and no separate kernel is needed for skewed pairs;
//   * a group whose ranges do not fit the stage (rare: > 5 sigma, or mis-tuned tmax) is merged straight
//     from global memory by the same loop;
//   * counts: per-lane counters, one warp reduction (REDUX) and one atomicAdd per item.
// Bound: nominally HBM (algorithmic bytes 8 * (|A| + |B|) per pair, SURVEY 8d); the stored bytes are
// ~4.25 per key (low word + table share), see DESIGN.md section 4 for the measured limiter.
#include <cstdlib>

#include <cuda/atomic>

#include "gkd_internal.cuh"

namespace gkd {

// ---- mbarrier / TMA / shared-memory wrappers --------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    uint32_t spins = 0;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (++spins > (1u << 24)) __trap();  // a lost copy must not hang the GPU
    } while (!done);
}

template <typename LowT>
__device__ __forceinline__ LowT lds_low(uint32_t addr);
template <>
__device__ __forceinline__ uint32_t lds_low<uint32_t>(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
template <>
__device__ __forceinline__ uint64_t lds_low<uint64_t>(uint32_t addr) {
    uint64_t v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr));
    return v;
}

// decode pair index t of this call into set ids
__device__ __forceinline__ void decode_pair(const PairSource &src, uint64_t t, uint32_t &ida, uint32_t &idb) {
    if (src.mode == PAIRS_UPPER) {
        upper_pair(src.first + t, src.n, ida, idb);
    } else if (src.mode == PAIRS_RECT) {
        ida = src.a[t / src.n];
        idb = src.b[t % src.n];
    } else if (src.mode == PAIRS_LIST_VS_ONE) {
        ida = src.a[t];
        idb = src.n;
    } else {
        ida = src.a[t];
        idb = src.b[t];
    }
}

// ---- the merge loops -----------------------------------------------------------------------------------
// Two-pointer count of equal keys of two ascending runs.  Equal heads advance both runs; the loop ends
// as soon as either run is exhausted (the rest of the other run cannot match).
// The shared-memory version is written in PTX to pin its shape: per step two compares, two predicated
// pointer bumps, a step counter, two predicated loads and the exit test (10 instructions for 32 lanes;
// the compiler's version of the same C loop took 13-15).  Every step advances one run, or both when the
// heads are equal, so matches = advances - steps.  The loads run ahead of the exit test and may read
// the word just past a run, which is still inside the CTA's shared memory.
template <typename LowT>
__device__ __forceinline__ uint32_t merge_smem(uint32_t pa, uint32_t ea, uint32_t pb, uint32_t eb);

#ifndef GKD_MERGE_UNROLL2
#define GKD_MERGE_UNROLL2 1
#endif
#ifndef GKD_MERGE_ONE_LDS
#define GKD_MERGE_ONE_LDS 0  // measured on B200 (300 genomes): 345 ms against 284 ms for the two-load step
#endif

#if GKD_MERGE_ONE_LDS
// Experiment kept for the record: one shared-memory load per step (exactly one run advances; ties advance A and
// are counted there), a single LDS with a selected address serving every lane.  It cuts the shared-memory
// wavefronts (the kernel's co-limiter) by ~40 % but needs 10.5 instead of 8 instructions per step and puts two
// selects on the load's dependency chain: slower overall (issue-bound), so the two-load step below is the default.
#define GKD_MERGE_STEP(T, SZ)               \
    "setp.le." T " ple, a, b;\n"           \
    "setp.eq." T " peq, a, b;\n"           \
    "@peq add.u32 %2, %2, 1;\n"            \
    "@ple add.u32 %0, %0, " SZ ";\n"       \
    "@!ple add.u32 %1, %1, " SZ ";\n"      \
    "selp.u32 adr, %0, %1, ple;\n"         \
    "ld.shared." T " v, [adr];\n"          \
    "selp." T " a, v, a, ple;\n"           \
    "selp." T " b, b, v, ple;\n"
#define GKD_MERGE_REGS(T) ".reg .pred ple, peq, pgo;\n.reg ." T " a, b, v;\n.reg .u32 adr;\n"
#define GKD_MERGE_COUNT2 ""
#define GKD_MERGE_COUNT1 ""
#else
#define GKD_MERGE_STEP(T, SZ)               \
    "setp.gt." T " pgt, a, b;\n"           \
    "setp.lt." T " plt, a, b;\n"           \
    "@!pgt add.u32 %0, %0, " SZ ";\n"      \
    "@!plt add.u32 %1, %1, " SZ ";\n"      \
    "@!pgt ld.shared." T " a, [%0];\n"     \
    "@!plt ld.shared." T " b, [%1];\n"
#define GKD_MERGE_REGS(T) ".reg .pred pgt, plt, pgo;\n.reg ." T " a, b;\n"
#define GKD_MERGE_COUNT2 "add.u32 %2, %2, 2;\n"
#define GKD_MERGE_COUNT1 "add.u32 %2, %2, 1;\n"
#endif

// With GKD_MERGE_UNROLL2 the loop runs two steps per trip while both runs hold at least two more keys (no exit
// test between them), then finishes with the one-step loop.
#define GKD_MERGE_BODY(T, SZ, TAG)                                                          \
    "{\n"                                                                                   \
    GKD_MERGE_REGS(T)                                                                       \
    "ld.shared." T " a, [%0];\n"                                                            \
    "ld.shared." T " b, [%1];\n"                                                            \
    "setp.lt.u32 pgo, %0, %5;\n"                                                            \
    "setp.lt.and.u32 pgo, %1, %6, pgo;\n"                                                   \
    "@!pgo bra " TAG "_ONE_%=;\n"                                                           \
    TAG "_TWO_%=:\n"                                                                        \
    GKD_MERGE_STEP(T, SZ)                                                                   \
    GKD_MERGE_STEP(T, SZ)                                                                   \
    GKD_MERGE_COUNT2                                                                        \
    "setp.lt.u32 pgo, %0, %5;\n"                                                            \
    "setp.lt.and.u32 pgo, %1, %6, pgo;\n"                                                   \
    "@pgo bra " TAG "_TWO_%=;\n"                                                            \
    "setp.lt.u32 pgo, %0, %3;\n"                                                            \
    "setp.lt.and.u32 pgo, %1, %4, pgo;\n"                                                   \
    "@!pgo bra " TAG "_END_%=;\n"                                                           \
    TAG "_ONE_%=:\n"                                                                        \
    GKD_MERGE_STEP(T, SZ)                                                                   \
    GKD_MERGE_COUNT1                                                                        \
    "setp.lt.u32 pgo, %0, %3;\n"                                                            \
    "setp.lt.and.u32 pgo, %1, %4, pgo;\n"                                                   \
    "@pgo bra " TAG "_ONE_%=;\n"                                                            \
    TAG "_END_%=:\n"                                                                        \
    "}\n"

// what merge_smem returns from its three in/out operands (pa, pb, and the step counter or the match counter)
__device__ __forceinline__ uint32_t merge_result(uint32_t pa, uint32_t pb, uint32_t start, uint32_t counter, int shift) {
#if GKD_MERGE_ONE_LDS
    (void)pa, (void)pb, (void)start, (void)shift;
    return counter;  // matches counted directly
#else
    return ((pa + pb - start) >> shift) - counter;  // every step advances one run, or both on a match
#endif
}

template <>
__device__ __forceinline__ uint32_t merge_smem<uint32_t>(uint32_t pa, uint32_t ea, uint32_t pb, uint32_t eb) {
    if (pa >= ea || pb >= eb) return 0;
    const uint32_t start = pa + pb;
    uint32_t counter = 0;
    // two unchecked steps need two keys left in each run: pa < ea - 4 and pb < eb - 4 (the runs are not empty here)
    const uint32_t ea2 = GKD_MERGE_UNROLL2 ? ea - 4u : 0u, eb2 = GKD_MERGE_UNROLL2 ? eb - 4u : 0u;
    asm volatile(GKD_MERGE_BODY("u32", "4", "M32") : "+r"(pa), "+r"(pb), "+r"(counter) : "r"(ea), "r"(eb), "r"(ea2), "r"(eb2) : "memory");
    return merge_result(pa, pb, start, counter, 2);
}

template <>
__device__ __forceinline__ uint32_t merge_smem<uint64_t>(uint32_t pa, uint32_t ea, uint32_t pb, uint32_t eb) {
    if (pa >= ea || pb >= eb) return 0;
    const uint32_t start = pa + pb;
    uint32_t counter = 0;
    const uint32_t ea2 = GKD_MERGE_UNROLL2 ? ea - 8u : 0u, eb2 = GKD_MERGE_UNROLL2 ? eb - 8u : 0u;
    asm volatile(GKD_MERGE_BODY("u64", "8", "M64") : "+r"(pa), "+r"(pb), "+r"(counter) : "r"(ea), "r"(eb), "r"(ea2), "r"(eb2) : "memory");
    return merge_result(pa, pb, start, counter, 3);
}

template <typename LowT>
__device__ __forceinline__ uint32_t merge_global(const LowT *__restrict__ pa, const LowT *__restrict__ ea,
                                                 const LowT *__restrict__ pb, const LowT *__restrict__ eb) {
    uint32_t cnt = 0;
    if (pa < ea && pb < eb) {
        LowT a = __ldg(pa), b = __ldg(pb);
        for (;;) {
            const bool le = a <= b, ge = b <= a;
            cnt += (le && ge) ? 1u : 0u;
            if (le) pa++;
            if (ge) pb++;
            if (pa >= ea || pb >= eb) break;
            if (le) a = __ldg(pa);
            if (ge) b = __ldg(pb);
        }
    }
    return cnt;
}

// bounds [lo, hi) of lane bucket f (at walk level L) in a set whose table is at S.level
__device__ __forceinline__ void lane_run(const SubSet &S, uint32_t L, uint32_t f, bool active, uint32_t &lo,
                                         uint32_t &hi) {
    lo = hi = 0;
    if (!active) return;
    if (S.level >= L) {
        const uint32_t sh = S.level - L;
        lo = __ldg(S.offs + ((size_t)f << sh));
        hi = __ldg(S.offs + ((size_t)(f + 1) << sh));
    } else {  // coarser table: the lanes of 2^sh consecutive buckets share one bucket of this set
        const uint32_t c = f >> (L - S.level);
        lo = __ldg(S.offs + c);
        hi = __ldg(S.offs + c + 1);
    }
}

// Kernel configuration: CAP bytes per set per stage, STAGES stages per warp, WARPS warps per CTA,
// CTAS CTAs per SM.
template <int CAP_, int STAGES_, int WARPS_, int CTAS_>
struct BucketCfg {
    static constexpr int CAP = CAP_, STAGES = STAGES_, WARPS = WARPS_, CTAS = CTAS_;
    static constexpr uint32_t STAGE_BYTES = 2u * CAP;                      // A range + B range
    static constexpr uint32_t WARP_BYTES = STAGES * STAGE_BYTES;
    static constexpr uint32_t BAR_OFF = WARPS * WARP_BYTES;
    static constexpr uint32_t SMEM = BAR_OFF + WARPS * STAGES * 8u;
    static_assert(CAP % 16 == 0, "stages hold whole 16-byte TMA units");
    static_assert((size_t)(SMEM + 1024) * CTAS <= 227u * 1024u, "does not fit the SM");
    static_assert(WARPS * CTAS <= 64, "at most 64 warps per SM");
};

struct OffsRegs {  // bucket bounds of one lane for one group (key indices)
    uint32_t loA, hiA, loB, hiB;
};
struct StageRegs {  // where this lane's runs of one group are, once staged
    uint32_t pa, ea, pb, eb;  // shared-memory addresses (staged) or key indices (direct)
    uint32_t mode;            // 0 = nothing to merge, 1 = staged and a copy is in flight, 2 = direct from global
};

template <typename LowT, class C>
__global__ void __launch_bounds__(C::WARPS * 32, C::CTAS)
    k_intersect_bucket(const SetDesc *__restrict__ sets, PairSource src, int use_pal, IsectPlan plan,
                       uint32_t *__restrict__ counts, unsigned long long *__restrict__ work_counter) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr uint32_t KEYS16 = 16u / (uint32_t)sizeof(LowT);  // keys per 16-byte TMA unit
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t buf0 = smem_u32(smem_raw) + warp * C::WARP_BYTES;
    const uint32_t bar0 = smem_u32(smem_raw) + C::BAR_OFF + warp * (C::STAGES * 8u);
    if (lane == 0) {
        for (int i = 0; i < C::STAGES; i++) mbar_init(bar0 + i * 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    uint32_t phases = 0;  // bit s = parity to wait for on the barrier of stage s

    const uint64_t total_items = (src.count_ptr ? (uint64_t)*src.count_ptr : src.count) * (uint64_t)plan.items_per_pair;
    unsigned long long next_item = 0;
    if (lane == 0) next_item = atomicAdd(work_counter, 1ull);
    for (;;) {
        const uint64_t item = __shfl_sync(0xffffffffu, next_item, 0);
        if (item >= total_items) break;
        if (lane == 0) next_item = atomicAdd(work_counter, 1ull);  // fetched while this item is processed
        const uint64_t pair = item / plan.items_per_pair;
        const uint32_t chunk = (uint32_t)(item - pair * plan.items_per_pair);
        uint32_t ida, idb;
        decode_pair(src, pair, ida, idb);
        const SetDesc *da = sets + ida, *db = sets + idb;
        const SubSet SA = use_pal ? da->pal : da->main, SB = use_pal ? db->pal : db->main;
        if (SA.n == 0 || SB.n == 0) continue;
        // walk level: the larger set averages <= tmax keys per lane bucket
        const uint32_t nmax = SA.n > SB.n ? SA.n : SB.n, lmax = SA.level > SB.level ? SA.level : SB.level;
        uint32_t L = level_for(nmax, plan.tmax);
        if (L < plan.level_min) L = plan.level_min;
        if (L > lmax) L = lmax;
        const uint32_t n_buckets = 1u << L;
        const uint32_t n_groups = (n_buckets + 31u) >> 5;
        const uint32_t g0 = chunk * plan.groups_per_item;
        if (g0 >= n_groups) continue;
        const uint32_t g1 = (n_groups - g0 > plan.groups_per_item) ? g0 + plan.groups_per_item : n_groups;
        const LowT *lowsA = (const LowT *)SA.lows, *lowsB = (const LowT *)SB.lows;

        // phase O: this lane's bucket bounds of group g
        auto load_offs = [&](uint32_t g) {
            OffsRegs o;
            const uint32_t f = g * 32u + lane;
            const bool active = f < n_buckets;
            lane_run(SA, L, f, active, o.loA, o.hiA);
            lane_run(SB, L, f, active, o.loB, o.hiB);
            return o;
        };
        // phase T: request the group's two key ranges into stage s (or decide to merge from global)
        auto stage_group = [&](const OffsRegs &o, uint32_t g, uint32_t s) {
            StageRegs r;
            const uint32_t last = (n_buckets - g * 32u >= 32u) ? 31u : (n_buckets - g * 32u - 1u);
            const uint32_t a_lo = __shfl_sync(0xffffffffu, o.loA, 0), a_hi = __shfl_sync(0xffffffffu, o.hiA, last);
            const uint32_t b_lo = __shfl_sync(0xffffffffu, o.loB, 0), b_hi = __shfl_sync(0xffffffffu, o.hiB, last);
            const uint32_t a0 = a_lo & ~(KEYS16 - 1u), b0 = b_lo & ~(KEYS16 - 1u);
            const uint32_t bytesA = a_hi > a_lo ? (uint32_t)align16((uint64_t)(a_hi - a0) * sizeof(LowT)) : 0u;
            const uint32_t bytesB = b_hi > b_lo ? (uint32_t)align16((uint64_t)(b_hi - b0) * sizeof(LowT)) : 0u;
            if (bytesA == 0 || bytesB == 0) {  // one side has no key in this group: nothing can match
                r.pa = r.ea = r.pb = r.eb = 0;
                r.mode = 0;
            } else if (bytesA > (uint32_t)C::CAP || bytesB > (uint32_t)C::CAP) {
                r.pa = o.loA, r.ea = o.hiA, r.pb = o.loB, r.eb = o.hiB;
                r.mode = 2;
            } else {
                const uint32_t bufA = buf0 + s * C::STAGE_BYTES, bufB = bufA + C::CAP, bar = bar0 + s * 8u;
                if (lane == 0) {
                    mbar_expect_tx(bar, bytesA + bytesB);
                    tma_load_1d(bufA, lowsA + a0, bytesA, bar);
                    tma_load_1d(bufB, lowsB + b0, bytesB, bar);
                }
                r.pa = bufA + (o.loA - a0) * (uint32_t)sizeof(LowT);
                r.ea = bufA + (o.hiA - a0) * (uint32_t)sizeof(LowT);
                r.pb = bufB + (o.loB - b0) * (uint32_t)sizeof(LowT);
                r.eb = bufB + (o.hiB - b0) * (uint32_t)sizeof(LowT);
                r.mode = 1;
            }
            return r;
        };
        // phase M: wait for the stage and merge this lane's runs
        auto merge_group = [&](const StageRegs &r, uint32_t s) -> uint32_t {
            uint32_t c = 0;
            if (r.mode == 1) {
                mbar_wait(bar0 + s * 8u, (phases >> s) & 1u);
                phases ^= 1u << s;
                c = merge_smem<LowT>(r.pa, r.ea, r.pb, r.eb);
            } else if (r.mode == 2) {
                c = merge_global<LowT>(lowsA + r.pa, lowsA + r.ea, lowsB + r.pb, lowsB + r.eb);
            }
            __syncwarp();  // every lane is done reading the stage before it is requested again
            return c;
        };

        uint32_t cnt = 0, s = 0;
        OffsRegs on = load_offs(g0);
        StageRegs cur = stage_group(on, g0, 0);
        if (g0 + 1 < g1) on = load_offs(g0 + 1);
        for (uint32_t g = g0; g < g1; g++) {
            if (C::STAGES >= 2) {
                StageRegs nxt = cur;
                if (g + 1 < g1) {
                    nxt = stage_group(on, g + 1, s ^ 1u);
                    if (g + 2 < g1) on = load_offs(g + 2);
                }
                cnt += merge_group(cur, s);
                cur = nxt;
                s ^= 1u;
            } else {
                cnt += merge_group(cur, 0);
                if (g + 1 < g1) {
                    cur = stage_group(on, g + 1, 0);
                    if (g + 2 < g1) on = load_offs(g + 2);
                }
            }
        }
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0 && cnt) atomicAdd(&counts[pair], cnt);
    }
}

// Configurations (index selected with GKD_ISECT_CFG; see profiles/ for the sweep).  The stage must hold
// 32 lanes x tmax keys plus ~5 sigma of the bucket-occupancy noise and the 16-byte alignment slack.
using BCfg0 = BucketCfg<2560, 2, 4, 5>;   // tmax 16 (u32) / 8 (u64), double-buffered, 20 warps per SM
using BCfg1 = BucketCfg<2560, 1, 4, 10>;  // single stage, 40 warps per SM
using BCfg2 = BucketCfg<3840, 2, 4, 3>;   // tmax 24 / 12, double-buffered, 12 warps per SM
using BCfg3 = BucketCfg<3840, 1, 4, 7>;   // single stage, 28 warps per SM
using BCfg4 = BucketCfg<1536, 2, 4, 9>;   // tmax 8 / 4, double-buffered, 36 warps per SM
using BCfg5 = BucketCfg<1536, 1, 4, 16>;  // single stage, 64 warps per SM
using BCfg6 = BucketCfg<3072, 1, 4, 9>;   // tmax 24 with a tight stage, 36 warps per SM
using BCfg7 = BucketCfg<3328, 1, 4, 8>;   // tmax 24, 32 warps per SM
using BCfg8 = BucketCfg<5632, 1, 4, 4>;   // tmax 48 / 24, 16 warps per SM
using BCfg9 = BucketCfg<5632, 1, 2, 9>;   // tmax 48 / 24, 18 warps per SM
constexpr int N_BCFG = 10;
constexpr int DEFAULT_BCFG = 9;
static const uint32_t g_cfg_tmax32[N_BCFG] = {16, 16, 24, 24, 8, 8, 24, 24, 48, 48};

#define GKD_FOR_EACH_BCFG(X) \
    X(0, BCfg0) X(1, BCfg1) X(2, BCfg2) X(3, BCfg3) X(4, BCfg4) X(5, BCfg5) X(6, BCfg6) X(7, BCfg7) X(8, BCfg8) X(9, BCfg9)

static int env_cfg() {
    const char *e = getenv("GKD_ISECT_CFG");
    int c = e ? atoi(e) : DEFAULT_BCFG;
    return (c < 0 || c >= N_BCFG) ? DEFAULT_BCFG : c;
}

cudaError_t intersect_configure() {
    cudaError_t e;
#define X(i, C)                                                                                                          \
    if ((e = cudaFuncSetAttribute(k_intersect_bucket<uint32_t, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM))) \
        return e;                                                                                                        \
    if ((e = cudaFuncSetAttribute(k_intersect_bucket<uint64_t, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM))) \
        return e;
    GKD_FOR_EACH_BCFG(X)
#undef X
    return cudaSuccess;
}

uint32_t intersect_default_tmax(int low_bits) {
    const char *e = getenv("GKD_ISECT_TMAX");
    uint32_t t = e ? (uint32_t)atoi(e) : g_cfg_tmax32[env_cfg()];
    if (low_bits == 64 && !e) t /= 2;
    return t < 1 ? 1 : t;
}

uint32_t intersect_warps_per_sm(int) {
    const int c = env_cfg();
#define X(i, C) \
    if (c == i) return C::WARPS * C::CTAS;
    GKD_FOR_EACH_BCFG(X)
#undef X
    return 16;
}

template <typename LowT, class C>
static cudaError_t launch_bcfg(const SetDesc *sets, PairSource src, int use_pal, const IsectPlan &plan, uint32_t *counts,
                               unsigned long long *work_counter, int n_sms, cudaStream_t s) {
    const uint64_t items = src.count * (uint64_t)plan.items_per_pair;
    uint64_t grid = (uint64_t)n_sms * C::CTAS;  // persistent: every SM holds CTAS resident CTAs
    const uint64_t need = (items + C::WARPS - 1) / C::WARPS;
    if (grid > need) grid = need;
    k_intersect_bucket<LowT, C><<<(unsigned)grid, C::WARPS * 32, C::SMEM, s>>>(sets, src, use_pal, plan, counts, work_counter);
    return cudaGetLastError();
}

cudaError_t launch_intersect(const SetDesc *sets, PairSource src, int use_pal, const IsectPlan &plan, uint32_t *counts,
                             unsigned long long *work_counter, int n_sms, cudaStream_t s) {
    if (src.count == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), s);
    if (e != cudaSuccess) return e;
    const int c = env_cfg();
#define X(i, C)                                                                                               \
    if (c == i)                                                                                               \
        return plan.low_bits == 32 ? launch_bcfg<uint32_t, C>(sets, src, use_pal, plan, counts, work_counter, n_sms, s) \
                                   : launch_bcfg<uint64_t, C>(sets, src, use_pal, plan, counts, work_counter, n_sms, s);
    GKD_FOR_EACH_BCFG(X)
#undef X
    return cudaErrorInvalidValue;
}

// ---- kernel 5: distance epilogue ----------------------------------------------------------------------
// SequenceKmers.similarity / distance of one pair from the canonical counts (c = |C_A n C_B|, cp = palindromic part) and
// the literal k-mers (li shared, la and lb of each set; 0 outside GKD_AMBIG_LITERAL)
__device__ __forceinline__ void pair_result(const SetDesc *__restrict__ sets, uint32_t ida, uint32_t idb, uint64_t c, uint64_t cp,
                                            uint32_t li, uint32_t la, uint32_t lb, int both_strands, uint64_t &I, uint64_t &sa,
                                            uint64_t &sb, double &dist) {
    const uint32_t nA = __ldg(&sets[ida].main.n), nB = __ldg(&sets[idb].main.n);
    const uint32_t pA = __ldg(&sets[ida].pal.n), pB = __ldg(&sets[idb].pal.n);
    if (both_strands) {
        // the reference's sets hold both strands: |S| = 2|C| - P, I = 2|C_A n C_B| - P(C_A n C_B)
        I = 2 * c - cp;
        sa = 2ull * nA - pA;
        sb = 2ull * nB - pB;
    } else {
        I = c;
        sa = nA;
        sb = nB;
    }
    I += li;
    sa += la;
    sb += lb;
    dist = 1.0;
    const double similarity = (double)I;
    if (similarity > 0) {
        // (this.size() + other.size()) is a Java int addition
        const int32_t sum = (int32_t)((uint32_t)sa + (uint32_t)sb);
        const double uni = (double)sum - similarity;
        dist = 1.0 - similarity / uni;
    }
}

// everything it reads is constant while kernel 5 runs: read-only cache loads
__device__ __forceinline__ void PairCounts::value(uint64_t t, uint32_t ida, uint32_t idb, uint64_t &I, uint64_t &sa,
                                                  uint64_t &sb, double &dist) const {
    pair_result(sets, ida, idb, __ldg(counts + t), pal_counts ? __ldg(pal_counts + t) : 0, lit_inter ? __ldg(lit_inter + t) : 0,
                lit_size ? __ldg(lit_size + ida) : 0, lit_size ? __ldg(lit_size + idb) : 0, both, I, sa, sb, dist);
}

__global__ void __launch_bounds__(256) k_epilogue(PairSource src, PairCounts pc, EpilogueOut out) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= src.count) return;
    uint32_t ida, idb;
    decode_pair(src, t, ida, idb);
    uint64_t I, sa, sb;
    double d;
    pc.value(t, ida, idb, I, sa, sb, d);
    if (out.inter) out.inter[t] = I;
    if (out.dist) out.dist[t] = d;
    if (out.contain_a) out.contain_a[t] = sa ? (double)I / (double)sa : 0.0;
    if (out.contain_b) out.contain_b[t] = sb ? (double)I / (double)sb : 0.0;
}

// ---- kernel 5, selection forms: only the chosen pairs leave the device ------------------------------------------
// Both compute every pair with decode_pair + PairCounts::value, so a selected pair's inter and dist are the dense call's.
//
// Within: pairs with dist <= max_dist, compacted in enumeration order.  A CTA owns a tile of SEL_TILE consecutive
// pairs; pass 1 counts its hits, one CTA scans the tile totals (exclusive offsets + the launch total), and pass 2
// recomputes the tile and writes each hit at tile offset + ballot/popc rank.  No atomics, so the order and the
// output are deterministic.  Hits at positions >= cap are counted but not written.
constexpr int SEL_THREADS = 256, SEL_ITEMS = 8;
constexpr uint64_t SEL_TILE = (uint64_t)SEL_THREADS * SEL_ITEMS;

uint64_t select_within_ctas(uint64_t count) { return (count + SEL_TILE - 1) / SEL_TILE; }

template <bool WRITE>
__global__ void __launch_bounds__(SEL_THREADS)
    k_select_within(PairSource src, PairCounts pc, double max_dist, uint32_t a_base, uint64_t cap, HitsOut out,
                    unsigned long long *__restrict__ cta) {
    __shared__ uint32_t s_warp[SEL_THREADS / 32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t tile0 = (uint64_t)blockIdx.x * SEL_TILE;
    unsigned long long base = WRITE ? cta[blockIdx.x] : 0ull;
    uint32_t mine = 0;
    for (int it = 0; it < SEL_ITEMS; it++) {
        const uint64_t t = tile0 + (uint64_t)it * SEL_THREADS + threadIdx.x;
        bool hit = false;
        uint32_t ida = 0, idb = 0;
        uint64_t I = 0;
        double d = 1.0;
        if (t < src.count) {
            decode_pair(src, t, ida, idb);
            uint64_t sa, sb;
            pc.value(t, ida, idb, I, sa, sb, d);
            hit = d <= max_dist;
        }
        if (!WRITE) {
            mine += hit ? 1u : 0u;
            continue;
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < SEL_THREADS / 32; w++) {
            const uint32_t v = s_warp[w];
            before += w < (int)warp ? v : 0u;
            total += v;
        }
        __syncthreads();  // s_warp is rewritten by the next item
        if (hit) {
            const unsigned long long at = base + before + __popc(bal & ((1u << lane) - 1u));
            if (at < cap) {
                const bool rect = src.mode == PAIRS_RECT;
                if (out.a) out.a[at] = rect ? a_base + (uint32_t)(t / src.n) : ida;
                if (out.b) out.b[at] = rect ? (uint32_t)(t % src.n) : idb;
                if (out.inter) out.inter[at] = I;
                if (out.dist) out.dist[at] = d;
            }
        }
        base += total;
    }
    if (!WRITE) {
        mine = __reduce_add_sync(0xffffffffu, mine);
        if (lane == 0) s_warp[warp] = mine;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t sum = 0;
            for (int w = 0; w < SEL_THREADS / 32; w++) sum += s_warp[w];
            cta[blockIdx.x] = sum;
        }
    }
}

// tile hit counts -> exclusive offsets in place, and the launch total (one CTA; thread x owns a contiguous run of tiles)
__global__ void __launch_bounds__(1024) k_select_scan(unsigned long long *__restrict__ cta, uint64_t n, unsigned long long *__restrict__ total) {
    __shared__ unsigned long long s_w[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t per = (n + 1023) / 1024;
    const uint64_t lo = min(n, (uint64_t)threadIdx.x * per), hi = min(n, lo + per);
    unsigned long long sum = 0;
    for (uint64_t i = lo; i < hi; i++) sum += cta[i];
    unsigned long long x = sum;  // inclusive scan over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= (uint32_t)o) x += y;
    }
    if (lane == 31) s_w[warp] = x;
    __syncthreads();
    if (warp == 0) {
        unsigned long long v = s_w[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= (uint32_t)o) v += y;
        }
        s_w[lane] = v;
    }
    __syncthreads();
    unsigned long long run = x - sum + (warp ? s_w[warp - 1] : 0ull);
    for (uint64_t i = lo; i < hi; i++) {
        const unsigned long long v = cta[i];
        cta[i] = run;
        run += v;
    }
    if (threadIdx.x == 1023) *total = run;
}

cudaError_t launch_select_within(PairSource src, const PairCounts &pc, double max_dist, uint32_t a_base, uint64_t cap,
                                 HitsOut out, unsigned long long *cta, unsigned long long *total, cudaStream_t s) {
    if (src.count == 0) return cudaMemsetAsync(total, 0, sizeof(unsigned long long), s);
    const uint64_t blocks = select_within_ctas(src.count);
    k_select_within<false><<<(unsigned)blocks, SEL_THREADS, 0, s>>>(src, pc, max_dist, a_base, cap, out, cta);
    k_select_scan<<<1, 1024, 0, s>>>(cta, blocks, total);
    if (cap) k_select_within<true><<<(unsigned)blocks, SEL_THREADS, 0, s>>>(src, pc, max_dist, a_base, cap, out, cta);
    return cudaGetLastError();
}

// Nearest: one CTA per query row of a PAIRS_RECT launch.  Slots [0, 256) of shared memory hold the row's best list
// (sorted by (distance bits, reference position); distances are non-negative, so their IEEE bits order like the
// values), slots [256, 512) the candidates of one round of 256 references: a reference is a candidate when it is
// within max_dist and beats the current k-th best.  A round with candidates ends with a bitonic sort of all 512
// slots, after which slots >= k are cleared.  Nothing leaves the CTA until the row is done.
constexpr int NEAR_THREADS = 256, NEAR_SLOTS = 512;
constexpr unsigned long long NEAR_NONE = ~0ull;  // sorts after every distance

// bitonic sort of the 512 slots by (distance bits, position), then slots >= k are cleared; the caller synchronises
// before it reads the list
__device__ __forceinline__ void near_sort_keep(unsigned long long *s_key, unsigned long long *s_inter, uint32_t *s_pos,
                                               uint32_t k, uint32_t tid) {
    for (uint32_t size = 2; size <= NEAR_SLOTS; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            const uint32_t i = (tid / stride) * 2u * stride + (tid % stride), l = i + stride;
            const bool up = (i & size) == 0;
            const unsigned long long ki = s_key[i], kl = s_key[l];
            const uint32_t pi = s_pos[i], pl = s_pos[l];
            const bool gt = ki > kl || (ki == kl && pi > pl);
            if (gt == up) {
                s_key[i] = kl, s_key[l] = ki;
                s_pos[i] = pl, s_pos[l] = pi;
                const unsigned long long t2 = s_inter[i];
                s_inter[i] = s_inter[l], s_inter[l] = t2;
            }
            __syncthreads();
        }
    }
    for (uint32_t i = k + tid; i < NEAR_SLOTS; i += NEAR_THREADS) {
        s_key[i] = NEAR_NONE;
        s_inter[i] = 0;
        s_pos[i] = 0xFFFFFFFFu;
    }
}

// list slots [0, k) -> row `row` of out (k <= NEAR_THREADS: thread i writes slot i); unused slots as gkd.h documents
__device__ __forceinline__ void near_write(const unsigned long long *s_key, const unsigned long long *s_inter,
                                           const uint32_t *s_pos, uint32_t k, uint32_t tid, uint32_t row, NearestOut out) {
    const bool valid = tid < k && s_pos[tid] != 0xFFFFFFFFu;
    if (tid < k) {
        const uint64_t o = (uint64_t)row * k + tid;
        if (out.ref_pos) out.ref_pos[o] = s_pos[tid];
        if (out.inter) out.inter[o] = valid ? s_inter[tid] : 0ull;
        if (out.dist) out.dist[o] = valid ? __longlong_as_double((long long)s_key[tid]) : -1.0;
    }
    const int found = __syncthreads_count(valid);
    if (tid == 0 && out.n_found) out.n_found[row] = (uint32_t)found;
}

__global__ void __launch_bounds__(NEAR_THREADS)
    k_select_nearest(PairSource src, PairCounts pc, double max_dist, uint32_t k, int exclude_self, NearestOut out) {
    __shared__ unsigned long long s_key[NEAR_SLOTS];
    __shared__ unsigned long long s_inter[NEAR_SLOTS];
    __shared__ uint32_t s_pos[NEAR_SLOTS];
    __shared__ uint32_t s_n;
    const uint32_t tid = threadIdx.x, row = blockIdx.x, nr = src.n;
    for (uint32_t i = tid; i < NEAR_SLOTS; i += NEAR_THREADS) {
        s_key[i] = NEAR_NONE;
        s_inter[i] = 0;
        s_pos[i] = 0xFFFFFFFFu;
    }
    if (tid == 0) s_n = 0;
    __syncthreads();
    unsigned long long thr = NEAR_NONE;  // distance bits of the k-th best so far
    for (uint32_t j0 = 0; j0 < nr; j0 += NEAR_THREADS) {
        const uint32_t j = j0 + tid;
        if (j < nr) {
            const uint64_t t = (uint64_t)row * nr + j;
            uint32_t ida, idb;
            decode_pair(src, t, ida, idb);
            if (!(exclude_self && ida == idb)) {
                uint64_t I, sa, sb;
                double d;
                pc.value(t, ida, idb, I, sa, sb, d);
                const unsigned long long key = (unsigned long long)__double_as_longlong(d);
                // a later reference with the k-th best distance loses the tie: strictly smaller only
                if (d <= max_dist && key < thr) {
                    const uint32_t slot = NEAR_THREADS + atomicAdd(&s_n, 1u);
                    s_key[slot] = key;
                    s_inter[slot] = I;
                    s_pos[slot] = j;
                }
            }
        }
        __syncthreads();
        const uint32_t n_cand = s_n;
        __syncthreads();  // everyone has read s_n before it is reset
        if (n_cand == 0) continue;
        near_sort_keep(s_key, s_inter, s_pos, k, tid);
        if (tid == 0) s_n = 0;
        __syncthreads();
        thr = s_key[k - 1];
    }
    near_write(s_key, s_inter, s_pos, k, tid, row, out);
}

cudaError_t launch_select_nearest(PairSource src, uint32_t rows, const PairCounts &pc, double max_dist, uint32_t k,
                                  int exclude_self, NearestOut out, cudaStream_t s) {
    if (rows == 0) return cudaSuccess;
    k_select_nearest<<<rows, NEAR_THREADS, 0, s>>>(src, pc, max_dist, k, exclude_self, out);
    return cudaGetLastError();
}

// Nearest, accumulating form: per-target lists of k slots that live in HBM (`state`, the layout of NearestOut) across
// the chunks and launches of one call.  One CTA per target loads its list into the slots [0, 256) of the layout above,
// gathers the target's pairs of this launch in rounds of 256 candidates and writes the list back if a round changed it.
//   UPPER chunk [first, first+count) with rows i0..i1: target i takes its row segment (i, j), target j the column
//     entries (i, j), i0 <= i < j, whose position is inside the chunk.  Targets are i0..n-1.
//   RECT launch: target = reference column j; it takes counts[row * nr + j] of every query row, neighbour a_base + row.
// A candidate enters when (distance bits, position) is below the k-th entry: unlike k_select_nearest, positions do not
// arrive in ascending order (the column side of a later chunk may tie the k-th distance with a smaller position).
// The lists outlive the launch, so a launch whose block join overflowed (it is redone by the merge kernel) must not
// touch them: the flag is read here, on the stream after kernel 4, rather than on the host afterwards.
__device__ __forceinline__ uint64_t upper_row_start(uint64_t i, uint64_t n) { return i * (2 * n - i - 1) / 2; }

__global__ void __launch_bounds__(NEAR_THREADS)
    k_nearest_absorb(PairSource src, PairCounts pc, double max_dist, uint32_t k, int exclude_self, uint32_t i0, uint32_t i1,
                     uint32_t a_base, const uint32_t *__restrict__ join_err, NearestOut state) {
    if (join_err && *join_err) return;
    __shared__ unsigned long long s_key[NEAR_SLOTS];
    __shared__ unsigned long long s_inter[NEAR_SLOTS];
    __shared__ uint32_t s_pos[NEAR_SLOTS];
    __shared__ uint32_t s_n;
    const uint32_t tid = threadIdx.x;
    const bool upper = src.mode == PAIRS_UPPER;
    const uint32_t tg = (upper ? i0 : 0u) + blockIdx.x;
    const uint64_t n = src.n, first = src.first, end = src.first + src.count;
    uint64_t rs = 0, row_lo = 0;
    uint32_t n_row = 0, n_col;
    if (upper) {
        rs = upper_row_start(tg, n);
        if (tg <= i1) {
            const uint64_t lo = max(rs, first), hi = min(rs + (n - tg - 1), end);
            if (hi > lo) row_lo = lo, n_row = (uint32_t)(hi - lo);
        }
        n_col = tg > i0 ? min(i1, tg - 1) - i0 + 1 : 0u;
    } else {
        n_col = (uint32_t)(src.count / src.n);
    }
    const uint32_t total = n_row + n_col;
    if (total == 0) return;

    const uint64_t base = (uint64_t)tg * k;
    for (uint32_t i = tid; i < NEAR_SLOTS; i += NEAR_THREADS) {
        const uint32_t p = i < k ? state.ref_pos[base + i] : 0xFFFFFFFFu;
        const bool used = p != 0xFFFFFFFFu;
        s_key[i] = used ? (unsigned long long)__double_as_longlong(state.dist[base + i]) : NEAR_NONE;
        s_inter[i] = used ? state.inter[base + i] : 0ull;
        s_pos[i] = p;
    }
    if (tid == 0) s_n = 0;
    __syncthreads();
    unsigned long long thr = s_key[k - 1];
    uint32_t thr_pos = s_pos[k - 1];
    bool changed = false;
    for (uint32_t u0 = 0; u0 < total; u0 += NEAR_THREADS) {
        const uint32_t u = u0 + tid;
        bool have = false;
        uint64_t t = 0;
        uint32_t ida = 0, idb = 0, nb = 0;
        if (u < n_row) {  // (tg, j): the row segment is contiguous
            const uint64_t p = row_lo + u;
            t = p - first;
            ida = tg, idb = tg + 1 + (uint32_t)(p - rs), nb = idb;
            have = true;
        } else if (u < total && upper) {  // (i, tg), i < tg: one entry per earlier row
            const uint32_t i = i0 + (u - n_row);
            const uint64_t p = upper_row_start(i, n) + (tg - i - 1);
            if (p >= first && p < end) {
                t = p - first;
                ida = i, idb = tg, nb = i;
                have = true;
            }
        } else if (u < total) {  // RECT: query row u against reference tg
            t = (uint64_t)u * src.n + tg;
            decode_pair(src, t, ida, idb);
            nb = a_base + u;
            have = !(exclude_self && ida == idb);
        }
        if (have) {
            uint64_t I, sa, sb;
            double d;
            pc.value(t, ida, idb, I, sa, sb, d);
            const unsigned long long key = (unsigned long long)__double_as_longlong(d);
            if (d <= max_dist && (key < thr || (key == thr && nb < thr_pos))) {
                const uint32_t slot = NEAR_THREADS + atomicAdd(&s_n, 1u);
                s_key[slot] = key;
                s_inter[slot] = I;
                s_pos[slot] = nb;
            }
        }
        __syncthreads();
        const uint32_t n_cand = s_n;
        __syncthreads();
        if (n_cand == 0) continue;
        near_sort_keep(s_key, s_inter, s_pos, k, tid);
        if (tid == 0) s_n = 0;
        __syncthreads();
        thr = s_key[k - 1];
        thr_pos = s_pos[k - 1];
        changed = true;
    }
    if (changed) near_write(s_key, s_inter, s_pos, k, tid, tg, state);
}

cudaError_t launch_nearest_absorb(PairSource src, const PairCounts &pc, double max_dist, uint32_t k, int exclude_self,
                                  uint32_t a_base, const uint32_t *join_err, NearestOut state, cudaStream_t s) {
    if (src.count == 0) return cudaSuccess;
    uint32_t i0 = 0, i1 = 0, j = 0, targets = src.n;
    if (src.mode == PAIRS_UPPER) {
        upper_pair(src.first, src.n, i0, j);
        upper_pair(src.first + src.count - 1, src.n, i1, j);
        targets = src.n - i0;
    }
    k_nearest_absorb<<<targets, NEAR_THREADS, 0, s>>>(src, pc, max_dist, k, exclude_self, i0, i1, a_base, join_err, state);
    return cudaGetLastError();
}

// Clusters, accumulating form: single linkage at max_dist as a union-find forest `parent` over the call's nodes in HBM,
// kept across the chunks and launches of one call like the nearest lists.  Invariant parent[x] <= x, so a root is the
// smallest node of its tree and the flattened forest is the label the API returns.
//   link:  find both roots, hook the larger under the smaller with a CAS that succeeds only while it is still a root;
//          a failed CAS means another thread hooked that root, so the loop resumes from the value it returned.
//   find:  path halving; its stores only ever write a smaller ancestor of the same tree (a non-root stays a
//          non-root, a root is only written by the CAS), so racing finds and links keep the forest valid.
// Loads go through device-scope relaxed atomics: a plain load may be served by a stale L1 line of another SM's write.
// No thread waits for another, so every loop ends.  Like k_nearest_absorb, a launch whose block join overflowed links
// nothing (the chunk is redone by the merge kernel): an overflowed attempt could only undercount, but this way every
// link is decided on final counts.
constexpr int CLUSTER_THREADS = 256;

__device__ __forceinline__ uint32_t uf_load(uint32_t *p) {
    return cuda::atomic_ref<uint32_t, cuda::thread_scope_device>(*p).load(cuda::memory_order_relaxed);
}

__device__ __forceinline__ void uf_store(uint32_t *p, uint32_t v) {
    cuda::atomic_ref<uint32_t, cuda::thread_scope_device>(*p).store(v, cuda::memory_order_relaxed);
}

__device__ __forceinline__ uint32_t uf_find(uint32_t *__restrict__ parent, uint32_t x) {
    uint32_t p = uf_load(parent + x);
    while (p != x) {
        const uint32_t gp = uf_load(parent + p);
        if (gp != p) uf_store(parent + x, gp);
        x = gp;
        p = uf_load(parent + x);
    }
    return x;
}

__device__ __forceinline__ void uf_union(uint32_t *__restrict__ parent, uint32_t a, uint32_t b) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    while (a != b) {
        const uint32_t hi = max(a, b), lo = min(a, b);
        const uint32_t old = atomicCAS(parent + hi, hi, lo);
        if (old == hi) return;
        a = uf_find(parent, old);
        b = uf_find(parent, lo);
    }
}

__global__ void __launch_bounds__(CLUSTER_THREADS)
    k_cluster_link(PairSource src, PairCounts pc, double max_dist, uint32_t a_base, uint32_t b_base,
                   const uint32_t *__restrict__ join_err, uint32_t *__restrict__ parent) {
    if (join_err && *join_err) return;
    const bool rect = src.mode == PAIRS_RECT;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < src.count; t += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t ida, idb;
        decode_pair(src, t, ida, idb);
        uint64_t I, sa, sb;
        double d;
        pc.value(t, ida, idb, I, sa, sb, d);
        if (!(d <= max_dist)) continue;
        if (rect) uf_union(parent, a_base + (uint32_t)(t / src.n), b_base + (uint32_t)(t % src.n));
        else uf_union(parent, ida, idb);
    }
}

// the root of x without writing: every value read is an ancestor of x or its root, so the walk ends at the root
__device__ __forceinline__ uint32_t uf_root(uint32_t *__restrict__ parent, uint32_t x) {
    for (uint32_t p = uf_load(parent + x); p != x; p = uf_load(parent + x)) x = p;
    return x;
}

// every node to its root, *n_roots += roots.  The labels live in `parent`, so only thread x writes parent[x], and it
// writes its root: a path-halving find here could store a stale ancestor over a node's label after that node's own
// thread had written the root.
__global__ void __launch_bounds__(CLUSTER_THREADS) k_cluster_flatten(uint32_t *__restrict__ parent, uint32_t n, uint32_t *__restrict__ n_roots) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    bool root = false;
    if (x < n) {
        const uint32_t r = uf_root(parent, x);
        root = r == x;
        if (!root) uf_store(parent + x, r);
    }
    const uint32_t roots = __popc(__ballot_sync(0xffffffffu, root));
    if ((threadIdx.x & 31) == 0 && roots) atomicAdd(n_roots, roots);
}

__global__ void __launch_bounds__(CLUSTER_THREADS) k_cluster_init(uint32_t *__restrict__ parent, uint32_t n) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < n) parent[x] = x;
    if (x == n) parent[x] = 0;  // the root counter of k_cluster_flatten
}

cudaError_t launch_cluster_init(uint32_t *parent, uint32_t n, cudaStream_t s) {
    k_cluster_init<<<(unsigned)(((uint64_t)n + CLUSTER_THREADS) / CLUSTER_THREADS), CLUSTER_THREADS, 0, s>>>(parent, n);
    return cudaGetLastError();
}

cudaError_t launch_cluster_link(PairSource src, const PairCounts &pc, double max_dist, uint32_t a_base, uint32_t b_base,
                                const uint32_t *join_err, uint32_t *parent, cudaStream_t s) {
    if (src.count == 0) return cudaSuccess;
    const uint64_t need = (src.count + CLUSTER_THREADS - 1) / CLUSTER_THREADS;  // grid-stride beyond 8192 CTAs
    const uint64_t blocks = need < 8192 ? need : 8192;
    k_cluster_link<<<(unsigned)blocks, CLUSTER_THREADS, 0, s>>>(src, pc, max_dist, a_base, b_base, join_err, parent);
    return cudaGetLastError();
}

cudaError_t launch_cluster_flatten(uint32_t *parent, uint32_t n, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    k_cluster_flatten<<<(unsigned)(((uint64_t)n + CLUSTER_THREADS - 1) / CLUSTER_THREADS), CLUSTER_THREADS, 0, s>>>(parent, n,
                                                                                                                  parent + n);
    return cudaGetLastError();
}

// Linkage, Boruvka form: the minimum spanning forest of an edge list (a chunk's edges within max_dist, compacted by
// k_select_within, followed by the forest of the earlier chunks) under the strict order (distance bits, min key, max key).
// Every round starts from the components of the previous one (comp[x] = root):
//   edges 0:  every edge between two components offers its distance bits to both roots' best_d (atomicMin);
//   edges 1:  an edge with the winning distance offers its key pair to best_k;
//   edges 2:  the one edge with both (the order is strict) writes its index to best_e;
//   hook:     every root with a best edge hooks under the root at its other end and appends the edge to the new forest;
//             of a mutual pair (both roots chose the same edge) only the larger root hooks, so each edge enters once and
//             the hooks form trees;
//   relabel:  each root jumps its own hook pointer to its tree's root (only thread x writes hook[x]; every value read
//             is an ancestor, so the walk ends), every node takes its root's final root, and best_* are reset.
// Every component with a crossing edge merges in a round, so ceil(log2 nodes) rounds finish the forest.  The host
// queues them all; a round whose predecessor hooked nothing (hooked[r] == 0) exits at once.
constexpr int LINK_THREADS = 256;

__device__ __forceinline__ unsigned long long link_load64(unsigned long long *p) {
    return cuda::atomic_ref<unsigned long long, cuda::thread_scope_device>(*p).load(cuda::memory_order_relaxed);
}

// atomicMin only when it can lower the value: most offers lose, and the relaxed load keeps them off the atomic unit
__device__ __forceinline__ void link_offer(unsigned long long *p, unsigned long long v) {
    if (v < link_load64(p)) atomicMin(p, v);
}

__device__ __forceinline__ unsigned long long link_keys(const LinkGraph &g, uint32_t na, uint32_t nb) {
    const uint32_t ka = g.key ? g.key[na] : na, kb = g.key ? g.key[nb] : nb;
    return (unsigned long long)min(ka, kb) << 32 | max(ka, kb);
}

__global__ void __launch_bounds__(LINK_THREADS) k_link_init(LinkState st, uint32_t rounds) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x < st.nodes) {
        st.comp[x] = st.hook[x] = x;
        st.best_d[x] = st.best_k[x] = ~0ull;
        st.best_e[x] = LINK_NONE;
    }
    if (x <= rounds) st.hooked[x] = x == 0 ? 1u : 0u;
    if (x == 0) *st.n_forest = 0;
}

template <int PHASE>
__global__ void __launch_bounds__(LINK_THREADS) k_link_edges(LinkGraph g, LinkState st, uint32_t round) {
    if (st.hooked[round] == 0) return;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < g.n_edges; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t na = g.a[e], nb = g.b[e] + g.b_off;
        const uint32_t ca = st.comp[na], cb = st.comp[nb];
        if (ca == cb) continue;
        const unsigned long long d = (unsigned long long)__double_as_longlong(g.dist[e]);
        if (PHASE == 0) {
            link_offer(st.best_d + ca, d);
            link_offer(st.best_d + cb, d);
            continue;
        }
        const bool at_a = st.best_d[ca] == d, at_b = st.best_d[cb] == d;
        if (!at_a && !at_b) continue;
        const unsigned long long kp = link_keys(g, na, nb);
        if (PHASE == 1) {
            if (at_a) link_offer(st.best_k + ca, kp);
            if (at_b) link_offer(st.best_k + cb, kp);
        } else {
            if (at_a && st.best_k[ca] == kp) st.best_e[ca] = (uint32_t)e;
            if (at_b && st.best_k[cb] == kp) st.best_e[cb] = (uint32_t)e;
        }
    }
}

__global__ void __launch_bounds__(LINK_THREADS) k_link_hook(LinkGraph g, LinkState st, LinkForest f, uint32_t round) {
    if (st.hooked[round] == 0) return;
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t e = LINK_NONE, y = x;
    if (x < st.nodes && st.comp[x] == x) e = st.best_e[x];
    if (e != LINK_NONE) {
        const uint32_t ca = st.comp[g.a[e]], cb = st.comp[g.b[e] + g.b_off];
        y = ca == x ? cb : ca;
        if (st.best_e[y] == e && x < y) e = LINK_NONE;  // mutual: the smaller root stays a root
    }
    const bool hooks = e != LINK_NONE;
    const uint32_t lane = threadIdx.x & 31, mask = __ballot_sync(0xffffffffu, hooks);
    if (!mask) return;
    uint32_t at = 0;
    if (lane == 0) at = atomicAdd(st.n_forest, (uint32_t)__popc(mask));
    at = __shfl_sync(0xffffffffu, at, 0) + __popc(mask & ((1u << lane) - 1u));
    if (!hooks) return;
    st.hook[x] = y;
    f.a[at] = g.a[e];
    f.b[at] = g.b[e];
    f.inter[at] = g.inter[e];
    f.dist[at] = g.dist[e];
    if (lane == __ffs(mask) - 1) st.hooked[round + 1] = 1u;
}

__global__ void __launch_bounds__(LINK_THREADS) k_link_relabel(LinkState st, uint32_t round) {
    if (st.hooked[round + 1] == 0) return;  // nothing merged: the labels stand and the later rounds exit
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= st.nodes) return;
    uint32_t r = st.comp[x];
    if (r == x) {
        for (uint32_t p = uf_load(st.hook + x), gp = uf_load(st.hook + p); gp != p; gp = uf_load(st.hook + p)) {
            p = gp;
            uf_store(st.hook + x, p);
        }
        r = uf_load(st.hook + x);
    } else {
        for (uint32_t p = uf_load(st.hook + r); p != r; p = uf_load(st.hook + r)) r = p;
    }
    st.comp[x] = r;
    st.best_d[x] = st.best_k[x] = ~0ull;
    st.best_e[x] = LINK_NONE;
}

uint64_t link_state_bytes(uint32_t nodes) { return (uint64_t)nodes * (16 + 16) + (LINK_MAX_ROUNDS + 2) * 4 + 16; }

LinkState link_state_at(void *base, uint32_t nodes) {
    LinkState st{};
    char *p = (char *)base;
    st.best_d = (unsigned long long *)p;
    st.best_k = st.best_d + nodes;
    st.best_e = (uint32_t *)(st.best_k + nodes);
    st.comp = st.best_e + nodes;
    st.hook = st.comp + nodes;
    st.key = st.hook + nodes;
    st.hooked = st.key + nodes;
    st.n_forest = st.hooked + LINK_MAX_ROUNDS + 1;
    st.nodes = nodes;
    return st;
}

cudaError_t launch_link_rounds(const LinkGraph &g, const LinkState &st, const LinkForest &f, uint32_t rounds, cudaStream_t s) {
    const unsigned node_blocks = (unsigned)(((uint64_t)st.nodes + LINK_THREADS - 1) / LINK_THREADS);
    const uint64_t need = (g.n_edges + LINK_THREADS - 1) / LINK_THREADS;  // grid-stride beyond 8192 CTAs
    const unsigned edge_blocks = (unsigned)(need < 8192 ? (need ? need : 1) : 8192);
    k_link_init<<<(unsigned)((std::max<uint64_t>(st.nodes, rounds + 1) + LINK_THREADS - 1) / LINK_THREADS), LINK_THREADS, 0, s>>>(st, rounds);
    for (uint32_t r = 0; r < rounds; r++) {
        k_link_edges<0><<<edge_blocks, LINK_THREADS, 0, s>>>(g, st, r);
        k_link_edges<1><<<edge_blocks, LINK_THREADS, 0, s>>>(g, st, r);
        k_link_edges<2><<<edge_blocks, LINK_THREADS, 0, s>>>(g, st, r);
        k_link_hook<<<node_blocks, LINK_THREADS, 0, s>>>(g, st, f, r);
        k_link_relabel<<<node_blocks, LINK_THREADS, 0, s>>>(st, r);
    }
    return cudaGetLastError();
}

// Greedy representative pass (DistanceRepsProcessor.java:185-201, FastaDistanceRepsProcessor.java:124-146): the
// candidate was intersected with every current representative (counts[t] for reps[t]); it joins the list unless
// one of them is within max_dist.  The list and its length live on the device, so the host queues the launches
// of every candidate back to back without reading anything.  The sets have no literal k-mers: gkd_greedy_reps runs the
// dense calls for those.
__global__ void __launch_bounds__(256)
    k_greedy_decide(const SetDesc *__restrict__ sets, uint32_t *__restrict__ reps, uint32_t *__restrict__ n_reps, uint32_t cand,
                    uint32_t visit, uint32_t *__restrict__ counts, uint32_t *__restrict__ pal_counts, int both_strands,
                    double max_dist, uint8_t *__restrict__ is_rep) {
    __shared__ int s_found;
    if (threadIdx.x == 0) s_found = 0;
    __syncthreads();
    const uint32_t n = *n_reps;
    int found = 0;
    for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) {
        uint64_t I, sa, sb;
        double d;
        pair_result(sets, reps[t], cand, counts[t], pal_counts ? pal_counts[t] : 0, 0, 0, 0, both_strands, I, sa, sb, d);
        found |= d <= max_dist ? 1 : 0;
        counts[t] = 0;  // ready for the next candidate
        if (pal_counts) pal_counts[t] = 0;
    }
    if (found) atomicOr(&s_found, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        is_rep[visit] = s_found ? 0 : 1;
        if (!s_found) {
            reps[n] = cand;
            *n_reps = n + 1;
        }
    }
}

cudaError_t launch_greedy_decide(const SetDesc *sets, uint32_t *reps, uint32_t *n_reps, uint32_t cand, uint32_t visit,
                                 uint32_t *counts, uint32_t *pal_counts, int both_strands, double max_dist, uint8_t *is_rep,
                                 cudaStream_t s) {
    k_greedy_decide<<<1, 256, 0, s>>>(sets, reps, n_reps, cand, visit, counts, pal_counts, both_strands, max_dist, is_rep);
    return cudaGetLastError();
}

cudaError_t launch_epilogue(PairSource src, const PairCounts &pc, EpilogueOut out, cudaStream_t s) {
    if (src.count == 0) return cudaSuccess;
    uint64_t blocks = (src.count + 255) / 256;
    k_epilogue<<<(unsigned)blocks, 256, 0, s>>>(src, pc, out);
    return cudaGetLastError();
}

}  // namespace gkd
