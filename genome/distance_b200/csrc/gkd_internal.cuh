// gkd_internal.cuh -- shared constants, layouts and launcher declarations of libgkd.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "gkd.h"

namespace gkd {

// ------------------------------------------------------------------------------------------------
// Layout contracts
// ------------------------------------------------------------------------------------------------
// Key that is never a valid k-mer: the canonical form of t..t is a..a = 0, and eight 0xFF bytes are
// not text.  Used for invalid k-mer slots before the sort.  The key mix below maps it to itself.
constexpr uint64_t KEY_SENTINEL = 0xFFFFFFFFFFFFFFFFull;

// ---- hashed key order ----------------------------------------------------------------------------
// Sets are kept sorted by h = mix(key), a BIJECTION on the key_bits-bit keys (2K bits for DNA/RNA, 8K
// for protein), not by the key itself.  Intersection only needs the two sets in the same total order,
// and the mixed order makes every set uniform over the key space whatever the composition of the
// genome (canonical k-mers are skewed towards a.. / c..; real genomes have GC bias and repeats), so
// equal-width key ranges ("buckets") hold equal shares of every set: the merge partition of kernel 4
// becomes a table lookup instead of a search, and kernel 3 can bucket by the top bits.
// xorshift / odd-multiply rounds are each invertible modulo 2^bits; unmix() undoes them for export.
struct MixParams {
    uint64_t mask;  // 2^bits - 1
    uint64_t fix;   // XOR constant that makes mix(all-ones key) == all-ones: that key is never valid (t..t is
                    // canonically a..a; 0xFF bytes are not text), so no valid h shares the low bits of the sentinel
    int bits;
    int shift;      // ceil(bits / 2): x ^= x >> shift is then its own inverse
};

constexpr uint64_t MIX_C1 = 0xff51afd7ed558ccdull, MIX_C2 = 0xc4ceb9fe1a85ec53ull;
constexpr uint64_t MIX_I1 = 0x4f74430c22a54005ull, MIX_I2 = 0x9cb4b2f8129337dbull;  // inverses modulo 2^64

__host__ __device__ inline uint64_t mix_rounds(uint64_t x, uint64_t mask, int s) {
    x ^= x >> s;
    x = (x * MIX_C1) & mask;
    x ^= x >> s;
    x = (x * MIX_C2) & mask;
    x ^= x >> s;
    return x;
}
__host__ __device__ inline uint64_t mix_key(uint64_t key, const MixParams &p) {
    return mix_rounds(key, p.mask, p.shift) ^ p.fix;
}
__host__ __device__ inline uint64_t unmix_key(uint64_t h, const MixParams &p) {
    uint64_t x = h ^ p.fix;
    x ^= x >> p.shift;
    x = (x * MIX_I2) & p.mask;
    x ^= x >> p.shift;
    x = (x * MIX_I1) & p.mask;
    x ^= x >> p.shift;
    return x;
}
inline MixParams make_mix(int bits) {
    MixParams p;
    p.bits = bits;
    p.mask = bits >= 64 ? ~0ull : ((1ull << bits) - 1ull);
    p.shift = (bits + 1) / 2;
    if (p.shift < 1) p.shift = 1;
    if (p.shift > 63) p.shift = 63;
    p.fix = mix_rounds(p.mask, p.mask, p.shift) ^ p.mask;
    return p;
}

// ---- bucketed set -----------------------------------------------------------------------------------
// A finished set in HBM is
//     offs[0 .. 2^level]  uint32   offs[b] = number of keys whose bucket (top `level` bits of h) is < b
//     lows[0 .. n)        LowT     the keys in ascending h order, each stored as its low 32 bits
//                                  (key_bits <= 42: a bucket at level >= key_bits-32 pins the rest) or
//                                  as the full 64-bit h (wider keys)
// `level` grows with the set so that a bucket holds at most `table_tmax` keys on average; levels are
// nested powers of two, so any two sets can be walked bucket by bucket at the coarser of their levels
// or any level below.  No sentinel tails: every run is bounded by its offsets.  Arrays start on 16-byte
// boundaries and are followed by 16 readable bytes (TMA bulk copies move whole 16-byte units).
struct SubSet {
    const void *lows;
    const uint32_t *offs;
    uint32_t n;
    uint32_t level;
};
// main = the canonical keys; pal = its reverse-palindromic members (even K, both-strand mode only)
struct SetDesc {
    SubSet main, pal;
};

constexpr uint32_t SET_LEVEL_MAX = 26;

__host__ __device__ inline uint32_t ceil_log2_u32(uint32_t q) {  // smallest L with 2^L >= q
    if (q <= 1) return 0;
#ifdef __CUDA_ARCH__
    return 32u - (uint32_t)__clz((int)(q - 1));
#else
    return 32u - (uint32_t)__builtin_clz(q - 1);
#endif
}
// smallest level at which buckets of a set of n keys average at most tmax keys
__host__ __device__ inline uint32_t level_for(uint32_t n, uint32_t tmax) { return ceil_log2_u32((n + tmax - 1) / tmax); }
// lowest usable level of a context: the low word must pin every bit below the bucket bits
__host__ __device__ inline uint32_t level_min(int key_bits, int low_bits) {
    return key_bits > low_bits ? (uint32_t)(key_bits - low_bits) : 0u;
}
__host__ __device__ inline uint32_t level_cap(int key_bits) {
    return (uint32_t)key_bits < SET_LEVEL_MAX ? (uint32_t)key_bits : SET_LEVEL_MAX;
}
__host__ __device__ inline uint32_t set_level(uint32_t n, uint32_t tmax, int key_bits, int low_bits) {
    uint32_t l = level_for(n, tmax), lo = level_min(key_bits, low_bits), hi = level_cap(key_bits);
    if (l < lo) l = lo;
    if (l > hi) l = hi;
    return l;
}
// 32-bit lows serve keys up to 42 bits (DNA/RNA K <= 21, protein K <= 5): the smallest table then has
// 2^10 entries; wider keys keep the whole 64-bit h per key.
inline int low_bits_for(int key_bits) { return key_bits <= 42 ? 32 : 64; }

__host__ __device__ inline uint64_t align16(uint64_t x) { return (x + 15ull) & ~15ull; }

// Packed residue streams.  A genome is one stream: its contigs joined by one separator position.
// DNA/RNA: 2-bit codes a=0 c=1 g=2 t=3, 32 per uint64, position p at bits [2(p%32), +2) of word p/32,
// plus a 1-bit "invalid" mask, 32 per uint32 (non-acgt characters, separators, tail padding).
// Protein: raw bytes, plus the same mask (separators and padding only).
constexpr int PACK_POS_PER_WORD = 32;
constexpr char STREAM_SEPARATOR = 0;  // byte written between contigs in the staged text

// Sort geometry
constexpr int SORT_THREADS = 256;
constexpr int SORT_ITEMS = 16;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;  // 4096 keys per tile
constexpr int RADIX_BITS = 8;               // widest digit of a pass; widths are evened out (42-bit keys: six 7-bit passes)
constexpr int RADIX_BINS = 1 << RADIX_BITS;  // row stride of the per-tile histogram table

// Encode geometry (tile == sort tile so one table of tiles serves both)
constexpr int ENC_THREADS = 256;
constexpr int ENC_PER_THREAD = 16;
constexpr int ENC_TILE = ENC_THREADS * ENC_PER_THREAD;
static_assert(ENC_TILE == SORT_TILE, "encode and sort share the tile table");

// One genome inside a build batch (device-visible).
struct BatchGenome {
    const uint64_t *codes;   // DNA: packed 2-bit words; protein: raw bytes (as uint8_t*)
    const uint32_t *mask;    // invalid bits
    uint64_t raw_off;        // offset (keys) of this genome's slots in the batch key buffers
    uint32_t n_pos;          // stream positions
    uint32_t n_slots;        // k-mer slots = max(0, n_pos - k + 1)
    uint32_t tile_first;     // first tile index of this genome in the batch tile table
    uint32_t n_tiles;
};

// Pair enumeration modes of the intersect kernel
enum PairMode : int { PAIRS_LIST = 0, PAIRS_UPPER = 1, PAIRS_RECT = 2, PAIRS_LIST_VS_ONE = 3 };

struct PairSource {
    int mode;
    uint32_t n;          // UPPER: number of sets; RECT: number of refs (columns); LIST_VS_ONE: the one set id
    uint64_t first;      // UPPER: linear index of the first pair of this call
    uint64_t count;      // pairs in this call (an upper bound when count_ptr is set)
    const uint32_t *a;   // LIST / LIST_VS_ONE: a ids; RECT: query ids; UPPER: nullptr (ids are 0..n-1)
    const uint32_t *b;   // LIST: b ids; RECT: ref ids
    const uint32_t *count_ptr;  // device-resident pair count (greedy pass: the list grows on the device), or nullptr
};

// ------------------------------------------------------------------------------------------------
// Launchers (each returns the cudaError of the launch; all work is stream-ordered)
// ------------------------------------------------------------------------------------------------
// kernel 1
cudaError_t launch_pack_dna(const char *text, uint64_t n_pos, uint64_t *codes, uint32_t *mask, int rna,
                            cudaStream_t s);
cudaError_t launch_pack_prot(const char *text, uint64_t n_pos, uint8_t *codes, uint32_t *mask, cudaStream_t s);
// kernel 2: writes h = mix(canonical key) per k-mer slot (KEY_SENTINEL for invalid slots)
cudaError_t launch_encode(const BatchGenome *genomes, uint32_t n_genomes, uint32_t n_tiles, int alphabet, int k,
                          MixParams mix, uint64_t *keys_out, cudaStream_t s);
// kernel 3: segmented LSD radix sort of each genome's slots, then unique/compact into bucketed sets
struct SortPlan {
    uint32_t n_genomes, n_tiles;
    int key_bits;
    uint64_t *keys_a, *keys_b;      // ping-pong buffers (batch raw size)
    uint32_t *tile_hist;            // [n_tiles][RADIX_BINS] digit counts, reused as offsets
    uint64_t *tile_uniq;            // [n_tiles] packed (pal << 32 | uniq) counts -> exclusive offsets
    uint64_t *genome_counts;        // [n_genomes] packed totals
};
cudaError_t sort_configure();  // per-device function attributes; call once per context after cudaSetDevice
cudaError_t launch_sort(const BatchGenome *genomes, const SortPlan &plan, uint64_t **sorted_out, uint32_t *passes,
                        cudaStream_t s);
cudaError_t launch_unique_count(const BatchGenome *genomes, const SortPlan &plan, const uint64_t *sorted, int alphabet,
                                int k, MixParams mix, cudaStream_t s);
// where the unique pass writes one set (device pointers into the set arena)
struct SetBuild {
    void *lows;          // LowT[n]
    uint32_t *offs;      // uint32[2^level + 1]
    uint64_t *pal_h;     // scratch: full h of the palindromic members (n_pal entries), or nullptr
    void *pal_lows;      // LowT[n_pal]
    uint32_t *pal_offs;  // uint32[2^pal_level + 1]
    uint32_t n, level, n_pal, pal_level;
};
cudaError_t launch_unique_write(const BatchGenome *genomes, const SortPlan &plan, const uint64_t *sorted,
                                const SetBuild *dst, int alphabet, int k, MixParams mix, int low_bits, cudaStream_t s);
// kernel 3, fast path (sort_msd.cu): MSD partition by the top bits of h fused into kernel 2 + one
// in-shared-memory sort per bin
constexpr uint32_t MSD_BIN_AVG = 8192;  // a genome gets 2^p bins, p smallest with n_slots <= MSD_BIN_AVG << p
constexpr uint32_t MSD_BIN_CAP = 9024;  // most keys a bin region / a bin-sort CTA holds (8192 + 8 sigma + 64, rounded)
constexpr uint32_t MSD_MAX_P = 12, MSD_SORT_BITS = 12;  // 4096 sort-buckets per bin: ~1-2 keys each
struct MsdGenome {
    uint32_t bin_first;  // index of the genome's first bin in the batch bin arrays
    uint32_t p;          // bin bits
    uint32_t s;          // sort-bucket bits inside a bin
    uint32_t level;      // table level of the finished set (>= p)
    uint32_t cap;        // keys a bin region of this genome holds
    uint32_t pad_;
    uint64_t bins_off;   // offset (keys) of the genome's bin 0 in the bin buffer; bin b starts at bins_off + b * cap
    void *lows;          // arena destinations
    uint32_t *offs;
};
struct MsdPlan {
    uint32_t n_bins, max_p;
    int key_bits;
    uint64_t *bins;            // fixed-capacity bin regions
    uint32_t *bin_cursor;      // [n_bins] keys in every bin
    unsigned long long *status;  // [n_bins] look-back descriptors
    uint32_t *genome_valid, *genome_maxbin, *genome_unique, *overflow;
};
cudaError_t msd_configure();
// keys_in == nullptr: encode the genomes (kernel 2) straight into the bins; else partition the given keys
cudaError_t launch_encode_scatter(const BatchGenome *genomes, uint32_t n_genomes, uint32_t n_tiles, const MsdGenome *msd,
                                  uint32_t max_p, int alphabet, int k, MixParams mix, const uint64_t *keys_in, uint64_t *bins_out,
                                  uint32_t *bin_cursor, uint32_t *overflow, cudaStream_t s);
cudaError_t launch_msd_totals(const MsdGenome *msd, uint32_t n_genomes, const MsdPlan &plan, cudaStream_t s);
cudaError_t launch_msd_binsort(const MsdGenome *msd, uint32_t n_genomes, const MsdPlan &plan, int low_bits, bool narrow,
                               cudaStream_t s);
// in-place key -> h for imported key arrays (keys outside the key space become KEY_SENTINEL)
cudaError_t launch_mix_keys(uint64_t *keys, uint64_t n, MixParams mix, cudaStream_t s);
// bucketed set -> original keys (unsorted: ascending h order), for export
cudaError_t launch_unmix_set(SubSet set, MixParams mix, int low_bits, uint64_t *keys_out, cudaStream_t s);
cudaError_t launch_fill_u64(uint64_t *dst, uint64_t n, uint64_t value, cudaStream_t s);
// kernels 4 + 5
struct IsectPlan {
    int low_bits;             // 32 or 64: lows type of the context
    uint32_t tmax;            // lane target: a pair is walked at the smallest level where the larger set averages <= tmax keys per bucket
    uint32_t level_min;       // lowest usable level of the context
    uint32_t groups_per_item; // 32-bucket groups per work item
    uint32_t items_per_pair;  // work items reserved per pair (items past a pair's last group exit at once)
};
cudaError_t intersect_configure();  // per-device function attributes; call once per context after cudaSetDevice
uint32_t intersect_default_tmax(int low_bits);  // lane target the kernel is tuned for (sets the table resolution)
uint32_t intersect_warps_per_sm(int low_bits);  // resident warps per SM of the selected configuration
cudaError_t launch_intersect(const SetDesc *sets, PairSource src, int use_pal, const IsectPlan &plan, uint32_t *counts,
                             unsigned long long *work_counter, int n_sms, cudaStream_t s);
// kernel 4, block-join form (join.cu): 32 row sets share one shared-memory hash table per key range
struct JoinClass {          // the row blocks whose sizes call for 2^level key ranges
    uint32_t level;
    uint32_t blk_first;     // first block of the class in rows[] (block b = rows[R b .. R b + R), R = join_cfg_rows(cfg))
    uint32_t n_blocks;
    uint32_t pad_;
    unsigned long long task_first;  // tasks of the class: n_blocks << level, range-major
};
constexpr int JOIN_MAX_CLASSES = 32;
struct JoinPlan {
    int mode;               // PAIRS_UPPER or PAIRS_RECT
    int key_bits;
    int cfg;                // geometry index (join_pick_cfg)
    uint32_t n_cols;        // UPPER: number of sets (columns are set ids 0..n-1); RECT: entries of col_ids
    uint32_t n_classes;
    unsigned long long n_tasks;
    unsigned long long first, count;        // UPPER: linear pair range of the call
    unsigned long long stride_r, stride_c;  // RECT: result slot = row position * stride_r + column position * stride_c
    const uint32_t *rows;     // blocks of R rows: UPPER set ids, RECT positions in row_ids; 0xFFFFFFFF pads a class
    const uint32_t *row_ids;  // RECT: ids of the row side; UPPER: nullptr
    const uint32_t *col_ids;  // RECT: ids of the column side; UPPER: nullptr
    JoinClass cls[JOIN_MAX_CLASSES];
};
cudaError_t join_configure();    // per-device function attributes
int join_pick_cfg(uint32_t n_rows, uint32_t n_cols, int low_bits);  // table geometry for a call (GKD_JOIN_CFG pins one)
uint32_t join_cfg_slots(int cfg);  // slots of the shared-memory table
uint32_t join_cfg_rows(int cfg);   // rows per block (32 or 64)
cudaError_t launch_join(const SetDesc *sets, const JoinPlan &plan, uint32_t *counts, unsigned long long *work_counter,
                        uint32_t *err, int n_sms, cudaStream_t s);
// What kernel 5 values the pairs of a chunk from: kernel 4's counts, indexed by chunk position t like the pair source,
// and the sets.  GKD_AMBIG_LITERAL sets also hold literal k-mers (collected and intersected on the host), which add to
// I and to both sizes.
struct PairCounts {
    const SetDesc *sets;
    const uint32_t *counts;      // |C_A n C_B|
    const uint32_t *pal_counts;  // its palindromic part, or nullptr (not needed)
    const uint32_t *lit_size;    // per set id: literal k-mers of the set, or nullptr (no set of the call has any)
    const uint32_t *lit_inter;   // per chunk position: literal k-mers both sets share, or nullptr (none in the chunk)
    int both;                    // GKD_STRAND_BOTH on nucleotides
#ifdef __CUDACC__
    // I, |A|, |B| and SequenceKmers.distance of pair t, sets ida and idb (intersect.cu)
    __device__ void value(uint64_t t, uint32_t ida, uint32_t idb, uint64_t &I, uint64_t &sa, uint64_t &sb, double &dist) const;
#endif
};
struct EpilogueOut {
    uint64_t *inter;     // similarity() of the reference: |A n B| (both strands under GKD_STRAND_BOTH)
    double *dist;        // SequenceKmers.distance
    double *contain_a;   // I / |A|  (0 when |A| == 0)
    double *contain_b;   // I / |B|
};
cudaError_t launch_epilogue(PairSource src, const PairCounts &pc, EpilogueOut out, cudaStream_t s);
// kernel 5, selection forms (replace launch_epilogue for the within / nearest calls)
struct HitsOut {         // any member may be nullptr
    uint32_t *a, *b;     // UPPER / LIST: set ids; RECT: a_base + query row, reference position
    uint64_t *inter;
    double *dist;
};
constexpr uint32_t NEAREST_MAX_K = 256;
struct NearestOut {      // rows * k row-major, n_found per row; any member may be nullptr
    uint32_t *ref_pos;
    uint64_t *inter;
    double *dist;
    uint32_t *n_found;
};
uint64_t select_within_ctas(uint64_t count);  // entries of the `cta` scratch array of launch_select_within
// pairs with dist <= max_dist compacted in enumeration order into out[0 .. min(hits, cap)); *total = hits of the launch
cudaError_t launch_select_within(PairSource src, const PairCounts &pc, double max_dist, uint32_t a_base, uint64_t cap,
                                 HitsOut out, unsigned long long *cta, unsigned long long *total, cudaStream_t s);
// PAIRS_RECT only: per query row the <= k (<= NEAREST_MAX_K) nearest references within max_dist, ties by position
cudaError_t launch_select_nearest(PairSource src, uint32_t rows, const PairCounts &pc, double max_dist, uint32_t k,
                                  int exclude_self, NearestOut out, cudaStream_t s);
// PAIRS_UPPER or PAIRS_RECT: merge the launch into per-target lists that persist across launches (`state`, every member
// set; targets * k slots, filled with the unused entry before the first launch).  UPPER: every pair (i, j) is offered
// to target i (neighbour j) and target j (neighbour i); RECT: to reference column j, neighbour a_base + query row.
// Writes nothing when join_err (may be nullptr) reads nonzero on the stream.
cudaError_t launch_nearest_absorb(PairSource src, const PairCounts &pc, double max_dist, uint32_t k, int exclude_self,
                                  uint32_t a_base, const uint32_t *join_err, NearestOut state, cudaStream_t s);
// Single-linkage clusters: a union-find forest parent[0, n) in device memory (invariant parent[x] <= x) followed by
// one root counter parent[n].  init: parent[x] = x and the counter 0.  link: every pair within max_dist joins its two
// nodes (UPPER: the set ids; RECT: a_base + query row and b_base + reference column); nothing when join_err (may be
// nullptr) reads nonzero on the stream.  flatten: parent[x] = the smallest node of x's cluster (a read-only walk;
// only thread x writes parent[x]), counter = clusters.
cudaError_t launch_cluster_init(uint32_t *parent, uint32_t n, cudaStream_t s);
cudaError_t launch_cluster_link(PairSource src, const PairCounts &pc, double max_dist, uint32_t a_base, uint32_t b_base,
                                const uint32_t *join_err, uint32_t *parent, cudaStream_t s);
cudaError_t launch_cluster_flatten(uint32_t *parent, uint32_t n, cudaStream_t s);
// The same forest on the host (the group's merge of its members' components): a link hooks the larger root under the
// smaller, so find() is the smallest node of the cluster.
struct HostForest {
    std::vector<uint32_t> parent;
    explicit HostForest(uint32_t n) : parent(n) {
        for (uint32_t x = 0; x < n; x++) parent[x] = x;
    }
    uint32_t find(uint32_t x) {
        while (parent[x] != x) x = parent[x] = parent[parent[x]];
        return x;
    }
    void link(uint32_t a, uint32_t b) {
        a = find(a);
        b = find(b);
        if (a < b) parent[b] = a;
        else if (b < a) parent[a] = b;
    }
};
// Single-linkage hierarchy: the minimum spanning forest (MSF) of the pairs within max_dist under the strict order
// (distance bits, min key, max key) of the two nodes.  One Boruvka pass (launch_link_rounds) replaces the device forest F
// with MSF(F u E) for a graph whose edge list is E_chunk followed by F, copied there by the caller.
struct LinkGraph {
    const uint32_t *a, *b;  // as launch_select_within writes them; the nodes are a and b + b_off
    const uint64_t *inter;
    const double *dist;
    uint64_t n_edges;       // < LINK_NONE
    uint32_t b_off;         // RECT: nq (reference column j is node nq + j); UPPER: 0
    const uint32_t *key;    // key of every node (nullptr: the node itself)
};
constexpr uint32_t LINK_NONE = 0xFFFFFFFFu;
// O(nodes) device state of one call, carved from one buffer of link_state_bytes(nodes)
struct LinkState {
    unsigned long long *best_d, *best_k;  // per component root: the minimum crossing edge's distance bits, then key pair
    uint32_t *best_e;                     // ... and its edge index
    uint32_t *comp, *hook;                // component root of every node; the root a root hooks under in this round
    uint32_t *hooked;                     // hooked[r] != 0: round r - 1 hooked something (hooked[0] = 1)
    uint32_t *n_forest;                   // edges written to the new forest
    uint32_t *key;                        // node keys, when the caller passed any
    uint32_t nodes;
};
struct LinkForest {  // the new forest: <= nodes - 1 edges
    uint32_t *a, *b;
    uint64_t *inter;
    double *dist;
};
constexpr uint32_t LINK_MAX_ROUNDS = 32;
uint64_t link_state_bytes(uint32_t nodes);
LinkState link_state_at(void *base, uint32_t nodes);
// rounds = ceil(log2(nodes)) Boruvka rounds, queued without a host read; a round after one that hooked nothing exits
// at once.  On return *st.n_forest (device) is the number of edges of the new forest f.
cudaError_t launch_link_rounds(const LinkGraph &g, const LinkState &st, const LinkForest &f, uint32_t rounds, cudaStream_t s);
// The same forest on the host: Kruskal in the strict order.  Used to sort the device forest at the end of a call (a
// forest keeps every edge), and for the group's merge of its members' forests.
struct LinkEdge {
    uint64_t dbits, keys;  // distance bits, (min key << 32) | max key
    uint32_t na, nb;       // nodes
    uint32_t a, b;         // as reported
    uint64_t inter;
    double dist;
};
inline LinkEdge link_edge(uint32_t a, uint32_t b, uint64_t inter, double dist, uint32_t na, uint32_t nb, uint32_t ka, uint32_t kb) {
    LinkEdge e{0, (uint64_t)std::min(ka, kb) << 32 | std::max(ka, kb), na, nb, a, b, inter, dist};
    std::memcpy(&e.dbits, &dist, 8);
    return e;
}
// edges <- MSF(edges) over nodes [0, nodes), ascending
inline void host_msf(std::vector<LinkEdge> &edges, uint32_t nodes) {
    std::sort(edges.begin(), edges.end(), [](const LinkEdge &x, const LinkEdge &y) {
        return x.dbits < y.dbits || (x.dbits == y.dbits && x.keys < y.keys);
    });
    HostForest f(nodes);
    size_t kept = 0;
    for (const LinkEdge &e : edges) {
        if (f.find(e.na) == f.find(e.nb)) continue;
        f.link(e.na, e.nb);
        edges[kept++] = e;
    }
    edges.resize(kept);
}
// Complete / average linkage (agglomerate.cu): reciprocal-nearest-neighbour rounds over an n x n matrix in HBM.  Slot
// x holds the cluster labelled x while it is active (size[x] != 0).  Entry (x, y) is one word lo (complete: the max of
// d 2^53) or two words lo, hi (average: S = sum of d 2^53 as a 128-bit integer), stored at [x n + y] and [y n + x].  A
// cluster distance is the exact rational S / (N 2^53) with N = 1 (complete) or |A| |B| (average); pairs are ordered by
// the strict key (S / N, smaller slot, larger slot).
struct AggMerge {  // one merge as the device appends it (unordered): slots a < b, their sizes, S of the pair
    uint32_t a, b, sa, sb;
    uint64_t lo, hi;
};
enum AggCounter : uint32_t { AGG_N_STALE = 0, AGG_N_SURV, AGG_N_MERGES, AGG_ROUND_MERGES, AGG_DONE, AGG_ROUNDS, AGG_BAD, AGG_COUNTERS };
constexpr uint32_t AGG_NONE = 0xFFFFFFFFu;
struct AggState {
    uint32_t n;
    int average;
    uint64_t *lo, *hi;              // the matrix (hi: average only)
    uint32_t *size, *nn, *mate;     // per slot: cluster size (0 = inactive), nearest active slot, merge partner this round
    uint64_t *nn_lo, *nn_hi;        // per slot: S of the nearest pair (N follows from the sizes)
    uint32_t *stale, *surv;         // rows to rescan; survivors (smaller slot of a merge) of this round
    unsigned long long *ctr;        // AggCounter; AGG_BAD: the smallest pair index of an invalid input value (~0: none)
    AggMerge *merges;               // <= n - 1
};
struct AggThreshold {  // v <= max_dist  <=>  S <= (m N) << shift (shift < 0: >> -shift); all: every value passes
    uint64_t m;
    int shift;
    int all;
};
uint64_t agg_state_bytes(uint32_t n, int average);  // the matrix and the O(n) state, in one buffer
AggState agg_state_at(void *base, uint32_t n, int average);
cudaError_t launch_agg_init(const AggState &st, cudaStream_t s);
// An n x n matrix the distances of a call are scattered into, entry (i, j) at [i n + j] and [j n + i]: w = d 2^53 (T =
// uint64_t, agglomeration; hi, when not nullptr, gets the zero high words of the average sums) or w = d (T = double,
// neighbour joining).
template <typename T>
struct Square {
    T *w;
    uint64_t *hi;
    uint32_t n;
    unsigned long long *bad;  // atomicMin of the pair index of a value that is not a valid entry
};
Square<uint64_t> agg_square(const AggState &st);
// entries [first, first + count) of the row-major strict upper triangle of n, as doubles in src (device), into the
// matrix; a value that is not a valid entry (uint64_t: a multiple of 2^-53 in [0, 2]; double: in [0, 2], so not NaN)
// is recorded in *bad.  Nothing when join_err (may be nullptr) reads nonzero on the stream: the chunk is redone.
template <typename T>
cudaError_t launch_square_scatter(const Square<T> &sq, const double *src, uint64_t first, uint64_t count, const uint32_t *join_err,
                                  cudaStream_t s);
// `rounds` rounds queued without a host read; a round after one that merged nothing exits at once (AGG_DONE)
cudaError_t launch_agg_rounds(const AggState &st, AggThreshold thr, uint32_t rounds, int n_sms, cudaStream_t s);
// the device bytes a dense agglomeration may take on the current device: the free memory, capped by the environment
// variable GKD_AGG_MAX_BYTES when it is set (a test pin that reaches the GKD_ENOMEM path at small n)
uint64_t agg_dense_room();
// The O(n) state alone (lo and hi nullptr, complete linkage), for the sparse form below
uint64_t agg_nodes_bytes(uint32_t n);
AggState agg_nodes_at(void *base, uint32_t n);
// Complete linkage from the pairs within max_dist (gkd_*_complete_linkage): the same rounds over one CSR row per slot
// instead of the matrix.  A pair absent from the rows is beyond max_dist, which complete linkage treats as +inf.  Row x
// holds its neighbours in ascending order, nbr[off[x] .. off[x + 1]), and their words w = d 2^53; a pair that stops
// being one (a partner merged away, or the merged distance became +inf) is a tombstone: w = CS_TOMB, its neighbour
// kept so that binary searches stay valid.  24 B per pair (both directions of 4 + 8 B) and 8 B per slot.
constexpr uint64_t CS_TOMB = ~0ull;
struct CsRows {
    const uint64_t *off;
    const uint32_t *nbr;
    uint64_t *w;
};
struct CsList {  // the pairs of a call as they arrive: a < b and w (16 B per pair)
    uint32_t *a, *b;
    uint64_t *w;
};
// count pairs (a[t], b[t], dist[t]) (device) to dst[at + t] as (min, max, d 2^53); a pair with an id >= n, two equal
// ids or a distance that is not a multiple of 2^-53 in [0, 2] stores CS_TOMB and records its index at in *bad
// (atomicMin)
cudaError_t launch_cs_append(const uint32_t *a, const uint32_t *b, const double *dist, uint64_t count, uint32_t n, CsList dst,
                             uint64_t at, unsigned long long *bad, cudaStream_t s);
// scratch bytes of the radix sort of launch_cs_rows
cudaError_t cs_sort_temp_bytes(uint64_t pairs, uint32_t n, size_t &bytes);
// the rows of `pairs` pairs of l: both directions to keys[0] / vals[0] (2 pairs entries each), one radix sort by (row,
// neighbour) that leaves keys[current] / vals[current] sorted (keys[1] may alias l), then off (n + 1) and nbr.  A key
// that occurs twice (a pair listed twice) is recorded in *dup (atomicMin; the caller sets it to ~0 first).
cudaError_t launch_cs_rows(CsList l, uint64_t pairs, uint32_t n, uint64_t *keys[2], uint64_t *vals[2], void *temp,
                           size_t temp_bytes, uint64_t *off, uint32_t *nbr, unsigned long long *dup, int &current,
                           cudaStream_t s);
// launch_agg_rounds over the rows (st from agg_nodes_at)
cudaError_t launch_cs_rounds(const AggState &st, CsRows r, AggThreshold thr, uint32_t rounds, int n_sms, cudaStream_t s);
// S1 / N1 < S2 / N2 exactly (S 128-bit as lo, hi; 192-bit cross products)
__host__ __device__ inline int agg_cmp(uint64_t lo1, uint64_t hi1, uint64_t n1, uint64_t lo2, uint64_t hi2, uint64_t n2) {
    // (lo + hi 2^64) * n as three words w0 + w1 2^64 + w2 2^128
    auto mul = [](uint64_t lo, uint64_t hi, uint64_t n, uint64_t &w0, uint64_t &w1, uint64_t &w2) {
        const unsigned __int128 p0 = (unsigned __int128)lo * n, p1 = (unsigned __int128)hi * n + (uint64_t)(p0 >> 64);
        w0 = (uint64_t)p0;
        w1 = (uint64_t)p1;
        w2 = (uint64_t)(p1 >> 64);
    };
    uint64_t a0, a1, a2, b0, b1, b2;
    mul(lo1, hi1, n2, a0, a1, a2);
    mul(lo2, hi2, n1, b0, b1, b2);
    if (a2 != b2) return a2 < b2 ? -1 : 1;
    if (a1 != b1) return a1 < b1 ? -1 : 1;
    if (a0 != b0) return a0 < b0 ? -1 : 1;
    return 0;
}
// Neighbour joining (nj.cu, gkd_*_nj): the distances of the active clusters in an n x n matrix of doubles in HBM.  The
// r active clusters of a round hold the slots 0 .. r - 1: when g leaves, the last active slot's row, column, sum and
// label move into g's slot, so a round reads only the r x r corner.  label[slot] is the cluster's label (its smallest
// id); Q and its ties are defined on labels, so the layout does not change the result.
// BIONJ (gkd_*_bionj) runs on the same matrix: d(x, y) stays in the upper triangle, [min n + max], and the variance
// V(x, y) lives in the lower one, [max n + min].  The fill writes d to both, so V starts equal to d.
struct NjCand {  // a candidate pair: Q, labels a < b, and the slots of the two clusters
    double q;
    uint32_t a, b, sa, sb;
};
struct NjState {
    uint32_t n;
    double *d;                  // the matrix, entry (x, y) at [x n + y] and [y n + x] (BIONJ: d above, V below)
    double *R;                  // per slot: the row sum of the start, then as the rounds update it
    double *S;                  // BIONJ only (else nullptr): per slot, the row sum of V, kept as R is
    double *lambda;             // BIONJ only: the current round's weight of f, set by the pick
    uint32_t *label;            // per slot
    NjCand *part;               // per CTA of the row scan: its best candidate
    uint32_t *pick;             // the slots of f and g of the current round
    unsigned int *ticket;       // CTAs of the row scan done (the last one picks)
    unsigned long long *bad;    // the smallest pair index of an invalid input value (~0: none)
    uint32_t *ra, *rb;          // the output rows (n - 1 each)
    double *la, *lb;
};
constexpr uint32_t NJ_MAX_CTAS = 2048;  // row-scan CTAs of one round
uint64_t nj_state_bytes(uint32_t n);     // the matrix and the O(n) state, in one buffer
uint64_t bionj_state_bytes(uint32_t n);  // nj_state_bytes plus S and lambda
NjState nj_state_at(void *base, uint32_t n, bool bionj);
inline Square<double> nj_square(const NjState &st) { return {st.d, nullptr, st.n, st.bad}; }
// the start sums and all n - 1 rounds (n >= 2) of NJ, or of BIONJ when st.S is set, queued without a host read:
// 3 (n - 2) + 2 launches; the rows are then in ra, rb, la, lb.  *ticket must be 0 (the scatter's init sets it).
cudaError_t launch_nj_rounds(const NjState &st, int n_sms, cudaStream_t s);
inline uint64_t nj_launches(uint32_t n) { return n < 2 ? 0 : 3ull * (n - 2) + 2; }
// Balanced minimum-evolution NNIs (bme.cu, gkd_*_bme): an M x M table of subtree averages, M = 2n - 2 (n >= 2), whose
// leaf block is d.  The distances are scattered into the NJ matrix placed in the table's rows n .. (not yet built),
// copied into the leaf block, and the NJ or BIONJ rounds (when the call starts from them) run there.
constexpr double BME_EPS = 0x1p-40;  // GKD_BME_EPS
inline uint64_t bme_max_swaps(uint32_t n) { return 4ull * n; }
uint64_t bme_table_bytes(uint32_t n);  // the table, with room for the NJ state inside it
uint64_t bme_state_bytes(uint32_t n);  // the table and the O(n) state, in one buffer
NjState bme_nj_state_at(void *base, uint32_t n, bool bionj);
cudaError_t launch_bme_leaves(void *base, uint32_t n, cudaStream_t s);  // the NJ matrix's d into the leaf block
struct BmeRun {
    std::vector<uint32_t> a, b;  // the rows, as gkd_joins holds them
    std::vector<double> la, lb;
    uint64_t swaps = 0, launches = 0, h2d = 0, d2h = 0;
};
// the search from the tree of the rows (a, b) (host, n - 1 each, checked), then the lengths and the rows
cudaError_t bme_search(void *base, uint32_t n, const uint32_t *a, const uint32_t *b, cudaStream_t s, BmeRun &r);
// greedy representative pass, decision step: candidate `cand` (visit index `visit`) joins reps[0..*n_reps) unless
// some representative is within max_dist; clears the counts it consumed
cudaError_t launch_greedy_decide(const SetDesc *sets, uint32_t *reps, uint32_t *n_reps, uint32_t cand, uint32_t visit,
                                 uint32_t *counts, uint32_t *pal_counts, int both_strands, double max_dist, uint8_t *is_rep,
                                 cudaStream_t s);
// MinHash sketches (sketch.cu)
constexpr uint32_t SKETCH_CAP = 32768;        // candidate codes one CTA sorts in shared memory
constexpr uint32_t SKETCH_MAX_WIDTH = 4096;   // widest signature (the reference's commands use 360 and 2000)
cudaError_t sketch_configure();
cudaError_t launch_sketch_filter(SubSet set, MixParams mix, int low_bits, int alphabet, int k, int both, int kind,
                                 uint32_t thresh, uint32_t *cand, uint32_t cap, uint32_t *n_cand, cudaStream_t s);
cudaError_t launch_sketch_finish(const uint32_t *cand, uint32_t n, uint32_t width, int32_t *out, uint32_t *n_out,
                                 uint32_t *n_distinct, cudaStream_t s);
cudaError_t launch_sketch_distance(const int32_t *sig, const uint32_t *len, uint32_t width, const uint32_t *a,
                                   const uint32_t *b, uint64_t n_pairs, double *dist, cudaStream_t s);
// synthetic data
cudaError_t launch_synth(char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member, double rate,
                         int protein, cudaStream_t s);
void synth_host(char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member, double rate, int protein);

#ifdef __CUDACC__
// which genome of a batch owns tile `tile` (tile_first is ascending)
__device__ __forceinline__ uint32_t find_genome(const BatchGenome *__restrict__ g, uint32_t n, uint32_t tile) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (g[mid].tile_first <= tile) lo = mid;
        else hi = mid;
    }
    return lo;
}

// reverse the order of the 32 two-bit groups of x (base order of a packed k-mer)
__device__ __forceinline__ uint64_t reverse_pairs(uint64_t x) {
    uint64_t y = __brevll(x);
    return ((y >> 1) & 0x5555555555555555ull) | ((y & 0x5555555555555555ull) << 1);
}
#endif

// decode the linear index of the row-major strict upper triangle of an n x n matrix
__host__ __device__ inline void upper_pair(uint64_t t, uint32_t n, uint32_t &i, uint32_t &j) {
    // row i starts at S(i) = i*(2n-i-1)/2 ; solve with a float guess and fix up
    double nn = (double)n - 0.5;
    double disc = nn * nn - 2.0 * (double)t;
    if (disc < 0) disc = 0;
    long long ii = (long long)(nn - sqrt(disc));
    if (ii < 0) ii = 0;
    if (ii > (long long)n - 2) ii = (long long)n - 2;
    auto start = [n](long long r) { return (uint64_t)r * (2ull * n - (uint64_t)r - 1ull) / 2ull; };
    while (ii > 0 && start(ii) > t) ii--;
    while (ii < (long long)n - 2 && start(ii + 1) <= t) ii++;
    i = (uint32_t)ii;
    j = (uint32_t)(t - start(ii)) + i + 1;
}

}  // namespace gkd
