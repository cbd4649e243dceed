/*
 * gkd.h -- C ABI of libgkd.so, the B200 (sm_100a) k-mer set distance engine.
 *
 * This is the drop-in boundary for ONE path of SEEDtk/genome.distance: building per-genome k-mer
 * sets and computing pairwise |A n B| and the reference's k-mer distance.  The reference (pure Java)
 * has no FFI for this path; the boundary it exposes upward is the object API of the external
 * org.theseed.sequence classes that its processors call.  Each entry point below names the
 * reference call site(s) it stands behind (paths relative to
 * /root/reference/src/main/java/org/theseed/genome/distance/).  Because one JNI crossing + one launch
 * per SequenceKmers.distance() would be launch-bound, the engine is batched: the Java shim hands it
 * whole genome lists and receives count/distance blocks (see INTEGRATION.md for the JNI binding).
 *
 * Conventions
 *   - plain C types only; no exceptions or exit() cross the ABI; every call returns a gkd_status
 *     (0 = OK, negative = error class) and leaves a message retrievable with gkd_last_error().
 *   - caller owns every buffer it passes; pageable host inputs are consumed (copied) before the call
 *     returns, pinned-host and device sequence text by the next gkd_build_sets (see gkd_add_sequences);
 *     outputs are caller-allocated.  Input sequence pointers may be pageable host, pinned host, or
 *     device memory (detected with cudaPointerGetAttributes).
 *   - genomes/sequences are referred to by dense uint32 ids in insertion order.
 *   - a context is single-caller (not thread-safe); different contexts are independent.
 *   - there is NO CPU fallback: every entry point that computes fails with GKD_ECUDA when no
 *     sm_100-class device is usable.
 */
#ifndef GKD_H
#define GKD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GKD_ABI_VERSION 2

typedef enum gkd_status {
    GKD_OK = 0,
    GKD_EINVAL = -1, /* bad argument; the Java shim maps this to ParseFailureException */
    GKD_EIO = -2,    /* unreadable input; maps to FileNotFoundException / IOException */
    GKD_ENOMEM = -3, /* host or device allocation failed */
    GKD_ECUDA = -4,  /* CUDA runtime / launch failure, or no usable device (sticky: poisons the ctx) */
    GKD_ESTATE = -5  /* call made in the wrong phase (e.g. distances before gkd_build_sets) */
} gkd_status;

/* KmerType members (KmerType.DNA is the only constant visible in-tree, FastaDistanceProcessor.java:89;
 * RNA reads u as t and is otherwise DNA; PROT is ProteinKmers) */
typedef enum gkd_alphabet { GKD_DNA = 0, GKD_PROT = 1, GKD_RNA = 2 } gkd_alphabet;

/* How set sizes and intersections are counted for nucleotide alphabets:
 *   GKD_STRAND_BOTH      - reference semantics: the set holds the k-mers of the sequence and of its
 *                          reverse complement, so |S| = 2|C| - P and I = 2|C_A n C_B| - P_I where C
 *                          are canonical k-mers and P counts reverse-palindromic ones (even K only)
 *   GKD_STRAND_CANONICAL - plain Jaccard over canonical k-mers.  For odd K (no palindromes) the
 *                          distances equal GKD_STRAND_BOTH's bit for bit while |C_A| + |C_B| < 2^30:
 *                          the both-strand Java int sum 2(|C_A| + |C_B|) wraps at 2^31 before the
 *                          canonical sum does (not tested: it needs about 10^9 keys)               */
typedef enum gkd_strand_mode { GKD_STRAND_BOTH = 0, GKD_STRAND_CANONICAL = 1 } gkd_strand_mode;

/* What to do with a nucleotide k-mer that contains a character outside acgt (after lower-casing; u reads
 * as t for RNA).  The reference does not pin this (SURVEY section 8c: "low / unpinned"), so it is a switch:
 *   GKD_AMBIG_SKIP    - the k-mer and its reverse complement are not members of the set
 *   GKD_AMBIG_LITERAL - kept as a literal string (recalled upstream behaviour): the lower-cased window is
 *                       a member and so is its reverse complement, in which the complement of an unknown
 *                       base is 'n'.  Such k-mers are rare, so they live in a per-set side list that is
 *                       built and intersected on the host; requires host-readable or device input text. */
typedef enum gkd_ambig_policy { GKD_AMBIG_SKIP = 0, GKD_AMBIG_LITERAL = 1 } gkd_ambig_policy;

typedef struct gkd_config {
    int32_t device;            /* CUDA device ordinal */
    int32_t k;                 /* k-mer size; 0 = type default (21 DNA/RNA, 8 protein;
                                  FastaDistanceProcessor.java:43,95-96).  DNA/RNA 1..32, protein 1..8 */
    int32_t alphabet;          /* gkd_alphabet */
    int32_t strand_mode;       /* gkd_strand_mode */
    uint64_t workspace_bytes;  /* device scratch for set construction (0 = default 8 GiB cap) */
    uint32_t segment_keys;     /* approximate keys (of both sets together) per work item of the intersect
                                  kernel (0 = choose from the workload) */
    int32_t ambig_policy;      /* gkd_ambig_policy (nucleotide alphabets only) */
    uint32_t reserved[6];
} gkd_config;

typedef struct gkd_ctx gkd_ctx;

/* Throughput/byte counters of the last build / distance call (the numbers bench.py reports). */
typedef struct gkd_metrics {
    double pack_ms, encode_ms, sort_ms, unique_ms; /* kernels 1-3, CUDA-event time on the ctx stream */
    double intersect_ms, epilogue_ms;              /* kernels 4-5 */
    double h2d_ms, d2h_ms;                         /* host<->device copies issued by the engine */
    uint64_t residues_packed;   /* bases / residues seen by kernel 1 */
    uint64_t kmer_positions;    /* k-mer positions encoded by kernel 2 */
    uint64_t keys_sorted;       /* keys through the radix sort (kernel 3 input) */
    uint32_t sort_passes;       /* LSD passes per key */
    uint32_t intersect_kernel;  /* kernel 4 variant of the last distance call: 3 = bucket merge on 32-bit low words, 4 = on 64-bit keys, 5 = block join (32 or 64 rows per shared-memory table) */
    uint64_t keys_unique;       /* sum of |C| over the sets built */
    uint64_t pairs;             /* pairs intersected by the last distance call */
    uint64_t intersect_bytes;   /* ALGORITHMIC bytes of the last distance call: 8*(|C_A|+|C_B|) per pair */
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t launches;          /* kernels launched by this ctx since creation */
    uint64_t intersect_launches;
    uint64_t total_pairs;            /* the three "last distance call" figures summed since gkd_create / gkd_reset */
    uint64_t total_intersect_bytes;
    double total_intersect_ms;
    uint64_t agglomerate_rounds;  /* rounds that merged something in the last gkd_*_agglomerate call */
    uint64_t reserved[2];
} gkd_metrics;

/* ---- lifecycle --------------------------------------------------------------------------- */
/* new KmerType/GenomeKmers configuration: K is per-context instead of the reference's static
 * GenomeKmers.setKmerSize / ProteinKmers.setKmerSize (GenomeProcessor.java:86, ProteinKmerReader.java:92) */
int gkd_create(gkd_ctx **out, const gkd_config *cfg);
int gkd_destroy(gkd_ctx *ctx);
/* drop every genome and set but keep device pools warm (used between bench steps) */
int gkd_reset(gkd_ctx *ctx);
/* drop the sets with id >= n_keep (e.g. a streamed column panel that has been intersected) and
 * recycle their arena; ids below n_keep stay valid */
int gkd_truncate(gkd_ctx *ctx, uint32_t n_keep);
/* message of the last failure on ctx (ctx may be NULL for a failed gkd_create) */
const char *gkd_last_error(const gkd_ctx *ctx);
int gkd_abi_version(void);

/* ---- ingest: kernel 1 --------------------------------------------------------------------- */
/* One genome / sequence record from n_contigs pieces; k-mers never span pieces.
 * Pageable host text is consumed before the call returns.  Pinned-host and device text is read by
 * stream-ordered copies: it must stay valid and unchanged until the next gkd_build_sets returns.
 * Stands behind: new GenomeKmers(genome) (GenomeProcessor.java:109,139 - one piece per contig),
 * KmerType.createKmers(seq, K) (FastaDistanceProcessor.java:153,184 - one piece),
 * new ProteinKmers(str) (ProteinKmerReader.java:100-101 - one piece; or one piece per protein for a
 * per-genome protein set).  Pointers may be host or device memory. */
int gkd_add_sequences(gkd_ctx *ctx, const char *const *contigs, const uint64_t *lens, uint32_t n_contigs,
                      uint32_t *out_id);
/* FastaInputStream(File) (FastaDistanceProcessor.java:104-108,119-131): per_record=1 makes each FASTA
 * record a unit (fastaDist); per_record=0 makes the whole file one genome, one contig per record. */
int gkd_add_fasta_file(gkd_ctx *ctx, const char *path, int per_record, uint32_t *first_id, uint32_t *n_added);
/* Sequence.getLabel()/getComment() (FastaDistanceProcessor.java:189-190); "" when not from FASTA */
const char *gkd_label(const gkd_ctx *ctx, uint32_t id);
const char *gkd_comment(const gkd_ctx *ctx, uint32_t id);
uint32_t gkd_count(const gkd_ctx *ctx);
/* attach a label and comment to a set that did not come from a FASTA file (copied) */
int gkd_set_label(gkd_ctx *ctx, uint32_t id, const char *label, const char *comment);

/* ---- set construction: kernels 2 + 3 ------------------------------------------------------- */
/* Build the sorted unique canonical uint64 key set of every genome added since the last build. */
int gkd_build_sets(gkd_ctx *ctx);
/* n_both = the reference's HashSet size (2|C|-P for DNA), n_canonical = |C|, n_palindromic = P */
int gkd_set_size(const gkd_ctx *ctx, uint32_t id, uint64_t *n_both, uint64_t *n_canonical, uint64_t *n_palindromic);
/* copy the keys of one set, sorted ascending, to host memory (cap in keys); *n receives |C|.  (The set is
 * stored in mixed-key order; export un-mixes and sorts, so this is a test / cache path, not a fast one.) */
int gkd_export_set(gkd_ctx *ctx, uint32_t id, uint64_t *keys, uint64_t cap, uint64_t *n);
/* adopt a key array (host or device pointer; copied; any order, duplicates allowed) as a new set.  The
 * keys go through the same mix / sort / unique pass as freshly encoded ones; values outside the key
 * space of the context are dropped. */
int gkd_import_set(gkd_ctx *ctx, const uint64_t *keys, uint64_t n, uint32_t *out_id);
/* same for n_sets arrays stored back to back: set i is keys[offsets[i] .. offsets[i+1]) (offsets is a
 * HOST array of n_sets+1 entries; keys may be host or device memory).  ids first_id ..
 * first_id+n_sets-1 are assigned in order. */
int gkd_import_sets(gkd_ctx *ctx, const uint64_t *keys, const uint64_t *offsets, uint32_t n_sets, uint32_t *first_id);

/* ---- set exchange between contexts / ranks (multi-GPU, SURVEY section 8e) ----------------------------
 * Finished sets live in "arenas": one contiguous device allocation per build batch, sets back to back in
 * id order, each set a position-independent block (bucket offset table + key low words, see DESIGN.md
 * section 3).  A host layer moves whole arenas (or the byte range of consecutive sets) between GPUs with
 * NCCL or peer copies and the receiver ADOPTS the bytes in place: no unpack, no second copy. */
typedef struct gkd_packed_set {
    uint64_t offs_off, lows_off;          /* byte offsets from the arena base: bucket table, key low words */
    uint64_t pal_offs_off, pal_lows_off;  /* same for the palindrome sub-set (even K, both strands); 0 if none */
    uint32_t n, n_pal;                    /* |C| and number of reverse-palindromic members */
    uint32_t level, pal_level;            /* table levels: the tables have 2^level + 1 entries */
} gkd_packed_set;
uint32_t gkd_arena_count(const gkd_ctx *ctx);
/* arena `arena` holds the sets first_id .. first_id+n_sets-1 in [base, base+bytes) on the context's device */
int gkd_arena_info(const gkd_ctx *ctx, uint32_t arena, uint32_t *first_id, uint32_t *n_sets, const void **base,
                   uint64_t *bytes);
/* layout of n_sets consecutive sets of ONE arena, offsets relative to that arena's base */
int gkd_describe_sets(const gkd_ctx *ctx, uint32_t first_id, uint32_t n_sets, gkd_packed_set *table);
/* register n_sets sets whose bytes the caller placed at device address `base` (e.g. a received arena);
 * `table` offsets are relative to `base`.  Nothing is copied: the caller keeps [base, base+bytes) alive and
 * unchanged until the sets are dropped with gkd_truncate / gkd_reset / gkd_destroy.  The sets must come
 * from a context with the same k, alphabet and strand mode. */
int gkd_adopt_sets(gkd_ctx *ctx, const void *base, uint64_t bytes, const gkd_packed_set *table, uint32_t n_sets,
                   uint32_t *first_id);

/* persisted sorted-set cache (".kset"): every set of the context with its label and comment, so a
 * reference panel is built once (SURVEY section 8f row 2).  Loading appends the sets as new ids and
 * fails with GKD_EINVAL if the file was written for a different k / alphabet. */
int gkd_save_sets(gkd_ctx *ctx, const char *path);
int gkd_load_sets(gkd_ctx *ctx, const char *path, uint32_t *first_id, uint32_t *n_loaded);

/* ---- distances: kernels 4 + 5 --------------------------------------------------------------- */
/* All pairs i<j in id order, row-major strict upper triangle of length N*(N-1)/2
 * (FastaDistanceProcessor.runReporter/computePairs :141-162,174-194).  inter receives the reference's
 * similarity() value (both-strand count under GKD_STRAND_BOTH); either output may be NULL. */
int gkd_all_vs_all(gkd_ctx *ctx, uint64_t *inter, double *dist);
/* Every q[i] against every r[j], row-major nq*nr (GenomeProcessor.runReporter :129-147). */
int gkd_query_vs_ref(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr,
                     uint64_t *inter, double *dist);
/* Arbitrary pair list (the primitive the two calls above and the multi-GPU tile sharding use). */
int gkd_pairs(gkd_ctx *ctx, const uint32_t *a, const uint32_t *b, uint64_t n_pairs, uint64_t *inter, double *dist);
/* Sub-range [first, first+count) of the row-major strict-upper-triangle pair enumeration of the
 * first n sets: the per-rank slice of the all-vs-all matrix. */
int gkd_all_vs_all_range(gkd_ctx *ctx, uint32_t n, uint64_t first, uint64_t count, uint64_t *inter, double *dist);
/* The same three calls with every output the epilogue can produce.  Any member may be NULL.
 * contain_a = I / |A| and contain_b = I / |B| are the containment indices of the pair (0 for an empty set);
 * they have no counterpart in the reference (north star: "Jaccard/containment"). */
typedef struct gkd_outputs {
    uint64_t *inter;
    double *dist;
    double *contain_a;
    double *contain_b;
} gkd_outputs;
int gkd_all_vs_all_range_ex(gkd_ctx *ctx, uint32_t n, uint64_t first, uint64_t count, const gkd_outputs *out);
int gkd_query_vs_ref_ex(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr,
                        const gkd_outputs *out);
int gkd_pairs_ex(gkd_ctx *ctx, const uint32_t *a, const uint32_t *b, uint64_t n_pairs, const gkd_outputs *out);
/* Greedy representative selection, pass 1 of DistanceRepsProcessor (:185-201) and the loop of
 * FastaDistanceRepsProcessor (:117-147): the sets order[0..n) are visited in that order; a set becomes a
 * representative unless some CURRENT representative is within max_dist (distance <= max_dist).  is_rep[i]
 * receives 1 when order[i] became a representative, else 0.  The whole pass runs on the device: the
 * representative list and its length stay in HBM and the launches of all candidates are queued back to back
 * (no per-candidate id upload, result download or synchronisation).  Unlike the reference's anyMatch there is no
 * early exit inside a candidate; the result is the same. */
int gkd_greedy_reps(gkd_ctx *ctx, const uint32_t *order, uint32_t n, double max_dist, uint8_t *is_rep);
/* SequenceKmers.distance(other) for one pair (DistanceRepsProcessor.java:101,190;
 * FastaDistanceRepsProcessor.java:128); uni = |A|+|B|-I */
int gkd_pair(gkd_ctx *ctx, uint32_t a, uint32_t b, uint64_t *inter, uint64_t *uni, double *dist);

/* ---- selections: only the chosen pairs leave the device (kernel 5 replaced by a selection epilogue) ----------
 * Pairs whose distance is <= max_dist (the comparison gkd_greedy_reps uses), in the enumeration order of the call.
 * Any array may be NULL; pointers may be host or device memory, like gkd_outputs (host memory only for a
 * GKD_AMBIG_LITERAL context, whose shared literal k-mers are counted on the host). */
typedef struct gkd_hits {
    uint32_t *a;      /* all-vs-all: id i (i < j);  query_vs_ref: position of the query in q */
    uint32_t *b;      /* all-vs-all: id j;          query_vs_ref: position of the reference in r */
    uint64_t *inter;  /* similarity(), as gkd_all_vs_all */
    double *dist;     /* bit-identical to the dense call's double for the same pair */
    uint64_t cap;     /* entries each non-NULL array can hold */
    uint64_t n;       /* out: number of qualifying pairs in the call; only the first min(n, cap) are written */
} gkd_hits;
/* The pairs of gkd_all_vs_all_range within max_dist: dereplication, clustering and relatives over one FASTA file
 * (FastaDistanceProcessor.runReporter :141-194 followed by a distance filter; DistanceRepsProcessor.java:185-201 applies
 * the same <= test one candidate at a time).  A cap smaller than the number of hits is not an error: n is the total,
 * so a caller that got n > cap can call again with cap = n. */
int gkd_all_vs_all_range_within(gkd_ctx *ctx, uint32_t n, uint64_t first, uint64_t count, double max_dist, gkd_hits *out);
/* The pairs of gkd_query_vs_ref within max_dist (GenomeProcessor.runReporter :129-147 with its -m/--maxDist applied). */
int gkd_query_vs_ref_within(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr,
                            double max_dist, gkd_hits *out);
/* For every query, its <= k nearest references with distance <= max_dist: ascending distance, ties broken by the
 * smaller position in r (the left-biased merge of DistanceRepsProcessor :120-122).  Outputs are nq*k row-major;
 * n_found[i] <= k; unused slots hold ref_pos = UINT32_MAX, inter = 0, dist = -1.0.  1 <= k <= 256.
 * exclude_self != 0 skips pairs whose two ids are equal (q == r == all sets gives each set's neighbours).
 * Pass 2 of DistanceRepsProcessor (:220-262, closest representative: k = 1, max_dist = 1.0) and classification
 * against a reference panel.  Any output may be NULL; pointers may be host or device memory as for gkd_hits. */
int gkd_query_vs_ref_nearest(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr,
                             uint32_t k, double max_dist, int exclude_self,
                             uint32_t *ref_pos, uint64_t *inter, double *dist, uint32_t *n_found);

/* k-nearest-neighbour lists: rows*k row-major (n_found: rows).  Any member may be NULL; pointers may be host or device
 * memory as for gkd_hits.  Unused slots hold pos = UINT32_MAX, inter = 0, dist = -1.0 (as gkd_query_vs_ref_nearest). */
typedef struct gkd_neighbors {
    uint32_t *pos;      /* neighbour: set id (all-vs-all) or position in the other list (query_vs_ref) */
    uint64_t *inter;    /* similarity(), as gkd_all_vs_all */
    double *dist;       /* bit-identical to the dense call's double for the same pair */
    uint32_t *n_found;  /* entries used per row, <= k */
} gkd_neighbors;
/* The k-nearest-neighbour graph of one collection (the exact form of what MashProcessor.java:150, getClosest(kmers, n,
 * maxDist), estimates): each of the first n sets gets its <= k nearest OTHER sets within max_dist, ascending distance,
 * ties by the smaller id.  Every pair i < j is intersected once and offered to both of its rows, so this costs half the
 * kernel-4 work of the rectangle and is equal, bit for bit, to gkd_query_vs_ref_nearest(q = r = 0..n-1, exclude_self = 1).
 * 1 <= k <= 256; out may not be NULL. */
int gkd_all_vs_all_nearest(gkd_ctx *ctx, uint32_t n, uint32_t k, double max_dist, const gkd_neighbors *out);
/* One query x reference pass, both directions: q_side = gkd_query_vs_ref_nearest's result; r_side = each reference's
 * <= k nearest queries (positions in q, ties by the smaller position), equal to gkd_query_vs_ref_nearest(r, q).
 * Either side may be NULL, but not both. */
int gkd_query_vs_ref_nearest_ex(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, uint32_t k,
                                double max_dist, int exclude_self, const gkd_neighbors *q_side, const gkd_neighbors *r_side);

/* Single-linkage clusters of the first n sets at max_dist: i and j are in one cluster when a chain of pairs, each with
 * distance <= max_dist (the comparison of gkd_*_within), joins them.  label[i] = the smallest id of i's cluster;
 * *n_clusters (may be NULL; host memory) = number of clusters.  Every pair i < j is intersected once; only the labels
 * leave the device.  label may be host or device memory (host only for GKD_AMBIG_LITERAL).  A negative max_dist gives
 * singletons. */
int gkd_all_vs_all_clusters(gkd_ctx *ctx, uint32_t n, double max_dist, uint32_t *label, uint32_t *n_clusters);
/* The components of one query x reference pass: node i is q[i], node nq + j is r[j] (positions, also when an id is on
 * both sides); the links are the pairs (q[i], r[j]) within max_dist.  q_label[i] / r_label[j] = the smallest node of the
 * component.  Either output may be NULL, not both; host or device memory as for gkd_all_vs_all_clusters. */
int gkd_query_vs_ref_clusters(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr,
                              double max_dist, uint32_t *q_label, uint32_t *r_label);

/* The single-linkage hierarchy of the first n sets up to max_dist: the minimum spanning forest of the pairs i < j with
 * distance <= max_dist (the comparison of gkd_*_within), under the strict order (distance bits, a, b).  out receives its
 * edges in ascending order, which is the merge order of single-linkage agglomeration; a, b (a < b), inter and dist are
 * bit-identical to the dense call's.  out->n = n - (clusters at max_dist); only the first min(n, cap) are written, so
 * cap = n - 1 always suffices.  For every t <= max_dist the components of the edges with dist <= t are the clusters of
 * gkd_all_vs_all_clusters(t).  Any array may be NULL; host or device memory as for gkd_hits.  A negative max_dist gives
 * no edges, max_dist = 1.0 a spanning tree.  Every pair is intersected once.  Device memory: one chunk of compacted
 * edges (24 B x 64 Mi pairs = 1.5 GiB at most) and O(n) forest state (56 B per node); only the forest leaves the
 * device. */
int gkd_all_vs_all_linkage(gkd_ctx *ctx, uint32_t n, double max_dist, gkd_hits *out);
/* The same over one query x reference pass, with the nodes of gkd_query_vs_ref_clusters: node i is q[i], node nq + j is
 * r[j]; an edge (a = i, b = j) joins them when dist(q[i], r[j]) <= max_dist.  Ties are broken by (min key, max key) of
 * the two nodes; the key of node i is q_key[i] and of node nq + j is r_key[j] (host arrays), or the node itself when the
 * array is NULL.  Keys must be distinct (GKD_EINVAL otherwise).  out->n <= nq + nr - 1. */
int gkd_query_vs_ref_linkage(gkd_ctx *ctx, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr,
                             double max_dist, const uint32_t *q_key, const uint32_t *r_key, gkd_hits *out);

/* Complete- and average-linkage (UPGMA) hierarchies of the first n sets up to max_dist.  d(x, y) is the dense call's
 * double; a cluster's label is its smallest id.  Cluster distance v(A, B): complete = max d(a, b); average =
 * S(A, B) / (|A| |B|) with S = the sum of d(a, b) 2^53 as an exact integer (every distance of kernel 5 is a multiple of
 * 2^-53 in [0, 2]; a value that is not fails the call with GKD_EINVAL).  The result is the sequential agglomeration that
 * repeatedly merges the pair of current clusters with the smallest strict key (v, min label, max label) while
 * v <= max_dist: one entry per merge, in that order, with a < b the two labels, height = v (average: v rounded to the
 * nearest double, ties to even) and size = |A| + |B|.  out->n = n - (clusters at max_dist); only the first min(n, cap)
 * entries are written, so cap = n - 1 always suffices.  For every t <= max_dist the clusters at t are the components of
 * the merges with v <= t.  Any array may be NULL; host or device memory as for gkd_hits.  A negative max_dist gives no
 * merges.  Single linkage is gkd_all_vs_all_linkage.
 * Device memory: an n x n matrix of 8 B (complete) or 16 B (average) entries, and O(n) state; the call fails with
 * GKD_ENOMEM, naming the bytes, when that exceeds the free device memory.  Only the merges (32 B each) leave the
 * device. */
typedef enum gkd_link_method { GKD_LINK_COMPLETE = 1, GKD_LINK_AVERAGE = 2 } gkd_link_method;
typedef struct gkd_merges {
    uint32_t *a, *b;  /* labels of the two clusters, a < b */
    double *height;
    uint32_t *size;   /* |A| + |B| */
    uint64_t cap;     /* entries each non-NULL array can hold */
    uint64_t n;       /* out: number of merges; only the first min(n, cap) are written */
} gkd_merges;
/* Every pair i < j is intersected once and its distance written straight into the matrix on the device. */
int gkd_all_vs_all_agglomerate(gkd_ctx *ctx, uint32_t n, int method, double max_dist, gkd_merges *out);
/* The same agglomeration over a caller's row-major strict upper triangle of n(n-1)/2 distances (host or device memory;
 * read, not modified), on the context's device.  n is not tied to the context's sets.  One gkd_all_vs_all serves
 * several methods or thresholds this way. */
int gkd_agglomerate(gkd_ctx *ctx, uint32_t n, const double *dist, int method, double max_dist, gkd_merges *out);

/* ---- several GPUs in one process ------------------------------------------------------------------------
 * A group is one context per listed device (an ordinal may be listed more than once) driven by one host thread
 * per member.  The pair matrix of FastaDistanceProcessor.runReporter (:141-194) is cut into member blocks, the
 * set arenas of the peers a member needs are pulled with peer copies (copy engines over NVLink; staged through
 * the host where peer access is unavailable) while earlier blocks are being intersected, and adopted in place.
 * There is no reduction.  Genomes get global ids in insertion order and must be added member by member
 * (member 0 first), so every member owns a contiguous block of ids; results are indexed by global id exactly
 * like gkd_all_vs_all, so a report produced through a group equals the single-GPU report byte for byte. */
typedef struct gkd_group gkd_group;
int gkd_group_create(gkd_group **out, const gkd_config *cfg /* device field ignored */, const int32_t *devices,
                     uint32_t n_devices);
int gkd_group_destroy(gkd_group *g);
const char *gkd_group_last_error(const gkd_group *g);
uint32_t gkd_group_size(const gkd_group *g);   /* members */
uint32_t gkd_group_count(const gkd_group *g);  /* genomes */
gkd_ctx *gkd_group_member(gkd_group *g, uint32_t member);
int gkd_group_set_panel(gkd_group *g, uint32_t sets_per_panel);  /* sets moved per peer copy (default 128) */
int gkd_group_add_sequences(gkd_group *g, uint32_t member, const char *const *contigs, const uint64_t *lens,
                            uint32_t n_contigs, uint32_t *global_id);
/* every record of a FASTA file, block-distributed over the members (FastaInputStream, per-record units) */
int gkd_group_add_fasta_file(gkd_group *g, const char *path, uint32_t *n_added);
const char *gkd_group_label(const gkd_group *g, uint32_t global_id);
const char *gkd_group_comment(const gkd_group *g, uint32_t global_id);
int gkd_group_build(gkd_group *g);  /* kernels 1-3 on every member concurrently */
/* all pairs i < j over global ids, row-major strict upper triangle (either output may be NULL) */
int gkd_group_all_vs_all(gkd_group *g, uint64_t *inter, double *dist);
/* the group form of gkd_all_vs_all_range_within over all global ids: hits ordered by (a, b), equal to one context's.
 * Every member selects on its own device; only the hits reach the host.  The arrays of out are host memory. */
int gkd_group_all_vs_all_within(gkd_group *g, double max_dist, gkd_hits *out);
/* gkd_all_vs_all_nearest over all global ids (pos holds global ids), equal to one context's result.  Every member
 * selects its diagonal block and both directions of its ring blocks on its own device; the host merges the partial
 * lists of every id.  The arrays of out are host memory, N*k (n_found: N). */
int gkd_group_all_vs_all_nearest(gkd_group *g, uint32_t k, double max_dist, const gkd_neighbors *out);
/* gkd_all_vs_all_clusters over all global ids; equal to one context's labels.  Every member clusters its diagonal block
 * and each ring block on its own device; the host joins the components of every call (O(rows + columns) per call).
 * label is host memory (N entries); *n_clusters may be NULL. */
int gkd_group_all_vs_all_clusters(gkd_group *g, double max_dist, uint32_t *label, uint32_t *n_clusters);
/* gkd_all_vs_all_linkage over all global ids; equal to one context's forest, bit for bit.  Every member computes the
 * forest of its diagonal block and of each ring call (keyed by global id) on its own device; the host merges them by
 * Kruskal in the order (distance bits, global a, global b).  The arrays of out are host memory. */
int gkd_group_all_vs_all_linkage(gkd_group *g, double max_dist, gkd_hits *out);
/* gkd_all_vs_all_agglomerate over all global ids; equal to one context's merges, bit for bit.  The members fill a host
 * triangle of all N(N-1)/2 distances as gkd_group_all_vs_all does (8 B per pair of host memory), then member 0 runs
 * gkd_agglomerate on it (its device needs the matrix of gkd_agglomerate).  The arrays of out are host memory. */
int gkd_group_all_vs_all_agglomerate(gkd_group *g, int method, double max_dist, gkd_merges *out);

/* ---- MinHash sketches (SURVEY section 8f row 4) ---------------------------------------------------------
 * SequenceKmers.hashSet(width) and Sketch.distance (SketchProcessor.java:91, WidthProcessor.java:177-183,
 * MashProcessor.java:116-150).  The implementing classes are external and the hash they use is NOT pinned by
 * the reference tree, so it is a switch: java.lang.String.hashCode of the k-mer string, or murmur3_x86_32
 * (seed 0) of its bytes (build.xml:30 ships a murmur3 jar next to the sequence module). */
typedef enum gkd_sketch_hash { GKD_HASH_JAVA_STRING = 0, GKD_HASH_MURMUR3 = 1 } gkd_sketch_hash;
/* hashSet(width): the `width` (<= 4096) smallest distinct hash codes of the set's k-mer strings (both strands
 * for nucleotide sets under GKD_STRAND_BOTH), ascending as signed Java ints; *n_out <= width entries are
 * written to out (fewer when the set has fewer distinct codes). */
int gkd_hash_set(gkd_ctx *ctx, uint32_t id, uint32_t width, int hash, int32_t *out, uint32_t *n_out);
/* Sketch.distance for a pair list: the sketches of the sets involved are built (hashSet(width)) and compared
 * on the device with the bottom-w estimator: over the w = min(|A|,|B|) smallest codes of the union, m are in
 * both; distance = 1 - m / w (1.0 for an empty signature). */
int gkd_sketch_distances(gkd_ctx *ctx, uint32_t width, int hash, const uint32_t *a, const uint32_t *b, uint64_t n_pairs,
                         double *dist);

/* ---- text + metrics --------------------------------------------------------------------------- */
/* java.lang.Double.toString layout ("" + distance, FastaDistanceProcessor.java:189-190,
 * GenomeProcessor.java:144); returns the length written, excluding the NUL */
int gkd_format_double(double v, char *buf, size_t cap);
int gkd_get_metrics(const gkd_ctx *ctx, gkd_metrics *out);
/* the cudaStream_t every kernel and copy of this context is issued on (so a caller can bracket
 * calls with its own CUDA events) */
void *gkd_stream(const gkd_ctx *ctx);

/* ---- synthetic genomes (bench/test utility; SURVEY section 8d generator) ----------------------- */
/* Writes `len` lower-case bases of descendant `member` of ancestor `family` (per-base substitution
 * probability sub_rate) to dst, which may be host or device memory.  Counter-based, so the host and
 * device paths produce identical bytes. */
int gkd_synth_dna(int device, char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member,
                  double sub_rate);
/* Same for a protein over the 20 standard amino-acid letters. */
int gkd_synth_protein(int device, char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member,
                      double sub_rate);

#ifdef __cplusplus
}
#endif
#endif /* GKD_H */
