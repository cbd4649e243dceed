// gkd_api.cu -- context, memory plan and the extern "C" ABI of libgkd.so (see include/gkd.h).
// One context = one CUDA device, one stream.  No CPU fallback: without a usable device every
// computing entry point fails with GKD_ECUDA.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "gkd_internal.cuh"

using namespace gkd;

// host FASTA scanner (fasta.cpp)
struct FastaPiece {
    const char *ptr;
    uint64_t len;
};
struct FastaRecord {
    std::string label, comment;
    std::vector<FastaPiece> lines;  // sequence lines, to be concatenated
};
int gkd_parse_fasta_file(const char *path, std::vector<char> &storage, std::vector<FastaRecord> &records,
                         std::string &err);

namespace {

thread_local std::string g_create_error;

constexpr uint64_t PACK_SLAB_BYTES = 256ull << 20;
constexpr uint64_t STAGE_BYTES = 32ull << 20;  // text staged per piece (multiple of 32 positions)
constexpr int N_STAGE = 3;    // pinned bounce buffers (pageable input)
constexpr int N_DSTAGE = 8;   // device staging buffers: the copies may run this many pieces ahead of kernel 1
constexpr uint64_t DEFAULT_WORKSPACE = 8ull << 30;
constexpr uint64_t PAIR_CHUNK = 64ull << 20;  // pairs per distance launch
constexpr uint64_t SET_BLOCK_ALIGN = 256;     // every set block of an arena starts on this boundary

struct Part {  // a run of residue text; new_contig starts a new contig (k-mers do not span contigs)
    const char *ptr;
    uint64_t len;
    bool new_contig;
};

struct GenomeRec {
    std::string label, comment;
    uint64_t n_pos = 0;         // stream positions (residues + separators)
    void *d_codes = nullptr;    // packed stream (slab memory)
    uint32_t *d_mask = nullptr;
    cudaEvent_t ready = nullptr;  // recorded on the ingest stream behind this genome's copy + pack (nullptr: nothing pending)
    bool built = false;
    SetDesc desc{{nullptr, nullptr, 0, 0}, {nullptr, nullptr, 0, 0}};
    gkd_packed_set packed{};    // layout relative to the base of `arena`
    int arena = -1;
    std::vector<uint32_t> lit;  // GKD_AMBIG_LITERAL: sorted ids (context dictionary) of the literal k-mers
};

struct Slab {
    char *base;
    uint64_t size, used;
};

struct DevBuf {  // grow-only scratch buffer
    void *p = nullptr;
    uint64_t cap = 0;
};

struct Arena {  // finished sets of one build / import batch, or an adopted buffer
    char *base;
    uint64_t bytes;  // bytes in use (owned: <= capacity)
    uint64_t capacity;
    uint32_t first_id, n_sets;
    bool owned;
};

struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

}  // namespace

struct gkd_ctx {
    gkd_config cfg{};
    int k = 0;
    int n_sms = 148;
    int key_bits = 0, low_bits = 32;
    uint32_t lvl_min = 0;
    uint32_t table_tmax = 16, isect_tmax = 16;
    MixParams mix{};
    cudaStream_t stream = nullptr;
    // ingest (host->device copies of the text + kernel 1) runs on its own two streams, so the copies of later genomes
    // overlap the set construction of earlier build batches; a batch waits for the `ready` event of its last genome
    cudaStream_t copy_stream = nullptr;  // the copies of the text into the staging buffers
    cudaStream_t pack_stream = nullptr;  // kernel 1 (staging buffer -> packed stream in the slab), behind each copy
    cudaEvent_t slab_ev = nullptr;
    std::vector<cudaEvent_t> ev_pool;
    bool poisoned = false;
    std::string err;

    std::vector<GenomeRec> genomes;
    uint32_t built_upto = 0;

    std::vector<Slab> slabs;
    std::vector<Arena> arenas;                              // live, in id order
    std::vector<std::pair<void *, uint64_t>> free_arenas;  // owned arenas released by reset/truncate, reused best-fit

    char *bounce[N_STAGE] = {nullptr, nullptr, nullptr};
    cudaEvent_t bounce_ev[N_STAGE] = {nullptr, nullptr, nullptr};
    char *stage_dev[N_DSTAGE] = {};
    cudaEvent_t copied[N_DSTAGE] = {}, packed[N_DSTAGE] = {};  // staging buffer s: text has landed / kernel 1 has consumed it
    bool packed_valid[N_DSTAGE] = {};
    int stage_next = 0, dstage_next = 0;

    DevBuf keys_a, keys_b, tile_hist, tile_uniq, genome_counts, batch_genomes, set_build;
    DevBuf d_sets, counts, pal_counts, d_inter, d_dist, d_ca, d_cb, ids_a, ids_b, work_counter;
    DevBuf sk_cand, sk_misc, sk_sig, sk_len, sk_out;
    DevBuf msd_genomes, msd_bins32, msd_bins64, msd_gstat;
    DevBuf gr_reps, gr_flags;
    DevBuf join_rows, join_err;
    DevBuf hit_a, hit_b, sel_cta;  // selection epilogues: hit ids / positions (nearest: ref_pos, n_found), tile offsets + total
    DevBuf nn_pos, nn_inter, nn_dist, nn_found;  // accumulating nearest selection: per-target lists of one call
    DevBuf uf_parent;  // cluster selection: the union-find forest of one call and its root counter
    DevBuf lk_forest, lk_state;  // linkage selection: the spanning forest of one call and its Boruvka state
    DevBuf lit_size, lit_inter;  // GKD_AMBIG_LITERAL: literal k-mers per set, and per pair of a chunk those both sets share
    int isect_algo = 0;  // GKD_ISECT_ALGO: 0 = choose per call, 1 = bucket merge only, 2 = block join whenever it applies
    bool use_msd = true;  // GKD_SORT_ALGO=lsd pins the LSD path
    bool sets_dirty = true;

    std::unordered_map<std::string, uint32_t> lit_dict;  // GKD_AMBIG_LITERAL: literal k-mer -> dense id

    cudaEvent_t ev[8] = {};
    gkd_metrics m{};
};

namespace {

int fail(gkd_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    else g_create_error = buf;
    return code;
}

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            c->poisoned = true;                                                                          \
            return fail(c, e__ == cudaErrorMemoryAllocation ? GKD_ENOMEM : GKD_ECUDA, "%s: %s (%s:%d)", #call, \
                        cudaGetErrorString(e__), __FILE__, __LINE__);                                    \
        }                                                                                                \
    } while (0)

#define CHECK_CTX(c)                                                                   \
    do {                                                                               \
        if (!(c)) return GKD_EINVAL;                                                   \
        if ((c)->poisoned) return fail((c), GKD_ECUDA, "context poisoned by an earlier CUDA error: %s", (c)->err.c_str()); \
    } while (0)

// no C++ exception may cross the ABI (gkd.h): bodies that allocate host memory run inside this guard
#define ABI_GUARD_BEGIN try {
#define ABI_GUARD_END(c)                                                        \
    }                                                                           \
    catch (const std::bad_alloc &) { return fail((c), GKD_ENOMEM, "out of host memory"); } \
    catch (const std::exception &ex__) { return fail((c), GKD_EINVAL, "internal error: %s", ex__.what()); }

int ensure(gkd_ctx *c, DevBuf &b, uint64_t bytes) {
    if (bytes <= b.cap) return GKD_OK;
    if (b.p) CK(cudaFreeAsync(b.p, c->stream));
    b.p = nullptr;
    b.cap = 0;
    uint64_t want = bytes + bytes / 8 + 256;
    CK(cudaMallocAsync(&b.p, want, c->stream));
    b.cap = want;
    return GKD_OK;
}

int slab_alloc(gkd_ctx *c, uint64_t bytes, void **out) {
    bytes = (bytes + 255) & ~255ull;
    for (auto &s : c->slabs) {
        if (s.size - s.used >= bytes) {
            *out = s.base + s.used;
            s.used += bytes;
            return GKD_OK;
        }
    }
    Slab s;
    s.size = std::max<uint64_t>(PACK_SLAB_BYTES, bytes);
    s.used = bytes;
    void *p = nullptr;
    CK(cudaMallocAsync(&p, s.size, c->stream));
    // the ingest stream writes the slab: order it behind the allocation
    CK(cudaEventRecord(c->slab_ev, c->stream));
    CK(cudaStreamWaitEvent(c->pack_stream, c->slab_ev, 0));
    s.base = (char *)p;
    c->slabs.push_back(s);
    *out = s.base;
    return GKD_OK;
}

enum MemKind { MEM_PAGEABLE = 0, MEM_PINNED = 1, MEM_DEVICE = 2 };

MemKind classify(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return MEM_PAGEABLE;
    }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return MEM_DEVICE;
    if (a.type == cudaMemoryTypeHost) return MEM_PINNED;
    return MEM_PAGEABLE;
}

double elapsed(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return ms;
}

// ---- GKD_AMBIG_LITERAL: literal k-mers of one genome (host side) ----------------------------------------
// Restates the recalled upstream behaviour (SURVEY 8c, "low / unpinned"): the lower-cased window that
// holds a character outside acgt is a set member as a literal string, and so is the window of the reverse
// complement strand, where the complement of an unknown base is 'n'.  These strings can never equal a
// pure-acgt k-mer, so they form a side set that is disjoint from the canonical keys.  They are rare
// (2(K-1)+1 distinct strings per run of unknown bases), so each genome keeps the sorted ids of its
// strings in a per-context dictionary and pairs are completed on the host.
inline char fold_nuc(char ch, bool rna) {
    if (ch >= 'A' && ch <= 'Z') ch = (char)(ch + 32);
    if (rna && ch == 'u') ch = 't';
    return ch;
}
inline char complement_nuc(char ch) {
    switch (ch) {
    case 'a': return 't';
    case 'c': return 'g';
    case 'g': return 'c';
    case 't': return 'a';
    default: return 'n';
    }
}

void literal_kmers_of_contig(gkd_ctx *c, const std::string &ct, std::vector<uint32_t> &ids) {
    const size_t k = (size_t)c->k, len = ct.size();
    if (len < k) return;
    std::string fwd(k, ' '), rc(k, ' ');
    size_t next_w = 0;  // first window start not yet emitted
    for (size_t p = 0; p < len; p++) {
        const char ch = ct[p];
        if (ch == 'a' || ch == 'c' || ch == 'g' || ch == 't') continue;
        size_t w0 = p + 1 >= k ? p + 1 - k : 0, w1 = std::min(p, len - k);
        if (w0 < next_w) w0 = next_w;
        for (size_t w = w0; w <= w1; w++) {
            for (size_t i = 0; i < k; i++) {
                fwd[i] = ct[w + i];
                rc[i] = complement_nuc(ct[w + k - 1 - i]);
            }
            for (const std::string *s : {&fwd, &rc}) {
                auto it = c->lit_dict.find(*s);
                uint32_t id;
                if (it == c->lit_dict.end()) {
                    id = (uint32_t)c->lit_dict.size();
                    c->lit_dict.emplace(*s, id);
                } else id = it->second;
                ids.push_back(id);
            }
        }
        if (w1 + 1 > next_w) next_w = w1 + 1;
    }
}

int collect_literals(gkd_ctx *c, const std::vector<Part> &parts, MemKind kind, std::vector<uint32_t> &ids) {
    const bool rna = c->cfg.alphabet == GKD_RNA;
    std::string ct;
    std::vector<char> tmp;
    auto flush = [&]() {
        if (!ct.empty()) literal_kmers_of_contig(c, ct, ids);
        ct.clear();
    };
    for (size_t i = 0; i < parts.size(); i++) {
        const Part &p = parts[i];
        if (p.new_contig) flush();
        const char *src = p.ptr;
        if (kind == MEM_DEVICE && p.len) {
            tmp.resize(p.len);
            CK(cudaMemcpyAsync(tmp.data(), p.ptr, p.len, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            src = tmp.data();
        }
        const size_t at = ct.size();
        ct.resize(at + p.len);
        for (uint64_t j = 0; j < p.len; j++) ct[at + j] = fold_nuc(src[j], rna);
    }
    flush();
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    return GKD_OK;
}

uint64_t literal_intersection(const std::vector<uint32_t> &a, const std::vector<uint32_t> &b) {
    uint64_t n = 0;
    size_t i = 0, j = 0;
    while (i < a.size() && j < b.size()) {
        if (a[i] < b[j]) i++;
        else if (b[j] < a[i]) j++;
        else n++, i++, j++;
    }
    return n;
}

// ---- ingest -------------------------------------------------------------------------------------------
int add_genome(gkd_ctx *c, const std::vector<Part> &parts, const std::string &label, const std::string &comment,
               uint32_t *out_id) {
    NvtxRange nvtx("gkd kernel 1: ingest + pack");
    const bool prot = c->cfg.alphabet == GKD_PROT;
    uint64_t n_pos = 0;
    bool first = true;
    for (auto &p : parts) {
        if (p.new_contig && !first) n_pos += 1;  // separator position between contigs
        n_pos += p.len;
        first = false;
    }
    if (n_pos >= 0xFFFF0000ull) return fail(c, GKD_EINVAL, "sequence of %llu residues exceeds the 2^32 position limit", (unsigned long long)n_pos);
    GenomeRec g;
    g.label = label;
    g.comment = comment;
    g.n_pos = n_pos;
    const uint64_t n_words = (n_pos + PACK_POS_PER_WORD - 1) / PACK_POS_PER_WORD + 2;
    void *codes = nullptr, *mask = nullptr;
    int rc = slab_alloc(c, n_words * (prot ? 32 : 8), &codes);
    if (rc) return rc;
    rc = slab_alloc(c, n_words * 4, &mask);
    if (rc) return rc;
    g.d_codes = codes;
    g.d_mask = (uint32_t *)mask;

    // memory kind of the inputs (all parts of one call are assumed to live in the same kind)
    MemKind kind = MEM_PAGEABLE;
    if (!parts.empty()) {
        kind = classify(parts.front().ptr);
        if (parts.size() > 1 && classify(parts.back().ptr) != kind)
            return fail(c, GKD_EINVAL, "all sequence pieces of one call must be in the same kind of memory");
    }
    if (!prot && c->cfg.ambig_policy == GKD_AMBIG_LITERAL && (rc = collect_literals(c, parts, kind, g.lit))) return rc;
    // walk the stream in pieces of at most STAGE_BYTES positions
    size_t pi = 0;          // current part
    uint64_t pofs = 0;      // offset inside current part
    bool pending_sep = false;
    uint64_t q0 = 0;
    do {
        const uint64_t q1 = std::min<uint64_t>(n_pos, q0 + STAGE_BYTES);
        const uint64_t plen = q1 - q0;
        const int s = c->dstage_next;
        c->dstage_next = (c->dstage_next + 1) % N_DSTAGE;
        char *dev = c->stage_dev[s];
        // the staging buffer is free again once kernel 1 has consumed its previous piece
        if (c->packed_valid[s]) CK(cudaStreamWaitEvent(c->copy_stream, c->packed[s], 0));
        if (kind == MEM_PAGEABLE) {
            const int bs = c->stage_next;
            c->stage_next = (c->stage_next + 1) % N_STAGE;
            CK(cudaEventSynchronize(c->bounce_ev[bs]));
            char *dst = c->bounce[bs];
            uint64_t w = 0;
            while (w < plen) {
                if (pending_sep) {
                    dst[w++] = STREAM_SEPARATOR;
                    pending_sep = false;
                    continue;
                }
                const Part &p = parts[pi];
                uint64_t take = std::min<uint64_t>(p.len - pofs, plen - w);
                memcpy(dst + w, p.ptr + pofs, take);
                w += take;
                pofs += take;
                if (pofs == p.len) {
                    pi++;
                    pofs = 0;
                    if (pi < parts.size() && parts[pi].new_contig) pending_sep = true;
                }
            }
            if (plen) CK(cudaMemcpyAsync(dev, dst, plen, cudaMemcpyHostToDevice, c->copy_stream));
            CK(cudaEventRecord(c->bounce_ev[bs], c->copy_stream));
            c->m.h2d_bytes += plen;
        } else {
            // pinned host or device memory: copy each run straight into the staged text; the
            // separators are the zero fill
            if (plen) CK(cudaMemsetAsync(dev, STREAM_SEPARATOR, plen, c->copy_stream));
            uint64_t w = 0;
            while (w < plen) {
                if (pending_sep) {
                    w++;
                    pending_sep = false;
                    continue;
                }
                const Part &p = parts[pi];
                uint64_t take = std::min<uint64_t>(p.len - pofs, plen - w);
                if (take) CK(cudaMemcpyAsync(dev + w, p.ptr + pofs, take, cudaMemcpyDefault, c->copy_stream));
                w += take;
                pofs += take;
                if (pofs == p.len) {
                    pi++;
                    pofs = 0;
                    if (pi < parts.size() && parts[pi].new_contig) pending_sep = true;
                }
            }
            if (kind == MEM_PINNED) c->m.h2d_bytes += plen;
        }
        // kernel 1 on this piece (q0 is a multiple of 32 positions), on its own stream behind the copy: the next
        // copies do not wait for it
        CK(cudaEventRecord(c->copied[s], c->copy_stream));
        CK(cudaStreamWaitEvent(c->pack_stream, c->copied[s], 0));
        if (prot)
            CK(launch_pack_prot(dev, plen, (uint8_t *)codes + q0, (uint32_t *)mask + q0 / 32, c->pack_stream));
        else
            CK(launch_pack_dna(dev, plen, (uint64_t *)codes + q0 / 32, (uint32_t *)mask + q0 / 32,
                               c->cfg.alphabet == GKD_RNA, c->pack_stream));
        CK(cudaEventRecord(c->packed[s], c->pack_stream));
        c->packed_valid[s] = true;
        c->m.launches++;
        q0 = q1;
    } while (q0 < n_pos);
    // contract (gkd.h): pageable text was copied into the bounce buffers before this returns; pinned and
    // device text is read by the stream-ordered copies above and must stay valid until gkd_build_sets
    // (which waits for them and synchronises) -- no per-genome synchronisation here.
    if (c->ev_pool.empty()) {
        cudaEvent_t e = nullptr;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->ev_pool.push_back(e);
    }
    g.ready = c->ev_pool.back();
    c->ev_pool.pop_back();
    CK(cudaEventRecord(g.ready, c->pack_stream));
    c->m.residues_packed += n_pos;
    if (out_id) *out_id = (uint32_t)c->genomes.size();
    c->genomes.push_back(std::move(g));
    return GKD_OK;
}

// ---- set construction ------------------------------------------------------------------------------------
bool has_pal_lists(const gkd_ctx *c) { return c->cfg.alphabet != GKD_PROT && (c->k % 2 == 0); }

// device allocation for a batch of finished sets: best-fitting parked arena, else a fresh one (parked
// arenas that were too small are released first so a streamed run does not creep up in memory)
int arena_alloc(gkd_ctx *c, uint64_t need, void **out, uint64_t *cap) {
    int best = -1;
    for (size_t i = 0; i < c->free_arenas.size(); i++)
        if (c->free_arenas[i].second >= need && (best < 0 || c->free_arenas[i].second < c->free_arenas[best].second))
            best = (int)i;
    if (best >= 0) {
        *out = c->free_arenas[best].first;
        *cap = c->free_arenas[best].second;
        c->free_arenas.erase(c->free_arenas.begin() + best);
        return GKD_OK;
    }
    for (auto &a : c->free_arenas) CK(cudaFreeAsync(a.first, c->stream));
    c->free_arenas.clear();
    CK(cudaMallocAsync(out, need, c->stream));
    *cap = need;
    return GKD_OK;
}

void set_desc_from_packed(GenomeRec &g, const char *base) {
    const gkd_packed_set &p = g.packed;
    g.desc.main.offs = (const uint32_t *)(base + p.offs_off);
    g.desc.main.lows = base + p.lows_off;
    g.desc.main.n = p.n;
    g.desc.main.level = p.level;
    const bool pal = p.pal_offs_off != 0 || p.pal_lows_off != 0;
    g.desc.pal.offs = pal ? (const uint32_t *)(base + p.pal_offs_off) : nullptr;
    g.desc.pal.lows = pal ? base + p.pal_lows_off : nullptr;
    g.desc.pal.n = p.n_pal;
    g.desc.pal.level = p.pal_level;
}

// unique/compact the sorted slots of a batch into a fresh set arena and record the descriptors
int finish_batch(gkd_ctx *c, const std::vector<BatchGenome> &bg, const std::vector<uint32_t> &ids, const SortPlan &plan,
                 const uint64_t *sorted) {
    const uint32_t n = (uint32_t)bg.size();
    CK(launch_unique_count((const BatchGenome *)c->batch_genomes.p, plan, sorted, c->cfg.alphabet, c->k, c->mix, c->stream));
    c->m.launches += 2;
    std::vector<uint64_t> counts(n);
    CK(cudaMemcpyAsync(counts.data(), plan.genome_counts, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    const bool pal = has_pal_lists(c);
    const uint64_t lsz = c->low_bits / 8;
    // layout: per set [offs][lows][pal offs][pal lows][pal scratch], every piece a multiple of 16 bytes
    std::vector<gkd_packed_set> packed(n);
    std::vector<uint64_t> palh_off(n, 0);
    uint64_t cur = 0;
    for (uint32_t i = 0; i < n; i++) {
        gkd_packed_set &p = packed[i];
        p = gkd_packed_set{};
        p.n = (uint32_t)counts[i];
        p.n_pal = (uint32_t)(counts[i] >> 32);
        p.level = set_level(p.n, c->table_tmax, c->key_bits, c->low_bits);
        cur = (cur + SET_BLOCK_ALIGN - 1) & ~(SET_BLOCK_ALIGN - 1);
        p.offs_off = cur;
        cur += align16(((1ull << p.level) + 1) * 4);
        p.lows_off = cur;
        cur += align16((uint64_t)p.n * lsz) + 16;
        if (pal) {
            p.pal_level = set_level(p.n_pal, c->table_tmax, c->key_bits, c->low_bits);
            p.pal_offs_off = cur;
            cur += align16(((1ull << p.pal_level) + 1) * 4);
            p.pal_lows_off = cur;
            cur += align16((uint64_t)p.n_pal * lsz) + 16;
            palh_off[i] = cur;
            cur += align16((uint64_t)p.n_pal * 8);
        }
    }
    const uint64_t need = cur + 256;
    void *arena = nullptr;
    uint64_t cap = 0;
    int rc = arena_alloc(c, need, &arena, &cap);
    if (rc) return rc;
    c->arenas.push_back(Arena{(char *)arena, need, cap, ids.empty() ? 0u : ids.front(), n, true});
    const int arena_idx = (int)c->arenas.size() - 1;
    std::vector<SetBuild> dst(n);
    char *base = (char *)arena;
    for (uint32_t i = 0; i < n; i++) {
        const gkd_packed_set &p = packed[i];
        SetBuild &d = dst[i];
        d.offs = (uint32_t *)(base + p.offs_off);
        d.lows = base + p.lows_off;
        d.n = p.n;
        d.level = p.level;
        d.n_pal = p.n_pal;
        d.pal_level = p.pal_level;
        d.pal_offs = pal ? (uint32_t *)(base + p.pal_offs_off) : nullptr;
        d.pal_lows = pal ? (void *)(base + p.pal_lows_off) : nullptr;
        d.pal_h = pal ? (uint64_t *)(base + palh_off[i]) : nullptr;
        GenomeRec &g = c->genomes[ids[i]];
        g.packed = p;
        g.arena = arena_idx;
        set_desc_from_packed(g, base);
        g.built = true;
        c->m.keys_unique += p.n;
    }
    if ((rc = ensure(c, c->set_build, n * sizeof(SetBuild)))) return rc;
    CK(cudaMemcpyAsync(c->set_build.p, dst.data(), n * sizeof(SetBuild), cudaMemcpyHostToDevice, c->stream));
    CK(launch_unique_write((const BatchGenome *)c->batch_genomes.p, plan, sorted, (const SetBuild *)c->set_build.p,
                           c->cfg.alphabet, c->k, c->mix, c->low_bits, c->stream));
    c->m.launches += 2;
    // the host vectors above are pageable: make sure the copies were consumed before they die
    CK(cudaStreamSynchronize(c->stream));
    c->sets_dirty = true;
    return GKD_OK;
}

void record_set(gkd_ctx *c, uint32_t id, const gkd_packed_set &p, int arena_idx, const char *base) {
    GenomeRec &g = c->genomes[id];
    g.packed = p;
    g.arena = arena_idx;
    set_desc_from_packed(g, base);
    g.built = true;
    c->m.keys_unique += p.n;
}

// Kernel 3, fast path (sort_msd.cu).  keys_in == nullptr: kernel 2 encodes the batch straight into fixed-capacity
// bins (fused pass); else the given h values (imports) are partitioned.  Returns GKD_OK and *done = true when the
// sets were built; *done = false when the batch has to take the LSD path (a bin overflowed: heavily repeated
// k-mers, or a key space too small to bucket).
int build_batch_msd(gkd_ctx *c, const std::vector<BatchGenome> &bg, const std::vector<uint32_t> &ids, uint32_t n_tiles,
                    const uint64_t *keys_in, bool *done) {
    *done = false;
    const uint32_t n = (uint32_t)bg.size();
    std::vector<MsdGenome> msd(n);
    uint32_t n_bins = 0, max_p = 0;
    uint64_t bin_keys = 0;
    bool narrow = true;  // key_bits - p <= 32 everywhere: the bin sort keeps 32-bit keys in shared memory
    for (uint32_t i = 0; i < n; i++) {
        uint32_t p = level_for(bg[i].n_slots, MSD_BIN_AVG);
        // big genomes get at least key_bits - 32 bin bits, so the bin sort can keep 32-bit keys in shared memory
        if (bg[i].n_slots >= (1u << 18) && c->key_bits > 32) p = std::max<uint32_t>(p, (uint32_t)c->key_bits - 32);
        p = std::min<uint32_t>(std::min<uint32_t>(p, MSD_MAX_P), (uint32_t)c->key_bits);
        const double mean = (double)bg[i].n_slots / (double)(1u << p);
        uint32_t cap = (uint32_t)(mean + 8.0 * std::sqrt(mean) + 64.0);
        cap = std::min<uint32_t>((cap + 3) & ~3u, MSD_BIN_CAP);
        if (mean > MSD_BIN_AVG) return GKD_OK;  // more than 2^MSD_MAX_P full bins: LSD path
        MsdGenome &M = msd[i];
        M = MsdGenome{};
        M.bin_first = n_bins;
        M.p = p;
        M.s = std::min<uint32_t>(MSD_SORT_BITS, (uint32_t)c->key_bits - p);
        M.cap = cap;
        M.bins_off = bin_keys;
        n_bins += 1u << p;
        bin_keys += (uint64_t)cap << p;
        max_p = std::max(max_p, p);
        narrow = narrow && (c->key_bits - (int)p <= 32);
    }
    int rc;
    if ((rc = ensure(c, c->keys_b, std::max<uint64_t>(bin_keys, 16) * 8))) return rc;
    if ((rc = ensure(c, c->msd_genomes, n * sizeof(MsdGenome)))) return rc;
    if ((rc = ensure(c, c->msd_bins32, (uint64_t)n_bins * 4 + 16))) return rc;  // bin_cursor | overflow flag
    if ((rc = ensure(c, c->msd_bins64, (uint64_t)n_bins * 8))) return rc;       // look-back status
    if ((rc = ensure(c, c->msd_gstat, (uint64_t)n * 12))) return rc;            // valid | maxbin | unique
    MsdPlan mp{};
    mp.n_bins = n_bins;
    mp.max_p = max_p;
    mp.key_bits = c->key_bits;
    mp.bins = (uint64_t *)c->keys_b.p;
    mp.bin_cursor = (uint32_t *)c->msd_bins32.p;
    mp.overflow = mp.bin_cursor + n_bins;
    mp.status = (unsigned long long *)c->msd_bins64.p;
    mp.genome_valid = (uint32_t *)c->msd_gstat.p;
    mp.genome_maxbin = mp.genome_valid + n;
    mp.genome_unique = mp.genome_maxbin + n;
    CK(cudaMemcpyAsync(c->msd_genomes.p, msd.data(), n * sizeof(MsdGenome), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(mp.bin_cursor, 0, (size_t)n_bins * 4 + 16, c->stream));
    CK(cudaMemsetAsync(mp.status, 0, (size_t)n_bins * 8, c->stream));
    nvtxRangePushA(keys_in ? "gkd kernel 3: partition into bins" : "gkd kernels 2+3: encode + mix + partition into bins");
    CK(launch_encode_scatter((const BatchGenome *)c->batch_genomes.p, n, n_tiles, (const MsdGenome *)c->msd_genomes.p, max_p,
                             c->cfg.alphabet, c->k, c->mix, keys_in, mp.bins, mp.bin_cursor, mp.overflow, c->stream));
    nvtxRangePop();
    CK(launch_msd_totals((const MsdGenome *)c->msd_genomes.p, n, mp, c->stream));
    c->m.launches += 2;
    std::vector<uint32_t> stat(2 * (size_t)n);
    uint32_t overflow = 0;
    CK(cudaMemcpyAsync(stat.data(), mp.genome_valid, 2 * (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&overflow, mp.overflow, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaEventRecord(c->ev[1], c->stream));
    CK(cudaEventRecord(c->ev[2], c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (overflow) return GKD_OK;  // *done stays false: LSD path
    // arena: the distinct count is only known after the bin sort, so the low words get room for every valid slot
    // (duplicates are a fraction of a percent of a genome's k-mers) and the table level comes from that bound
    const uint64_t lsz = c->low_bits / 8;
    std::vector<gkd_packed_set> packed(n);
    uint64_t cur = 0;
    for (uint32_t i = 0; i < n; i++) {
        gkd_packed_set &p = packed[i];
        p = gkd_packed_set{};
        const uint32_t n_valid = stat[i];
        p.level = std::max(set_level(n_valid, c->table_tmax, c->key_bits, c->low_bits), msd[i].p);
        msd[i].level = p.level;
        cur = (cur + SET_BLOCK_ALIGN - 1) & ~(SET_BLOCK_ALIGN - 1);
        p.offs_off = cur;
        cur += align16(((1ull << p.level) + 1) * 4);
        p.lows_off = cur;
        cur += align16((uint64_t)n_valid * lsz) + 16;
    }
    const uint64_t need = cur + 256;
    void *arena = nullptr;
    uint64_t cap = 0;
    if ((rc = arena_alloc(c, need, &arena, &cap))) return rc;
    c->arenas.push_back(Arena{(char *)arena, need, cap, ids.empty() ? 0u : ids.front(), n, true});
    const int arena_idx = (int)c->arenas.size() - 1;
    char *base = (char *)arena;
    for (uint32_t i = 0; i < n; i++) {
        msd[i].offs = (uint32_t *)(base + packed[i].offs_off);
        msd[i].lows = base + packed[i].lows_off;
    }
    CK(cudaMemcpyAsync(c->msd_genomes.p, msd.data(), n * sizeof(MsdGenome), cudaMemcpyHostToDevice, c->stream));
    nvtxRangePushA("gkd kernel 3: bin sort + unique + bucket tables");
    CK(launch_msd_binsort((const MsdGenome *)c->msd_genomes.p, n, mp, c->low_bits, narrow, c->stream));
    nvtxRangePop();
    c->m.launches++;
    std::vector<uint32_t> uniq(n);
    CK(cudaMemcpyAsync(uniq.data(), mp.genome_unique, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (uint32_t i = 0; i < n; i++) {
        packed[i].n = uniq[i];
        record_set(c, ids[i], packed[i], arena_idx, base);
    }
    c->sets_dirty = true;
    c->m.sort_passes = 1;
    *done = true;
    return GKD_OK;
}

// raw slots in plan.keys_a -> finished sets on the LSD path: radix sort + unique
int sort_and_finish_lsd(gkd_ctx *c, const std::vector<BatchGenome> &bg, const std::vector<uint32_t> &ids, const SortPlan &plan) {
    uint64_t *sorted = nullptr;
    uint32_t passes = 0;
    nvtxRangePushA("gkd kernel 3: LSD radix sort");
    CK(launch_sort((const BatchGenome *)c->batch_genomes.p, plan, &sorted, &passes, c->stream));
    nvtxRangePop();
    c->m.launches += 3ull * passes;
    c->m.sort_passes = passes;
    CK(cudaEventRecord(c->ev[2], c->stream));
    NvtxRange nvtx("gkd kernel 3: unique + bucket tables");
    return finish_batch(c, bg, ids, plan, sorted);
}

bool msd_applies(const gkd_ctx *c) { return c->use_msd && !has_pal_lists(c); }

int plan_batch(gkd_ctx *c, std::vector<BatchGenome> &bg, SortPlan &plan, uint64_t raw_keys, uint32_t n_tiles) {
    int rc;
    if ((rc = ensure(c, c->keys_a, raw_keys * 8))) return rc;
    if ((rc = ensure(c, c->keys_b, raw_keys * 8))) return rc;
    if ((rc = ensure(c, c->tile_hist, (uint64_t)std::max(n_tiles, 1u) * RADIX_BINS * 4))) return rc;
    if ((rc = ensure(c, c->tile_uniq, (uint64_t)std::max(n_tiles, 1u) * 8))) return rc;
    if ((rc = ensure(c, c->genome_counts, bg.size() * 8))) return rc;
    if ((rc = ensure(c, c->batch_genomes, bg.size() * sizeof(BatchGenome)))) return rc;
    CK(cudaMemcpyAsync(c->batch_genomes.p, bg.data(), bg.size() * sizeof(BatchGenome), cudaMemcpyHostToDevice, c->stream));
    plan.n_genomes = (uint32_t)bg.size();
    plan.n_tiles = n_tiles;
    plan.key_bits = c->key_bits;
    plan.keys_a = (uint64_t *)c->keys_a.p;
    plan.keys_b = (uint64_t *)c->keys_b.p;
    plan.tile_hist = (uint32_t *)c->tile_hist.p;
    plan.tile_uniq = (uint64_t *)c->tile_uniq.p;
    plan.genome_counts = (uint64_t *)c->genome_counts.p;
    return GKD_OK;
}

int build_batch(gkd_ctx *c, uint32_t first, uint32_t last) {
    std::vector<BatchGenome> bg;
    std::vector<uint32_t> ids;
    uint64_t raw = 0;
    uint32_t tiles = 0;
    for (uint32_t id = first; id < last; id++) {
        GenomeRec &g = c->genomes[id];
        BatchGenome b;
        b.codes = (const uint64_t *)g.d_codes;
        b.mask = g.d_mask;
        b.n_pos = (uint32_t)g.n_pos;
        b.n_slots = g.n_pos >= (uint64_t)c->k ? (uint32_t)(g.n_pos - c->k + 1) : 0;
        b.raw_off = raw;
        b.tile_first = tiles;
        b.n_tiles = (b.n_slots + SORT_TILE - 1) / SORT_TILE;
        raw += ((uint64_t)b.n_slots + 15) & ~15ull;
        tiles += b.n_tiles;
        bg.push_back(b);
        ids.push_back(id);
        c->m.kmer_positions += b.n_slots;
    }
    // the packed streams of this batch come from the ingest stream (in order: the last pending event covers all)
    for (uint32_t id = last; id-- > first;)
        if (c->genomes[id].ready) {
            CK(cudaStreamWaitEvent(c->stream, c->genomes[id].ready, 0));
            break;
        }
    SortPlan plan{};
    int rc = plan_batch(c, bg, plan, std::max<uint64_t>(raw, 16), tiles);
    if (rc) return rc;
    CK(cudaEventRecord(c->ev[0], c->stream));
    c->m.keys_sorted += raw;
    bool done = false;
    if (msd_applies(c)) {
        // fast path: kernel 2 writes straight into the bins of kernel 3 (ev[1] == ev[2]: the partition is part of
        // the encode time, the bin sort is reported as unique_ms)
        rc = build_batch_msd(c, bg, ids, tiles, nullptr, &done);
        if (rc) return rc;
        plan.keys_b = (uint64_t *)c->keys_b.p;  // the bin buffer may have been re-allocated larger
    }
    if (!done) {
        nvtxRangePushA("gkd kernel 2: canonical encode + mix");
        CK(launch_encode((const BatchGenome *)c->batch_genomes.p, plan.n_genomes, tiles, c->cfg.alphabet, c->k, c->mix,
                         plan.keys_a, c->stream));
        nvtxRangePop();
        if (tiles) c->m.launches++;
        CK(cudaEventRecord(c->ev[1], c->stream));
        rc = sort_and_finish_lsd(c, bg, ids, plan);
        if (rc) return rc;
    }
    CK(cudaEventRecord(c->ev[3], c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->m.encode_ms += elapsed(c->ev[0], c->ev[1]);
    c->m.sort_ms += elapsed(c->ev[1], c->ev[2]);
    c->m.unique_ms += elapsed(c->ev[2], c->ev[3]);
    return GKD_OK;
}

int upload_sets(gkd_ctx *c) {
    if (!c->sets_dirty) return GKD_OK;
    const size_t n = c->genomes.size();
    std::vector<SetDesc> h(n);
    std::vector<uint32_t> lit(n);
    bool any_lit = false;
    for (size_t i = 0; i < n; i++) {
        h[i] = c->genomes[i].desc;
        lit[i] = (uint32_t)c->genomes[i].lit.size();
        any_lit = any_lit || lit[i];
    }
    int rc = ensure(c, c->d_sets, std::max<size_t>(n, 1) * sizeof(SetDesc));
    if (rc) return rc;
    if (n) CK(cudaMemcpyAsync(c->d_sets.p, h.data(), n * sizeof(SetDesc), cudaMemcpyHostToDevice, c->stream));
    if (any_lit) {
        if ((rc = ensure(c, c->lit_size, n * 4))) return rc;
        CK(cudaMemcpyAsync(c->lit_size.p, lit.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));
    c->sets_dirty = false;
    return GKD_OK;
}

// adopt key arrays (device memory, back to back at offsets[]) as new sets: mix, sort, unique
int import_device_batch(gkd_ctx *c, const uint64_t *keys, const uint64_t *offsets, uint32_t i0, uint32_t i1, bool on_device) {
    const uint32_t id0 = (uint32_t)c->genomes.size();
    std::vector<BatchGenome> bg(i1 - i0);
    std::vector<uint32_t> ids(i1 - i0);
    uint32_t tiles = 0;
    const uint64_t k0 = offsets[i0], total = offsets[i1] - k0;
    for (uint32_t i = i0; i < i1; i++) {
        BatchGenome &b = bg[i - i0];
        b.codes = nullptr;
        b.mask = nullptr;
        b.raw_off = offsets[i] - k0;
        b.n_pos = 0;
        b.n_slots = (uint32_t)(offsets[i + 1] - offsets[i]);
        b.tile_first = tiles;
        b.n_tiles = (b.n_slots + SORT_TILE - 1) / SORT_TILE;
        tiles += b.n_tiles;
        ids[i - i0] = id0 + (i - i0);
    }
    SortPlan plan{};
    int rc = plan_batch(c, bg, plan, std::max<uint64_t>(total, 16), tiles);
    if (rc) return rc;
    if (total) {
        CK(cudaMemcpyAsync(plan.keys_a, keys + k0, total * 8, cudaMemcpyDefault, c->stream));
        if (!on_device) c->m.h2d_bytes += total * 8;
        CK(launch_mix_keys(plan.keys_a, total, c->mix, c->stream));
        c->m.launches++;
    }
    for (uint32_t i = i0; i < i1; i++) c->genomes.push_back(GenomeRec());
    bool done = false;
    rc = GKD_OK;
    if (msd_applies(c)) {
        rc = build_batch_msd(c, bg, ids, tiles, plan.keys_a, &done);
        plan.keys_b = (uint64_t *)c->keys_b.p;  // the bin buffer may have been re-allocated larger
    }
    if (!rc && !done) rc = sort_and_finish_lsd(c, bg, ids, plan);
    if (rc) c->genomes.resize(id0);
    return rc;
}

// ---- distances ------------------------------------------------------------------------------------------
// host copy of the pair source (ids live on the host here)
struct HostPairs {
    int mode;
    uint32_t n;
    uint64_t first, count;
    const uint32_t *a, *b;
    uint32_t na, nb;  // lengths of a / b arrays (LIST: count each; RECT: nq, nr)
};

int check_built(gkd_ctx *c, uint32_t id) {
    if (id >= c->genomes.size()) return fail(c, GKD_EINVAL, "set id %u out of range (have %zu)", id, c->genomes.size());
    if (!c->genomes[id].built) return fail(c, GKD_ESTATE, "set %u has not been built; call gkd_build_sets first", id);
    return GKD_OK;
}

uint64_t both_size(const gkd_ctx *c, const GenomeRec &g) {
    const bool both = c->cfg.alphabet != GKD_PROT && c->cfg.strand_mode == GKD_STRAND_BOTH;
    return (both ? 2ull * g.desc.main.n - g.desc.pal.n : g.desc.main.n) + g.lit.size();
}

void host_pair_ids(const HostPairs &hp, uint64_t t, uint32_t &a, uint32_t &b) {
    if (hp.mode == PAIRS_UPPER) upper_pair(hp.first + t, hp.n, a, b);
    else if (hp.mode == PAIRS_RECT) a = hp.a[t / hp.nb], b = hp.b[t % hp.nb];
    else a = hp.a[t], b = hp.b[t];
}

// Block-join planning (join.cu).  Decides whether the chunk [first, first+count) of an UPPER call, or a RECT
// call, is served by the block join and lays out its row blocks: rows are grouped by the number of key ranges
// their size calls for (so that 32 rows fill ~30 % of the table in every range), largest class first, a class
// padded to whole blocks.  Returns false when the merge kernel should run.
bool plan_join(gkd_ctx *c, const HostPairs &hp, uint64_t first, uint64_t count, JoinPlan &plan, std::vector<uint32_t> &rows,
               bool &swapped) {
    swapped = false;
    if (c->isect_algo == 1 || count == 0) return false;
    if (hp.mode != PAIRS_UPPER && hp.mode != PAIRS_RECT) return false;
    const bool forced = c->isect_algo == 2;
    // 32-bit low words identify a key only inside a range of at most 2^31 values; 64-bit keys are stored whole
    const uint32_t lt_min = c->low_bits == 32 ? (uint32_t)std::max(1, c->key_bits - 31) : 1u;
    const uint32_t lt_max = std::min<uint32_t>((uint32_t)c->key_bits - 1u, 30u);
    if (lt_min > lt_max) return false;
    uint32_t fill_pct = 30;
    if (const char *e = getenv("GKD_JOIN_FILL")) fill_pct = (uint32_t)std::min(45, std::max(5, atoi(e)));

    // candidate rows and the columns they meet
    std::vector<uint32_t> cand;  // UPPER: set ids; RECT: positions in the row-side id list
    const uint32_t *row_ids = nullptr;
    uint32_t n_cols = 0;
    if (hp.mode == PAIRS_UPPER) {
        uint32_t i0, j0, i1, j1;
        upper_pair(first, hp.n, i0, j0);
        upper_pair(first + count - 1, hp.n, i1, j1);
        for (uint32_t i = i0; i <= i1; i++) cand.push_back(i);
        n_cols = hp.n;
        // a thin slice of the triangle would stream every column for a few pairs
        if (!forced && count < (uint64_t)cand.size() * (hp.n - i0) / 4) return false;
    } else {
        // the table side needs whole blocks of rows, the streamed side many columns
        swapped = hp.na < 32 && hp.nb >= 32;
        const uint32_t nr = swapped ? hp.nb : hp.na;
        row_ids = swapped ? hp.b : hp.a;
        n_cols = swapped ? hp.na : hp.nb;
        for (uint32_t i = 0; i < nr; i++) cand.push_back(i);
    }
    const int cfg = join_pick_cfg((uint32_t)cand.size(), n_cols, c->low_bits);
    const uint64_t R = join_cfg_rows(cfg);
    const uint64_t fill = std::max<uint64_t>(32, (uint64_t)join_cfg_slots(cfg) * fill_pct / 100);
    auto size_at = [&](uint32_t e) -> uint64_t { return c->genomes[row_ids ? row_ids[e] : e].desc.main.n; };
    uint64_t n_max = 0;
    std::vector<std::pair<uint32_t, uint32_t>> byl;  // (level, entry)
    for (uint32_t e : cand) {
        const uint64_t n = size_at(e);
        if (n == 0) continue;  // nothing can match: the counts stay 0
        n_max = std::max(n_max, n);
        uint32_t L = ceil_log2_u32((uint32_t)std::min<uint64_t>(0xFFFFFFFFull, (R * n + fill - 1) / fill));
        L = std::min(std::max(L, lt_min), lt_max);
        byl.push_back({L, e});
    }
    if (byl.empty()) return false;
    if (!forced) {
        // enough rows to share a probe, enough columns to pay for building the tables, and sets large enough
        // that the tables of the coarsest usable range are not almost empty
        if (byl.size() < 16 || n_cols < 64) return false;
        if (R * n_max < (fill << lt_min) / 4) return false;
    }
    std::stable_sort(byl.begin(), byl.end(), [](const auto &x, const auto &y) { return x.first > y.first; });
    plan = JoinPlan{};
    plan.mode = hp.mode;
    plan.key_bits = c->key_bits;
    plan.cfg = cfg;
    plan.n_cols = n_cols;
    plan.first = first;
    plan.count = count;
    plan.stride_r = swapped ? 1ull : (unsigned long long)hp.nb;
    plan.stride_c = swapped ? (unsigned long long)hp.nb : 1ull;
    rows.clear();
    unsigned long long tasks = 0;
    for (size_t i = 0; i < byl.size();) {
        size_t j = i;
        while (j < byl.size() && byl[j].first == byl[i].first) j++;
        if (plan.n_classes >= (uint32_t)JOIN_MAX_CLASSES) return false;
        JoinClass &k = plan.cls[plan.n_classes++];
        k.level = byl[i].first;
        k.blk_first = (uint32_t)(rows.size() / R);
        for (size_t t = i; t < j; t++) rows.push_back(byl[t].second);
        while (rows.size() % R) rows.push_back(0xFFFFFFFFu);
        k.n_blocks = (uint32_t)(rows.size() / R) - k.blk_first;
        k.task_first = tasks;
        tasks += (unsigned long long)k.n_blocks << k.level;
        i = j;
    }
    plan.n_tasks = tasks;
    return true;
}

// The sets of one call: the largest sizes and levels (kernel 4's work split) and whether any has literal k-mers
struct SetScan {
    uint64_t max_n = 0, max_pal = 0;
    uint32_t max_level = 0, max_pal_level = 0;
    bool any_lit = false;
    int see(gkd_ctx *c, uint32_t id) {
        const int rc = check_built(c, id);
        if (rc) return rc;
        const GenomeRec &g = c->genomes[id];
        max_n = std::max<uint64_t>(max_n, g.desc.main.n);
        max_pal = std::max<uint64_t>(max_pal, g.desc.pal.n);
        max_level = std::max(max_level, g.desc.main.level);
        max_pal_level = std::max(max_pal_level, g.desc.pal.level);
        any_lit = any_lit || !g.lit.empty();
        return GKD_OK;
    }
};

// Kernel 4's work split for `pairs` pairs whose sets have at most nmax keys and level lmax: a pair is walked in
// 32-bucket groups at the level of its larger set; an item is a run of groups of one pair.  Few pairs -> small items so
// every warp has work; many pairs -> eight items per pair, so the warps that share a pair read neighbouring parts of its
// two key streams.  gkd_config.segment_keys, when set, fixes the item size instead.
IsectPlan make_plan(const gkd_ctx *c, uint64_t pairs, uint64_t nmax, uint32_t lmax, bool one_item) {
    IsectPlan p{};
    p.low_bits = c->low_bits;
    p.tmax = c->isect_tmax;
    p.level_min = c->lvl_min;
    uint32_t L = std::max(level_for((uint32_t)nmax, p.tmax), c->lvl_min);
    L = std::min(L, lmax);
    const uint64_t max_groups = ((1ull << L) + 31) >> 5;
    uint64_t gpi;
    if (one_item || max_groups <= 64) gpi = max_groups;  // tiny sets: a pair is one item (the per-item set-up would dominate)
    else if (c->cfg.segment_keys) gpi = std::max<uint64_t>(1, c->cfg.segment_keys / (64ull * p.tmax));
    else {
        const uint64_t warps = (uint64_t)c->n_sms * intersect_warps_per_sm(c->low_bits);
        const long double total_groups = (long double)pairs * max_groups;
        gpi = (uint64_t)std::min<long double>(total_groups / (long double)(warps * 8), (long double)(max_groups / 8));
    }
    gpi = std::min<uint64_t>(std::max<uint64_t>(gpi, 1), max_groups);
    p.groups_per_item = (uint32_t)gpi;
    p.items_per_pair = (uint32_t)((max_groups + gpi - 1) / gpi);
    return p;
}

// One chunk of run_pairs once its kernel-4 launches are queued: pairs done .. done + cnt of hp and their counts
struct Chunk {
    const HostPairs &hp;
    const PairSource &src;
    uint64_t done, cnt;
    PairCounts pc;
    const uint32_t *join_err;  // the block join's overflow flag on the device; nullptr when the merge kernel ran
};

// What a call computes from the counts of kernel 4: one form of kernel 5.  run_call owns the call (checks, start, chunk
// loop, finish), run_pairs the chunk loop and the redo of a chunk whose join table overflowed; the form owns its outputs,
// its state, its launches and its copies, and its answer to a call without pairs.  The bytes queue() and keep() read
// back are counted only for a chunk that is kept.
struct Form {
    uint32_t a_base = 0;  // RECT: position in the caller's q of this launch's first query row (run_rect)
    virtual ~Form() = default;
    // the caller's output buffers (unused entries nullptr)
    virtual std::array<const void *, 8> outputs() const = 0;
    // before the first chunk, also when the call has no pairs
    virtual int start(gkd_ctx *c) { return GKD_OK; }
    // the chunk's kernel-5 launches, then the reads the host needs once the stream is synchronised; records ev[7]
    virtual int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) = 0;
    // the join held: the chunk is kept
    virtual int keep(gkd_ctx *c, const Chunk &e, uint64_t &d2h) { return GKD_OK; }
    // after the last chunk, also when the call has no pairs
    virtual int finish(gkd_ctx *c) { return GKD_OK; }
};

// a read of `bytes` from the device into dst (host or device memory), skipped when dst is nullptr; counted in d2h
int read_back(gkd_ctx *c, void *dst, const void *src, uint64_t bytes, uint64_t &d2h) {
    if (!dst || !bytes) return GKD_OK;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, c->stream));
    d2h += bytes;
    return GKD_OK;
}

// gkd_all_vs_all*, gkd_query_vs_ref*, gkd_pairs*: every pair's values to the caller's outputs; a nullptr member of the
// outputs is not computed
struct Dense : Form {
    gkd_outputs out;
    explicit Dense(const gkd_outputs &o) : out(o) {}
    std::array<const void *, 8> outputs() const override { return {out.inter, out.dist, out.contain_a, out.contain_b}; }
    int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        // the chunk's part of out (RECT: from row a_base of the caller's block)
        const uint64_t t = (uint64_t)a_base * e.hp.nb + e.done;
        const gkd_outputs o{out.inter ? out.inter + t : nullptr, out.dist ? out.dist + t : nullptr,
                            out.contain_a ? out.contain_a + t : nullptr, out.contain_b ? out.contain_b + t : nullptr};
        int rc;
        if (o.inter && (rc = ensure(c, c->d_inter, e.cnt * 8))) return rc;
        if (o.dist && (rc = ensure(c, c->d_dist, e.cnt * 8))) return rc;
        if (o.contain_a && (rc = ensure(c, c->d_ca, e.cnt * 8))) return rc;
        if (o.contain_b && (rc = ensure(c, c->d_cb, e.cnt * 8))) return rc;
        EpilogueOut eo{o.inter ? (uint64_t *)c->d_inter.p : nullptr, o.dist ? (double *)c->d_dist.p : nullptr,
                       o.contain_a ? (double *)c->d_ca.p : nullptr, o.contain_b ? (double *)c->d_cb.p : nullptr};
        nvtxRangePushA("gkd kernel 5: distance epilogue");
        CK(launch_epilogue(e.src, e.pc, eo, c->stream));
        nvtxRangePop();
        c->m.launches++;
        CK(cudaEventRecord(c->ev[7], c->stream));
        // queued before the overflow flag is read: a redo rewrites the same slots
        if ((rc = read_back(c, o.inter, c->d_inter.p, e.cnt * 8, d2h)) || (rc = read_back(c, o.dist, c->d_dist.p, e.cnt * 8, d2h)) ||
            (rc = read_back(c, o.contain_a, c->d_ca.p, e.cnt * 8, d2h)) || (rc = read_back(c, o.contain_b, c->d_cb.p, e.cnt * 8, d2h)))
            return rc;
        return GKD_OK;
    }
};

int run_pairs(gkd_ctx *c, const HostPairs &hp, Form &f) {
    int rc = upload_sets(c);
    if (rc) return rc;
    const bool nuc = c->cfg.alphabet != GKD_PROT;
    const bool both = nuc && c->cfg.strand_mode == GKD_STRAND_BOTH;
    const bool need_pal = both && (c->k % 2 == 0);
    c->m.pairs = hp.count;
    c->m.intersect_bytes = 0;
    c->m.intersect_ms = c->m.epilogue_ms = 0;

    // validate ids, gather sizes for the work split and the byte accounting
    SetScan s;
    long double sum_bytes = 0;
    auto size_of = [&](uint32_t id) -> uint64_t { return c->genomes[id].desc.main.n; };
    if (hp.mode == PAIRS_UPPER) {
        for (uint32_t i = 0; i < hp.n; i++)
            if ((rc = s.see(c, i))) return rc;
        // bytes of the requested range, row by row
        uint32_t i0 = 0, j0 = 1;
        if (hp.count) upper_pair(hp.first, hp.n, i0, j0);
        uint64_t left = hp.count;
        std::vector<uint64_t> prefix(hp.n + 1, 0);
        for (uint32_t i = 0; i < hp.n; i++) prefix[i + 1] = prefix[i] + size_of(i);
        for (uint32_t i = i0, j = j0; left > 0 && i + 1 < hp.n; i++, j = i + 1) {
            uint64_t in_row = std::min<uint64_t>(left, hp.n - j);
            sum_bytes += 8.0L * ((long double)in_row * size_of(i) + (long double)(prefix[j + in_row] - prefix[j]));
            left -= in_row;
        }
    } else if (hp.mode == PAIRS_RECT) {
        uint64_t sq = 0, sr = 0;
        for (uint32_t i = 0; i < hp.na; i++) {
            if ((rc = s.see(c, hp.a[i]))) return rc;
            sq += size_of(hp.a[i]);
        }
        for (uint32_t i = 0; i < hp.nb; i++) {
            if ((rc = s.see(c, hp.b[i]))) return rc;
            sr += size_of(hp.b[i]);
        }
        sum_bytes = 8.0L * ((long double)sq * hp.nb + (long double)sr * hp.na);
    } else {
        for (uint64_t t = 0; t < hp.count; t++) {
            if ((rc = s.see(c, hp.a[t])) || (rc = s.see(c, hp.b[t]))) return rc;
            sum_bytes += 8.0L * (size_of(hp.a[t]) + size_of(hp.b[t]));
        }
    }
    c->m.intersect_bytes = (uint64_t)sum_bytes;
    c->m.total_intersect_bytes += (uint64_t)sum_bytes;
    c->m.total_pairs += hp.count;
    if (hp.count == 0) return GKD_OK;
    const IsectPlan plan = make_plan(c, hp.count, s.max_n, s.max_level, false);
    const IsectPlan pal_plan = make_plan(c, hp.count, s.max_pal, s.max_pal_level, true);

    // device id arrays
    PairSource src{};
    src.mode = hp.mode;
    src.n = hp.n;
    if (hp.mode != PAIRS_UPPER) {
        if ((rc = ensure(c, c->ids_a, (uint64_t)hp.na * 4))) return rc;
        if ((rc = ensure(c, c->ids_b, (uint64_t)hp.nb * 4))) return rc;
        CK(cudaMemcpyAsync(c->ids_a.p, hp.a, (uint64_t)hp.na * 4, cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemcpyAsync(c->ids_b.p, hp.b, (uint64_t)hp.nb * 4, cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    if ((rc = ensure(c, c->work_counter, 8))) return rc;

    bool join_banned = false;  // set when a join table overflowed: the chunk is redone by the merge kernel
    JoinPlan jplan{};
    std::vector<uint32_t> jrows, lit_inter;
    for (uint64_t done = 0; done < hp.count;) {
        const uint64_t cnt = std::min<uint64_t>(PAIR_CHUNK, hp.count - done);
        src.count = cnt;
        bool jswapped = false;
        const bool use_join = !join_banned && plan_join(c, hp, hp.mode == PAIRS_UPPER ? hp.first + done : 0, cnt, jplan, jrows, jswapped);
        if (hp.mode == PAIRS_UPPER) {
            src.first = hp.first + done;
            src.a = src.b = nullptr;
        } else if (hp.mode == PAIRS_RECT) {
            // run_rect splits by query rows, so a rectangle always fits one launch
            src.first = 0;
            src.a = (const uint32_t *)c->ids_a.p;
            src.b = (const uint32_t *)c->ids_b.p;
            if (hp.count > PAIR_CHUNK) return fail(c, GKD_EINVAL, "query x reference block larger than %llu pairs", (unsigned long long)PAIR_CHUNK);
        } else {
            src.first = 0;
            src.a = (const uint32_t *)c->ids_a.p + done;
            src.b = (const uint32_t *)c->ids_b.p + done;
        }
        if ((rc = ensure(c, c->counts, cnt * 4))) return rc;
        CK(cudaMemsetAsync(c->counts.p, 0, cnt * 4, c->stream));
        if (need_pal) {
            if ((rc = ensure(c, c->pal_counts, cnt * 4))) return rc;
            CK(cudaMemsetAsync(c->pal_counts.p, 0, cnt * 4, c->stream));
        }

        if (use_join) {
            if ((rc = ensure(c, c->join_rows, jrows.size() * 4))) return rc;
            if ((rc = ensure(c, c->join_err, 4))) return rc;
            CK(cudaMemcpyAsync(c->join_rows.p, jrows.data(), jrows.size() * 4, cudaMemcpyHostToDevice, c->stream));
            CK(cudaMemsetAsync(c->join_err.p, 0, 4, c->stream));
            jplan.rows = (const uint32_t *)c->join_rows.p;
            if (hp.mode == PAIRS_RECT) {
                jplan.row_ids = (const uint32_t *)(jswapped ? c->ids_b.p : c->ids_a.p);
                jplan.col_ids = (const uint32_t *)(jswapped ? c->ids_a.p : c->ids_b.p);
            }
        }
        CK(cudaEventRecord(c->ev[4], c->stream));
        if (use_join) {
            nvtxRangePushA("gkd kernel 4: block join");
            CK(launch_join((const SetDesc *)c->d_sets.p, jplan, (uint32_t *)c->counts.p,
                           (unsigned long long *)c->work_counter.p, (uint32_t *)c->join_err.p, c->n_sms, c->stream));
        } else {
            nvtxRangePushA("gkd kernel 4: bucket-merge intersect");
            CK(launch_intersect((const SetDesc *)c->d_sets.p, src, 0, plan, (uint32_t *)c->counts.p,
                                (unsigned long long *)c->work_counter.p, c->n_sms, c->stream));
        }
        nvtxRangePop();
        CK(cudaEventRecord(c->ev[5], c->stream));
        c->m.intersect_kernel = use_join ? 5u : (c->low_bits == 32 ? 3u : 4u);
        uint32_t join_err = 0;
        if (use_join) {
            // a table that would overflow flags the launch; the chunk is then redone by the merge kernel
            CK(cudaMemcpyAsync(&join_err, c->join_err.p, 4, cudaMemcpyDeviceToHost, c->stream));
        }
        c->m.launches++;
        c->m.intersect_launches++;
        if (need_pal && s.max_pal) {
            CK(launch_intersect((const SetDesc *)c->d_sets.p, src, 1, pal_plan, (uint32_t *)c->pal_counts.p,
                                (unsigned long long *)c->work_counter.p, c->n_sms, c->stream));
            c->m.launches++;
        }
        CK(cudaEventRecord(c->ev[6], c->stream));
        PairCounts pc{(const SetDesc *)c->d_sets.p, (const uint32_t *)c->counts.p,
                      need_pal ? (const uint32_t *)c->pal_counts.p : nullptr, s.any_lit ? (const uint32_t *)c->lit_size.p : nullptr,
                      nullptr, both ? 1 : 0};
        if (s.any_lit) {
            // GKD_AMBIG_LITERAL: the literal k-mers live on the host, so the part of I they share is counted here while
            // kernel 4 runs; kernel 5 adds it, and the sizes, to the counts
            lit_inter.resize(cnt);
            bool shared = false;
            for (uint64_t t = 0; t < cnt; t++) {
                uint32_t a, b;
                host_pair_ids(hp, done + t, a, b);
                lit_inter[t] = (uint32_t)literal_intersection(c->genomes[a].lit, c->genomes[b].lit);
                shared = shared || lit_inter[t];
            }
            if (shared) {
                if ((rc = ensure(c, c->lit_inter, cnt * 4))) return rc;
                CK(cudaMemcpyAsync(c->lit_inter.p, lit_inter.data(), cnt * 4, cudaMemcpyHostToDevice, c->stream));
                c->m.h2d_bytes += cnt * 4;
                pc.lit_inter = (const uint32_t *)c->lit_inter.p;
            }
        }
        const Chunk e{hp, src, done, cnt, pc, use_join ? (const uint32_t *)c->join_err.p : nullptr};
        uint64_t d2h = 0;
        if ((rc = f.queue(c, e, d2h))) return rc;
        CK(cudaStreamSynchronize(c->stream));
        if (join_err) {  // the attempt keeps nothing
            join_banned = true;
            continue;
        }
        if ((rc = f.keep(c, e, d2h))) return rc;
        c->m.d2h_bytes += d2h;
        const double ims = elapsed(c->ev[4], c->ev[5]);
        c->m.intersect_ms += ims;
        c->m.total_intersect_ms += ims;
        c->m.epilogue_ms += elapsed(c->ev[6], c->ev[7]);
        done += PAIR_CHUNK;
    }
    return GKD_OK;
}

// A query x reference block with at least one pair (hp: q = a, nq = na, r = b, nr = nb), split by query rows so that
// each launch stays under PAIR_CHUNK pairs and every row is complete in one launch; f.a_base is the launch's first row.
// The call's metrics add up its launches.
int run_rect(gkd_ctx *c, const HostPairs &hp, Form &f) {
    const uint32_t nq = hp.na, nr = hp.nb;
    const uint32_t rows_per = (uint32_t)std::max<uint64_t>(1, PAIR_CHUNK / nr);
    uint64_t pairs = 0, bytes = 0;
    double ims = 0, ems = 0;
    for (uint32_t q0 = 0; q0 < nq; q0 += rows_per) {
        const uint32_t rows = std::min(rows_per, nq - q0);
        const HostPairs part{PAIRS_RECT, nr, 0, (uint64_t)rows * nr, hp.a + q0, hp.b, rows, nr};
        f.a_base = q0;
        const int rc = run_pairs(c, part, f);
        if (rc) return rc;
        pairs += c->m.pairs;
        bytes += c->m.intersect_bytes;
        ims += c->m.intersect_ms;
        ems += c->m.epilogue_ms;
    }
    c->m.pairs = pairs;
    c->m.intersect_bytes = bytes;
    c->m.intersect_ms = ims;
    c->m.epilogue_ms = ems;
    return GKD_OK;
}

// ---- selection forms --------------------------------------------------------------------------------------------
// gkd_*_within: the pairs with dist <= max_dist, in enumeration order, to the caller's hits.  hits.n counts every hit so
// far and is the next write position, so a chunk's hits are read back only once the chunk is kept.
struct Within : Form {
    double max_dist;
    gkd_hits &h;
    uint64_t wcap = 0;  // hits of the chunk the device buffers hold
    unsigned long long chunk_hits = 0;
    Within(double d, gkd_hits &hits) : max_dist(d), h(hits) {}
    std::array<const void *, 8> outputs() const override { return {h.a, h.b, h.inter, h.dist}; }
    int start(gkd_ctx *c) override {
        h.n = 0;
        return GKD_OK;
    }
    int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        const bool any_out = h.a || h.b || h.inter || h.dist;
        wcap = (any_out && h.n < h.cap) ? std::min<uint64_t>(e.cnt, h.cap - h.n) : 0;
        const uint64_t nctas = select_within_ctas(e.cnt);
        int rc;
        if ((rc = ensure(c, c->sel_cta, (nctas + 1) * 8))) return rc;
        if (h.a && (rc = ensure(c, c->hit_a, wcap * 4))) return rc;
        if (h.b && (rc = ensure(c, c->hit_b, wcap * 4))) return rc;
        if (h.inter && (rc = ensure(c, c->d_inter, wcap * 8))) return rc;
        if (h.dist && (rc = ensure(c, c->d_dist, wcap * 8))) return rc;
        const HitsOut ho{h.a ? (uint32_t *)c->hit_a.p : nullptr, h.b ? (uint32_t *)c->hit_b.p : nullptr,
                         h.inter ? (uint64_t *)c->d_inter.p : nullptr, h.dist ? (double *)c->d_dist.p : nullptr};
        unsigned long long *cta = (unsigned long long *)c->sel_cta.p;
        nvtxRangePushA("gkd kernel 5: within selection");
        CK(launch_select_within(e.src, e.pc, max_dist, a_base, wcap, ho, cta, cta + nctas, c->stream));
        nvtxRangePop();
        c->m.launches += wcap ? 3 : 2;
        CK(cudaEventRecord(c->ev[7], c->stream));
        CK(cudaMemcpyAsync(&chunk_hits, cta + nctas, 8, cudaMemcpyDeviceToHost, c->stream));
        d2h += 8;
        return GKD_OK;
    }
    int keep(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        const uint64_t w = std::min<uint64_t>(chunk_hits, wcap);
        int rc;
        if ((rc = read_back(c, h.a ? h.a + h.n : nullptr, c->hit_a.p, w * 4, d2h)) ||
            (rc = read_back(c, h.b ? h.b + h.n : nullptr, c->hit_b.p, w * 4, d2h)) ||
            (rc = read_back(c, h.inter ? h.inter + h.n : nullptr, c->d_inter.p, w * 8, d2h)) ||
            (rc = read_back(c, h.dist ? h.dist + h.n : nullptr, c->d_dist.p, w * 8, d2h)))
            return rc;
        CK(cudaStreamSynchronize(c->stream));
        h.n += chunk_hits;
        return GKD_OK;
    }
};

// gkd_*_nearest: the k nearest within max_dist by (distance bits, position).  rows (RECT only): each of the n_rows query
// rows' list, complete in every launch (k_select_nearest) and read back once the chunk is kept.  lists: per-target lists
// on the device (c->nn_*) that the launches merge into (k_nearest_absorb; UPPER: both ends of every pair, RECT: each
// reference's nearest queries), read once by finish().  A list nothing was offered to is unused: every slot pos
// 0xFFFFFFFF, inter 0, dist -1.0, and n_found 0.
struct Nearest : Form {
    uint32_t k;
    double max_dist;
    int exclude_self;
    const gkd_neighbors *rows, *lists;  // either may be nullptr
    uint32_t n_rows, targets;
    bool rows_kept = false;
    Nearest(uint32_t k_, double d, int excl, const gkd_neighbors *rows_, uint32_t n_rows_, const gkd_neighbors *lists_,
            uint32_t targets_)
        : k(k_), max_dist(d), exclude_self(excl), rows(rows_), lists(lists_), n_rows(n_rows_), targets(targets_) {}
    std::array<const void *, 8> outputs() const override {
        const gkd_neighbors none{};
        const gkd_neighbors &a = rows ? *rows : none, &b = lists ? *lists : none;
        return {a.pos, a.inter, a.dist, a.n_found, b.pos, b.inter, b.dist, b.n_found};
    }
    // the device buffers of one side's lists
    struct Bufs {
        DevBuf &pos, &inter, &dist, &found;
    };
    static Bufs row_bufs(gkd_ctx *c) { return {c->hit_a, c->d_inter, c->d_dist, c->hit_b}; }
    static Bufs list_bufs(gkd_ctx *c) { return {c->nn_pos, c->nn_inter, c->nn_dist, c->nn_found}; }
    // n unused lists in d
    int fill_unused(gkd_ctx *c, const Bufs &d, uint64_t n) {
        if (n == 0) return GKD_OK;
        const uint64_t slots = n * k;
        int rc;
        if ((rc = ensure(c, d.pos, slots * 4)) || (rc = ensure(c, d.inter, slots * 8)) || (rc = ensure(c, d.dist, slots * 8)) ||
            (rc = ensure(c, d.found, n * 4)))
            return rc;
        const double none = -1.0;
        uint64_t none_bits;
        std::memcpy(&none_bits, &none, 8);
        CK(cudaMemsetAsync(d.pos.p, 0xFF, slots * 4, c->stream));
        CK(cudaMemsetAsync(d.inter.p, 0, slots * 8, c->stream));
        CK(cudaMemsetAsync(d.found.p, 0, n * 4, c->stream));
        CK(launch_fill_u64((uint64_t *)d.dist.p, slots, none_bits, c->stream));
        c->m.launches++;
        return GKD_OK;
    }
    // lists [0, n) of d to lists [at, at + n) of out, then the stream is synchronised
    int read_lists(gkd_ctx *c, const Bufs &d, uint64_t n, const gkd_neighbors &out, uint64_t at, uint64_t &d2h) {
        const uint64_t slots = n * k, o = at * k;
        int rc;
        if ((rc = read_back(c, out.pos ? out.pos + o : nullptr, d.pos.p, slots * 4, d2h)) ||
            (rc = read_back(c, out.inter ? out.inter + o : nullptr, d.inter.p, slots * 8, d2h)) ||
            (rc = read_back(c, out.dist ? out.dist + o : nullptr, d.dist.p, slots * 8, d2h)) ||
            (rc = read_back(c, out.n_found ? out.n_found + at : nullptr, d.found.p, n * 4, d2h)))
            return rc;
        CK(cudaStreamSynchronize(c->stream));
        return GKD_OK;
    }
    int start(gkd_ctx *c) override { return lists ? fill_unused(c, list_bufs(c), targets) : GKD_OK; }
    int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        int rc;
        if (rows) {
            const uint64_t slots = (uint64_t)e.hp.na * k;
            if (rows->pos && (rc = ensure(c, c->hit_a, slots * 4))) return rc;
            if (rows->n_found && (rc = ensure(c, c->hit_b, (uint64_t)e.hp.na * 4))) return rc;
            if (rows->inter && (rc = ensure(c, c->d_inter, slots * 8))) return rc;
            if (rows->dist && (rc = ensure(c, c->d_dist, slots * 8))) return rc;
            const NearestOut no{rows->pos ? (uint32_t *)c->hit_a.p : nullptr, rows->inter ? (uint64_t *)c->d_inter.p : nullptr,
                                rows->dist ? (double *)c->d_dist.p : nullptr, rows->n_found ? (uint32_t *)c->hit_b.p : nullptr};
            nvtxRangePushA("gkd kernel 5: nearest selection");
            CK(launch_select_nearest(e.src, e.hp.na, e.pc, max_dist, k, exclude_self, no, c->stream));
            nvtxRangePop();
            c->m.launches++;
        }
        if (lists) {
            // the lists outlive this chunk: the kernel itself skips a chunk whose join overflowed
            const NearestOut st{(uint32_t *)c->nn_pos.p, (uint64_t *)c->nn_inter.p, (double *)c->nn_dist.p, (uint32_t *)c->nn_found.p};
            nvtxRangePushA("gkd kernel 5: nearest absorb");
            CK(launch_nearest_absorb(e.src, e.pc, max_dist, k, exclude_self, a_base, e.join_err, st, c->stream));
            nvtxRangePop();
            c->m.launches++;
        }
        CK(cudaEventRecord(c->ev[7], c->stream));
        return GKD_OK;
    }
    int keep(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        if (!rows) return GKD_OK;
        rows_kept = true;
        return read_lists(c, row_bufs(c), e.hp.na, *rows, a_base, d2h);
    }
    // the lists to the caller, once, at the end of the call; rows no launch reached (no reference) are unused
    int finish(gkd_ctx *c) override {
        int rc;
        uint64_t d2h = 0;
        if (rows && !rows_kept &&
            ((rc = fill_unused(c, row_bufs(c), n_rows)) || (rc = read_lists(c, row_bufs(c), n_rows, *rows, 0, d2h))))
            return rc;
        if (lists && (rc = read_lists(c, list_bufs(c), targets, *lists, 0, d2h))) return rc;
        c->m.d2h_bytes += d2h;
        return GKD_OK;
    }
};

// gkd_*_clusters: the pairs within max_dist link their nodes in the union-find forest c->uf_parent (k_cluster_link;
// RECT: query row r is node a_base + r, reference column j is node b_base + j).  Nothing is read back before finish(),
// which writes the labels of nodes [0, na) to a_out and of [na, nodes) to b_out (either may be NULL).
struct Clusters : Form {
    double max_dist;
    uint32_t nodes, b_base, na;
    uint32_t *a_out, *b_out, *n_clusters;
    Clusters(double d, uint32_t nodes_, uint32_t b_base_, uint32_t *a_out_, uint32_t na_, uint32_t *b_out_,
             uint32_t *n_clusters_)
        : max_dist(d), nodes(nodes_), b_base(b_base_), na(na_), a_out(a_out_), b_out(b_out_), n_clusters(n_clusters_) {}
    std::array<const void *, 8> outputs() const override { return {a_out, b_out}; }
    int start(gkd_ctx *c) override {  // every node its own root
        const int rc = ensure(c, c->uf_parent, ((uint64_t)nodes + 1) * 4);
        if (rc) return rc;
        CK(launch_cluster_init((uint32_t *)c->uf_parent.p, nodes, c->stream));
        c->m.launches++;
        return GKD_OK;
    }
    int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        // the forest outlives this chunk: the kernel itself skips a chunk whose join overflowed
        nvtxRangePushA("gkd kernel 5: cluster link");
        CK(launch_cluster_link(e.src, e.pc, max_dist, a_base, b_base, e.join_err, (uint32_t *)c->uf_parent.p, c->stream));
        nvtxRangePop();
        c->m.launches++;
        CK(cudaEventRecord(c->ev[7], c->stream));
        return GKD_OK;
    }
    // the labels to the caller, once, at the end of the call
    int finish(gkd_ctx *c) override {
        uint32_t *parent = (uint32_t *)c->uf_parent.p;
        CK(cudaEventRecord(c->ev[6], c->stream));
        CK(launch_cluster_flatten(parent, nodes, c->stream));
        CK(cudaEventRecord(c->ev[7], c->stream));
        c->m.launches++;
        uint32_t roots = 0;
        const uint32_t nb = nodes - na;
        if (a_out && na) CK(cudaMemcpyAsync(a_out, parent, (uint64_t)na * 4, cudaMemcpyDefault, c->stream));
        if (b_out && nb) CK(cudaMemcpyAsync(b_out, parent + na, (uint64_t)nb * 4, cudaMemcpyDefault, c->stream));
        CK(cudaMemcpyAsync(&roots, parent + nodes, 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        c->m.d2h_bytes += (a_out ? (uint64_t)na * 4 : 0) + (b_out ? (uint64_t)nb * 4 : 0) + 4;
        c->m.epilogue_ms += elapsed(c->ev[6], c->ev[7]);
        if (n_clusters) *n_clusters = roots;
        return GKD_OK;
    }
};

// gkd_*_linkage: the call's forest so far is replaced, chunk by chunk, with MSF(forest u the chunk's pairs within
// max_dist).  Node of a reported edge (a, b): a and b + b_off.
struct Linkage : Form {
    double max_dist;
    uint32_t nodes, b_off;
    std::vector<uint32_t> key;        // key of every node (empty: the node itself); uploaded to c->lk_state when not empty
    uint32_t n_dev = 0;               // edges of the device forest c->lk_forest
    unsigned long long chunk_hits = 0;
    gkd_hits *out;
    Linkage(double d, uint32_t nodes_, uint32_t b_off_, std::vector<uint32_t> key_, gkd_hits *out_)
        : max_dist(d), nodes(nodes_), b_off(b_off_), key(std::move(key_)), out(out_) {}
    std::array<const void *, 8> outputs() const override { return {out->a, out->b, out->inter, out->dist}; }
    LinkEdge edge(uint32_t a, uint32_t b, uint64_t inter, double dist) const {
        const uint32_t na = a, nb = b + b_off;
        return link_edge(a, b, inter, dist, na, nb, key.empty() ? na : key[na], key.empty() ? nb : key[nb]);
    }
    int start(gkd_ctx *c) override {  // an empty forest on the device, and the node keys there when the caller passed any
        out->n = 0;
        int rc;
        if ((rc = ensure(c, c->lk_forest, (uint64_t)nodes * 24)) || (rc = ensure(c, c->lk_state, link_state_bytes(nodes))))
            return rc;
        if (!key.empty())
            CK(cudaMemcpyAsync(link_state_at(c->lk_state.p, nodes).key, key.data(), (uint64_t)nodes * 4, cudaMemcpyHostToDevice,
                               c->stream));
        n_dev = 0;
        return GKD_OK;
    }
    int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        // every edge of the chunk within max_dist, with room behind them for the forest so far (keep)
        const uint64_t room = e.cnt + nodes;
        const uint64_t nctas = select_within_ctas(e.cnt);
        int rc;
        if ((rc = ensure(c, c->sel_cta, (nctas + 1) * 8))) return rc;
        if ((rc = ensure(c, c->hit_a, room * 4)) || (rc = ensure(c, c->hit_b, room * 4))) return rc;
        if ((rc = ensure(c, c->d_inter, room * 8)) || (rc = ensure(c, c->d_dist, room * 8))) return rc;
        const HitsOut ho{(uint32_t *)c->hit_a.p, (uint32_t *)c->hit_b.p, (uint64_t *)c->d_inter.p, (double *)c->d_dist.p};
        unsigned long long *cta = (unsigned long long *)c->sel_cta.p;
        nvtxRangePushA("gkd kernel 5: linkage edges");
        CK(launch_select_within(e.src, e.pc, max_dist, a_base, e.cnt, ho, cta, cta + nctas, c->stream));
        nvtxRangePop();
        c->m.launches += 3;
        CK(cudaMemcpyAsync(&chunk_hits, cta + nctas, 8, cudaMemcpyDeviceToHost, c->stream));
        d2h += 8;
        return GKD_OK;
    }
    // The chunk's chunk_hits edges are compacted at the front of hit_a / hit_b / d_inter / d_dist: the forest so far is
    // copied behind them and the Boruvka rounds replace it with MSF(forest u chunk).  The forest outlives the chunk, so
    // the rounds start only once the host has seen that the join held.  Records ev[7] after the rounds and reads the new
    // forest's size (4 bytes).
    int keep(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        d2h += 4;
        if (chunk_hits == 0) {  // the forest stands
            CK(cudaEventRecord(c->ev[7], c->stream));
            CK(cudaStreamSynchronize(c->stream));
            return GKD_OK;
        }
        const uint32_t N = nodes;
        uint64_t *fi = (uint64_t *)c->lk_forest.p;  // 24 B per node: inter, dist, a, b
        double *fd = (double *)(fi + N);
        uint32_t *fa = (uint32_t *)(fd + N), *fb = fa + N;
        const uint64_t f = n_dev;
        if (f) {
            CK(cudaMemcpyAsync((uint32_t *)c->hit_a.p + chunk_hits, fa, f * 4, cudaMemcpyDeviceToDevice, c->stream));
            CK(cudaMemcpyAsync((uint32_t *)c->hit_b.p + chunk_hits, fb, f * 4, cudaMemcpyDeviceToDevice, c->stream));
            CK(cudaMemcpyAsync((uint64_t *)c->d_inter.p + chunk_hits, fi, f * 8, cudaMemcpyDeviceToDevice, c->stream));
            CK(cudaMemcpyAsync((double *)c->d_dist.p + chunk_hits, fd, f * 8, cudaMemcpyDeviceToDevice, c->stream));
        }
        const LinkState st = link_state_at(c->lk_state.p, N);
        const LinkGraph g{(const uint32_t *)c->hit_a.p, (const uint32_t *)c->hit_b.p, (const uint64_t *)c->d_inter.p,
                          (const double *)c->d_dist.p, chunk_hits + f, b_off, key.empty() ? nullptr : st.key};
        if (g.n_edges >= LINK_NONE) return fail(c, GKD_EINVAL, "linkage: %llu edges in one pass", (unsigned long long)g.n_edges);
        uint32_t rounds = 1;
        while (rounds < LINK_MAX_ROUNDS && (1ull << rounds) < N) rounds++;
        nvtxRangePushA("gkd kernel 5: linkage rounds");
        CK(launch_link_rounds(g, st, LinkForest{fa, fb, fi, fd}, rounds, c->stream));
        nvtxRangePop();
        c->m.launches += 1 + 5 * rounds;
        uint32_t n_forest = 0;
        CK(cudaEventRecord(c->ev[7], c->stream));
        CK(cudaMemcpyAsync(&n_forest, st.n_forest, 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        n_dev = n_forest;
        return GKD_OK;
    }
    // The forest to the caller, once, at the end of the call: the device forest is copied to the host and sorted there by
    // one Kruskal pass (a forest keeps every edge).
    int finish(gkd_ctx *c) override {
        std::vector<LinkEdge> edges;
        const uint64_t f = n_dev, N = nodes;
        if (f) {
            std::vector<uint64_t> in(f);
            std::vector<double> d(f);
            std::vector<uint32_t> a(f), b(f);
            const uint64_t *fi = (const uint64_t *)c->lk_forest.p;
            const double *fd = (const double *)(fi + N);
            const uint32_t *fa = (const uint32_t *)(fd + N), *fb = fa + N;
            CK(cudaMemcpyAsync(in.data(), fi, f * 8, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaMemcpyAsync(d.data(), fd, f * 8, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaMemcpyAsync(a.data(), fa, f * 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaMemcpyAsync(b.data(), fb, f * 4, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            c->m.d2h_bytes += f * 24;
            for (uint64_t t = 0; t < f; t++) edges.push_back(edge(a[t], b[t], in[t], d[t]));
        }
        host_msf(edges, nodes);
        out->n = edges.size();
        const uint64_t w = std::min<uint64_t>(out->n, out->cap);
        if (w == 0) return GKD_OK;
        std::vector<uint32_t> a(w), b(w);
        std::vector<uint64_t> in(w);
        std::vector<double> d(w);
        for (uint64_t t = 0; t < w; t++) a[t] = edges[t].a, b[t] = edges[t].b, in[t] = edges[t].inter, d[t] = edges[t].dist;
        if (out->a) CK(cudaMemcpyAsync(out->a, a.data(), w * 4, cudaMemcpyDefault, c->stream));
        if (out->b) CK(cudaMemcpyAsync(out->b, b.data(), w * 4, cudaMemcpyDefault, c->stream));
        if (out->inter) CK(cudaMemcpyAsync(out->inter, in.data(), w * 8, cudaMemcpyDefault, c->stream));
        if (out->dist) CK(cudaMemcpyAsync(out->dist, d.data(), w * 8, cudaMemcpyDefault, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        return GKD_OK;
    }
};

// ---- complete / average linkage ------------------------------------------------------------------------------------
// S / (N 2^53) rounded to the nearest double, ties to even (S = lo + hi 2^64, N >= 1)
double agg_round(uint64_t lo, uint64_t hi, uint64_t N) {
    const unsigned __int128 S = (unsigned __int128)hi << 64 | lo;
    unsigned __int128 q = S / N, r = S % N;
    if (q == 0 && r == 0) return 0.0;
    int e = -53;  // value = (q + r / N) 2^e
    while (q < ((unsigned __int128)1 << 55)) {  // at least 56 quotient bits: 53 kept, a round bit and two more
        r <<= 1;
        q = q << 1 | (r >= N ? 1 : 0);
        if (r >= N) r -= N;
        e--;
    }
    int bits = 0;
    for (unsigned __int128 t = q; t; t >>= 1) bits++;
    const int drop = bits - 53;
    uint64_t keep = (uint64_t)(q >> drop);
    const unsigned __int128 rest = q & (((unsigned __int128)1 << drop) - 1), half = (unsigned __int128)1 << (drop - 1);
    if (rest > half || (rest == half && (r != 0 || (keep & 1)))) keep++;
    return std::ldexp((double)keep, e + drop);
}

// One complete- or average-linkage agglomeration on the context's device (gkd_all_vs_all_agglomerate, gkd_agglomerate):
// start() checks the free memory and sets up the matrix and state of agglomerate.cu in one buffer of the call; the
// distances are scattered into it (scatter); finish() runs the rounds, reads the merges back and writes them to out in
// the sequential order.
struct Agglomeration {
    const char *fn;
    uint32_t n;
    int average;
    double max_dist;
    gkd_merges *out;
    void *buf = nullptr;
    cudaStream_t stream = nullptr;
    AggState st{};
    Agglomeration(const char *fn_, uint32_t n_, int method, double d, gkd_merges *out_)
        : fn(fn_), n(n_), average(method == GKD_LINK_AVERAGE), max_dist(d), out(out_) {}
    ~Agglomeration() {
        if (buf) cudaFreeAsync(buf, stream);
    }
    std::array<const void *, 8> outputs() const { return {out->a, out->b, out->height, out->size}; }
    int start(gkd_ctx *c) {
        out->n = 0;
        c->m.agglomerate_rounds = 0;
        if (n < 2) return GKD_OK;
        const uint64_t need = agg_state_bytes(n, average);
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        if (need > free_b)
            return fail(c, GKD_ENOMEM, "%s: %s linkage of %u sets needs %llu bytes of device memory; %llu are free", fn,
                        average ? "average" : "complete", n, (unsigned long long)need, (unsigned long long)free_b);
        stream = c->stream;
        CK(cudaMallocAsync(&buf, need, c->stream));
        st = agg_state_at(buf, n, average);
        CK(launch_agg_init(st, c->stream));
        c->m.launches++;
        return GKD_OK;
    }
    // entries [first, first + count) of the triangle, as doubles in device memory
    int scatter(gkd_ctx *c, const double *src, uint64_t first, uint64_t count, const uint32_t *join_err) {
        CK(launch_agg_scatter(st, src, first, count, join_err, c->stream));
        c->m.launches++;
        return GKD_OK;
    }
    int finish(gkd_ctx *c) {
        if (n < 2) return GKD_OK;
        unsigned long long ctr[AGG_COUNTERS];
        CK(cudaMemcpyAsync(ctr, st.ctr, sizeof(ctr), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        c->m.d2h_bytes += sizeof(ctr);
        if (ctr[AGG_BAD] != ~0ull) {
            uint32_t i, j;
            upper_pair(ctr[AGG_BAD], n, i, j);
            return fail(c, GKD_EINVAL, "%s: the distance of pair (%u, %u) is not a multiple of 2^-53 in [0, 2]", fn, i, j);
        }
        if (max_dist < 0) return GKD_OK;
        AggThreshold thr{0, 0, max_dist >= 2.0 ? 1 : 0};
        if (!thr.all) {
            int e = 0;
            const double fr = std::frexp(max_dist, &e);  // max_dist = m 2^(e - 53)
            thr.m = (uint64_t)std::ldexp(fr, 53);
            thr.shift = e;
        }
        // batches of rounds without a host read in between; a batch that ends with AGG_DONE set is the last
        CK(cudaEventRecord(c->ev[6], c->stream));
        uint64_t queued = 0;
        for (uint32_t batch = 8;; batch = std::min<uint32_t>(batch * 2, 512)) {
            CK(launch_agg_rounds(st, thr, batch, c->n_sms, c->stream));
            c->m.launches += 4ull * batch;
            queued += batch;
            CK(cudaMemcpyAsync(ctr, st.ctr, sizeof(ctr), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            c->m.d2h_bytes += sizeof(ctr);
            if (ctr[AGG_DONE]) break;
            // every round but the last merges at least one pair
            if (queued > (uint64_t)n + 1024) return fail(c, GKD_EINVAL, "internal error: %s did not finish in %llu rounds", fn,
                                                          (unsigned long long)queued);
        }
        CK(cudaEventRecord(c->ev[7], c->stream));
        const uint64_t m = ctr[AGG_N_MERGES];
        std::vector<AggMerge> ms(m);
        if (m) CK(cudaMemcpyAsync(ms.data(), st.merges, m * sizeof(AggMerge), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        c->m.d2h_bytes += m * sizeof(AggMerge);
        c->m.epilogue_ms += elapsed(c->ev[6], c->ev[7]);
        c->m.agglomerate_rounds = ctr[AGG_ROUNDS];
        // the merge keys strictly increase in the sequential order
        auto N = [&](const AggMerge &x) -> uint64_t { return average ? (uint64_t)x.sa * x.sb : 1; };
        std::sort(ms.begin(), ms.end(), [&](const AggMerge &x, const AggMerge &y) {
            const int k = agg_cmp(x.lo, x.hi, N(x), y.lo, y.hi, N(y));
            return k < 0 || (k == 0 && (x.a < y.a || (x.a == y.a && x.b < y.b)));
        });
        out->n = m;
        const uint64_t w = std::min<uint64_t>(m, out->cap);
        if (w == 0) return GKD_OK;
        std::vector<uint32_t> a(w), b(w), size(w);
        std::vector<double> h(w);
        for (uint64_t t = 0; t < w; t++) {
            const AggMerge &x = ms[t];
            a[t] = x.a;
            b[t] = x.b;
            size[t] = x.sa + x.sb;
            h[t] = average ? agg_round(x.lo, x.hi, N(x)) : std::ldexp((double)x.lo, -53);
        }
        if (out->a) CK(cudaMemcpyAsync(out->a, a.data(), w * 4, cudaMemcpyDefault, c->stream));
        if (out->b) CK(cudaMemcpyAsync(out->b, b.data(), w * 4, cudaMemcpyDefault, c->stream));
        if (out->height) CK(cudaMemcpyAsync(out->height, h.data(), w * 8, cudaMemcpyDefault, c->stream));
        if (out->size) CK(cudaMemcpyAsync(out->size, size.data(), w * 4, cudaMemcpyDefault, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        return GKD_OK;
    }
};

// gkd_all_vs_all_agglomerate: each chunk's distances (the dense epilogue's doubles) go straight into the matrix; a chunk
// whose join overflowed writes nothing and its redo writes the same entries, so the rounds in finish() see final values.
struct Agglomerate : Form {
    Agglomeration g;
    Agglomerate(uint32_t n, int method, double d, gkd_merges *out) : g("gkd_all_vs_all_agglomerate", n, method, d, out) {}
    std::array<const void *, 8> outputs() const override { return g.outputs(); }
    int start(gkd_ctx *c) override { return g.start(c); }
    int queue(gkd_ctx *c, const Chunk &e, uint64_t &d2h) override {
        int rc = ensure(c, c->d_dist, e.cnt * 8);
        if (rc) return rc;
        nvtxRangePushA("gkd kernel 5: agglomerate matrix");
        CK(launch_epilogue(e.src, e.pc, EpilogueOut{nullptr, (double *)c->d_dist.p, nullptr, nullptr}, c->stream));
        c->m.launches++;
        rc = g.scatter(c, (const double *)c->d_dist.p, e.src.first, e.cnt, e.join_err);
        nvtxRangePop();
        if (rc) return rc;
        CK(cudaEventRecord(c->ev[7], c->stream));
        return GKD_OK;
    }
    int finish(gkd_ctx *c) override { return g.finish(c); }
};

// the triangle over the first n sets, and the block of queries q x references r
HostPairs triangle(uint32_t n) { return {PAIRS_UPPER, n, 0, (uint64_t)n * (n - 1) / 2, nullptr, nullptr, 0, 0}; }
HostPairs block(const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr) {
    return {PAIRS_RECT, nr, 0, (uint64_t)nq * nr, q, r, nq, nr};
}

// gkd.h publishes host memory as the only output memory of a GKD_AMBIG_LITERAL context, so device buffers are refused in
// that mode
int host_outputs_ok(gkd_ctx *c, const char *fn, const std::array<const void *, 8> &ps) {
    if (c->cfg.ambig_policy != GKD_AMBIG_LITERAL) return GKD_OK;
    for (const void *p : ps)
        if (p && classify(p) == MEM_DEVICE) return fail(c, GKD_EINVAL, "%s: GKD_AMBIG_LITERAL needs host output buffers", fn);
    return GKD_OK;
}

// One pair call on one device, for every form: the context, the shape of the pairs (messages start with fn), the
// caller's outputs, every id the call names (also when it has no pairs), then the form's start, the chunks and the
// form's finish.  RECT: hp is the caller's whole block.
int run_call(gkd_ctx *c, const char *fn, const HostPairs &hp, Form &f) {
    CHECK_CTX(c);
    CK(cudaSetDevice(c->cfg.device));
    if (hp.mode == PAIRS_UPPER) {
        if (hp.n > c->genomes.size()) return fail(c, GKD_EINVAL, "%s: %u sets but only %zu exist", fn, hp.n, c->genomes.size());
        const uint64_t total = (uint64_t)hp.n * (hp.n - 1) / 2;
        if (hp.first > total || hp.count > total - hp.first)
            return fail(c, GKD_EINVAL, "%s: pair range [%llu, +%llu) outside 0..%llu", fn, (unsigned long long)hp.first,
                        (unsigned long long)hp.count, (unsigned long long)total);
    } else {
        if ((hp.na && !hp.a) || (hp.nb && !hp.b)) return fail(c, GKD_EINVAL, "%s: null id array", fn);
        if (hp.mode == PAIRS_LIST && hp.count > 0xFFFFFFFFull)
            return fail(c, GKD_EINVAL, "%s: more than 2^32 pairs in one call", fn);
    }
    int rc = host_outputs_ok(c, fn, f.outputs());
    if (rc) return rc;
    // the metrics of this call alone (run_pairs sets them again for each launch)
    c->m.pairs = c->m.intersect_bytes = 0;
    c->m.intersect_ms = c->m.epilogue_ms = 0;
    ABI_GUARD_BEGIN
    if (hp.mode == PAIRS_UPPER) {
        for (uint32_t i = 0; i < hp.n; i++)
            if ((rc = check_built(c, i))) return rc;
    } else if (hp.mode == PAIRS_RECT) {
        for (uint32_t i = 0; i < hp.na; i++)
            if ((rc = check_built(c, hp.a[i]))) return rc;
        for (uint32_t j = 0; j < hp.nb; j++)
            if ((rc = check_built(c, hp.b[j]))) return rc;
    } else {
        for (uint64_t t = 0; t < hp.count; t++)
            if ((rc = check_built(c, hp.a[t])) || (rc = check_built(c, hp.b[t]))) return rc;
    }
    if ((rc = f.start(c))) return rc;
    if (hp.count && (rc = hp.mode == PAIRS_RECT ? run_rect(c, hp, f) : run_pairs(c, hp, f))) return rc;
    return f.finish(c);
    ABI_GUARD_END(c)
}

int default_k(int alphabet) { return alphabet == GKD_PROT ? 8 : 21; }

}  // namespace

// =============================================================================================================
// extern "C" ABI
// =============================================================================================================
extern "C" {

int gkd_abi_version(void) { return GKD_ABI_VERSION; }

const char *gkd_last_error(const gkd_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int gkd_create(gkd_ctx **out, const gkd_config *cfg) {
    if (!out || !cfg) return fail(nullptr, GKD_EINVAL, "gkd_create: null argument");
    *out = nullptr;
    if (cfg->alphabet < GKD_DNA || cfg->alphabet > GKD_RNA) return fail(nullptr, GKD_EINVAL, "unknown alphabet %d", cfg->alphabet);
    int k = cfg->k == 0 ? default_k(cfg->alphabet) : cfg->k;
    int kmax = cfg->alphabet == GKD_PROT ? 8 : 32;
    if (k < 1 || k > kmax)
        return fail(nullptr, GKD_EINVAL, "kmer size %d is outside the exact-key range 1..%d of this alphabet", k, kmax);
    if (cfg->strand_mode != GKD_STRAND_BOTH && cfg->strand_mode != GKD_STRAND_CANONICAL)
        return fail(nullptr, GKD_EINVAL, "unknown strand mode %d", cfg->strand_mode);
    if (cfg->ambig_policy != GKD_AMBIG_SKIP && cfg->ambig_policy != GKD_AMBIG_LITERAL)
        return fail(nullptr, GKD_EINVAL, "unknown ambiguity policy %d", cfg->ambig_policy);
    if (cfg->ambig_policy == GKD_AMBIG_LITERAL && cfg->alphabet != GKD_PROT && cfg->strand_mode != GKD_STRAND_BOTH)
        return fail(nullptr, GKD_EINVAL, "literal ambiguous k-mers are defined for the both-strand sets only");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, GKD_ECUDA, "no CUDA device available (%s); libgkd has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, GKD_EINVAL, "device %d out of range (have %d)", cfg->device, ndev);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess)
        return fail(nullptr, GKD_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, GKD_ECUDA, "device %d is sm_%d%d; libgkd is built for sm_100a (B200) only", cfg->device, prop.major, prop.minor);
    gkd_ctx *c = new (std::nothrow) gkd_ctx();
    if (!c) return fail(nullptr, GKD_ENOMEM, "out of host memory");
    c->cfg = *cfg;
    c->k = k;
    c->cfg.k = k;
    if (c->cfg.workspace_bytes == 0) c->cfg.workspace_bytes = DEFAULT_WORKSPACE;
    c->n_sms = prop.multiProcessorCount;
    c->key_bits = cfg->alphabet == GKD_PROT ? 8 * k : 2 * k;
    c->low_bits = low_bits_for(c->key_bits);
    c->lvl_min = level_min(c->key_bits, c->low_bits);
    c->mix = make_mix(c->key_bits);
    c->isect_tmax = intersect_default_tmax(c->low_bits);
    c->table_tmax = c->isect_tmax;
    if (const char *t = getenv("GKD_TABLE_TMAX")) c->table_tmax = (uint32_t)std::max(1, atoi(t));
#define CK_CREATE(call)                                                                        \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            fail(nullptr, GKD_ECUDA, "%s: %s", #call, cudaGetErrorString(e__));                \
            delete c;                                                                          \
            return GKD_ECUDA;                                                                  \
        }                                                                                      \
    } while (0)
    CK_CREATE(cudaSetDevice(cfg->device));
    CK_CREATE(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    {
        // highest priority: the pack kernels are tiny and sit between the copies, so they must not queue behind the
        // grids of a running build batch (the next copy of the stream could not start)
        int prio_lo = 0, prio_hi = 0;
        CK_CREATE(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CK_CREATE(cudaStreamCreateWithPriority(&c->copy_stream, cudaStreamNonBlocking, prio_hi));
        CK_CREATE(cudaStreamCreateWithPriority(&c->pack_stream, cudaStreamNonBlocking, prio_hi));
    }
    CK_CREATE(cudaEventCreateWithFlags(&c->slab_ev, cudaEventDisableTiming));
    cudaMemPool_t pool;
    CK_CREATE(cudaDeviceGetDefaultMemPool(&pool, cfg->device));
    uint64_t thresh = UINT64_MAX;
    CK_CREATE(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh));
    for (int i = 0; i < N_STAGE; i++) {
        CK_CREATE(cudaMallocHost((void **)&c->bounce[i], STAGE_BYTES));
        CK_CREATE(cudaEventCreateWithFlags(&c->bounce_ev[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < N_DSTAGE; i++) {
        CK_CREATE(cudaMalloc((void **)&c->stage_dev[i], STAGE_BYTES + 256));
        CK_CREATE(cudaEventCreateWithFlags(&c->copied[i], cudaEventDisableTiming));
        CK_CREATE(cudaEventCreateWithFlags(&c->packed[i], cudaEventDisableTiming));
    }
    for (auto &ev : c->ev) CK_CREATE(cudaEventCreate(&ev));
    // function attributes are per device: every context sets them for its own device
    CK_CREATE(intersect_configure());
    CK_CREATE(join_configure());
    CK_CREATE(sort_configure());
    CK_CREATE(sketch_configure());
    CK_CREATE(msd_configure());
    if (const char *a = getenv("GKD_SORT_ALGO")) c->use_msd = !(a[0] == 'l' || a[0] == 'L');
    if (const char *a = getenv("GKD_ISECT_ALGO")) c->isect_algo = (a[0] == 'm' || a[0] == 'M') ? 1 : (a[0] == 'j' || a[0] == 'J') ? 2 : 0;
#undef CK_CREATE
    *out = c;
    return GKD_OK;
}

static void release_arenas_from(gkd_ctx *c, size_t first_dropped) {
    for (size_t i = first_dropped; i < c->arenas.size(); i++)
        if (c->arenas[i].owned) c->free_arenas.push_back({c->arenas[i].base, c->arenas[i].capacity});
    c->arenas.resize(first_dropped);
}

static int trim_free_arenas(gkd_ctx *c, size_t keep) {
    // keep at most a handful of spare arenas; release the smallest ones beyond that
    while (c->free_arenas.size() > keep) {
        size_t small = 0;
        for (size_t i = 1; i < c->free_arenas.size(); i++)
            if (c->free_arenas[i].second < c->free_arenas[small].second) small = i;
        CK(cudaFreeAsync(c->free_arenas[small].first, c->stream));
        c->free_arenas.erase(c->free_arenas.begin() + small);
    }
    return GKD_OK;
}

// the `ready` events of genomes first.. go back to the pool (both streams are idle when this is called)
static void recycle_events(gkd_ctx *c, size_t first) {
    for (size_t i = first; i < c->genomes.size(); i++)
        if (c->genomes[i].ready) {
            c->ev_pool.push_back(c->genomes[i].ready);
            c->genomes[i].ready = nullptr;
        }
}

int gkd_reset(gkd_ctx *c) {
    CHECK_CTX(c);
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaStreamSynchronize(c->copy_stream));
    CK(cudaStreamSynchronize(c->pack_stream));
    CK(cudaStreamSynchronize(c->stream));
    recycle_events(c, 0);
    release_arenas_from(c, 0);
    int rc = trim_free_arenas(c, 16);
    if (rc) return rc;
    for (auto &s : c->slabs) s.used = 0;
    c->genomes.clear();
    c->lit_dict.clear();
    c->built_upto = 0;
    c->sets_dirty = true;
    uint64_t launches = c->m.launches, il = c->m.intersect_launches;
    c->m = gkd_metrics{};
    c->m.launches = launches;
    c->m.intersect_launches = il;
    return GKD_OK;
}

int gkd_truncate(gkd_ctx *c, uint32_t n_keep) {
    CHECK_CTX(c);
    if (n_keep >= c->genomes.size()) return GKD_OK;
    CK(cudaSetDevice(c->cfg.device));
    CK(cudaStreamSynchronize(c->copy_stream));
    CK(cudaStreamSynchronize(c->pack_stream));
    CK(cudaStreamSynchronize(c->stream));
    recycle_events(c, n_keep);
    // arenas are created in id order, one per build/import/adopt batch: recycle those that hold only dropped sets
    size_t keep = c->arenas.size();
    while (keep > 0 && c->arenas[keep - 1].first_id >= n_keep) keep--;
    release_arenas_from(c, keep);
    int rc = trim_free_arenas(c, 16);
    if (rc) return rc;
    c->genomes.resize(n_keep);
    if (c->built_upto > n_keep) c->built_upto = n_keep;
    c->sets_dirty = true;
    return GKD_OK;
}

int gkd_destroy(gkd_ctx *c) {
    if (!c) return GKD_EINVAL;
    cudaSetDevice(c->cfg.device);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->pack_stream) cudaStreamSynchronize(c->pack_stream);
    cudaStreamSynchronize(c->stream);
    recycle_events(c, 0);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    if (c->slab_ev) cudaEventDestroy(c->slab_ev);
    for (auto &a : c->arenas)
        if (a.owned) cudaFreeAsync(a.base, c->stream);
    for (auto &a : c->free_arenas) cudaFreeAsync(a.first, c->stream);
    for (auto &s : c->slabs) cudaFreeAsync(s.base, c->stream);
    DevBuf *bufs[] = {&c->keys_a, &c->keys_b, &c->tile_hist, &c->tile_uniq, &c->genome_counts, &c->batch_genomes,
                      &c->set_build, &c->d_sets, &c->counts, &c->pal_counts, &c->d_inter, &c->d_dist, &c->d_ca,
                      &c->d_cb, &c->ids_a, &c->ids_b, &c->work_counter, &c->sk_cand, &c->sk_misc, &c->sk_sig,
                      &c->sk_len, &c->sk_out, &c->msd_genomes, &c->msd_bins32, &c->msd_bins64, &c->msd_gstat,
                      &c->gr_reps, &c->gr_flags, &c->join_rows, &c->join_err, &c->hit_a, &c->hit_b, &c->sel_cta, &c->nn_pos, &c->nn_inter,
                      &c->nn_dist, &c->nn_found, &c->uf_parent, &c->lk_forest, &c->lk_state, &c->lit_size, &c->lit_inter};
    for (DevBuf *b : bufs)
        if (b->p) cudaFreeAsync(b->p, c->stream);
    cudaStreamSynchronize(c->stream);
    for (int i = 0; i < N_STAGE; i++) {
        if (c->bounce[i]) cudaFreeHost(c->bounce[i]);
        if (c->bounce_ev[i]) cudaEventDestroy(c->bounce_ev[i]);
    }
    for (int i = 0; i < N_DSTAGE; i++) {
        if (c->stage_dev[i]) cudaFree(c->stage_dev[i]);
        if (c->copied[i]) cudaEventDestroy(c->copied[i]);
        if (c->packed[i]) cudaEventDestroy(c->packed[i]);
    }
    for (auto &ev : c->ev)
        if (ev) cudaEventDestroy(ev);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->pack_stream) cudaStreamDestroy(c->pack_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    cudaGetLastError();
    delete c;
    return GKD_OK;
}

int gkd_add_sequences(gkd_ctx *c, const char *const *contigs, const uint64_t *lens, uint32_t n_contigs, uint32_t *out_id) {
    CHECK_CTX(c);
    if (n_contigs && (!contigs || !lens)) return fail(c, GKD_EINVAL, "gkd_add_sequences: null contig array");
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    std::vector<Part> parts;
    parts.reserve(n_contigs);
    for (uint32_t i = 0; i < n_contigs; i++) {
        if (lens[i] && !contigs[i]) return fail(c, GKD_EINVAL, "gkd_add_sequences: contig %u is null", i);
        parts.push_back(Part{contigs[i], lens[i], true});
    }
    return add_genome(c, parts, "", "", out_id);
    ABI_GUARD_END(c)
}

int gkd_add_fasta_file(gkd_ctx *c, const char *path, int per_record, uint32_t *first_id, uint32_t *n_added) {
    CHECK_CTX(c);
    if (!path) return fail(c, GKD_EINVAL, "gkd_add_fasta_file: null path");
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    std::vector<char> storage;
    std::vector<FastaRecord> recs;
    std::string err;
    if (gkd_parse_fasta_file(path, storage, recs, err)) return fail(c, GKD_EIO, "%s", err.c_str());
    uint32_t first = (uint32_t)c->genomes.size(), added = 0;
    if (per_record) {
        for (auto &r : recs) {
            std::vector<Part> parts;
            bool firstp = true;
            for (auto &l : r.lines) {
                parts.push_back(Part{l.ptr, l.len, firstp});
                firstp = false;
            }
            int rc = add_genome(c, parts, r.label, r.comment, nullptr);
            if (rc) return rc;
            added++;
        }
    } else {
        std::vector<Part> parts;
        for (auto &r : recs) {
            bool firstp = true;
            for (auto &l : r.lines) {
                parts.push_back(Part{l.ptr, l.len, firstp});
                firstp = false;
            }
            if (r.lines.empty()) parts.push_back(Part{"", 0, true});
        }
        std::string label = recs.empty() ? "" : recs[0].label, comment = recs.empty() ? "" : recs[0].comment;
        int rc = add_genome(c, parts, label, comment, nullptr);
        if (rc) return rc;
        added = 1;
    }
    // the staged pieces reference `storage` (pageable): they were consumed by memcpy before add_genome returned
    if (first_id) *first_id = first;
    if (n_added) *n_added = added;
    return GKD_OK;
    ABI_GUARD_END(c)
}

const char *gkd_label(const gkd_ctx *c, uint32_t id) { return (c && id < c->genomes.size()) ? c->genomes[id].label.c_str() : ""; }
const char *gkd_comment(const gkd_ctx *c, uint32_t id) { return (c && id < c->genomes.size()) ? c->genomes[id].comment.c_str() : ""; }
uint32_t gkd_count(const gkd_ctx *c) { return c ? (uint32_t)c->genomes.size() : 0; }

int gkd_set_label(gkd_ctx *c, uint32_t id, const char *label, const char *comment) {
    if (!c) return GKD_EINVAL;
    if (id >= c->genomes.size()) return fail(c, GKD_EINVAL, "set id %u out of range (have %zu)", id, c->genomes.size());
    ABI_GUARD_BEGIN
    c->genomes[id].label = label ? label : "";
    c->genomes[id].comment = comment ? comment : "";
    return GKD_OK;
    ABI_GUARD_END(c)
}

int gkd_build_sets(gkd_ctx *c) {
    CHECK_CTX(c);
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    const uint32_t n = (uint32_t)c->genomes.size();
    // skip sets that were imported ready-made
    while (c->built_upto < n) {
        if (c->genomes[c->built_upto].built) {
            c->built_upto++;
            continue;
        }
        // greedy batch under the workspace cap (two key buffers of 8 B per slot)
        const uint64_t cap_keys = std::max<uint64_t>(c->cfg.workspace_bytes / 16, SORT_TILE);
        uint64_t raw = 0;
        uint32_t last = c->built_upto;
        while (last < n && !c->genomes[last].built) {
            uint64_t slots = c->genomes[last].n_pos >= (uint64_t)c->k ? c->genomes[last].n_pos - c->k + 1 : 0;
            slots = (slots + 15) & ~15ull;
            if (last > c->built_upto && raw + slots > cap_keys) break;
            raw += slots;
            last++;
        }
        int rc = build_batch(c, c->built_upto, last);
        if (rc) return rc;
        c->built_upto = last;
    }
    // pinned / device input text of gkd_add_sequences may be released by the caller from here on
    CK(cudaStreamSynchronize(c->stream));
    return upload_sets(c);
    ABI_GUARD_END(c)
}

int gkd_set_size(const gkd_ctx *c, uint32_t id, uint64_t *n_both, uint64_t *n_canonical, uint64_t *n_palindromic) {
    if (!c) return GKD_EINVAL;
    if (id >= c->genomes.size() || !c->genomes[id].built) return GKD_ESTATE;
    const GenomeRec &g = c->genomes[id];
    if (n_both) *n_both = both_size(c, g);
    if (n_canonical) *n_canonical = g.desc.main.n;
    if (n_palindromic) *n_palindromic = g.desc.pal.n;
    return GKD_OK;
}

int gkd_export_set(gkd_ctx *c, uint32_t id, uint64_t *keys, uint64_t cap, uint64_t *n) {
    CHECK_CTX(c);
    int rc = check_built(c, id);
    if (rc) return rc;
    const SetDesc &d = c->genomes[id].desc;
    if (n) *n = d.main.n;
    if (!keys) return GKD_OK;
    if (cap < d.main.n) return fail(c, GKD_EINVAL, "export buffer holds %llu keys, set has %u", (unsigned long long)cap, d.main.n);
    if (d.main.n == 0) return GKD_OK;
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    // un-mix into the sort workspace, sort ascending by key, copy out
    std::vector<BatchGenome> bg(1);
    bg[0] = BatchGenome{nullptr, nullptr, 0, 0, d.main.n, 0, (d.main.n + SORT_TILE - 1) / SORT_TILE};
    SortPlan plan{};
    if ((rc = plan_batch(c, bg, plan, d.main.n, bg[0].n_tiles))) return rc;
    CK(launch_unmix_set(d.main, c->mix, c->low_bits, plan.keys_a, c->stream));
    uint64_t *sorted = nullptr;
    uint32_t passes = 0;
    CK(launch_sort((const BatchGenome *)c->batch_genomes.p, plan, &sorted, &passes, c->stream));
    c->m.launches += 1 + 3ull * passes;
    CK(cudaMemcpyAsync(keys, sorted, (uint64_t)d.main.n * 8, cudaMemcpyDefault, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->m.d2h_bytes += (uint64_t)d.main.n * 8;
    return GKD_OK;
    ABI_GUARD_END(c)
}

int gkd_import_sets(gkd_ctx *c, const uint64_t *keys, const uint64_t *offsets, uint32_t n_sets, uint32_t *first_id) {
    CHECK_CTX(c);
    if (first_id) *first_id = (uint32_t)c->genomes.size();
    if (n_sets == 0) return GKD_OK;
    if (!offsets) return fail(c, GKD_EINVAL, "gkd_import_sets: null offsets");
    const uint64_t total = offsets[n_sets] - offsets[0];
    if (total && !keys) return fail(c, GKD_EINVAL, "gkd_import_sets: null keys");
    for (uint32_t i = 0; i < n_sets; i++)
        if (offsets[i + 1] < offsets[i] || offsets[i + 1] - offsets[i] >= 0xFFFF0000ull)
            return fail(c, GKD_EINVAL, "gkd_import_sets: bad offsets at set %u", i);
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    const bool on_device = total && classify(keys) == MEM_DEVICE;
    // batches under the workspace cap, like gkd_build_sets
    const uint64_t cap_keys = std::max<uint64_t>(c->cfg.workspace_bytes / 16, SORT_TILE);
    const uint32_t id0 = (uint32_t)c->genomes.size();
    for (uint32_t i0 = 0; i0 < n_sets;) {
        uint32_t i1 = i0 + 1;
        while (i1 < n_sets && offsets[i1 + 1] - offsets[i0] <= cap_keys) i1++;
        int rc = import_device_batch(c, keys, offsets, i0, i1, on_device);
        if (rc) {
            gkd_truncate(c, id0);
            return rc;
        }
        i0 = i1;
    }
    return GKD_OK;
    ABI_GUARD_END(c)
}

int gkd_import_set(gkd_ctx *c, const uint64_t *keys, uint64_t n, uint32_t *out_id) {
    uint64_t offsets[2] = {0, n};
    return gkd_import_sets(c, keys, offsets, 1, out_id);
}

// ---- set exchange ---------------------------------------------------------------------------------------
uint32_t gkd_arena_count(const gkd_ctx *c) { return c ? (uint32_t)c->arenas.size() : 0; }

int gkd_arena_info(const gkd_ctx *c, uint32_t arena, uint32_t *first_id, uint32_t *n_sets, const void **base, uint64_t *bytes) {
    if (!c || arena >= c->arenas.size()) return GKD_EINVAL;
    const Arena &a = c->arenas[arena];
    if (first_id) *first_id = a.first_id;
    if (n_sets) *n_sets = a.n_sets;
    if (base) *base = a.base;
    if (bytes) *bytes = a.bytes;
    return GKD_OK;
}

int gkd_describe_sets(const gkd_ctx *cc, uint32_t first_id, uint32_t n_sets, gkd_packed_set *table) {
    gkd_ctx *c = const_cast<gkd_ctx *>(cc);
    if (!c) return GKD_EINVAL;
    if (n_sets == 0) return GKD_OK;
    if (!table) return fail(c, GKD_EINVAL, "gkd_describe_sets: null table");
    if ((uint64_t)first_id + n_sets > c->genomes.size()) return fail(c, GKD_EINVAL, "gkd_describe_sets: ids out of range");
    const int arena = c->genomes[first_id].arena;
    for (uint32_t i = 0; i < n_sets; i++) {
        const GenomeRec &g = c->genomes[first_id + i];
        if (!g.built) return fail(c, GKD_ESTATE, "set %u has not been built", first_id + i);
        if (g.arena != arena) return fail(c, GKD_EINVAL, "sets %u..%u span more than one arena", first_id, first_id + n_sets - 1);
        if (!g.lit.empty()) return fail(c, GKD_EINVAL, "set %u has literal ambiguous k-mers, which live on the host and are not exchanged", first_id + i);
        table[i] = g.packed;
    }
    return GKD_OK;
}

int gkd_adopt_sets(gkd_ctx *c, const void *base, uint64_t bytes, const gkd_packed_set *table, uint32_t n_sets, uint32_t *first_id) {
    CHECK_CTX(c);
    if (first_id) *first_id = (uint32_t)c->genomes.size();
    if (n_sets == 0) return GKD_OK;
    if (!base || !table) return fail(c, GKD_EINVAL, "gkd_adopt_sets: null argument");
    if (((uintptr_t)base & 15) != 0) return fail(c, GKD_EINVAL, "gkd_adopt_sets: base must be 16-byte aligned");
    if (classify(base) != MEM_DEVICE) return fail(c, GKD_EINVAL, "gkd_adopt_sets: base must be device memory");
    const uint64_t lsz = c->low_bits / 8;
    const bool pal = has_pal_lists(c);
    ABI_GUARD_BEGIN
    for (uint32_t i = 0; i < n_sets; i++) {
        const gkd_packed_set &p = table[i];
        auto piece_ok = [&](uint64_t off, uint64_t len) { return (off & 15) == 0 && off <= bytes && len <= bytes - off; };
        bool ok = p.level >= c->lvl_min && p.level <= level_cap(c->key_bits) &&
                  piece_ok(p.offs_off, ((1ull << p.level) + 1) * 4) && piece_ok(p.lows_off, align16((uint64_t)p.n * lsz));
        if (ok && pal)
            ok = p.pal_level >= c->lvl_min && p.pal_level <= level_cap(c->key_bits) && p.pal_lows_off != 0 &&
                 piece_ok(p.pal_offs_off, ((1ull << p.pal_level) + 1) * 4) &&
                 piece_ok(p.pal_lows_off, align16((uint64_t)p.n_pal * lsz));
        if (ok && !pal) ok = p.n_pal == 0;
        if (!ok) return fail(c, GKD_EINVAL, "gkd_adopt_sets: descriptor %u does not fit the buffer or this context (k, alphabet)", i);
    }
    const uint32_t id0 = (uint32_t)c->genomes.size();
    c->arenas.push_back(Arena{(char *)const_cast<void *>(base), bytes, bytes, id0, n_sets, false});
    for (uint32_t i = 0; i < n_sets; i++) {
        GenomeRec g;
        g.packed = table[i];
        if (!pal) g.packed.pal_offs_off = g.packed.pal_lows_off = 0;
        g.arena = (int)c->arenas.size() - 1;
        set_desc_from_packed(g, (const char *)base);
        g.built = true;
        c->genomes.push_back(std::move(g));
    }
    c->sets_dirty = true;
    return GKD_OK;
    ABI_GUARD_END(c)
}

// .kset layout (little-endian): "GKDKSET1", u32 k, u32 alphabet, u32 n_sets, u32 0; then per set:
// u64 n_keys, u32 label_len, u32 comment_len, label bytes, comment bytes, n_keys x u64 keys ascending.
int gkd_save_sets(gkd_ctx *c, const char *path) {
    CHECK_CTX(c);
    if (!path) return fail(c, GKD_EINVAL, "gkd_save_sets: null path");
    CK(cudaSetDevice(c->cfg.device));
    for (uint32_t i = 0; i < c->genomes.size(); i++) {
        int rc = check_built(c, i);
        if (rc) return rc;
        if (!c->genomes[i].lit.empty()) return fail(c, GKD_EINVAL, "set %u has literal ambiguous k-mers, which the .kset cache cannot hold", i);
    }
    ABI_GUARD_BEGIN
    FILE *f = fopen(path, "wb");
    if (!f) return fail(c, GKD_EIO, "Cannot open %s for writing.", path);
    uint32_t hdr[4] = {(uint32_t)c->k, (uint32_t)c->cfg.alphabet, (uint32_t)c->genomes.size(), 0};
    bool ok = fwrite("GKDKSET1", 1, 8, f) == 8 && fwrite(hdr, 4, 4, f) == 4;
    std::vector<uint64_t> host;
    for (uint32_t i = 0; ok && i < c->genomes.size(); i++) {
        const GenomeRec &g = c->genomes[i];
        uint64_t n = g.desc.main.n;
        uint32_t ll[2] = {(uint32_t)g.label.size(), (uint32_t)g.comment.size()};
        host.resize(n);
        int rc = gkd_export_set(c, i, host.data(), n, nullptr);
        if (rc) {
            fclose(f);
            return rc;
        }
        ok = fwrite(&n, 8, 1, f) == 1 && fwrite(ll, 4, 2, f) == 2 &&
             fwrite(g.label.data(), 1, ll[0], f) == ll[0] && fwrite(g.comment.data(), 1, ll[1], f) == ll[1] &&
             fwrite(host.data(), 8, n, f) == n;
    }
    ok = (fclose(f) == 0) && ok;
    return ok ? GKD_OK : fail(c, GKD_EIO, "Write error on %s.", path);
    ABI_GUARD_END(c)
}

int gkd_load_sets(gkd_ctx *c, const char *path, uint32_t *first_id, uint32_t *n_loaded) {
    CHECK_CTX(c);
    if (!path) return fail(c, GKD_EINVAL, "gkd_load_sets: null path");
    ABI_GUARD_BEGIN
    FILE *f = fopen(path, "rb");
    if (!f) return fail(c, GKD_EIO, "Input file %s is not found or unreadable.", path);
    struct Closer {
        FILE *f;
        ~Closer() { fclose(f); }
    } closer{f};
    char magic[8];
    uint32_t hdr[4];
    if (fread(magic, 1, 8, f) != 8 || memcmp(magic, "GKDKSET1", 8) != 0 || fread(hdr, 4, 4, f) != 4)
        return fail(c, GKD_EIO, "%s is not a .kset file.", path);
    if ((int)hdr[0] != c->k || (int)hdr[1] != c->cfg.alphabet)
        return fail(c, GKD_EINVAL, "%s holds k=%u alphabet=%u sets; this context is k=%d alphabet=%d", path, hdr[0], hdr[1],
                    c->k, c->cfg.alphabet);
    // the file is untrusted: every count is bounded by the bytes that are actually left in it
    long here = ftell(f);
    if (here < 0 || fseek(f, 0, SEEK_END) != 0) return fail(c, GKD_EIO, "%s is not seekable.", path);
    const uint64_t file_size = (uint64_t)ftell(f);
    fseek(f, here, SEEK_SET);
    uint64_t left = file_size - (uint64_t)here;
    const uint32_t n = hdr[2];
    if ((uint64_t)n * 16 > left) return fail(c, GKD_EIO, "%s is truncated or corrupt.", path);
    std::vector<uint64_t> keys, offsets(1, 0);
    std::vector<std::string> labels(n), comments(n);
    bool ok = true;
    for (uint32_t i = 0; ok && i < n; i++) {
        uint64_t nk;
        uint32_t ll[2];
        ok = fread(&nk, 8, 1, f) == 1 && fread(ll, 4, 2, f) == 2;
        if (!ok) break;
        left -= 16;
        ok = nk < 0xFFFF0000ull && (uint64_t)ll[0] + ll[1] <= left && nk <= (left - ll[0] - ll[1]) / 8;
        if (!ok) break;
        labels[i].resize(ll[0]);
        comments[i].resize(ll[1]);
        ok = fread(&labels[i][0], 1, ll[0], f) == ll[0] && fread(&comments[i][0], 1, ll[1], f) == ll[1];
        if (!ok) break;
        size_t at = keys.size();
        keys.resize(at + nk);
        ok = fread(keys.data() + at, 8, nk, f) == nk;
        left -= (uint64_t)ll[0] + ll[1] + nk * 8;
        offsets.push_back(keys.size());
    }
    if (!ok) return fail(c, GKD_EIO, "%s is truncated or corrupt.", path);
    uint32_t first = 0;
    int rc = gkd_import_sets(c, keys.data(), offsets.data(), n, &first);
    if (rc) return rc;
    for (uint32_t i = 0; i < n; i++) {
        c->genomes[first + i].label = labels[i];
        c->genomes[first + i].comment = comments[i];
    }
    if (first_id) *first_id = first;
    if (n_loaded) *n_loaded = n;
    return GKD_OK;
    ABI_GUARD_END(c)
}

// ---- distances --------------------------------------------------------------------------------------------
int gkd_all_vs_all_range_ex(gkd_ctx *c, uint32_t n, uint64_t first, uint64_t count, const gkd_outputs *out) {
    if (!out) return fail(c, GKD_EINVAL, "gkd_all_vs_all_range_ex: null outputs");
    Dense f(*out);
    return run_call(c, "gkd_all_vs_all_range_ex", HostPairs{PAIRS_UPPER, n, first, count, nullptr, nullptr, 0, 0}, f);
}

int gkd_all_vs_all_range(gkd_ctx *c, uint32_t n, uint64_t first, uint64_t count, uint64_t *inter, double *dist) {
    gkd_outputs o{inter, dist, nullptr, nullptr};
    return gkd_all_vs_all_range_ex(c, n, first, count, &o);
}

int gkd_all_vs_all(gkd_ctx *c, uint64_t *inter, double *dist) {
    CHECK_CTX(c);
    uint32_t n = (uint32_t)c->genomes.size();
    return gkd_all_vs_all_range(c, n, 0, n < 2 ? 0 : (uint64_t)n * (n - 1) / 2, inter, dist);
}

int gkd_query_vs_ref_ex(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, const gkd_outputs *out) {
    if (!out) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_ex: null outputs");
    Dense f(*out);
    return run_call(c, "gkd_query_vs_ref_ex", block(q, nq, r, nr), f);
}

int gkd_query_vs_ref(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, uint64_t *inter, double *dist) {
    gkd_outputs o{inter, dist, nullptr, nullptr};
    return gkd_query_vs_ref_ex(c, q, nq, r, nr, &o);
}

int gkd_pairs_ex(gkd_ctx *c, const uint32_t *a, const uint32_t *b, uint64_t n_pairs, const gkd_outputs *out) {
    if (!out) return fail(c, GKD_EINVAL, "gkd_pairs_ex: null outputs");
    Dense f(*out);
    return run_call(c, "gkd_pairs_ex", HostPairs{PAIRS_LIST, 0, 0, n_pairs, a, b, (uint32_t)n_pairs, (uint32_t)n_pairs}, f);
}

int gkd_pairs(gkd_ctx *c, const uint32_t *a, const uint32_t *b, uint64_t n_pairs, uint64_t *inter, double *dist) {
    gkd_outputs o{inter, dist, nullptr, nullptr};
    return gkd_pairs_ex(c, a, b, n_pairs, &o);
}

int gkd_greedy_reps(gkd_ctx *c, const uint32_t *order, uint32_t n, double max_dist, uint8_t *is_rep) {
    CHECK_CTX(c);
    if (n == 0) return GKD_OK;
    if (!order || !is_rep) return fail(c, GKD_EINVAL, "gkd_greedy_reps: null argument");
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    int rc = upload_sets(c);
    if (rc) return rc;
    const bool nuc = c->cfg.alphabet != GKD_PROT;
    const bool both = nuc && c->cfg.strand_mode == GKD_STRAND_BOTH;
    const bool need_pal = both && (c->k % 2 == 0);
    SetScan s;
    for (uint32_t i = 0; i < n; i++)
        if ((rc = s.see(c, order[i]))) return rc;
    if (s.any_lit) {
        // the shared literal k-mers of a pair are counted on the host per chunk, which the device-resident list below
        // cannot wait for: one batched call per candidate
        std::vector<uint32_t> reps, cand;
        std::vector<double> dist;
        for (uint32_t i = 0; i < n; i++) {
            bool found = false;
            if (!reps.empty()) {
                cand.assign(reps.size(), order[i]);
                dist.assign(reps.size(), 1.0);
                Dense f(gkd_outputs{nullptr, dist.data(), nullptr, nullptr});
                HostPairs hp{PAIRS_LIST, 0, 0, reps.size(), reps.data(), cand.data(), (uint32_t)reps.size(), (uint32_t)reps.size()};
                if ((rc = run_pairs(c, hp, f))) return rc;
                for (double d : dist) found = found || d <= max_dist;
            }
            is_rep[i] = found ? 0 : 1;
            if (!found) reps.push_back(order[i]);
        }
        return GKD_OK;
    }
    // device state: representative ids, their count, per-visit flags, counts (zeroed once; the decision kernel
    // clears what it consumed)
    if ((rc = ensure(c, c->gr_reps, (uint64_t)n * 4 + 16))) return rc;
    if ((rc = ensure(c, c->gr_flags, (uint64_t)n))) return rc;
    if ((rc = ensure(c, c->counts, (uint64_t)n * 4))) return rc;
    if (need_pal && (rc = ensure(c, c->pal_counts, (uint64_t)n * 4))) return rc;
    if ((rc = ensure(c, c->work_counter, 8))) return rc;
    uint32_t *d_reps = (uint32_t *)c->gr_reps.p, *d_nreps = d_reps + n;
    CK(cudaMemsetAsync(d_nreps, 0, 16, c->stream));
    CK(cudaMemsetAsync(c->counts.p, 0, (uint64_t)n * 4, c->stream));
    if (need_pal) CK(cudaMemsetAsync(c->pal_counts.p, 0, (uint64_t)n * 4, c->stream));
    CK(cudaEventRecord(c->ev[4], c->stream));
    NvtxRange nvtx("gkd greedy representatives (kernels 4+5 per candidate, device-resident list)");
    for (uint32_t i = 0; i < n; i++) {
        if (i > 0) {  // at most i representatives so far
            PairSource src{};
            src.mode = PAIRS_LIST_VS_ONE;
            src.n = order[i];
            src.count = i;
            src.a = d_reps;
            src.count_ptr = d_nreps;
            CK(launch_intersect((const SetDesc *)c->d_sets.p, src, 0, make_plan(c, i, s.max_n, s.max_level, false), (uint32_t *)c->counts.p,
                                (unsigned long long *)c->work_counter.p, c->n_sms, c->stream));
            c->m.launches++;
            c->m.intersect_launches++;
            if (need_pal && s.max_pal) {
                CK(launch_intersect((const SetDesc *)c->d_sets.p, src, 1, make_plan(c, i, s.max_pal, s.max_pal_level, true),
                                    (uint32_t *)c->pal_counts.p, (unsigned long long *)c->work_counter.p, c->n_sms, c->stream));
                c->m.launches++;
            }
        }
        CK(launch_greedy_decide((const SetDesc *)c->d_sets.p, d_reps, d_nreps, order[i], i, (uint32_t *)c->counts.p,
                                need_pal ? (uint32_t *)c->pal_counts.p : nullptr, both ? 1 : 0, max_dist,
                                (uint8_t *)c->gr_flags.p, c->stream));
        c->m.launches++;
    }
    CK(cudaEventRecord(c->ev[5], c->stream));
    CK(cudaMemcpyAsync(is_rep, c->gr_flags.p, n, cudaMemcpyDefault, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->m.d2h_bytes += n;
    c->m.intersect_ms = elapsed(c->ev[4], c->ev[5]);
    c->m.total_intersect_ms += c->m.intersect_ms;
    return GKD_OK;
    ABI_GUARD_END(c)
}

int gkd_pair(gkd_ctx *c, uint32_t a, uint32_t b, uint64_t *inter, uint64_t *uni, double *dist) {
    uint64_t I = 0;
    double d = 1.0;
    int rc = gkd_pairs(c, &a, &b, 1, &I, &d);
    if (rc) return rc;
    if (inter) *inter = I;
    if (dist) *dist = d;
    if (uni) {
        uint64_t sa = 0, sb = 0;
        gkd_set_size(c, a, &sa, nullptr, nullptr);
        gkd_set_size(c, b, &sb, nullptr, nullptr);
        *uni = sa + sb - I;
    }
    return GKD_OK;
}

// ---- selections ---------------------------------------------------------------------------------------------
int gkd_all_vs_all_range_within(gkd_ctx *c, uint32_t n, uint64_t first, uint64_t count, double max_dist, gkd_hits *out) {
    if (!out) return fail(c, GKD_EINVAL, "gkd_all_vs_all_range_within: null hits");
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "gkd_all_vs_all_range_within: max_dist is NaN");
    Within f(max_dist, *out);
    return run_call(c, "gkd_all_vs_all_range_within", HostPairs{PAIRS_UPPER, n, first, count, nullptr, nullptr, 0, 0}, f);
}

int gkd_query_vs_ref_within(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, double max_dist,
                            gkd_hits *out) {
    if (!out) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_within: null hits");
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_within: max_dist is NaN");
    Within f(max_dist, *out);
    return run_call(c, "gkd_query_vs_ref_within", block(q, nq, r, nr), f);
}

static int nearest_args_ok(gkd_ctx *c, const char *fn, uint32_t k, double max_dist) {
    if (k < 1 || k > NEAREST_MAX_K) return fail(c, GKD_EINVAL, "%s: k = %u is outside 1..%u", fn, k, NEAREST_MAX_K);
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "%s: max_dist is NaN", fn);
    return GKD_OK;
}

int gkd_query_vs_ref_nearest(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, uint32_t k,
                             double max_dist, int exclude_self, uint32_t *ref_pos, uint64_t *inter, double *dist,
                             uint32_t *n_found) {
    const gkd_neighbors qs{ref_pos, inter, dist, n_found};
    return gkd_query_vs_ref_nearest_ex(c, q, nq, r, nr, k, max_dist, exclude_self, &qs, nullptr);
}

// the q side as row lists (complete in every launch), the r side through the per-target lists across the launches
int gkd_query_vs_ref_nearest_ex(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, uint32_t k,
                                double max_dist, int exclude_self, const gkd_neighbors *q_side, const gkd_neighbors *r_side) {
    const char *fn = "gkd_query_vs_ref_nearest_ex";
    int rc = nearest_args_ok(c, fn, k, max_dist);
    if (rc) return rc;
    if (!q_side && !r_side) return fail(c, GKD_EINVAL, "%s: both sides are NULL", fn);
    Nearest f(k, max_dist, exclude_self ? 1 : 0, q_side, nq, r_side, nr);
    return run_call(c, fn, block(q, nq, r, nr), f);
}

int gkd_all_vs_all_nearest(gkd_ctx *c, uint32_t n, uint32_t k, double max_dist, const gkd_neighbors *out) {
    int rc = nearest_args_ok(c, "gkd_all_vs_all_nearest", k, max_dist);
    if (rc) return rc;
    if (!out) return fail(c, GKD_EINVAL, "gkd_all_vs_all_nearest: null output");
    Nearest f(k, max_dist, 0, nullptr, 0, out, n);
    return run_call(c, "gkd_all_vs_all_nearest", triangle(n), f);
}

// ---- single-linkage clusters ----------------------------------------------------------------------------------
int gkd_all_vs_all_clusters(gkd_ctx *c, uint32_t n, double max_dist, uint32_t *label, uint32_t *n_clusters) {
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "gkd_all_vs_all_clusters: max_dist is NaN");
    if (!label) return fail(c, GKD_EINVAL, "gkd_all_vs_all_clusters: null label");
    Clusters f(max_dist, n, 0, label, n, nullptr, n_clusters);
    return run_call(c, "gkd_all_vs_all_clusters", triangle(n), f);
}

int gkd_query_vs_ref_clusters(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, double max_dist,
                              uint32_t *q_label, uint32_t *r_label) {
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_clusters: max_dist is NaN");
    if (!q_label && !r_label) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_clusters: both outputs are NULL");
    if ((uint64_t)nq + nr >= 0xFFFFFFFFull) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_clusters: %u + %u nodes", nq, nr);
    Clusters f(max_dist, nq + nr, nq, q_label, nq, r_label, nullptr);
    return run_call(c, "gkd_query_vs_ref_clusters", block(q, nq, r, nr), f);
}

// ---- single-linkage hierarchy --------------------------------------------------------------------------------
// node keys of a rectangle: q_key[i] for node i and r_key[j] for node nq + j, or the node itself where an array is NULL.
// key stays empty when both are NULL.  Checked before the context is used: the keys must be distinct.
static int link_keys(gkd_ctx *c, const uint32_t *q_key, uint32_t nq, const uint32_t *r_key, uint32_t nr,
                     std::vector<uint32_t> &key) {
    if (!q_key && !r_key) return GKD_OK;
    ABI_GUARD_BEGIN
    key.resize((uint64_t)nq + nr);
    for (uint32_t i = 0; i < nq; i++) key[i] = q_key ? q_key[i] : i;
    for (uint32_t j = 0; j < nr; j++) key[(uint64_t)nq + j] = r_key ? r_key[j] : nq + j;
    std::vector<uint32_t> sorted(key);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
        return fail(c, GKD_EINVAL, "gkd_query_vs_ref_linkage: node keys are not distinct");
    return GKD_OK;
    ABI_GUARD_END(c)
}

int gkd_all_vs_all_linkage(gkd_ctx *c, uint32_t n, double max_dist, gkd_hits *out) {
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "gkd_all_vs_all_linkage: max_dist is NaN");
    if (!out) return fail(c, GKD_EINVAL, "gkd_all_vs_all_linkage: null out");
    Linkage f(max_dist, n, 0, {}, out);
    return run_call(c, "gkd_all_vs_all_linkage", triangle(n), f);
}

int gkd_query_vs_ref_linkage(gkd_ctx *c, const uint32_t *q, uint32_t nq, const uint32_t *r, uint32_t nr, double max_dist,
                             const uint32_t *q_key, const uint32_t *r_key, gkd_hits *out) {
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_linkage: max_dist is NaN");
    if (!out) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_linkage: null out");
    if ((uint64_t)nq + nr >= 0xFFFFFFFFull) return fail(c, GKD_EINVAL, "gkd_query_vs_ref_linkage: %u + %u nodes", nq, nr);
    std::vector<uint32_t> key;
    int rc = link_keys(c, q_key, nq, r_key, nr, key);
    if (rc) return rc;
    Linkage f(max_dist, nq + nr, nq, std::move(key), out);
    return run_call(c, "gkd_query_vs_ref_linkage", block(q, nq, r, nr), f);
}

// ---- complete / average linkage -------------------------------------------------------------------------------
static int agglomerate_args_ok(gkd_ctx *c, const char *fn, int method, double max_dist, const gkd_merges *out) {
    if (max_dist != max_dist) return fail(c, GKD_EINVAL, "%s: max_dist is NaN", fn);
    if (method != GKD_LINK_COMPLETE && method != GKD_LINK_AVERAGE) return fail(c, GKD_EINVAL, "%s: unknown method %d", fn, method);
    if (!out) return fail(c, GKD_EINVAL, "%s: null out", fn);
    return GKD_OK;
}

int gkd_all_vs_all_agglomerate(gkd_ctx *c, uint32_t n, int method, double max_dist, gkd_merges *out) {
    const int rc = agglomerate_args_ok(c, "gkd_all_vs_all_agglomerate", method, max_dist, out);
    if (rc) return rc;
    Agglomerate f(n, method, max_dist, out);
    return run_call(c, "gkd_all_vs_all_agglomerate", triangle(n), f);
}

int gkd_agglomerate(gkd_ctx *c, uint32_t n, const double *dist, int method, double max_dist, gkd_merges *out) {
    const char *fn = "gkd_agglomerate";
    int rc = agglomerate_args_ok(c, fn, method, max_dist, out);
    if (rc) return rc;
    if (!dist && n >= 2) return fail(c, GKD_EINVAL, "%s: null dist", fn);
    CHECK_CTX(c);
    CK(cudaSetDevice(c->cfg.device));
    Agglomeration g(fn, n, method, max_dist, out);
    if ((rc = host_outputs_ok(c, fn, g.outputs()))) return rc;
    c->m.pairs = c->m.intersect_bytes = 0;
    c->m.intersect_ms = c->m.epilogue_ms = 0;
    ABI_GUARD_BEGIN
    if ((rc = g.start(c))) return rc;
    const uint64_t total = (uint64_t)n * (n - (n > 0)) / 2;
    const bool on_device = total && classify(dist) == MEM_DEVICE;
    for (uint64_t first = 0; first < total; first += PAIR_CHUNK) {
        const uint64_t cnt = std::min<uint64_t>(PAIR_CHUNK, total - first);
        const double *src = dist + first;
        if (!on_device) {  // staged through the scatter's source buffer, in stream order
            if ((rc = ensure(c, c->d_dist, cnt * 8))) return rc;
            CK(cudaMemcpyAsync(c->d_dist.p, src, cnt * 8, cudaMemcpyHostToDevice, c->stream));
            c->m.h2d_bytes += cnt * 8;
            src = (const double *)c->d_dist.p;
        }
        if ((rc = g.scatter(c, src, first, cnt, nullptr))) return rc;
    }
    return g.finish(c);
    ABI_GUARD_END(c)
}

// ---- MinHash sketches ---------------------------------------------------------------------------------------
// hashSet(width) of one set into device memory `d_out` (width int32 slots); *n_out = entries written
static int sketch_one(gkd_ctx *c, uint32_t id, uint32_t width, int hash, int32_t *d_out, uint32_t *n_out) {
    const GenomeRec &g = c->genomes[id];
    const bool nuc = c->cfg.alphabet != GKD_PROT;
    const int both = nuc && c->cfg.strand_mode == GKD_STRAND_BOTH;
    if (!g.lit.empty()) return fail(c, GKD_EINVAL, "sketches of sets with literal ambiguous k-mers are not supported");
    int rc;
    if ((rc = ensure(c, c->sk_cand, (uint64_t)SKETCH_CAP * 4))) return rc;
    if ((rc = ensure(c, c->sk_misc, 16))) return rc;
    uint32_t *misc = (uint32_t *)c->sk_misc.p;  // [0] candidates seen, [1] entries written, [2] distinct candidates
    const uint64_t n_codes = (uint64_t)g.desc.main.n * (both ? 2 : 1);
    // codes are close to uniform over 2^32: keep about 2*width+64 of them; everything when the set is small
    const uint64_t want = 2ull * width + 64;
    uint64_t thresh = n_codes <= SKETCH_CAP / 2 ? 0xFFFFFFFFull : std::min<uint64_t>(0xFFFFFFFFull, (want << 32) / n_codes);
    for (int attempt = 0; attempt < 40; attempt++) {
        CK(launch_sketch_filter(g.desc.main, c->mix, c->low_bits, c->cfg.alphabet, c->k, both, hash, (uint32_t)thresh,
                                (uint32_t *)c->sk_cand.p, SKETCH_CAP, misc, c->stream));
        uint32_t seen = 0;
        CK(cudaMemcpyAsync(&seen, misc, 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        c->m.launches++;
        if (seen > SKETCH_CAP) {  // too many below the threshold (skewed codes): tighten
            thresh /= 4;
            continue;
        }
        CK(launch_sketch_finish((const uint32_t *)c->sk_cand.p, seen, width, d_out, misc + 1, misc + 2, c->stream));
        uint32_t res[2] = {0, 0};
        CK(cudaMemcpyAsync(res, misc + 1, 8, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        c->m.launches++;
        if (res[1] >= width || thresh >= 0xFFFFFFFFull) {  // enough distinct codes, or every code was considered
            *n_out = res[0];
            return GKD_OK;
        }
        thresh = std::min<uint64_t>(0xFFFFFFFFull, thresh * 4 + 1024);  // too few distinct codes: widen
    }
    return fail(c, GKD_EINVAL, "sketch threshold search did not converge for set %u", id);
}

int gkd_hash_set(gkd_ctx *c, uint32_t id, uint32_t width, int hash, int32_t *out, uint32_t *n_out) {
    CHECK_CTX(c);
    int rc = check_built(c, id);
    if (rc) return rc;
    if (width == 0 || width > SKETCH_MAX_WIDTH) return fail(c, GKD_EINVAL, "sketch width must be 1..%u", SKETCH_MAX_WIDTH);
    if (hash != GKD_HASH_JAVA_STRING && hash != GKD_HASH_MURMUR3) return fail(c, GKD_EINVAL, "unknown sketch hash %d", hash);
    if (!out || !n_out) return fail(c, GKD_EINVAL, "gkd_hash_set: null output");
    CK(cudaSetDevice(c->cfg.device));
    if ((rc = ensure(c, c->sk_out, (uint64_t)SKETCH_MAX_WIDTH * 4))) return rc;
    uint32_t n = 0;
    if ((rc = sketch_one(c, id, width, hash, (int32_t *)c->sk_out.p, &n))) return rc;
    if (n) CK(cudaMemcpyAsync(out, c->sk_out.p, (uint64_t)n * 4, cudaMemcpyDefault, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->m.d2h_bytes += (uint64_t)n * 4;
    *n_out = n;
    return GKD_OK;
}

int gkd_sketch_distances(gkd_ctx *c, uint32_t width, int hash, const uint32_t *a, const uint32_t *b, uint64_t n_pairs,
                         double *dist) {
    CHECK_CTX(c);
    if (width == 0 || width > SKETCH_MAX_WIDTH) return fail(c, GKD_EINVAL, "sketch width must be 1..%u", SKETCH_MAX_WIDTH);
    if (hash != GKD_HASH_JAVA_STRING && hash != GKD_HASH_MURMUR3) return fail(c, GKD_EINVAL, "unknown sketch hash %d", hash);
    if (n_pairs == 0) return GKD_OK;
    if (!a || !b || !dist) return fail(c, GKD_EINVAL, "gkd_sketch_distances: null argument");
    if (n_pairs > 0xFFFFFFFFull) return fail(c, GKD_EINVAL, "gkd_sketch_distances: more than 2^32 pairs in one call");
    CK(cudaSetDevice(c->cfg.device));
    ABI_GUARD_BEGIN
    // sketch every set that occurs in the list once, into a dense signature matrix
    const uint32_t n_sets = (uint32_t)c->genomes.size();
    std::vector<uint32_t> slot(n_sets, UINT32_MAX), order;
    std::vector<uint32_t> ra(n_pairs), rb(n_pairs);
    for (uint64_t t = 0; t < n_pairs; t++) {
        for (uint32_t id : {a[t], b[t]}) {
            int rc = check_built(c, id);
            if (rc) return rc;
            if (slot[id] == UINT32_MAX) {
                slot[id] = (uint32_t)order.size();
                order.push_back(id);
            }
        }
        ra[t] = slot[a[t]];
        rb[t] = slot[b[t]];
    }
    int rc;
    if ((rc = ensure(c, c->sk_sig, (uint64_t)order.size() * width * 4))) return rc;
    if ((rc = ensure(c, c->sk_len, (uint64_t)order.size() * 4))) return rc;
    std::vector<uint32_t> lens(order.size());
    for (size_t s = 0; s < order.size(); s++)
        if ((rc = sketch_one(c, order[s], width, hash, (int32_t *)c->sk_sig.p + s * width, &lens[s]))) return rc;
    if ((rc = ensure(c, c->ids_a, n_pairs * 4))) return rc;
    if ((rc = ensure(c, c->ids_b, n_pairs * 4))) return rc;
    if ((rc = ensure(c, c->d_dist, n_pairs * 8))) return rc;
    CK(cudaMemcpyAsync(c->sk_len.p, lens.data(), lens.size() * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ids_a.p, ra.data(), n_pairs * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->ids_b.p, rb.data(), n_pairs * 4, cudaMemcpyHostToDevice, c->stream));
    CK(launch_sketch_distance((const int32_t *)c->sk_sig.p, (const uint32_t *)c->sk_len.p, width, (const uint32_t *)c->ids_a.p,
                              (const uint32_t *)c->ids_b.p, n_pairs, (double *)c->d_dist.p, c->stream));
    c->m.launches++;
    CK(cudaMemcpyAsync(dist, c->d_dist.p, n_pairs * 8, cudaMemcpyDefault, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->m.d2h_bytes += n_pairs * 8;
    return GKD_OK;
    ABI_GUARD_END(c)
}

int gkd_get_metrics(const gkd_ctx *c, gkd_metrics *out) {
    if (!c || !out) return GKD_EINVAL;
    *out = c->m;
    return GKD_OK;
}

void *gkd_stream(const gkd_ctx *c) { return c ? (void *)c->stream : nullptr; }

// java.lang.Double.toString: shortest digits that round-trip, decimal layout for 1e-3 <= |v| < 1e7,
// otherwise d.dddE[-]n; always at least one digit after the point.
int gkd_format_double(double v, char *buf, size_t cap) {
    if (std::isnan(v)) return snprintf(buf, cap, "NaN");
    if (std::isinf(v)) return snprintf(buf, cap, v > 0 ? "Infinity" : "-Infinity");
    if (v == 0.0) return snprintf(buf, cap, std::signbit(v) ? "-0.0" : "0.0");
    char tmp[48];
    int prec = 17;
    for (int p = 1; p <= 17; p++) {
        snprintf(tmp, sizeof(tmp), "%.*e", p - 1, v);
        if (strtod(tmp, nullptr) == v) {
            prec = p;
            break;
        }
    }
    snprintf(tmp, sizeof(tmp), "%.*e", prec - 1, v);
    std::string mant;
    const char *e = strchr(tmp, 'e');
    for (const char *p = tmp; p < e; p++)
        if (*p >= '0' && *p <= '9') mant.push_back(*p);
    int ex = atoi(e + 1);
    while (mant.size() > 1 && mant.back() == '0') mant.pop_back();
    std::string out;
    if (v < 0) out.push_back('-');
    if (ex >= -3 && ex < 7) {
        if (ex >= 0) {
            std::string ip = mant.substr(0, std::min<size_t>(mant.size(), (size_t)ex + 1));
            while ((int)ip.size() < ex + 1) ip.push_back('0');
            std::string fp = mant.size() > (size_t)ex + 1 ? mant.substr((size_t)ex + 1) : "0";
            out += ip + "." + fp;
        } else {
            out += "0." + std::string((size_t)(-ex - 1), '0') + mant;
        }
    } else {
        out += mant.substr(0, 1) + "." + (mant.size() > 1 ? mant.substr(1) : std::string("0")) + "E" + std::to_string(ex);
    }
    return snprintf(buf, cap, "%s", out.c_str());
}

static int synth_any(int device, char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member, double rate,
                     int protein) {
    if (len && !dst) return GKD_EINVAL;
    if (device >= 0 && classify(dst) == MEM_DEVICE) {
        if (cudaSetDevice(device) != cudaSuccess) return GKD_ECUDA;
        if (launch_synth(dst, len, seed, family, member, rate, protein, 0) != cudaSuccess) return GKD_ECUDA;
        if (cudaStreamSynchronize(0) != cudaSuccess) return GKD_ECUDA;
        return GKD_OK;
    }
    synth_host(dst, len, seed, family, member, rate, protein);
    return GKD_OK;
}

int gkd_synth_dna(int device, char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member, double sub_rate) {
    return synth_any(device, dst, len, seed, family, member, sub_rate, 0);
}

int gkd_synth_protein(int device, char *dst, uint64_t len, uint64_t seed, uint32_t family, uint32_t member, double sub_rate) {
    return synth_any(device, dst, len, seed, family, member, sub_rate, 1);
}

}  // extern "C"
