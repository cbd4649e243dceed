// gkd_group.cu -- several devices behind the C ABI: a group of contexts (one per listed device) in ONE
// process, one host thread per member, set arenas moved with peer copies (copy engines over NVLink) and
// adopted in place.  Built entirely on the public single-device ABI (gkd.h) plus cudaMemcpyPeerAsync.
//
// Reference shape: FastaDistanceProcessor.runReporter / computePairs (:141-194) -- all pairs i < j of one
// FASTA file.  The pair matrix shards with no reduction (SURVEY section 8e): member x owns its diagonal
// block and the blocks (x, (x+s) mod R), s = 1..R/2 (the half-way block of an even ring is split between
// its two members), exactly the schedule of genome/distance_b200/sharding.py (the one-process-per-GPU
// torch.distributed layer); here the transport is a peer copy instead of NCCL send/recv.  The cluster and linkage
// forms also use the host union-find of gkd_internal.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "gkd.h"
#include "gkd_internal.cuh"  // HostForest, host_msf, NEAREST_MAX_K

// host FASTA scanner (fasta.cpp)
struct FastaPiece {
    const char *ptr;
    uint64_t len;
};
struct FastaRecord {
    std::string label, comment;
    std::vector<FastaPiece> lines;
};
int gkd_parse_fasta_file(const char *path, std::vector<char> &storage, std::vector<FastaRecord> &records,
                         std::string &err);

namespace {

struct ArenaMeta {  // snapshot of one arena of a member after the build (read-only during the ring)
    uint32_t first, n;
    const char *base;
    uint64_t bytes;
    std::vector<gkd_packed_set> table;  // offsets relative to base
};

struct Panel {  // sets [first, first+count) of a member: bytes [begin, end) of one of its arenas
    uint32_t arena, first, count;
    uint64_t begin, end;
    std::vector<gkd_packed_set> table;  // offsets relative to begin
};

struct Member {
    gkd_ctx *ctx = nullptr;
    int device = 0;
    std::vector<uint32_t> global_ids;  // local set id -> global id (ascending: members own contiguous id blocks)
    std::vector<ArenaMeta> arenas;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copy_done[2] = {nullptr, nullptr};
    void *recv[2] = {nullptr, nullptr};
    uint64_t recv_cap[2] = {0, 0};
    int rc = GKD_OK;
    std::string err;
};

thread_local std::string g_group_create_error;

}  // namespace

struct gkd_group {
    gkd_config cfg{};
    std::vector<Member> members;
    uint32_t n_genomes = 0;
    uint32_t panel_sets = 128;
    std::vector<std::pair<uint32_t, uint32_t>> where;  // global id -> (member, local id)
    std::string err;
};

namespace {

int gfail(gkd_group *g, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (g) g->err = buf;
    else g_group_create_error = buf;
    return code;
}

// plan_panels of sharding.py: never spans two arenas, at most max_sets sets, offsets rebased to `begin`
std::vector<Panel> plan_panels(const std::vector<ArenaMeta> &meta, uint32_t lo, uint32_t hi, uint32_t max_sets) {
    std::vector<Panel> out;
    for (uint32_t ai = 0; ai < meta.size(); ai++) {
        const ArenaMeta &A = meta[ai];
        uint32_t a = std::max(lo, A.first), b = std::min(hi, A.first + A.n);
        while (a < b) {
            const uint32_t m = std::min(b - a, std::max(1u, max_sets));
            Panel p;
            p.arena = ai;
            p.first = a;
            p.count = m;
            p.table.assign(A.table.begin() + (a - A.first), A.table.begin() + (a - A.first + m));
            p.begin = p.table[0].offs_off;
            p.end = (a + m == A.first + A.n) ? A.bytes : A.table[a - A.first + m].offs_off;
            for (auto &t : p.table) {
                t.offs_off -= p.begin;
                t.lows_off -= p.begin;
                if (t.pal_offs_off) t.pal_offs_off -= p.begin;
                if (t.pal_lows_off) t.pal_lows_off -= p.begin;
            }
            out.push_back(std::move(p));
            a += m;
        }
    }
    return out;
}

inline uint64_t row_start(uint64_t i, uint64_t n) { return i * (2 * n - i - 1) / 2; }

#define MCK(call)                                                                                         \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess) {                                                                         \
            char b__[256];                                                                                \
            snprintf(b__, sizeof(b__), "%s: %s", #call, cudaGetErrorString(e__));                         \
            M.err = b__;                                                                                  \
            M.rc = e__ == cudaErrorMemoryAllocation ? GKD_ENOMEM : GKD_ECUDA;                             \
            return;                                                                                       \
        }                                                                                                 \
    } while (0)
#define MGK(call)                                             \
    do {                                                      \
        int r__ = (call);                                     \
        if (r__ != GKD_OK) {                                  \
            M.rc = r__;                                       \
            M.err = gkd_last_error(M.ctx);                    \
            return;                                           \
        }                                                     \
    } while (0)

// What a group call computes: every member runs its own form over its diagonal block and over each of its ring calls
// (member_ring), in global ids, and the entry point merges the members' forms.
struct RingForm {
    virtual ~RingForm() = default;
    // the member's own sets, local ids 0 .. m-1 (m >= 2)
    virtual int diagonal(Member &M, uint32_t m) = 0;
    // the member's rows (local ids) x the adopted columns cols; col_gid: the global id of every column
    virtual int block(Member &M, const std::vector<uint32_t> &rows, const std::vector<uint32_t> &cols,
                      const std::vector<uint32_t> &col_gid) = 0;
};

// gkd_group_all_vs_all: every block scattered into the caller's triangle
struct RingDense : RingForm {
    uint64_t N;
    uint64_t *inter;
    double *dist;
    std::vector<uint64_t> bi;
    std::vector<double> bd;
    RingDense(uint64_t n, uint64_t *inter_, double *dist_) : N(n), inter(inter_), dist(dist_) {}
    void put(uint32_t ga, uint32_t gb, uint64_t t) {  // entry t of the call to pair (ga, gb)
        if (ga > gb) std::swap(ga, gb);
        const uint64_t o = row_start(ga, N) + (gb - ga - 1);
        if (inter) inter[o] = bi[t];
        if (dist) dist[o] = bd[t];
    }
    int diagonal(Member &M, uint32_t m) override {
        const uint64_t cnt = (uint64_t)m * (m - 1) / 2;
        bi.resize(cnt);
        bd.resize(cnt);
        const int rc = gkd_all_vs_all_range(M.ctx, m, 0, cnt, bi.data(), bd.data());
        if (rc != GKD_OK) return rc;
        uint64_t t = 0;
        for (uint32_t i = 0; i < m; i++)
            for (uint32_t j = i + 1; j < m; j++, t++) put(M.global_ids[i], M.global_ids[j], t);
        return GKD_OK;
    }
    int block(Member &M, const std::vector<uint32_t> &rows, const std::vector<uint32_t> &cols,
              const std::vector<uint32_t> &col_gid) override {
        bi.resize(rows.size() * cols.size());
        bd.resize(bi.size());
        const int rc = gkd_query_vs_ref(M.ctx, rows.data(), (uint32_t)rows.size(), cols.data(), (uint32_t)cols.size(), bi.data(), bd.data());
        if (rc != GKD_OK) return rc;
        for (size_t r = 0; r < rows.size(); r++)
            for (size_t c = 0; c < cols.size(); c++) put(M.global_ids[rows[r]], col_gid[c], r * cols.size() + c);
        return GKD_OK;
    }
};

// gkd_group_all_vs_all_within: a member's hits in global ids (a < b); no dense result exists on this path
struct GroupHit {
    uint32_t a, b;
    uint64_t inter;
    double dist;
};
// first capacity a member offers a within call; a call with more hits is repeated with the exact total
constexpr uint64_t WITHIN_FIRST_CAP = 4ull << 20;
struct RingWithin : RingForm {
    double max_dist;
    std::vector<GroupHit> hits;
    std::vector<uint32_t> ha, hb;  // hit positions of one call
    std::vector<uint64_t> bi;
    std::vector<double> bd;
    explicit RingWithin(double d) : max_dist(d) {}
    template <class Call>
    int fetch(uint64_t pairs, Call call, uint64_t &nh) {  // one within call, repeated once with cap = n if it was short
        uint64_t cap = std::min(pairs, WITHIN_FIRST_CAP);
        for (;;) {
            ha.resize(cap);
            hb.resize(cap);
            bi.resize(cap);
            bd.resize(cap);
            gkd_hits h{ha.data(), hb.data(), bi.data(), bd.data(), cap, 0};
            const int rc = call(h);
            if (rc != GKD_OK) return rc;
            nh = h.n;
            if (h.n <= cap) return GKD_OK;
            cap = h.n;
        }
    }
    int diagonal(Member &M, uint32_t m) override {
        const uint64_t cnt = (uint64_t)m * (m - 1) / 2;
        uint64_t nh = 0;
        const int rc = fetch(cnt, [&](gkd_hits &h) { return gkd_all_vs_all_range_within(M.ctx, m, 0, cnt, max_dist, &h); }, nh);
        if (rc != GKD_OK) return rc;
        for (uint64_t t = 0; t < nh; t++) hits.push_back({M.global_ids[ha[t]], M.global_ids[hb[t]], bi[t], bd[t]});
        return GKD_OK;
    }
    int block(Member &M, const std::vector<uint32_t> &rows, const std::vector<uint32_t> &cols,
              const std::vector<uint32_t> &col_gid) override {
        uint64_t nh = 0;
        const int rc = fetch((uint64_t)rows.size() * cols.size(), [&](gkd_hits &h) {
            return gkd_query_vs_ref_within(M.ctx, rows.data(), (uint32_t)rows.size(), cols.data(), (uint32_t)cols.size(), max_dist, &h);
        }, nh);
        if (rc != GKD_OK) return rc;
        for (uint64_t t = 0; t < nh; t++) {
            const uint32_t ga = M.global_ids[rows[ha[t]]], gb = col_gid[hb[t]];
            hits.push_back({std::min(ga, gb), std::max(ga, gb), bi[t], bd[t]});
        }
        return GKD_OK;
    }
};

// gkd_group_all_vs_all_nearest: a member's partial lists by global id.  A pair is computed once in the whole ring, so
// the global top k of an id, by (distance bits, global id), is the top k of the union of its partial top-k lists.
struct Neighbor {
    uint64_t key;  // distance bits (distances are non-negative: the bits order like the values)
    uint32_t id;
    uint64_t inter;
    bool operator<(const Neighbor &o) const { return key < o.key || (key == o.key && id < o.id); }
};
struct RingNearest : RingForm {
    uint32_t k;
    double max_dist;
    std::vector<std::vector<Neighbor>> lists;  // global id -> <= k entries after every call
    std::vector<uint32_t> qpos, qn, rpos, rn;  // the lists of one call, per side
    std::vector<uint64_t> qi, ri;
    std::vector<double> qd, rd;
    RingNearest(uint32_t k_, double d, uint32_t n) : k(k_), max_dist(d), lists(n) {}
    void add(uint32_t target, uint32_t id, uint64_t inter, double d) {
        uint64_t key;
        memcpy(&key, &d, 8);
        lists[target].push_back(Neighbor{key, id, inter});
    }
    void keep_best(uint32_t target) {
        std::vector<Neighbor> &l = lists[target];
        if (l.size() <= k) return;
        std::partial_sort(l.begin(), l.begin() + k, l.end());
        l.resize(k);
    }
    gkd_neighbors side(size_t rows, std::vector<uint32_t> &pos, std::vector<uint64_t> &in, std::vector<double> &d,
                       std::vector<uint32_t> &nf) {
        pos.resize(rows * k);
        in.resize(rows * k);
        d.resize(rows * k);
        nf.resize(rows);
        return gkd_neighbors{pos.data(), in.data(), d.data(), nf.data()};
    }
    int diagonal(Member &M, uint32_t m) override {
        const gkd_neighbors nb = side(m, qpos, qi, qd, qn);
        const int rc = gkd_all_vs_all_nearest(M.ctx, m, k, max_dist, &nb);
        if (rc != GKD_OK) return rc;
        for (uint32_t i = 0; i < m; i++)
            for (uint32_t s = 0; s < qn[i]; s++) {
                const uint64_t o = (uint64_t)i * k + s;
                add(M.global_ids[i], M.global_ids[qpos[o]], qi[o], qd[o]);
            }
        return GKD_OK;
    }
    int block(Member &M, const std::vector<uint32_t> &rows, const std::vector<uint32_t> &cols,
              const std::vector<uint32_t> &col_gid) override {
        // The lists break ties by position in the call, and a group of panels may span peers (x+1)%R, (x+2)%R, ...,
        // whose global ids are not ascending: order the columns by global id so that position order is id order.
        // The rows are this member's own ids, ascending.
        std::vector<uint32_t> order(cols.size());
        for (uint32_t c = 0; c < order.size(); c++) order[c] = c;
        std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return col_gid[a] < col_gid[b]; });
        std::vector<uint32_t> scols(cols.size()), sgid(cols.size());
        for (size_t c = 0; c < order.size(); c++) scols[c] = cols[order[c]], sgid[c] = col_gid[order[c]];
        const gkd_neighbors qs = side(rows.size(), qpos, qi, qd, qn), rs = side(cols.size(), rpos, ri, rd, rn);
        const int rc = gkd_query_vs_ref_nearest_ex(M.ctx, rows.data(), (uint32_t)rows.size(), scols.data(), (uint32_t)scols.size(),
                                                   k, max_dist, 0, &qs, &rs);
        if (rc != GKD_OK) return rc;
        for (size_t r = 0; r < rows.size(); r++) {
            const uint32_t target = M.global_ids[rows[r]];
            for (uint32_t s = 0; s < qn[r]; s++) {
                const uint64_t o = (uint64_t)r * k + s;
                add(target, sgid[qpos[o]], qi[o], qd[o]);
            }
            keep_best(target);
        }
        for (size_t c = 0; c < scols.size(); c++) {
            for (uint32_t s = 0; s < rn[c]; s++) {
                const uint64_t o = (uint64_t)c * k + s;
                add(sgid[c], M.global_ids[rows[rpos[o]]], ri[o], rd[o]);
            }
            keep_best(sgid[c]);
        }
        return GKD_OK;
    }
};

// gkd_group_all_vs_all_clusters: a member's links (global p, global label[p]) for every node p of its calls with
// label[p] != p.  A call's labels carry all the connectivity of its links, and the ring computes every pair once, so
// the union of these links over all members has the components of the whole triangle.
struct RingClusters : RingForm {
    double max_dist;
    std::vector<std::pair<uint32_t, uint32_t>> links;
    std::vector<uint32_t> ql, rl;  // the labels of one call
    explicit RingClusters(double d) : max_dist(d) {}
    int diagonal(Member &M, uint32_t m) override {
        ql.resize(m);
        const int rc = gkd_all_vs_all_clusters(M.ctx, m, max_dist, ql.data(), nullptr);
        if (rc != GKD_OK) return rc;
        for (uint32_t i = 0; i < m; i++)
            if (ql[i] != i) links.push_back({M.global_ids[i], M.global_ids[ql[i]]});
        return GKD_OK;
    }
    int block(Member &M, const std::vector<uint32_t> &rows, const std::vector<uint32_t> &cols,
              const std::vector<uint32_t> &col_gid) override {
        const uint32_t nr = (uint32_t)rows.size(), nc = (uint32_t)cols.size();
        auto gid = [&](uint32_t node) { return node < nr ? M.global_ids[rows[node]] : col_gid[node - nr]; };
        ql.resize(nr);
        rl.resize(nc);
        const int rc = gkd_query_vs_ref_clusters(M.ctx, rows.data(), nr, cols.data(), nc, max_dist, ql.data(), rl.data());
        if (rc != GKD_OK) return rc;
        for (uint32_t p = 0; p < nr; p++)
            if (ql[p] != p) links.push_back({gid(p), gid(ql[p])});
        for (uint32_t c = 0; c < nc; c++)
            if (rl[c] != nr + c) links.push_back({col_gid[c], gid(rl[c])});
        return GKD_OK;
    }
};

// gkd_group_all_vs_all_linkage: the forest edges of a member's calls in global ids (a < b).  The ring computes every
// pair once, so MSF(union of the calls' forests) = MSF(triangle) under one strict order: every call breaks ties by global
// ids (its keys), and an edge a call's forest left out is the maximum of a cycle of the whole graph.
struct RingLinkage : RingForm {
    double max_dist;
    std::vector<gkd::LinkEdge> edges;
    std::vector<uint32_t> ha, hb;
    std::vector<uint64_t> bi;
    std::vector<double> bd;
    explicit RingLinkage(double d) : max_dist(d) {}
    // the forest of one call, at most nodes - 1 edges
    template <class Call, class GidA, class GidB>
    int forest(uint64_t nodes, Call call, GidA gid_a, GidB gid_b) {
        ha.resize(nodes);
        hb.resize(nodes);
        bi.resize(nodes);
        bd.resize(nodes);
        gkd_hits h{ha.data(), hb.data(), bi.data(), bd.data(), nodes, 0};
        const int rc = call(h);
        if (rc != GKD_OK) return rc;
        for (uint64_t t = 0; t < h.n; t++) {
            const uint32_t ga = gid_a(ha[t]), gb = gid_b(hb[t]), lo = std::min(ga, gb), hi = std::max(ga, gb);
            edges.push_back(gkd::link_edge(lo, hi, bi[t], bd[t], lo, hi, lo, hi));
        }
        return GKD_OK;
    }
    int diagonal(Member &M, uint32_t m) override {
        auto own = [&](uint32_t i) { return M.global_ids[i]; };  // ascending, so local order is global order
        return forest(m, [&](gkd_hits &h) { return gkd_all_vs_all_linkage(M.ctx, m, max_dist, &h); }, own, own);
    }
    int block(Member &M, const std::vector<uint32_t> &rows, const std::vector<uint32_t> &cols,
              const std::vector<uint32_t> &col_gid) override {
        // keyed by global id: the columns may span peers on both sides of this member's ids, and ties must be broken
        // as one context over all ids breaks them
        const uint32_t nr = (uint32_t)rows.size(), nc = (uint32_t)cols.size();
        std::vector<uint32_t> row_gid(nr);
        for (uint32_t p = 0; p < nr; p++) row_gid[p] = M.global_ids[rows[p]];
        return forest((uint64_t)nr + nc - 1,
                      [&](gkd_hits &h) {
                          return gkd_query_vs_ref_linkage(M.ctx, rows.data(), nr, cols.data(), nc, max_dist, row_gid.data(),
                                                          col_gid.data(), &h);
                      },
                      [&](uint32_t p) { return row_gid[p]; }, [&](uint32_t c) { return col_gid[c]; });
    }
};

// The ring of one member (runs on its own host thread; no exception may leave the thread): its diagonal block while the
// first group of peer panels is in flight, then one call per group, each through the member's form.
void member_ring(gkd_group *g, uint32_t x, RingForm &f) {
    Member &M = g->members[x];
    const uint32_t R = (uint32_t)g->members.size();
    const uint32_t m = (uint32_t)M.global_ids.size();
    MCK(cudaSetDevice(M.device));
    // transfer slots: (panel to receive, its owner, my rows)
    struct Slot {
        Panel p;
        uint32_t src, row0, row1;
    };
    std::vector<Slot> slots;
    for (uint32_t s = 1; s <= R / 2; s++) {
        const uint32_t src = (x + s) % R;
        const bool half = (R % 2 == 0) && s == R / 2;
        const uint32_t ms = (uint32_t)g->members[src].global_ids.size();
        uint32_t row0 = 0, row1 = m, rc0 = 0, rc1 = ms;
        if (half) {  // block X x Y (X = lower member): lower computes X[:h] x Y, higher computes Y x X[h:]
            if (x < src) row1 = (m + 1) / 2;
            else rc0 = (ms + 1) / 2;
        }
        if (row1 <= row0) continue;
        for (auto &p : plan_panels(g->members[src].arenas, rc0, rc1, g->panel_sets)) slots.push_back(Slot{std::move(p), src, row0, row1});
    }
    // Panels are the unit of transfer; the unit of compute is a GROUP of consecutive panels that meet the same rows, up
    // to GROUP_SETS sets (possibly of several peers): kernel 4's block join builds one table per (64 rows, key range) and
    // probes every column of the call with it, so one call over many columns amortises the tables.
    constexpr uint32_t GROUP_SETS = 1024;
    struct Group {
        size_t s0, s1;  // slots [s0, s1)
        std::vector<uint64_t> off;  // byte offset of every panel in the receive buffer
        uint64_t bytes;
    };
    std::vector<Group> groups;
    for (size_t k = 0; k < slots.size();) {
        Group G{k, k, {}, 0};
        uint32_t sets = 0;
        while (G.s1 < slots.size() && slots[G.s1].row0 == slots[k].row0 && slots[G.s1].row1 == slots[k].row1 &&
               (G.s1 == k || sets + slots[G.s1].p.count <= GROUP_SETS)) {
            G.off.push_back(G.bytes);
            G.bytes += (slots[G.s1].p.end - slots[G.s1].p.begin + 255) & ~255ull;
            sets += slots[G.s1].p.count;
            G.s1++;
        }
        groups.push_back(std::move(G));
        k = groups.back().s1;
    }
    auto post = [&](size_t gi) {  // start the peer copies of group gi into receive buffer gi & 1
        const Group &G = groups[gi];
        const int b = (int)(gi & 1);
        if (G.bytes > M.recv_cap[b]) {
            if (M.recv[b]) MCK(cudaFree(M.recv[b]));
            M.recv[b] = nullptr;
            M.recv_cap[b] = 0;
            MCK(cudaMalloc(&M.recv[b], G.bytes + G.bytes / 8 + 256));
            M.recv_cap[b] = G.bytes + G.bytes / 8 + 256;
        }
        for (size_t k = G.s0; k < G.s1; k++) {
            const Slot &S = slots[k];
            const Member &O = g->members[S.src];
            const char *src_ptr = O.arenas[S.p.arena].base + S.p.begin;
            MCK(cudaMemcpyPeerAsync((char *)M.recv[b] + G.off[k - G.s0], M.device, src_ptr, O.device, S.p.end - S.p.begin, M.copy_stream));
        }
        MCK(cudaEventRecord(M.copy_done[b], M.copy_stream));
    };
    if (!groups.empty()) post(0);
    if (M.rc) return;
    if (m >= 2) MGK(f.diagonal(M, m));
    std::vector<uint32_t> rows, cols, col_gid;  // col_gid: global id of every column of the call
    for (size_t gi = 0; gi < groups.size(); gi++) {
        if (gi + 1 < groups.size()) {
            // buffer (gi+1)&1 was last used by group gi-1, whose sets were dropped (and the stream drained) below
            post(gi + 1);
            if (M.rc) return;
        }
        const Group &G = groups[gi];
        const int b = (int)(gi & 1);
        MCK(cudaEventSynchronize(M.copy_done[b]));
        const Slot &S0 = slots[G.s0];
        rows.clear();
        cols.clear();
        col_gid.clear();
        for (uint32_t r = S0.row0; r < S0.row1; r++) rows.push_back(r);
        for (size_t k = G.s0; k < G.s1; k++) {
            const Slot &S = slots[k];
            uint32_t first = 0;
            MGK(gkd_adopt_sets(M.ctx, (char *)M.recv[b] + G.off[k - G.s0], S.p.end - S.p.begin, S.p.table.data(), S.p.count, &first));
            for (uint32_t c = 0; c < S.p.count; c++) {
                cols.push_back(first + c);
                col_gid.push_back(g->members[S.src].global_ids[S.p.first + c]);
            }
        }
        MGK(f.block(M, rows, cols, col_gid));
        MGK(gkd_truncate(M.ctx, m));
    }
}

// Every member's ring with its own form forms[x], one host thread per member; the first member error is the group's
template <class Form>
int run_members(gkd_group *g, std::vector<Form> &forms) {
    for (auto &M : g->members)
        if (M.arenas.empty() && !M.global_ids.empty()) return gfail(g, GKD_ESTATE, "call gkd_group_build first");
    std::vector<std::thread> threads;
    for (uint32_t x = 0; x < g->members.size(); x++) {
        g->members[x].rc = GKD_OK;
        threads.emplace_back([g, x, &f = forms[x]]() {
            try {
                member_ring(g, x, f);
            } catch (const std::exception &ex) {
                g->members[x].rc = GKD_ENOMEM;
                g->members[x].err = ex.what();
            }
        });
    }
    for (auto &t : threads) t.join();
    for (size_t i = 0; i < g->members.size(); i++)
        if (g->members[i].rc != GKD_OK) return gfail(g, g->members[i].rc, "member %zu: %s", i, g->members[i].err.c_str());
    return GKD_OK;
}

// Every pair of the group within max_dist, in global ids, to all: one RingWithin ring, each member keeping all of its
// hits.  The members own disjoint pairs, so one sort by (a, b) gives the order of one context's row-major triangle.
int group_within(gkd_group *g, double max_dist, std::vector<GroupHit> &all) {
    std::vector<RingWithin> forms(g->members.size(), RingWithin(max_dist));
    const int rc = run_members(g, forms);
    if (rc != GKD_OK) return rc;
    for (auto &f : forms) {
        all.insert(all.end(), f.hits.begin(), f.hits.end());
        std::vector<GroupHit>().swap(f.hits);
    }
    std::sort(all.begin(), all.end(), [](const GroupHit &p, const GroupHit &q) { return p.a < q.a || (p.a == q.a && p.b < q.b); });
    return GKD_OK;
}

}  // namespace

extern "C" {

const char *gkd_group_last_error(const gkd_group *g) { return g ? g->err.c_str() : g_group_create_error.c_str(); }

int gkd_group_create(gkd_group **out, const gkd_config *cfg, const int32_t *devices, uint32_t n_devices) {
    if (!out || !cfg || !devices || n_devices == 0) return gfail(nullptr, GKD_EINVAL, "gkd_group_create: null or empty argument");
    *out = nullptr;
    gkd_group *g = new (std::nothrow) gkd_group();
    if (!g) return gfail(nullptr, GKD_ENOMEM, "out of host memory");
    try {
        g->cfg = *cfg;
        g->members.resize(n_devices);
        for (uint32_t i = 0; i < n_devices; i++) {
            Member &M = g->members[i];
            M.device = devices[i];
            gkd_config c = *cfg;
            c.device = devices[i];
            int rc = gkd_create(&M.ctx, &c);
            if (rc != GKD_OK) {
                gfail(nullptr, rc, "member %u (device %d): %s", i, devices[i], gkd_last_error(nullptr));
                gkd_group_destroy(g);
                return rc;
            }
            bool ok = cudaSetDevice(M.device) == cudaSuccess &&
                      cudaStreamCreateWithFlags(&M.copy_stream, cudaStreamNonBlocking) == cudaSuccess &&
                      cudaEventCreateWithFlags(&M.copy_done[0], cudaEventDisableTiming) == cudaSuccess &&
                      cudaEventCreateWithFlags(&M.copy_done[1], cudaEventDisableTiming) == cudaSuccess;
            if (!ok) {
                gfail(nullptr, GKD_ECUDA, "member %u (device %d): cannot create the copy stream", i, devices[i]);
                gkd_group_destroy(g);
                return GKD_ECUDA;
            }
        }
        // direct peer copies over NVLink where the hardware allows it (staged through the host otherwise)
        for (uint32_t i = 0; i < n_devices; i++)
            for (uint32_t j = 0; j < n_devices; j++) {
                if (devices[i] == devices[j]) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) == cudaSuccess && can) {
                    cudaSetDevice(devices[i]);
                    cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
                    if (e != cudaSuccess) cudaGetLastError();  // already enabled is fine
                }
            }
    } catch (const std::bad_alloc &) {
        gkd_group_destroy(g);
        return gfail(nullptr, GKD_ENOMEM, "out of host memory");
    }
    *out = g;
    return GKD_OK;
}

int gkd_group_destroy(gkd_group *g) {
    if (!g) return GKD_EINVAL;
    for (auto &M : g->members) {
        if (M.ctx) {
            cudaSetDevice(M.device);
            if (M.copy_stream) cudaStreamSynchronize(M.copy_stream);
            gkd_destroy(M.ctx);  // drops the adopted sets before their buffers go
        }
        cudaSetDevice(M.device);
        for (int b = 0; b < 2; b++) {
            if (M.recv[b]) cudaFree(M.recv[b]);
            if (M.copy_done[b]) cudaEventDestroy(M.copy_done[b]);
        }
        if (M.copy_stream) cudaStreamDestroy(M.copy_stream);
    }
    cudaGetLastError();
    delete g;
    return GKD_OK;
}

uint32_t gkd_group_size(const gkd_group *g) { return g ? (uint32_t)g->members.size() : 0; }
uint32_t gkd_group_count(const gkd_group *g) { return g ? g->n_genomes : 0; }
gkd_ctx *gkd_group_member(gkd_group *g, uint32_t member) { return (g && member < g->members.size()) ? g->members[member].ctx : nullptr; }

int gkd_group_set_panel(gkd_group *g, uint32_t sets_per_panel) {
    if (!g || sets_per_panel == 0) return GKD_EINVAL;
    g->panel_sets = sets_per_panel;
    return GKD_OK;
}

int gkd_group_add_sequences(gkd_group *g, uint32_t member, const char *const *contigs, const uint64_t *lens, uint32_t n_contigs,
                            uint32_t *global_id) {
    if (!g) return GKD_EINVAL;
    if (member >= g->members.size()) return gfail(g, GKD_EINVAL, "member %u out of range (have %zu)", member, g->members.size());
    // members own contiguous blocks of global ids: a genome may only go to the current member or a later one
    for (uint32_t later = member + 1; later < g->members.size(); later++)
        if (!g->members[later].global_ids.empty())
            return gfail(g, GKD_EINVAL, "genomes must be added member by member in ascending member order");
    try {
        Member &M = g->members[member];
        uint32_t local = 0;
        int rc = gkd_add_sequences(M.ctx, contigs, lens, n_contigs, &local);
        if (rc != GKD_OK) return gfail(g, rc, "%s", gkd_last_error(M.ctx));
        M.global_ids.push_back(g->n_genomes);
        g->where.push_back({member, local});
        if (global_id) *global_id = g->n_genomes;
        g->n_genomes++;
        return GKD_OK;
    } catch (const std::bad_alloc &) {
        return gfail(g, GKD_ENOMEM, "out of host memory");
    }
}

int gkd_group_add_fasta_file(gkd_group *g, const char *path, uint32_t *n_added) {
    if (!g || !path) return GKD_EINVAL;
    if (g->n_genomes != 0) return gfail(g, GKD_ESTATE, "gkd_group_add_fasta_file needs an empty group (it block-distributes the records)");
    try {
        std::vector<char> storage;
        std::vector<FastaRecord> recs;
        std::string err;
        if (gkd_parse_fasta_file(path, storage, recs, err)) return gfail(g, GKD_EIO, "%s", err.c_str());
        const uint32_t R = (uint32_t)g->members.size(), n = (uint32_t)recs.size();
        const uint32_t base = n / R, extra = n % R;  // block distribution, sizes differ by at most one
        uint32_t r = 0;
        for (uint32_t member = 0; member < R; member++) {
            const uint32_t take = base + (member < extra ? 1 : 0);
            for (uint32_t i = 0; i < take; i++, r++) {
                // one record = one genome whose sequence lines are pieces of ONE contig: hand the pieces through
                // the member context's FASTA-aware path by concatenating them (records are small relative to the file)
                std::string seq;
                for (auto &l : recs[r].lines) seq.append(l.ptr, l.len);
                const char *p = seq.data();
                uint64_t len = seq.size();
                int rc = gkd_group_add_sequences(g, member, &p, &len, 1, nullptr);
                if (rc != GKD_OK) return rc;
                gkd_set_label(g->members[member].ctx, g->where.back().second, recs[r].label.c_str(), recs[r].comment.c_str());
            }
        }
        if (n_added) *n_added = n;
        return GKD_OK;
    } catch (const std::bad_alloc &) {
        return gfail(g, GKD_ENOMEM, "out of host memory");
    }
}

const char *gkd_group_label(const gkd_group *g, uint32_t global_id) {
    if (!g || global_id >= g->where.size()) return "";
    return gkd_label(g->members[g->where[global_id].first].ctx, g->where[global_id].second);
}
const char *gkd_group_comment(const gkd_group *g, uint32_t global_id) {
    if (!g || global_id >= g->where.size()) return "";
    return gkd_comment(g->members[g->where[global_id].first].ctx, g->where[global_id].second);
}

int gkd_group_build(gkd_group *g) {
    if (!g) return GKD_EINVAL;
    try {
        std::vector<std::thread> threads;
        for (auto &M : g->members) {
            M.rc = GKD_OK;
            threads.emplace_back([&M]() {
                M.rc = gkd_build_sets(M.ctx);
                if (M.rc != GKD_OK) M.err = gkd_last_error(M.ctx);
            });
        }
        for (auto &t : threads) t.join();
        for (size_t i = 0; i < g->members.size(); i++)
            if (g->members[i].rc != GKD_OK) return gfail(g, g->members[i].rc, "member %zu: %s", i, g->members[i].err.c_str());
        // snapshot every member's arena layout: the ring reads its peers' layouts while they adopt and drop panels
        for (auto &M : g->members) {
            M.arenas.clear();
            const uint32_t na = gkd_arena_count(M.ctx);
            for (uint32_t a = 0; a < na; a++) {
                ArenaMeta A;
                const void *base = nullptr;
                int rc = gkd_arena_info(M.ctx, a, &A.first, &A.n, &base, &A.bytes);
                if (rc != GKD_OK) return gfail(g, rc, "gkd_arena_info failed");
                A.base = (const char *)base;
                A.table.resize(A.n);
                rc = gkd_describe_sets(M.ctx, A.first, A.n, A.table.data());
                if (rc != GKD_OK) return gfail(g, rc, "%s", gkd_last_error(M.ctx));
                M.arenas.push_back(std::move(A));
            }
        }
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_build: %s", ex.what());
    }
}

int gkd_group_all_vs_all(gkd_group *g, uint64_t *inter, double *dist) {
    if (!g) return GKD_EINVAL;
    try {
        std::vector<RingDense> forms(g->members.size(), RingDense(g->n_genomes, inter, dist));
        return run_members(g, forms);
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all: %s", ex.what());
    }
}

int gkd_group_all_vs_all_within(gkd_group *g, double max_dist, gkd_hits *out) {
    if (!out) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_within: null hits");
    if (max_dist != max_dist) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_within: max_dist is NaN");
    if (!g) return GKD_EINVAL;
    try {
        out->n = 0;
        std::vector<GroupHit> all;
        const int rc = group_within(g, max_dist, all);
        if (rc != GKD_OK) return rc;
        out->n = all.size();
        const uint64_t w = std::min<uint64_t>(all.size(), out->cap);
        for (uint64_t t = 0; t < w; t++) {
            if (out->a) out->a[t] = all[t].a;
            if (out->b) out->b[t] = all[t].b;
            if (out->inter) out->inter[t] = all[t].inter;
            if (out->dist) out->dist[t] = all[t].dist;
        }
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all_within: %s", ex.what());
    }
}

int gkd_group_all_vs_all_nearest(gkd_group *g, uint32_t k, double max_dist, const gkd_neighbors *out) {
    if (k < 1 || k > gkd::NEAREST_MAX_K)
        return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_nearest: k = %u is outside 1..%u", k, gkd::NEAREST_MAX_K);
    if (max_dist != max_dist) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_nearest: max_dist is NaN");
    if (!out) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_nearest: null output");
    if (!g) return GKD_EINVAL;
    try {
        const uint32_t N = g->n_genomes;
        std::vector<RingNearest> forms(g->members.size(), RingNearest(k, max_dist, N));
        const int rc = run_members(g, forms);
        if (rc != GKD_OK) return rc;
        std::vector<Neighbor> all;
        for (uint32_t t = 0; t < N; t++) {
            all.clear();
            for (auto &f : forms) {
                all.insert(all.end(), f.lists[t].begin(), f.lists[t].end());
                std::vector<Neighbor>().swap(f.lists[t]);
            }
            const size_t m = std::min<size_t>(all.size(), k);
            std::partial_sort(all.begin(), all.begin() + m, all.end());
            for (uint32_t i = 0; i < k; i++) {
                const uint64_t o = (uint64_t)t * k + i;
                double d = -1.0;
                if (i < m) memcpy(&d, &all[i].key, 8);
                if (out->pos) out->pos[o] = i < m ? all[i].id : 0xFFFFFFFFu;
                if (out->inter) out->inter[o] = i < m ? all[i].inter : 0;
                if (out->dist) out->dist[o] = d;
            }
            if (out->n_found) out->n_found[t] = (uint32_t)m;
        }
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all_nearest: %s", ex.what());
    }
}

int gkd_group_all_vs_all_clusters(gkd_group *g, double max_dist, uint32_t *label, uint32_t *n_clusters) {
    if (max_dist != max_dist) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_clusters: max_dist is NaN");
    if (!label) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_clusters: null label");
    if (!g) return GKD_EINVAL;
    try {
        std::vector<RingClusters> forms(g->members.size(), RingClusters(max_dist));
        const int rc = run_members(g, forms);
        if (rc != GKD_OK) return rc;
        const uint32_t N = g->n_genomes;
        gkd::HostForest forest(N);
        for (auto &f : forms)
            for (const auto &l : f.links) forest.link(l.first, l.second);
        uint32_t roots = 0;
        for (uint32_t i = 0; i < N; i++) {
            label[i] = forest.find(i);
            roots += label[i] == i ? 1u : 0u;
        }
        if (n_clusters) *n_clusters = roots;
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all_clusters: %s", ex.what());
    }
}

int gkd_group_all_vs_all_linkage(gkd_group *g, double max_dist, gkd_hits *out) {
    if (max_dist != max_dist) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_linkage: max_dist is NaN");
    if (!out) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_linkage: null out");
    if (!g) return GKD_EINVAL;
    try {
        std::vector<RingLinkage> forms(g->members.size(), RingLinkage(max_dist));
        const int rc = run_members(g, forms);
        if (rc != GKD_OK) return rc;
        std::vector<gkd::LinkEdge> edges;
        for (auto &f : forms) {
            edges.insert(edges.end(), f.edges.begin(), f.edges.end());
            std::vector<gkd::LinkEdge>().swap(f.edges);
        }
        gkd::host_msf(edges, g->n_genomes);
        out->n = edges.size();
        const uint64_t w = std::min<uint64_t>(out->n, out->cap);
        for (uint64_t t = 0; t < w; t++) {
            if (out->a) out->a[t] = edges[t].a;
            if (out->b) out->b[t] = edges[t].b;
            if (out->inter) out->inter[t] = edges[t].inter;
            if (out->dist) out->dist[t] = edges[t].dist;
        }
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all_linkage: %s", ex.what());
    }
}

// The host triangle of all N(N-1)/2 distances, filled through the dense ring, for an engine member 0 then runs on it
// with `need` bytes of device memory (what: the engine, for the message).  Both allocations are checked before any pair
// is intersected.
static int group_triangle(gkd_group *g, const char *fn, const char *what, uint64_t need, std::vector<double> &dist) {
    const uint64_t N = g->n_genomes;
    const uint64_t tri = N * (N - (N > 0)) / 2;
    try {
        dist.resize(tri);
    } catch (const std::bad_alloc &) {
        return gfail(g, GKD_ENOMEM, "%s: the host triangle of %llu sets needs %llu bytes", fn, (unsigned long long)N,
                     (unsigned long long)(tri * 8));
    }
    if (cudaSetDevice(g->members[0].device) != cudaSuccess) return gfail(g, GKD_ECUDA, "%s: cannot select the device of member 0", fn);
    const uint64_t room = gkd::agg_dense_room();
    if (N >= 2 && need > room)
        return gfail(g, GKD_ENOMEM, "%s: %s of %llu sets needs %llu bytes of device memory on member 0; %llu are free", fn, what,
                     (unsigned long long)N, (unsigned long long)need, (unsigned long long)room);
    return gkd_group_all_vs_all(g, nullptr, dist.data());
}

int gkd_group_all_vs_all_agglomerate(gkd_group *g, int method, double max_dist, gkd_merges *out) {
    if (max_dist != max_dist) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_agglomerate: max_dist is NaN");
    if (method != GKD_LINK_COMPLETE && method != GKD_LINK_AVERAGE)
        return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_agglomerate: unknown method %d", method);
    if (!out) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_agglomerate: null out");
    if (!g) return GKD_EINVAL;
    try {
        out->n = 0;
        std::vector<double> dist;
        int rc = group_triangle(g, "gkd_group_all_vs_all_agglomerate",
                                method == GKD_LINK_AVERAGE ? "average linkage" : "complete linkage",
                                gkd::agg_state_bytes(g->n_genomes, method == GKD_LINK_AVERAGE), dist);
        if (rc != GKD_OK) return rc;
        gkd_ctx *c0 = g->members[0].ctx;
        if ((rc = gkd_agglomerate(c0, g->n_genomes, dist.data(), method, max_dist, out)) != GKD_OK)
            return gfail(g, rc, "member 0: %s", gkd_last_error(c0));
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all_agglomerate: %s", ex.what());
    }
}

// a tree over all global ids: the host triangle through group_triangle, then `call` (gkd_nj or gkd_bionj) on member 0
// with `need` bytes of its device memory
static int group_joins(gkd_group *g, const char *fn, const char *what, uint64_t need,
                       int (*call)(gkd_ctx *, uint32_t, const double *, gkd_joins *), gkd_joins *out) {
    if (!out) return gfail(g, GKD_EINVAL, "%s: null out", fn);
    if (!g) return GKD_EINVAL;
    try {
        out->n = 0;
        std::vector<double> dist;
        int rc = group_triangle(g, fn, what, need, dist);
        if (rc != GKD_OK) return rc;
        gkd_ctx *c0 = g->members[0].ctx;
        if ((rc = call(c0, g->n_genomes, dist.data(), out)) != GKD_OK) return gfail(g, rc, "member 0: %s", gkd_last_error(c0));
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "%s: %s", fn, ex.what());
    }
}

int gkd_group_all_vs_all_nj(gkd_group *g, gkd_joins *out) {
    return group_joins(g, "gkd_group_all_vs_all_nj", "neighbour joining", g ? gkd::nj_state_bytes(g->n_genomes) : 0, gkd_nj, out);
}

int gkd_group_all_vs_all_bionj(gkd_group *g, gkd_joins *out) {
    return group_joins(g, "gkd_group_all_vs_all_bionj", "BIONJ", g ? gkd::bionj_state_bytes(g->n_genomes) : 0, gkd_bionj, out);
}

int gkd_group_all_vs_all_bme(gkd_group *g, int start, gkd_joins *out, uint64_t *n_swaps) {
    const char *fn = "gkd_group_all_vs_all_bme";
    if (start != GKD_TREE_NJ && start != GKD_TREE_BIONJ) return gfail(g, GKD_EINVAL, "%s: start %d is not GKD_TREE_NJ or GKD_TREE_BIONJ", fn, start);
    if (!out) return gfail(g, GKD_EINVAL, "%s: null out", fn);
    if (!g) return GKD_EINVAL;
    try {
        out->n = 0;
        if (n_swaps) *n_swaps = 0;
        std::vector<double> dist;
        int rc = group_triangle(g, fn, "balanced minimum evolution", gkd::bme_state_bytes(g->n_genomes), dist);
        if (rc != GKD_OK) return rc;
        gkd_ctx *c0 = g->members[0].ctx;
        if ((rc = gkd_bme(c0, g->n_genomes, dist.data(), start, out, n_swaps)) != GKD_OK)
            return gfail(g, rc, "member 0: %s", gkd_last_error(c0));
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "%s: %s", fn, ex.what());
    }
}

int gkd_group_all_vs_all_complete_linkage(gkd_group *g, double max_dist, gkd_merges *out) {
    if (max_dist != max_dist) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_complete_linkage: max_dist is NaN");
    if (!out) return gfail(g, GKD_EINVAL, "gkd_group_all_vs_all_complete_linkage: null out");
    if (!g) return GKD_EINVAL;
    try {
        out->n = 0;
        std::vector<GroupHit> all;
        int rc = group_within(g, max_dist, all);
        if (rc != GKD_OK) return rc;
        std::vector<uint32_t> a(all.size()), b(all.size());
        std::vector<double> d(all.size());
        for (size_t t = 0; t < all.size(); t++) a[t] = all[t].a, b[t] = all[t].b, d[t] = all[t].dist;
        std::vector<GroupHit>().swap(all);
        const gkd_hits h{a.data(), b.data(), nullptr, d.data(), a.size(), a.size()};
        gkd_ctx *c0 = g->members[0].ctx;
        if ((rc = gkd_complete_linkage(c0, g->n_genomes, &h, max_dist, out)) != GKD_OK)
            return gfail(g, rc, "member 0: %s", gkd_last_error(c0));
        return GKD_OK;
    } catch (const std::exception &ex) {
        return gfail(g, GKD_ENOMEM, "gkd_group_all_vs_all_complete_linkage: %s", ex.what());
    }
}

}  // extern "C"
