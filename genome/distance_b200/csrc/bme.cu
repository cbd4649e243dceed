// bme.cu -- balanced minimum-evolution NNIs on the device (kernel-5 forms of gkd_*_bme and gkd_bme_nni).
//
// The device holds the table of subtree averages Delta (gkd.h): an M x M matrix of doubles, M = 2n - 2, one row and one
// column per node of the tree rooted at the midpoint of its root edge (the root itself has none).  Cell (x, y) holds
// Delta(below x, below y) when neither node is an ancestor of the other, and Delta(above x, below y) when x is an
// ancestor of y (and the same value at (y, x)).  The leaf block (x, y < n) is d.  The host holds the topology (O(n)):
// for every side its size, label, height and two child sides in label order, and for every node its Euler interval,
// which it uploads after every change, so each cell finds its two sides and the two cells its formula reads in O(1).
//   build:   Delta(X, Y) reads cells of sides of smaller height, so level L = height(X) + height(Y) is one launch over
//            the cells, L = 1 .. 2 max height;
//   swap:    the gains of every internal edge and the pick (one CTA, a total order: largest gain, then the smaller edge
//            key, then swap B <-> C), read by the host; the host applies the swap to its topology and marks the sides
//            whose subtree holds the swapped edge, and lists the cells of the marked sides by level (O(n times the
//            diameter) of them); one launch per level recomputes exactly the listed cells;
//   lengths: one thread per edge, read back with the topology's rows.
// Every Delta, gain and length is one IEEE double operation per step in the order of gkd.h (the __d*_rn intrinsics
// are never contracted into an FMA), and a cell's value depends only on its two sides, so the incremental update gives
// the table a recomputation from scratch gives, bit for bit.
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "gkd_internal.cuh"

namespace gkd {

namespace {

constexpr int BME_THREADS = 256;
constexpr int PICK_THREADS = 1024;
constexpr uint32_t BME_NONE = 0xFFFFFFFFu;
constexpr uint32_t SIDE_VALID = 1, SIDE_CHANGED = 2;
constexpr uint64_t BME_CELL_CHUNK = 1u << 20;  // marked cells uploaded at once (8 MiB)

// six cells of an edge: internal AB, CD, AC, BD, AD, BC; pendant (i, A), (i, B), (A, B); leaf pair (i, j)
struct BmeEdge {
    uint64_t cell[6];
    uint32_t key_label, key_size;
    uint32_t kind;  // 0 internal, 1 pendant, 2 two leaves, 3 no edge
    uint32_t pad;
};

struct BmePick {
    double gain;
    uint32_t key_label, key_size, swap, edge;
};

// the side arrays, indexed by side id 2 node + (above ? 1 : 0), and the nodes' Euler intervals
struct BmeSides {
    const uint32_t *size, *label, *height, *kid0, *kid1, *flag;
    const uint32_t *tin, *tout;
};

struct BmeDev {
    double *T;
    uint32_t *side;  // 6 arrays of 2M, then tin and tout of M
    BmeEdge *edges;
    double *len;
    BmePick *pick;
    uint2 *cells;  // BME_CELL_CHUNK entries of a level's marked cells
};

__global__ void __launch_bounds__(BME_THREADS) k_bme_leaves(double *T, uint64_t M, const double *d, uint32_t n) {
    const uint32_t i = blockIdx.x, j = blockIdx.y * BME_THREADS + threadIdx.x;
    if (j < n) T[i * M + j] = d[(uint64_t)i * n + j];
}

// cells (a, b), a < b, of level L whose sides are both valid and one of them marked
__global__ void __launch_bounds__(BME_THREADS) k_bme_level(double *T, uint32_t M, BmeSides s, uint32_t L) {
    const uint32_t a = blockIdx.x, b = blockIdx.y * BME_THREADS + threadIdx.x;
    if (b >= M || b <= a) return;
    uint32_t X = 2 * a, Y = 2 * b;
    const uint32_t ta = __ldg(s.tin + a), tb = __ldg(s.tin + b);
    if (ta <= tb && tb <= __ldg(s.tout + a)) X++;       // a above b: Delta(above a, below b)
    else if (tb <= ta && ta <= __ldg(s.tout + b)) Y++;  // b above a
    const uint32_t fx = __ldg(s.flag + X), fy = __ldg(s.flag + Y);
    if (!(fx & fy & SIDE_VALID) || !((fx | fy) & SIDE_CHANGED)) return;
    if (__ldg(s.height + X) + __ldg(s.height + Y) != L) return;
    const uint32_t sx = __ldg(s.size + X), sy = __ldg(s.size + Y);
    const bool split_x = sx > sy || (sx == sy && __ldg(s.label + X) > __ldg(s.label + Y));
    const uint32_t Z = split_x ? X : Y, W = split_x ? Y : X;
    const uint64_t w = W >> 1;
    const double v1 = T[(uint64_t)(__ldg(s.kid0 + Z) >> 1) * M + w], v2 = T[(uint64_t)(__ldg(s.kid1 + Z) >> 1) * M + w];
    const double v = __dmul_rn(0.5, __dadd_rn(v1, v2));
    T[(uint64_t)a * M + b] = v;
    T[(uint64_t)b * M + a] = v;
}

// the cells of a list, all of one level: (X, Y) side ids of two disjoint sides; the formula of k_bme_level
__global__ void __launch_bounds__(BME_THREADS) k_bme_cells(double *T, uint32_t M, BmeSides s, const uint2 *__restrict__ cells,
                                                           uint32_t count) {
    const uint32_t t = blockIdx.x * BME_THREADS + threadIdx.x;
    if (t >= count) return;
    const uint2 c = cells[t];
    const uint32_t X = c.x, Y = c.y;
    const uint32_t sx = __ldg(s.size + X), sy = __ldg(s.size + Y);
    const bool split_x = sx > sy || (sx == sy && __ldg(s.label + X) > __ldg(s.label + Y));
    const uint32_t Z = split_x ? X : Y, W = split_x ? Y : X;
    const uint64_t w = W >> 1;
    const double v1 = T[(uint64_t)(__ldg(s.kid0 + Z) >> 1) * M + w], v2 = T[(uint64_t)(__ldg(s.kid1 + Z) >> 1) * M + w];
    const double v = __dmul_rn(0.5, __dadd_rn(v1, v2));
    T[(uint64_t)(X >> 1) * M + (Y >> 1)] = v;
    T[(uint64_t)(Y >> 1) * M + (X >> 1)] = v;
}

__device__ __forceinline__ bool pick_before(const BmePick &x, const BmePick &y) {
    if (x.gain != y.gain) return x.gain > y.gain;
    if (x.key_label != y.key_label) return x.key_label < y.key_label;
    if (x.key_size != y.key_size) return x.key_size < y.key_size;
    return x.swap < y.swap;
}

// gains = 0.25 ((D_AB + D_CD) - (D_AC + D_BD)) and 0.25 ((D_AB + D_CD) - (D_AD + D_BC)) of every internal edge; the
// largest in the total order of pick_before into *out
__global__ void __launch_bounds__(PICK_THREADS) k_bme_pick(const double *__restrict__ T, const BmeEdge *__restrict__ e,
                                                           uint32_t ne, BmePick *out) {
    __shared__ BmePick part[PICK_THREADS];
    BmePick best{-__longlong_as_double(0x7FF0000000000000ll), BME_NONE, BME_NONE, BME_NONE, BME_NONE};
    for (uint32_t t = threadIdx.x; t < ne; t += PICK_THREADS) {
        const BmeEdge &g = e[t];
        const double ab_cd = __dadd_rn(T[g.cell[0]], T[g.cell[1]]);
        const double g0 = __dmul_rn(0.25, __dsub_rn(ab_cd, __dadd_rn(T[g.cell[2]], T[g.cell[3]])));
        const double g1 = __dmul_rn(0.25, __dsub_rn(ab_cd, __dadd_rn(T[g.cell[4]], T[g.cell[5]])));
        const BmePick c0{g0, g.key_label, g.key_size, 0, t}, c1{g1, g.key_label, g.key_size, 1, t};
        if (pick_before(c0, best)) best = c0;
        if (pick_before(c1, best)) best = c1;
    }
    part[threadIdx.x] = best;
    __syncthreads();
    for (int w = PICK_THREADS / 2; w; w >>= 1) {
        if (threadIdx.x < w && pick_before(part[threadIdx.x + w], part[threadIdx.x])) part[threadIdx.x] = part[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = part[0];
}

// the BME length of edge slot t (gkd.h)
__global__ void __launch_bounds__(BME_THREADS) k_bme_lengths(const double *__restrict__ T, const BmeEdge *__restrict__ e,
                                                             uint32_t ne, double *len) {
    const uint32_t t = blockIdx.x * BME_THREADS + threadIdx.x;
    if (t >= ne) return;
    const BmeEdge &g = e[t];
    double l = 0.0;
    if (g.kind == 0) {
        const double x = __dadd_rn(__dadd_rn(__dadd_rn(T[g.cell[2]], T[g.cell[4]]), T[g.cell[5]]), T[g.cell[3]]);
        l = __dsub_rn(__dmul_rn(0.25, x), __dmul_rn(0.5, __dadd_rn(T[g.cell[0]], T[g.cell[1]])));
    } else if (g.kind == 1) {
        l = __dmul_rn(0.5, __dsub_rn(__dadd_rn(T[g.cell[0]], T[g.cell[1]]), T[g.cell[2]]));
    } else if (g.kind == 2) {
        l = T[g.cell[0]];
    }
    len[t] = l;
}

// ---- the topology, on the host -------------------------------------------------------------------------------------

struct Topology {
    uint32_t n, M, root;
    std::vector<uint32_t> par, kid;  // kid[2 v], kid[2 v + 1]
    std::vector<uint32_t> size, label, height, kid0, kid1, flag, tin, tout;  // sides: 2M; tin, tout: M

    uint32_t sib(uint32_t v) const {
        const uint32_t p = par[v];
        return kid[2 * p] == v ? kid[2 * p + 1] : kid[2 * p];
    }
    bool leaf(uint32_t v) const { return v < n; }
    uint32_t canon(uint32_t sid) const { return (sid & 1) && par[sid >> 1] == root ? 2 * sib(sid >> 1) : sid; }
    uint64_t cell(uint32_t x, uint32_t y) const { return (uint64_t)(x >> 1) * M + (y >> 1); }

    Topology(uint32_t n_, const uint32_t *a, const uint32_t *b) : n(n_), M(2 * n_ - 2), root(2 * n_ - 2) {
        par.assign(2 * n - 1, BME_NONE);
        kid.assign(2 * (2 * n - 1), BME_NONE);
        std::vector<uint32_t> cur(n);
        for (uint32_t i = 0; i < n; i++) cur[i] = i;
        for (uint32_t t = 0; t + 1 < n; t++) {
            const uint32_t v = n + t;
            kid[2 * v] = cur[a[t]];
            kid[2 * v + 1] = cur[b[t]];
            par[cur[a[t]]] = par[cur[b[t]]] = v;
            cur[a[t]] = v;
        }
        size.resize(2 * M);
        label.resize(2 * M);
        height.resize(2 * M);
        kid0.resize(2 * M);
        kid1.resize(2 * M);
        flag.resize(2 * M);
        tin.resize(M);
        tout.resize(M);
        sides();
    }

    void set_side(uint32_t sid, uint32_t x, uint32_t y) {
        if (label[y] < label[x]) std::swap(x, y);
        kid0[sid] = x;
        kid1[sid] = y;
        size[sid] = size[x] + size[y];
        label[sid] = label[x];
        height[sid] = 1 + std::max(height[x], height[y]);
    }

    // every side's size, label, height and children, and the Euler intervals, from par and kid
    void sides() {
        std::vector<uint32_t> pre;
        pre.reserve(M);
        std::vector<uint32_t> stack{kid[2 * root + 1], kid[2 * root]};
        uint32_t clock = 0;
        while (!stack.empty()) {
            const uint32_t v = stack.back();
            stack.pop_back();
            pre.push_back(v);
            tin[v] = clock++;
            if (!leaf(v)) {
                stack.push_back(kid[2 * v + 1]);
                stack.push_back(kid[2 * v]);
            }
        }
        for (uint32_t t = M; t-- > 0;) {  // below sides, children first
            const uint32_t v = pre[t], s = 2 * v;
            flag[s] = SIDE_VALID;
            if (leaf(v)) {
                size[s] = 1, label[s] = v, height[s] = 0, kid0[s] = kid1[s] = BME_NONE;
                tout[v] = tin[v];
            } else {
                set_side(s, 2 * kid[2 * v], 2 * kid[2 * v + 1]);
                tout[v] = std::max(tout[kid[2 * v]], tout[kid[2 * v + 1]]);
            }
        }
        for (uint32_t v : pre) {  // above sides, parents first
            const uint32_t s = 2 * v + 1, p = par[v];
            if (p == root) {
                flag[s] = 0;
                continue;
            }
            flag[s] = SIDE_VALID;
            set_side(s, 2 * sib(v), canon(2 * p + 1));
        }
    }

    // the four sides of the internal edge above v (v = root: the root edge), A B | C D named as gkd.h names them
    void name(uint32_t v, uint32_t q[4]) const {
        uint32_t g[4];
        if (v == root) {
            const uint32_t c0 = kid[2 * root], c1 = kid[2 * root + 1];
            g[0] = 2 * kid[2 * c0], g[1] = 2 * kid[2 * c0 + 1], g[2] = 2 * kid[2 * c1], g[3] = 2 * kid[2 * c1 + 1];
        } else {
            g[0] = 2 * kid[2 * v], g[1] = 2 * kid[2 * v + 1], g[2] = 2 * sib(v), g[3] = canon(2 * par[v] + 1);
        }
        auto lab = [&](uint32_t s) { return label[s]; };
        if (std::min(lab(g[2]), lab(g[3])) < std::min(lab(g[0]), lab(g[1]))) std::swap(g[0], g[2]), std::swap(g[1], g[3]);
        if (lab(g[1]) < lab(g[0])) std::swap(g[0], g[1]);
        if (lab(g[3]) < lab(g[2])) std::swap(g[2], g[3]);
        std::copy(g, g + 4, q);
    }

    BmeEdge internal_edge(uint32_t v) const {
        uint32_t q[4];
        name(v, q);
        const uint32_t A = q[0], B = q[1], C = q[2], D = q[3];
        return BmeEdge{{cell(A, B), cell(C, D), cell(A, C), cell(B, D), cell(A, D), cell(B, C)}, label[C], size[C] + size[D], 0, 0};
    }

    // the nodes v whose upper edge is internal, and root when the root edge is
    std::vector<uint32_t> internal_edges() const {
        std::vector<uint32_t> out;
        for (uint32_t v = n; v < M; v++)
            if (par[v] != root) out.push_back(v);
        if (!leaf(kid[2 * root]) && !leaf(kid[2 * root + 1])) out.push_back(root);
        return out;
    }

    // the edge slots of the lengths: slot v is the edge above v; the root edge is slot c0, slot c1 has none
    std::vector<BmeEdge> length_edges() const {
        std::vector<BmeEdge> out(M);
        const uint32_t c0 = kid[2 * root], c1 = kid[2 * root + 1];
        auto pendant = [&](uint32_t i) {
            const uint32_t o = canon(2 * i + 1), A = kid0[o], B = kid1[o];
            return BmeEdge{{cell(2 * i, A), cell(2 * i, B), cell(A, B), 0, 0, 0}, 0, 0, 1, 0};
        };
        for (uint32_t v = 0; v < M; v++) {
            if (v == c1) out[v] = BmeEdge{{0, 0, 0, 0, 0, 0}, 0, 0, 3, 0};
            else if (v == c0) {
                if (leaf(c0) && leaf(c1)) out[v] = BmeEdge{{cell(2 * c0, 2 * c1), 0, 0, 0, 0, 0}, 0, 0, 2, 0};
                else if (leaf(c1)) out[v] = pendant(c1);
                else if (leaf(c0)) out[v] = pendant(c0);
                else out[v] = internal_edge(root);
            } else out[v] = leaf(v) ? pendant(v) : internal_edge(v);
        }
        return out;
    }

    void exchange(uint32_t x, uint32_t y) {
        const uint32_t px = par[x], py = par[y];
        kid[kid[2 * px] == x ? 2 * px : 2 * px + 1] = y;
        kid[kid[2 * py] == y ? 2 * py : 2 * py + 1] = x;
        par[x] = py, par[y] = px;
    }

    // swap `sw` (0: B <-> C, 1: B <-> D) at the edge above v; the side towards the root never moves.  Then marks the
    // sides whose subtree holds the edge or hangs from it
    void apply(uint32_t v, uint32_t sw) {
        uint32_t q[4];
        name(v, q);
        const uint32_t A = q[0], B = q[1], C = q[2], D = q[3];
        const uint32_t mate[2][2] = {{A, C}, {A, D}};  // the new split pairs A with C (sw 0) or with D (sw 1)
        const uint32_t other = mate[sw][1];
        uint32_t x1, x2, y1, y2;
        if (v == root) {
            const uint32_t c0 = kid[2 * root], c1 = kid[2 * root + 1];
            x1 = 2 * kid[2 * c0], x2 = 2 * kid[2 * c0 + 1], y1 = 2 * kid[2 * c1], y2 = 2 * kid[2 * c1 + 1];
        } else {
            x1 = 2 * kid[2 * v], x2 = 2 * kid[2 * v + 1], y1 = 2 * sib(v), y2 = canon(2 * par[v] + 1);
        }
        // x1's new partner: A's new partner when x1 is A, A when x1 pairs with A, else the one of B, C, D left over
        uint32_t partner;
        if (x1 == A) partner = other;
        else if (x1 == other) partner = A;
        else partner = (x1 == B) ? (sw == 0 ? D : C) : B;
        if (v == root) exchange(x2 >> 1, (partner == y1 ? y1 : y2) >> 1);
        else exchange((partner == y1 ? x2 : x1) >> 1, y1 >> 1);
        sides();
        // below(y) changed iff y is at or above an end of the edge below the root; above(y) iff y is not strictly above
        std::vector<uint8_t> up(M, 0);
        const uint32_t ends[2] = {v == root ? kid[2 * root] : v, v == root ? kid[2 * root + 1] : v};
        for (uint32_t e : ends)
            for (uint32_t y = e; y != root; y = par[y]) up[y] = 1;
        for (uint32_t y = 0; y < M; y++) {
            if (up[y]) flag[2 * y] |= SIDE_CHANGED;
            const bool strictly_above = up[y] && y != ends[0] && y != ends[1];
            if ((flag[2 * y + 1] & SIDE_VALID) && !strictly_above) flag[2 * y + 1] |= SIDE_CHANGED;
        }
    }

    // the cells of the marked sides, ordered by level: every marked side X with every side Y inside its complement
    // (the complement and its descendant sides, which do not hold the swapped edge and so are not marked; the pair of
    // the swapped edge's two sides once).  start[L] .. start[L + 1] is level L.  O(n times the diameter) cells.
    void marked_cells(std::vector<uint2> &out, std::vector<uint64_t> &start) const {
        std::vector<uint2> cells;
        std::vector<uint32_t> stack;
        uint32_t top = 0;
        for (uint32_t X = 0; X < 2 * M; X++) {
            if ((flag[X] & (SIDE_VALID | SIDE_CHANGED)) != (SIDE_VALID | SIDE_CHANGED)) continue;
            stack.assign(1, (X & 1) ? X - 1 : canon(X + 1));
            while (!stack.empty()) {
                const uint32_t Y = stack.back();
                stack.pop_back();
                if (!(flag[Y] & SIDE_CHANGED) || X < Y) {
                    cells.push_back(make_uint2(X, Y));
                    top = std::max(top, height[X] + height[Y]);
                }
                if (kid0[Y] != BME_NONE) stack.push_back(kid0[Y]), stack.push_back(kid1[Y]);
            }
        }
        start.assign(top + 2, 0);
        for (const uint2 &c : cells) start[height[c.x] + height[c.y] + 1]++;
        for (uint32_t L = 1; L < start.size(); L++) start[L] += start[L - 1];
        out.resize(cells.size());
        std::vector<uint64_t> at(start.begin(), start.end() - 1);
        for (const uint2 &c : cells) out[at[height[c.x] + height[c.y]]++] = c;
    }

    uint32_t max_height(bool changed_only) const {
        uint32_t h = 0;
        for (uint32_t s = 0; s < 2 * M; s++)
            if ((flag[s] & SIDE_VALID) && (!changed_only || (flag[s] & SIDE_CHANGED))) h = std::max(h, height[s]);
        return h;
    }
};

#define BK(x)                                   \
    do {                                        \
        cudaError_t e_ = (x);                   \
        if (e_ != cudaSuccess) return e_;       \
    } while (0)

BmeDev bme_dev_at(void *base, uint32_t n) {
    const uint64_t M = 2ull * n - 2;
    BmeDev d{};
    d.T = (double *)base;
    char *p = (char *)base + bme_table_bytes(n);
    d.side = (uint32_t *)p;
    p += (6 * 2 * M + 2 * M) * 4;
    p = (char *)(((uintptr_t)p + 255) & ~(uintptr_t)255);
    d.edges = (BmeEdge *)p;
    d.len = (double *)(d.edges + M);
    d.pick = (BmePick *)(d.len + M);
    d.cells = (uint2 *)(((uintptr_t)(d.pick + 1) + 255) & ~(uintptr_t)255);
    return d;
}

BmeSides sides_of(const BmeDev &d, uint32_t M) {
    const uint32_t *s = d.side;
    const uint64_t S = 2ull * M;
    return BmeSides{s, s + S, s + 2 * S, s + 3 * S, s + 4 * S, s + 5 * S, s + 6 * S, s + 6 * S + M};
}

cudaError_t upload(const BmeDev &d, const Topology &t, cudaStream_t s, BmeRun &r) {
    const uint64_t S = 2ull * t.M;
    const std::vector<uint32_t> *arr[6] = {&t.size, &t.label, &t.height, &t.kid0, &t.kid1, &t.flag};
    for (int i = 0; i < 6; i++) {
        cudaError_t e = cudaMemcpyAsync(d.side + i * S, arr[i]->data(), S * 4, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return e;
    }
    cudaError_t e = cudaMemcpyAsync(d.side + 6 * S, t.tin.data(), t.M * 4ull, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d.side + 6 * S + t.M, t.tout.data(), t.M * 4ull, cudaMemcpyHostToDevice, s);
    r.h2d += (6 * S + 2 * t.M) * 4;
    return e;
}

// the marked cells, level by level, in chunks of at most BME_CELL_CHUNK: one launch per level and chunk.  A chunk's
// upload is queued after the launches that read the previous one.
cudaError_t update(const BmeDev &d, const Topology &t, uint64_t chunk, cudaStream_t s, BmeRun &r) {
    std::vector<uint2> cells;
    std::vector<uint64_t> start;
    t.marked_cells(cells, start);
    const BmeSides sd = sides_of(d, t.M);
    const uint64_t total = cells.size();
    for (uint64_t c0 = 0; c0 < total; c0 += chunk) {
        const uint64_t c1 = std::min(total, c0 + chunk);
        BK(cudaMemcpyAsync(d.cells, cells.data() + c0, (c1 - c0) * sizeof(uint2), cudaMemcpyHostToDevice, s));
        r.h2d += (c1 - c0) * sizeof(uint2);
        for (uint64_t L = 1; L + 1 < start.size(); L++) {
            const uint64_t lo = std::max(start[L], c0), hi = std::min(start[L + 1], c1);
            if (lo >= hi) continue;
            const uint32_t cnt = (uint32_t)(hi - lo);
            k_bme_cells<<<(cnt + BME_THREADS - 1) / BME_THREADS, BME_THREADS, 0, s>>>(d.T, t.M, sd, d.cells + (lo - c0), cnt);
            r.launches++;
        }
    }
    return cudaGetLastError();
}

// levels 1 .. top over every cell (the build)
cudaError_t levels(const BmeDev &d, const Topology &t, uint32_t top, cudaStream_t s, BmeRun &r) {
    const dim3 grid(t.M, (t.M + BME_THREADS - 1) / BME_THREADS);
    const BmeSides sd = sides_of(d, t.M);
    for (uint32_t L = 1; L <= top; L++) k_bme_level<<<grid, BME_THREADS, 0, s>>>(d.T, t.M, sd, L);
    r.launches += top;
    return cudaGetLastError();
}

}  // namespace

uint64_t bme_table_bytes(uint32_t n) {
    if (n < 2) return 0;
    const uint64_t N = n, M = 2 * N - 2;
    const uint64_t need = std::max(M * M * 8, N * M * 8 + bionj_state_bytes(n));
    return (need + 255) & ~255ull;
}

uint64_t bme_state_bytes(uint32_t n) {
    if (n < 2) return 0;
    const uint64_t M = 2ull * n - 2;
    return bme_table_bytes(n) + (8 * 2 * M) * 4 + 256 + M * sizeof(BmeEdge) + M * 8 + sizeof(BmePick) + 256 +
           std::min<uint64_t>(BME_CELL_CHUNK, M * M) * sizeof(uint2);
}

NjState bme_nj_state_at(void *base, uint32_t n, bool bionj) {
    return nj_state_at((char *)base + (uint64_t)n * (2ull * n - 2) * 8, n, bionj);
}

cudaError_t launch_bme_leaves(void *base, uint32_t n, cudaStream_t s) {
    const uint64_t M = 2ull * n - 2;
    const NjState st = bme_nj_state_at(base, n, false);
    k_bme_leaves<<<dim3(n, (n + BME_THREADS - 1) / BME_THREADS), BME_THREADS, 0, s>>>((double *)base, M, st.d, n);
    return cudaGetLastError();
}

cudaError_t bme_search(void *base, uint32_t n, const uint32_t *a, const uint32_t *b, cudaStream_t s, BmeRun &r) {
    const uint64_t cap = bme_max_swaps(n);
    r.swaps = 0;
    Topology t(n, a, b);
    const BmeDev d = bme_dev_at(base, n);
    for (uint32_t s2 = 0; s2 < 2 * t.M; s2++) t.flag[s2] |= SIDE_CHANGED;
    BK(upload(d, t, s, r));
    BK(levels(d, t, 2 * t.max_height(false), s, r));
    std::vector<BmeEdge> edges;
    while (r.swaps < cap) {
        const std::vector<uint32_t> at = t.internal_edges();
        if (at.empty()) break;
        edges.resize(at.size());
        for (size_t i = 0; i < at.size(); i++) edges[i] = t.internal_edge(at[i]);
        BK(cudaMemcpyAsync(d.edges, edges.data(), edges.size() * sizeof(BmeEdge), cudaMemcpyHostToDevice, s));
        r.h2d += edges.size() * sizeof(BmeEdge);
        k_bme_pick<<<1, PICK_THREADS, 0, s>>>(d.T, d.edges, (uint32_t)edges.size(), d.pick);
        r.launches++;
        BmePick p;
        BK(cudaMemcpyAsync(&p, d.pick, sizeof(p), cudaMemcpyDeviceToHost, s));
        BK(cudaStreamSynchronize(s));
        r.d2h += sizeof(p);
        if (!(p.gain > BME_EPS)) break;
        t.apply(at[p.edge], p.swap);
        BK(upload(d, t, s, r));
        BK(update(d, t, std::min<uint64_t>(BME_CELL_CHUNK, (uint64_t)t.M * t.M), s, r));
        r.swaps++;
    }
    // the lengths, then the rows in post-order from the root
    edges = t.length_edges();
    BK(cudaMemcpyAsync(d.edges, edges.data(), edges.size() * sizeof(BmeEdge), cudaMemcpyHostToDevice, s));
    r.h2d += edges.size() * sizeof(BmeEdge);
    k_bme_lengths<<<(t.M + BME_THREADS - 1) / BME_THREADS, BME_THREADS, 0, s>>>(d.T, d.edges, t.M, d.len);
    r.launches++;
    std::vector<double> len(t.M);
    BK(cudaMemcpyAsync(len.data(), d.len, t.M * 8ull, cudaMemcpyDeviceToHost, s));
    BK(cudaStreamSynchronize(s));
    r.d2h += t.M * 8ull;
    r.a.clear(), r.b.clear(), r.la.clear(), r.lb.clear();
    const uint32_t c0 = t.kid[2 * t.root], c1 = t.kid[2 * t.root + 1];
    auto lab = [&](uint32_t v) { return t.label[2 * v]; };
    std::vector<std::pair<uint32_t, bool>> stack;  // (node, children done)
    auto push_kids = [&](uint32_t v0, uint32_t v1) {  // the smaller label is emitted first
        if (lab(v1) < lab(v0)) std::swap(v0, v1);
        stack.push_back({v1, false});
        stack.push_back({v0, false});
    };
    push_kids(c0, c1);
    while (!stack.empty()) {
        auto [v, done] = stack.back();
        stack.pop_back();
        if (t.leaf(v)) continue;
        uint32_t k0 = t.kid[2 * v], k1 = t.kid[2 * v + 1];
        if (lab(k1) < lab(k0)) std::swap(k0, k1);
        if (done) {
            r.a.push_back(lab(k0)), r.b.push_back(lab(k1)), r.la.push_back(len[k0]), r.lb.push_back(len[k1]);
        } else {
            stack.push_back({v, true});
            push_kids(k0, k1);
        }
    }
    const double h = 0.5 * len[c0];  // exact: a product by 0.5 on the host rounds as on the device
    r.a.push_back(std::min(lab(c0), lab(c1))), r.b.push_back(std::max(lab(c0), lab(c1)));
    r.la.push_back(h), r.lb.push_back(h);
    return cudaSuccess;
}

}  // namespace gkd
