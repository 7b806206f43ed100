// Symbolic phase of the nested-dissection multifrontal solver (host only, no CUDA types).
//
// Replaces the analysis step MUMPS performs inside `factorMUMPS(Aii,1)` (MUMPSfuncs.jl:24-39, called from mt2DTE.jl:50-53):
// a fill-reducing ordering, the supernode (front) tree and the index maps of the extend-add.  The numeric phase
// (mf_kernels.cuh / mf_solver.cu) consumes the flat tables built here; they are identical for every system of a batch
// (all frequencies / modes / chains share one sparsity pattern).
//
//   * ordering      : geometric nested dissection of the nl x nf grid (closed-form line separators, mf_order_grid) for the MT
//                     stencil systems; recursive bisection by breadth-first level sets (mf_order_graph) for arbitrary symmetric
//                     patterns handed to the Level-1 shim.  Both return the supernode partition in elimination (post) order.
//   * symbolic      : structure of every front = [pivot columns | update rows], parent = supernode holding the first update
//                     row, depth from the roots.  Fronts of depth d+1 are exactly the children of fronts of depth d, so the
//                     numeric phase runs depth by depth with two ping-pong arenas.
//   * padding       : pivot and update counts are padded to multiples of 8 (the DMMA tile): padded pivots are identity rows.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <functional>
#include <numeric>
#include <queue>
#include <vector>

namespace hmcmt {
namespace mf {

constexpr int kTile = 8;
constexpr int kChunkMax = 96;      // pivots eliminated per step on a large front (diagonal block inverted in shared memory)

inline int pad8(int x) { return (x + 7) & ~7; }

// shared memory of the single-CTA front kernel (mf_kernels.cuh) for a front of nb tile rows of which npb are pivots:
// lower tiles + max(sweep scratch, M' buffer) + the pivot block inverse + flag
// (+ the front's record at the head, + relTotal ints: the row maps of all children, staged together ahead of the extend-add)
constexpr size_t kFrontDescBytes = 160;
constexpr int kSmallChildren = 4;
inline size_t mf_front_smem_bytes(int nb, int npb, int relTotal = 0) {
    const size_t nT = (size_t)nb * (nb + 1) / 2, nS = 2 * (size_t)npb, nM = (size_t)(nb - npb) * npb;
    return kFrontDescBytes + (nT + (nS > nM ? nS : nM) + 1) * 128 * sizeof(double) + 16 + (((size_t)relTotal + 1) & ~(size_t)1) * 2 * sizeof(int);
}
// The 8- and 16-warp instantiations (launches whose largest front has more than 64 rows) keep only the pivot columns: the
// pivot triangle and the F21 block, no F22 (gathered from the children straight into the registers of the Schur product),
// plus one inverse row map of the update rows per child (nChild x (nb - npb) * 8 ints).  M' = F21 (-G) stays in shared
// memory beside them (resident M').
inline size_t mf_mid_front_smem_bytes(int nb, int npb, int relTotal, int nChild) {
    const size_t nub = (size_t)(nb - npb), nT = (size_t)npb * (npb + 1) / 2 + nub * npb, nS = 2 * (size_t)npb, nM = nub * npb;
    return kFrontDescBytes + (nT + (nS > nM ? nS : nM) + 1) * 128 * sizeof(double) + 16 + (((size_t)relTotal + 1) & ~(size_t)1) * 2 * sizeof(int) +
           (size_t)nChild * nub * 8 * sizeof(int);
}
// The same layout without M' (streamed M', mf_small_stream_kernel): the products write M' to the factor arena as M and the
// Schur product reads it back from there (L2), so shared memory holds the pivot columns, the sweep scratch and the row maps.
inline size_t mf_stream_front_smem_bytes(int nb, int npb, int relTotal, int nChild) {
    const size_t nub = (size_t)(nb - npb), nT = (size_t)npb * (npb + 1) / 2 + nub * npb, nS = 2 * (size_t)npb;
    return kFrontDescBytes + (nT + nS + 1) * 128 * sizeof(double) + 16 + (((size_t)relTotal + 1) & ~(size_t)1) * 2 * sizeof(int) +
           (size_t)nChild * nub * 8 * sizeof(int);
}
constexpr size_t kFrontSmemMax = 227 * 1024;
// Fronts of up to kFullFrontMaxFp rows are classified on the whole-front layout (mf_front_smem_bytes), whatever instantiation
// later runs them.  Larger ones (up to fSmall) run in the pivot-column layout of the 8 / 16-warp instantiations: with M' in
// shared memory when that fits, else with M' streamed through the factor arena.
constexpr int kFullFrontMaxFp = 144;
inline bool mf_front_needs_stream(int nb, int npb, int relTotal, int nChild) {
    return mf_mid_front_smem_bytes(nb, npb, relTotal, nChild) > kFrontSmemMax;
}
inline size_t mf_large_front_smem_bytes(int nb, int npb, int relTotal, int nChild) {
    return mf_front_needs_stream(nb, npb, relTotal, nChild) ? mf_stream_front_smem_bytes(nb, npb, relTotal, nChild)
                                                            : mf_mid_front_smem_bytes(nb, npb, relTotal, nChild);
}

// lower-triangular entry of the original matrix (row >= col, original numbering) and where its value comes from
struct Entry {
    int row, col, src;      // src: index into the per-system value array handed to the numeric phase
};

struct OrigEntry {
    int lrow, lcol, src;    // position inside the front (local indices), src < 0: the constant 1 (identity padding)
};

struct Chunk {
    int p0, p1;             // pivot range [p0, p1) inside the front (multiples of 8)
    int64_t gOff, mOff;     // offsets (in doubles) into the per-system factor arena: G (sc x sc), M ((fp-p1) x sc)
};

struct Front {
    int s, sp, u, up;       // real / padded pivot and update counts; fp = sp + up
    int cbp;                // base of the pivots in the padded permuted numbering
    int rowPtr;             // offset of the update rows in Symbolic::rows / rel
    int parent, depth;
    int childPtr, nChild;   // into Symbolic::children
    int origPtr, nOrig;     // into Symbolic::orig
    int chunkPtr, nChunk;   // into Symbolic::chunks
    int isBig;              // 1: front lives in global memory (three-phase path), 0: one CTA, shared memory
    int64_t frontOff;       // big: offset of the fp x fp front in the depth-parity arena; small: offset of its up x up update matrix
    int64_t updOff;         // offset (complex entries) of its update vector in the solve workspace
    int fp() const { return sp + up; }
    // where the update matrix U = F22 lives: k-grouped matrix with `ldU` rows, first row / column `offU`
    int ldU() const { return isBig ? sp + up : up; }
    int offU() const { return isBig ? sp : 0; }
};

struct Symbolic {
    int N = 0, Np = 0, K = 0, maxDepth = 0;
    std::vector<int> pos2orig;          // [Np] padded permuted position -> original index (-1: padding)
    std::vector<int> orig2pos;          // [N]
    std::vector<Front> fronts;          // elimination order
    std::vector<int> rows;              // update rows of every front (padded permuted positions, ascending)
    std::vector<int> rel;               // same indexing: local index of that row inside the parent's front
    std::vector<int> children;
    std::vector<OrigEntry> orig;
    std::vector<Chunk> chunks;
    std::vector<std::vector<int>> byDepthSmall, byDepthBig;      // launch lists
    std::vector<int64_t> bigDoublesAtDepth;                      // leading part of the depth arena holding the large fronts
    int64_t factorDoubles = 0;          // per system
    int64_t arenaDoubles[2] = {0, 0};   // per system, depth parity
    int64_t updEntries = 0;             // per system: total update-vector entries (complex)
    int maxFpSmall = 0, maxFpBig = 0, maxFp = 0;
    double flops = 0.0;                 // real flops of one factorisation (padded sizes, sweep formulation)
};

// ------------------------------------------------------------------------------------------------------------------------
// orderings: each returns the supernodes (lists of original indices) in elimination order

// nl lines of nf unknowns, q = l*nf + f, 5-point coupling (q, q-1) inside a line and (q, q-nf) between lines
//   leaf  : boxes of at most `leaf` unknowns are eliminated as one dense supernode
//   cross : boxes whose longer side is at most `cross` are cut four ways by a cross-shaped separator (one supernode = the
//           middle line + the two halves of the middle column): half as many tree levels and no 3..6-unknown separators padded
//           to a whole 8-pivot tile at the bottom of the tree, where the fronts are bound by latency and not by flops
//   push  : a leaf box whose unknown count exceeds a multiple of 8 by at most `push` hands that excess (nodes next to the
//           separator above it) to the separator's supernode when that one has padding to spare: a 3 x 3 leaf then eliminates
//           8 unknowns in ONE 8-pivot tile instead of 9 in two (the second tile would be 1 pivot + 7 identity rows: a whole
//           inversion / barrier round, and a 16 x 16 instead of an 8 x 8 block in the factor), the 3-unknown separator takes the
//           ninth into its own padding.  Any partition is a valid elimination order; only the fill changes (marginally).
inline void mf_order_grid(int nl, int nf, int leaf, std::vector<std::vector<int>>& out, int cross = 0, int push = 0) {
    // returns the index in `out` of the supernode emitted last for the box (-1: none) and whether the box was a leaf
    std::function<int(int, int, int, int, bool&)> rec = [&](int l0, int l1, int f0, int f1, bool& isLeaf) -> int {
        const int nL = l1 - l0, nF = f1 - f0;
        isLeaf = false;
        if (nL <= 0 || nF <= 0) return -1;
        if (nL * nF <= leaf) {
            std::vector<int> v;
            v.reserve((size_t)nL * nF);
            for (int l = l0; l < l1; ++l)
                for (int f = f0; f < f1; ++f) v.push_back(l * nf + f);
            out.push_back(std::move(v));
            isLeaf = true;
            return (int)out.size() - 1;
        }
        std::vector<int> sep;
        bool la = false, lb = false, lc = false, ld = false;
        if (std::max(nL, nF) <= cross && std::min(nL, nF) >= 3) {
            const int ml = (l0 + l1) / 2, mf = (f0 + f1) / 2;
            rec(l0, ml, f0, mf, la);
            rec(l0, ml, mf + 1, f1, lb);
            rec(ml + 1, l1, f0, mf, lc);
            rec(ml + 1, l1, mf + 1, f1, ld);
            for (int f = f0; f < f1; ++f) sep.push_back(ml * nf + f);
            for (int l = l0; l < l1; ++l)
                if (l != ml) sep.push_back(l * nf + mf);
        } else {
            const bool byLine = nL >= nF;
            const int mid = byLine ? (l0 + l1) / 2 : (f0 + f1) / 2;
            const int a = byLine ? rec(l0, mid, f0, f1, la) : rec(l0, l1, f0, mid, la);
            const int b = byLine ? rec(mid + 1, l1, f0, f1, lb) : rec(l0, l1, mid + 1, f1, lb);
            if (byLine) for (int f = f0; f < f1; ++f) sep.push_back(mid * nf + f);
            else for (int l = l0; l < l1; ++l) sep.push_back(l * nf + mid);
            const int cap = pad8((int)sep.size());
            auto absorb = [&](int ci, bool childIsLeaf, int adj) {      // adj: line / column of the child next to the separator
                if (ci < 0 || !childIsLeaf || push <= 0) return;
                std::vector<int>& v = out[ci];
                const int s = (int)v.size(), e = s % 8;
                if (s <= 8 || e == 0 || e > push || (int)sep.size() + e > cap) return;
                int moved = 0;
                for (size_t i = 0; i < v.size() && moved < e;) {
                    const int q = v[i], l = q / nf, f = q - l * nf;
                    if ((byLine ? l : f) == adj) { sep.push_back(q); v.erase(v.begin() + i); ++moved; }
                    else ++i;
                }
            };
            absorb(a, la, mid - 1);
            absorb(b, lb, mid + 1);
        }
        out.push_back(std::move(sep));
        return (int)out.size() - 1;
    };
    bool dummy = false;
    rec(0, nl, 0, nf, dummy);
}

// general symmetric pattern (adjacency in CSR form without the diagonal): recursive bisection, the separator is the smallest
// breadth-first level between 35 % and 65 % of the region, start node = a pseudo-peripheral node of the region
inline void mf_order_graph(int n, const std::vector<int>& adjPtr, const std::vector<int>& adj, int leaf,
                           std::vector<std::vector<int>>& out) {
    std::vector<int> region(n, 0);      // region id of every node (-1: already ordered)
    std::vector<int> level(n, -1), queue;
    queue.reserve(n);
    int nextRegion = 1;
    // explicit stack of (region id, node list); post-order emission through a marker entry
    struct Item {
        std::vector<int> nodes;
        std::vector<int> sep;
        int stage;
    };
    std::vector<Item> stack;
    {
        Item it;
        it.nodes.resize(n);
        std::iota(it.nodes.begin(), it.nodes.end(), 0);
        it.stage = 0;
        stack.push_back(std::move(it));
    }
    auto bfs = [&](int start, int rid, const std::vector<int>& nodes, int& nLevels) {
        for (int v : nodes) level[v] = -1;
        queue.clear();
        queue.push_back(start);
        level[start] = 0;
        size_t head = 0;
        while (head < queue.size()) {
            const int v = queue[head++];
            for (int k = adjPtr[v]; k < adjPtr[v + 1]; ++k) {
                const int w = adj[k];
                if (region[w] == rid && level[w] < 0) {
                    level[w] = level[v] + 1;
                    queue.push_back(w);
                }
            }
        }
        nLevels = level[queue.back()] + 1;
    };
    while (!stack.empty()) {
        if (stack.back().stage == 1) {          // both parts emitted: now the separator
            if (!stack.back().sep.empty()) out.push_back(std::move(stack.back().sep));
            stack.pop_back();
            continue;
        }
        Item it = std::move(stack.back());
        stack.pop_back();
        std::vector<int>& nodes = it.nodes;
        if (nodes.empty()) continue;
        if ((int)nodes.size() <= leaf) {
            out.push_back(std::move(nodes));
            continue;
        }
        const int rid = nextRegion++;
        for (int v : nodes) region[v] = rid;
        int nLevels = 0;
        bfs(nodes[0], rid, nodes, nLevels);
        if (queue.size() < nodes.size()) {
            // disconnected: the component reached and the rest are independent parts, no separator
            Item a, b;
            a.stage = b.stage = 0;
            for (int v : nodes) (level[v] >= 0 ? a.nodes : b.nodes).push_back(v);
            Item marker;
            marker.stage = 1;
            stack.push_back(std::move(marker));
            stack.push_back(std::move(b));
            stack.push_back(std::move(a));
            continue;
        }
        // pseudo-peripheral start: restart twice from the last node reached
        for (int rep = 0; rep < 2; ++rep) {
            const int far = queue.back();
            bfs(far, rid, nodes, nLevels);
        }
        if (nLevels < 3) {      // (nearly) complete graph: one dense front
            out.push_back(std::move(nodes));
            continue;
        }
        std::vector<int> cnt(nLevels, 0);
        for (int v : nodes) ++cnt[level[v]];
        const double tot = (double)nodes.size();
        int best = -1;
        double acc = 0.0;
        for (int L = 0; L < nLevels; ++L) {
            const double before = acc;
            acc += cnt[L];
            if (L == 0 || L == nLevels - 1) continue;
            if (before >= 0.35 * tot && before <= 0.65 * tot)
                if (best < 0 || cnt[L] < cnt[best]) best = L;
        }
        if (best < 0) {
            // no level starts inside the window: take the level containing the median
            acc = 0.0;
            for (int L = 0; L < nLevels; ++L) {
                acc += cnt[L];
                if (acc >= 0.5 * tot) { best = std::min(std::max(L, 1), nLevels - 2); break; }
            }
        }
        Item a, b, marker;
        a.stage = b.stage = 0;
        marker.stage = 1;
        for (int v : nodes) {
            if (level[v] < best) a.nodes.push_back(v);
            else if (level[v] > best) b.nodes.push_back(v);
            else marker.sep.push_back(v);
        }
        for (int v : marker.sep) region[v] = -1;
        stack.push_back(std::move(marker));
        stack.push_back(std::move(b));
        stack.push_back(std::move(a));
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// symbolic factorisation for a given supernode partition + layout of the numeric phase
//   entries : lower-triangular pattern (row >= col) with value sources, must contain every diagonal entry
//   fSmall  : fronts with fp <= fSmall are handled by the single-CTA shared-memory kernel
inline bool mf_symbolic(int N, const std::vector<std::vector<int>>& snodes, const std::vector<Entry>& entries, int fSmall,
                        Symbolic& S) {
    S = Symbolic();
    S.N = N;
    const int K = (int)snodes.size();
    S.K = K;
    S.fronts.resize(K);
    S.orig2pos.assign(N, -1);
    std::vector<int> cbp(K + 1, 0);
    for (int k = 0; k < K; ++k) cbp[k + 1] = cbp[k] + pad8((int)snodes[k].size());
    S.Np = cbp[K];
    S.pos2orig.assign(S.Np, -1);
    std::vector<int> snOf(S.Np, -1);
    for (int k = 0; k < K; ++k) {
        for (int i = 0; i < (int)snodes[k].size(); ++i) {
            const int o = snodes[k][i];
            if (o < 0 || o >= N || S.orig2pos[o] >= 0) return false;
            S.orig2pos[o] = cbp[k] + i;
            S.pos2orig[cbp[k] + i] = o;
        }
        for (int p = cbp[k]; p < cbp[k + 1]; ++p) snOf[p] = k;
    }
    for (int o = 0; o < N; ++o) if (S.orig2pos[o] < 0) return false;
    // adjacency (strictly lower part, permuted): column lo -> rows hi
    std::vector<int> aPtr(S.Np + 1, 0);
    for (const Entry& e : entries) {
        const int a = S.orig2pos[e.row], b = S.orig2pos[e.col];
        if (a != b) ++aPtr[std::min(a, b) + 1];
    }
    for (int p = 0; p < S.Np; ++p) aPtr[p + 1] += aPtr[p];
    std::vector<int> aIdx(aPtr[S.Np]), fill(aPtr.begin(), aPtr.end() - 1);
    for (const Entry& e : entries) {
        const int a = S.orig2pos[e.row], b = S.orig2pos[e.col];
        if (a != b) aIdx[fill[std::min(a, b)]++] = std::max(a, b);
    }
    // structures
    std::vector<std::vector<int>> pending(K);      // update rows handed up by the children (may contain duplicates)
    std::vector<int> mark(S.Np, -1);
    S.rows.clear();
    std::vector<std::vector<int>> kids(K);
    for (int k = 0; k < K; ++k) {
        Front& F = S.fronts[k];
        F.s = (int)snodes[k].size();
        F.sp = pad8(F.s);
        F.cbp = cbp[k];
        const int c1 = cbp[k + 1];
        std::vector<int> st;
        for (int p = cbp[k]; p < cbp[k] + F.s; ++p)
            for (int q = aPtr[p]; q < aPtr[p + 1]; ++q) {
                const int r = aIdx[q];
                if (r >= c1 && mark[r] != k) { mark[r] = k; st.push_back(r); }
            }
        for (int r : pending[k])
            if (r >= c1 && mark[r] != k) { mark[r] = k; st.push_back(r); }
        std::vector<int>().swap(pending[k]);
        std::sort(st.begin(), st.end());
        F.u = (int)st.size();
        F.up = pad8(F.u);
        F.rowPtr = (int)S.rows.size();
        F.parent = -1;
        if (F.u) {
            F.parent = snOf[st[0]];
            kids[F.parent].push_back(k);
            std::vector<int>& pp = pending[F.parent];
            pp.insert(pp.end(), st.begin(), st.end());
        }
        S.rows.insert(S.rows.end(), st.begin(), st.end());
        // padded update rows: index -1 (never referenced: their matrix rows are zero)
        for (int i = F.u; i < F.up; ++i) S.rows.push_back(-1);
    }
    // depth, children table
    S.maxDepth = 0;
    for (int k = K - 1; k >= 0; --k) {
        Front& F = S.fronts[k];
        F.depth = F.parent < 0 ? 0 : S.fronts[F.parent].depth + 1;
        S.maxDepth = std::max(S.maxDepth, F.depth);
        F.childPtr = (int)S.children.size();
        F.nChild = (int)kids[k].size();
        S.children.insert(S.children.end(), kids[k].begin(), kids[k].end());
    }
    // relative positions inside the parent front
    S.rel.assign(S.rows.size(), -1);
    for (int k = 0; k < K; ++k) {
        const Front& F = S.fronts[k];
        if (F.parent < 0) continue;
        const Front& P = S.fronts[F.parent];
        const int* prow = S.rows.data() + P.rowPtr;
        for (int i = 0; i < F.u; ++i) {
            const int r = S.rows[F.rowPtr + i];
            int loc;
            if (r < P.cbp + P.sp) loc = r - P.cbp;
            else {
                const int* it = std::lower_bound(prow, prow + P.u, r);
                if (it == prow + P.u || *it != r) return false;
                loc = P.sp + (int)(it - prow);
            }
            S.rel[F.rowPtr + i] = loc;
        }
    }
    // original entries per front (+ identity on the padded pivots)
    {
        std::vector<int> cnt(K + 1, 0);
        for (const Entry& e : entries) {
            const int lo = std::min(S.orig2pos[e.row], S.orig2pos[e.col]);
            ++cnt[snOf[lo] + 1];
        }
        for (int k = 0; k < K; ++k) cnt[k + 1] += S.fronts[k].sp - S.fronts[k].s;
        for (int k = 0; k < K; ++k) cnt[k + 1] += cnt[k];
        S.orig.resize(cnt[K]);
        std::vector<int> at(cnt.begin(), cnt.end() - 1);
        for (int k = 0; k < K; ++k) {
            S.fronts[k].origPtr = cnt[k];
            S.fronts[k].nOrig = cnt[k + 1] - cnt[k];
        }
        for (const Entry& e : entries) {
            const int a = S.orig2pos[e.row], b = S.orig2pos[e.col];
            const int lo = std::min(a, b), hi = std::max(a, b);
            const int k = snOf[lo];
            const Front& F = S.fronts[k];
            int lrow;
            if (hi < F.cbp + F.sp) lrow = hi - F.cbp;
            else {
                const int* r0 = S.rows.data() + F.rowPtr;
                const int* it = std::lower_bound(r0, r0 + F.u, hi);
                if (it == r0 + F.u || *it != hi) return false;
                lrow = F.sp + (int)(it - r0);
            }
            S.orig[at[k]++] = OrigEntry{lrow, lo - F.cbp, e.src};
        }
        for (int k = 0; k < K; ++k)
            for (int i = S.fronts[k].s; i < S.fronts[k].sp; ++i) S.orig[at[k]++] = OrigEntry{i, i, -1};
    }
    // numeric layout: per depth the large fronts first (that part of the arena is written completely by the gather assembly), then the update
    // matrices of the small fronts
    S.byDepthSmall.assign(S.maxDepth + 1, {});
    S.byDepthBig.assign(S.maxDepth + 1, {});
    int64_t fac = 0, arena[2] = {0, 0}, upd = 0;
    std::vector<int64_t> arenaAtDepth(S.maxDepth + 1, 0);
    for (int k = 0; k < K; ++k) {
        Front& F = S.fronts[k];
        const int fp = F.fp();
        int relTotal = 0;
        for (int c = 0; c < F.nChild; ++c) relTotal += S.fronts[S.children[F.childPtr + c]].u;
        // (the single-CTA kernel's front record describes up to kSmallChildren children)
        const size_t smem = fp <= kFullFrontMaxFp ? mf_front_smem_bytes(fp / 8, F.sp / 8, relTotal)
                                                  : mf_large_front_smem_bytes(fp / 8, F.sp / 8, relTotal, F.nChild);
        F.isBig = (fp > fSmall || F.nChild > kSmallChildren || smem > kFrontSmemMax) ? 1 : 0;
        S.maxFp = std::max(S.maxFp, fp);
        (F.isBig ? S.maxFpBig : S.maxFpSmall) = std::max(F.isBig ? S.maxFpBig : S.maxFpSmall, fp);
        (F.isBig ? S.byDepthBig : S.byDepthSmall)[F.depth].push_back(k);
        F.updOff = upd;
        upd += F.up;
        F.chunkPtr = (int)S.chunks.size();
        const int cmax = F.isBig ? kChunkMax : F.sp;
        for (int p0 = 0; p0 < F.sp; p0 += cmax) {
            const int p1 = std::min(p0 + cmax, F.sp), sc = p1 - p0;
            Chunk c{p0, p1, fac, 0};
            fac += 2 * (int64_t)sc * sc;
            c.mOff = fac;
            fac += 2 * (int64_t)(fp - p1) * sc;
            S.chunks.push_back(c);
            const double a = sc, b = fp - p1;
            S.flops += 8.0 * (0.5 * a * a * a + a * a * b + 0.5 * a * b * b);
        }
        F.nChunk = (int)S.chunks.size() - F.chunkPtr;
    }
    S.bigDoublesAtDepth.assign(S.maxDepth + 1, 0);
    for (int d = 0; d <= S.maxDepth; ++d) {
        for (int k : S.byDepthBig[d]) {
            Front& F = S.fronts[k];
            F.frontOff = arenaAtDepth[d];
            arenaAtDepth[d] += 2 * (int64_t)F.fp() * F.fp();
        }
        S.bigDoublesAtDepth[d] = arenaAtDepth[d];
        for (int k : S.byDepthSmall[d]) {
            Front& F = S.fronts[k];
            F.frontOff = arenaAtDepth[d];
            arenaAtDepth[d] += 2 * (int64_t)F.up * F.up;
        }
    }
    for (int d = 0; d <= S.maxDepth; ++d) arena[d & 1] = std::max(arena[d & 1], arenaAtDepth[d]);
    S.factorDoubles = fac;
    S.arenaDoubles[0] = arena[0];
    S.arenaDoubles[1] = arena[1];
    S.updEntries = upd;
    return true;
}

// real update rows of all children of front k (entries of the staged row maps)
inline int mf_rel_total(const Symbolic& S, int k) {
    const Front& F = S.fronts[k];
    int n = 0;
    for (int c = 0; c < F.nChild; ++c) n += S.fronts[S.children[F.childPtr + c]].u;
    return n;
}

// ------------------------------------------------------------------------------------------------------------------------
// launch-schedule rules of the numeric phase (mf_solver.cu), kept here so that host tools can classify fronts without CUDA
constexpr int kSolveWarpMaxFp = 64;       // solves: warp-per-front kernels up to this front size
constexpr int kSolveMfThreads = 256;      // CTA-per-front solve kernels: upper bound, 128 where no front of the depth exceeds 144 rows

// tuning knobs read from the environment when a solver builds its schedule (and hashed into the Level-1 shim's cache key)
struct SchedKnobs {
    int fp1 = 40, fp2 = 40, fp4 = 64, fp8 = 96;      // HMCMT_MF_FP1/2/4/8: largest front of a launch per warp count
    int solveThreads = 0;                            // HMCMT_MF_SOLVE_THREADS: CTA-solve threads, 0 = by front size
    static SchedKnobs from_env() {
        auto knob = [](const char* name, int dflt) { const char* e = std::getenv(name); return e ? std::atoi(e) : dflt; };
        SchedKnobs k;
        k.fp1 = knob("HMCMT_MF_FP1", k.fp1); k.fp2 = knob("HMCMT_MF_FP2", k.fp2);
        k.fp4 = knob("HMCMT_MF_FP4", k.fp4); k.fp8 = knob("HMCMT_MF_FP8", k.fp8);
        k.solveThreads = knob("HMCMT_MF_SOLVE_THREADS", 0);
        return k;
    }
};

// warps per front of a single-CTA launch, by the largest front of the launch (measured optimum at cfg2; one warp per front needs
// no CTA barrier).  Fronts above kFullFrontMaxFp rows exist only in the pivot-column layout: at least 8 warps.
inline int mf_small_warps(int maxFp, const SchedKnobs& k) {
    const int w = maxFp <= k.fp1 ? 1 : (maxFp <= k.fp2 ? 2 : (maxFp <= k.fp4 ? 4 : (maxFp <= k.fp8 ? 8 : 16)));
    return maxFp > kFullFrontMaxFp && w < 8 ? 8 : w;
}
// a single-CTA launch streams M' (16 warps, mf_small_stream_kernel) when one of its fronts needs it
inline bool mf_small_stream(const Symbolic& S, const std::vector<int>& launch) {
    for (int k : launch) {
        const Front& F = S.fronts[k];
        if (F.fp() > kFullFrontMaxFp && mf_front_needs_stream(F.fp() / 8, F.sp / 8, mf_rel_total(S, k), F.nChild)) return true;
    }
    return false;
}
// solves: one warp per front (record-driven kernels) for small fronts with few children, one CTA per front otherwise
inline bool mf_solve_by_warp(const Front& F) { return !F.isBig && F.fp() <= kSolveWarpMaxFp && F.nChild <= kSmallChildren; }
// threads of the CTA-per-front solve kernels at a depth whose largest CTA-solved front has maxFp rows
inline int mf_solve_cta_threads(int maxFp, const SchedKnobs& k) {
    return k.solveThreads ? k.solveThreads : (maxFp <= 144 ? 128 : kSolveMfThreads);
}

// Level-1 analysis of a 1-based CSC pattern (n columns, colptr[n] - 1 entries, both triangles or one): the lower triangle
// (row >= col) is what the factorisation reads, entry k takes its value from nzval[k]; ordered by level-set bisection.
inline bool mf_analyse_csc(int64_t n, const int64_t* rowval, const int64_t* colptr, int leaf, int fSmall, Symbolic& S) {
    std::vector<Entry> ent;
    ent.reserve((size_t)(colptr[n] - 1) / 2 + n);
    std::vector<int> ptr(n + 1, 0);
    for (int64_t j = 0; j < n; ++j)
        for (int64_t k = colptr[j] - 1; k < colptr[j + 1] - 1; ++k) {
            const int64_t i = rowval[k] - 1;
            if (i < 0 || i >= n) return false;
            if (i < j) continue;
            ent.push_back(Entry{(int)i, (int)j, (int)k});
            if (i != j) { ++ptr[i + 1]; ++ptr[j + 1]; }
        }
    for (int64_t i = 0; i < n; ++i) ptr[i + 1] += ptr[i];
    std::vector<int> adj(ptr[n]), at(ptr.begin(), ptr.end() - 1);
    for (const Entry& e : ent)
        if (e.row != e.col) { adj[at[e.row]++] = e.col; adj[at[e.col]++] = e.row; }
    std::vector<std::vector<int>> sn;
    mf_order_graph((int)n, ptr, adj, leaf, sn);
    return mf_symbolic((int)n, sn, ent, fSmall, S);
}

// pattern of the MT stencil systems in the internal ordering (mt_kernels.cuh): value array = [diag N | e1 N | e2 N]
inline void mf_grid_entries(int nl, int nf, std::vector<Entry>& e) {
    const int N = nl * nf;
    e.clear();
    e.reserve((size_t)3 * N);
    for (int l = 0; l < nl; ++l)
        for (int f = 0; f < nf; ++f) {
            const int q = l * nf + f;
            e.push_back(Entry{q, q, q});
            if (f > 0) e.push_back(Entry{q, q - 1, N + q});
            if (l > 0) e.push_back(Entry{q, q - nf, 2 * N + q});
        }
}

}  // namespace mf
}  // namespace hmcmt
