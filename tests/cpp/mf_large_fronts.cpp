// Single-CTA fronts above 144 rows on the tables of mf_symbolic.h (host only): the classification of every front and the
// single-CTA launch of every depth as mf_solver.cu builds it, and a hash of the symbolic tables and of that schedule (layout-
// independent of the build: sizes, offsets and lists only), so that the tables at fSmall = 144 can be pinned.  Test
// infrastructure only.
//   usage: mf_large_fronts grid <nl> <nf> <leaf> <fSmall> <cross> <push>   (MT stencil pattern, the plan's ordering)
//          mf_large_fronts csc <pattern file> <leaf> <fSmall>                  (Level-1 analysis; file as for mf_classes.cpp)
//   output: one line per depth, then one per front of more than 144 rows, then the hash:
//     depth <d> nSmall <n> nBig <n> maxFpSmall <fp> warps <w> stream <0|1> smem <bytes>
//     front <k> depth <d> sp <sp> up <up> nChild <c> big <0|1> layout <resident|streamed|-> nChunk <n>
//     hash <16 hex digits>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../hmcmt2d_b200/csrc/mf_symbolic.h"

using namespace hmcmt::mf;

static uint64_t h = 1469598103934665603ull;
static void mix(int64_t v) {
    for (int i = 0; i < 8; ++i) { h ^= (uint64_t)((v >> (8 * i)) & 0xff); h *= 1099511628211ull; }
}

int main(int argc, char** argv) {
    Symbolic S;
    if (argc >= 8 && !strcmp(argv[1], "grid")) {
        const int nl = atoi(argv[2]), nf = atoi(argv[3]), leaf = atoi(argv[4]), fSmall = atoi(argv[5]);
        std::vector<Entry> ent;
        std::vector<std::vector<int>> sn;
        mf_grid_entries(nl, nf, ent);
        mf_order_grid(nl, nf, leaf, sn, atoi(argv[6]), atoi(argv[7]));
        if (!mf_symbolic(nl * nf, sn, ent, fSmall, S)) { printf("symbolic failed\n"); return 1; }
    } else if (argc >= 5 && !strcmp(argv[1], "csc")) {
        FILE* f = fopen(argv[2], "r");
        if (!f) return 2;
        long long n = 0;
        if (fscanf(f, "%lld", &n) != 1 || n < 1) return 2;
        std::vector<int64_t> colptr(n + 1);
        for (auto& v : colptr) if (fscanf(f, "%lld", (long long*)&v) != 1) return 2;
        std::vector<int64_t> rowval(colptr[n] - 1);
        for (auto& v : rowval) if (fscanf(f, "%lld", (long long*)&v) != 1) return 2;
        fclose(f);
        if (!mf_analyse_csc(n, rowval.data(), colptr.data(), atoi(argv[3]), atoi(argv[4]), S)) { printf("analysis failed\n"); return 1; }
    } else {
        return 2;
    }
    const SchedKnobs kn;      // the library's defaults
    for (const Front& F : S.fronts)
        for (int64_t v : {(int64_t)F.s, (int64_t)F.sp, (int64_t)F.u, (int64_t)F.up, (int64_t)F.cbp, (int64_t)F.rowPtr, (int64_t)F.parent,
                          (int64_t)F.depth, (int64_t)F.childPtr, (int64_t)F.nChild, (int64_t)F.origPtr, (int64_t)F.nOrig, (int64_t)F.chunkPtr,
                          (int64_t)F.nChunk, (int64_t)F.isBig, F.frontOff, F.updOff})
            mix(v);
    for (const Chunk& c : S.chunks) { mix(c.p0); mix(c.p1); mix(c.gOff); mix(c.mOff); }
    for (int v : S.rows) mix(v);
    for (int v : S.rel) mix(v);
    for (int v : S.children) mix(v);
    for (const OrigEntry& o : S.orig) { mix(o.lrow); mix(o.lcol); mix(o.src); }
    for (int64_t v : {S.factorDoubles, S.arenaDoubles[0], S.arenaDoubles[1], S.updEntries}) mix(v);
    for (int d = 0; d <= S.maxDepth; ++d) {
        const std::vector<int>& sm = S.byDepthSmall[d];
        int mx = 0;
        for (int k : sm) mx = std::max(mx, S.fronts[k].fp());
        // the launch as Solver::build() forms it
        const bool stream = !sm.empty() && mf_small_stream(S, sm);
        const int warps = sm.empty() ? 0 : (stream ? 16 : mf_small_warps(mx, kn));
        size_t smem = 0;
        for (int k : sm) {
            const Front& F = S.fronts[k];
            const int nb = F.fp() / 8, npb = F.sp / 8, rt = mf_rel_total(S, k);
            smem = std::max(smem, stream ? mf_stream_front_smem_bytes(nb, npb, rt, F.nChild)
                                         : warps >= 8 ? mf_mid_front_smem_bytes(nb, npb, rt, F.nChild) : mf_front_smem_bytes(nb, npb, rt));
        }
        for (int k : sm) mix(k);
        for (int k : S.byDepthBig[d]) mix(-1 - k);
        mix(warps); mix((int64_t)smem); mix(stream);
        printf("depth %d nSmall %d nBig %d maxFpSmall %d warps %d stream %d smem %zu\n", d, (int)sm.size(), (int)S.byDepthBig[d].size(), mx,
               warps, (int)stream, smem);
    }
    for (int k = 0; k < S.K; ++k) {
        const Front& F = S.fronts[k];
        if (F.fp() <= kFullFrontMaxFp) continue;
        const bool streamed = mf_front_needs_stream(F.fp() / 8, F.sp / 8, mf_rel_total(S, k), F.nChild);
        printf("front %d depth %d sp %d up %d nChild %d big %d layout %s nChunk %d\n", k, F.depth, F.sp, F.up, F.nChild, F.isBig,
               F.isBig ? "-" : (streamed ? "streamed" : "resident"), F.nChunk);
    }
    printf("hash %016llx\n", (unsigned long long)h);
    return 0;
}
