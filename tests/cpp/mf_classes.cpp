// Kernel classes of the multifrontal solver for a Level-1 matrix (host only, the analysis of mumps_shim.cu and the launch-schedule
// rules of mf_solver.cu, both from mf_symbolic.h): which kernel instantiation, layout and solve variant each front takes.  The GPU
// tests of the kernel classes (tests/test_gpu_mf_kernel_classes.py) declare the classes each of their matrices covers; the CPU
// test runs this program on the same matrices and checks the declarations, so that a change of thresholds or ordering that moves
// a matrix out of its class fails on any machine.  Test infrastructure only.
//   usage: mf_classes <pattern file> <leaf> <fSmall> <fp1> <fp2> <fp4> <fp8> <solveThreads>
//   pattern file: n, then the n + 1 entries of colptr, then the colptr[n] - 1 entries of rowval (1-based CSC, whitespace-separated)
//   output, one line per front then one per depth:
//     front <k> depth <d> s <s> sp <sp> u <u> fp <fp> nChild <c> big <0|1> why <-|fp|children|smem> nChunk <n> lastChunk <w>
//           warps <launch warps, 0: big> cpiv <p/cu,...|-> solve <warp|cta> width <warp-solve width, 0: cta>
//     depth <d> nSmall <n> nBig <n> warps <w> nSolveWarp <n> nSolveCta <n> threads <t>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../hmcmt2d_b200/csrc/mf_symbolic.h"

using namespace hmcmt::mf;

int main(int argc, char** argv) {
    if (argc < 9) return 2;
    FILE* f = fopen(argv[1], "r");
    if (!f) return 2;
    long long n = 0;
    if (fscanf(f, "%lld", &n) != 1 || n < 1) return 2;
    std::vector<int64_t> colptr(n + 1);
    for (auto& v : colptr) if (fscanf(f, "%lld", (long long*)&v) != 1) return 2;
    std::vector<int64_t> rowval(colptr[n] - 1);
    for (auto& v : rowval) if (fscanf(f, "%lld", (long long*)&v) != 1) return 2;
    fclose(f);
    const int leaf = atoi(argv[2]), fSmall = atoi(argv[3]);
    SchedKnobs kn;
    kn.fp1 = atoi(argv[4]); kn.fp2 = atoi(argv[5]); kn.fp4 = atoi(argv[6]); kn.fp8 = atoi(argv[7]); kn.solveThreads = atoi(argv[8]);
    Symbolic S;
    if (!mf_analyse_csc(n, rowval.data(), colptr.data(), leaf, fSmall, S)) { printf("analysis failed\n"); return 1; }

    std::vector<int> warpsAt(S.maxDepth + 1, 0), threadsAt(S.maxDepth + 1, 0), nWarp(S.maxDepth + 1, 0), nCta(S.maxDepth + 1, 0);
    for (int d = 0; d <= S.maxDepth; ++d) {
        int mx = 0, mxc = 0;
        for (int k : S.byDepthSmall[d]) mx = std::max(mx, S.fronts[k].fp());
        warpsAt[d] = S.byDepthSmall[d].empty() ? 0 : mf_small_warps(mx, kn);
        for (int k : S.byDepthBig[d]) { mxc = std::max(mxc, S.fronts[k].fp()); ++nCta[d]; }
        for (int k : S.byDepthSmall[d]) {
            if (mf_solve_by_warp(S.fronts[k])) ++nWarp[d];
            else { mxc = std::max(mxc, S.fronts[k].fp()); ++nCta[d]; }
        }
        threadsAt[d] = mf_solve_cta_threads(mxc, kn);
    }
    for (int k = 0; k < S.K; ++k) {
        const Front& F = S.fronts[k];
        const char* why = "-";
        if (F.isBig) why = F.fp() > fSmall ? "fp" : (F.nChild > kSmallChildren ? "children" : "smem");
        const Chunk& last = S.chunks[F.chunkPtr + F.nChunk - 1];
        std::string cpiv;
        if (!F.isBig)
            for (int c = 0; c < F.nChild; ++c) {      // SmallDesc::cPiv as mf_solver.cu computes it
                const Front& C = S.fronts[S.children[F.childPtr + c]];
                int piv = 0;
                while (piv < C.u && S.rel[C.rowPtr + piv] < F.sp) ++piv;
                cpiv += (cpiv.empty() ? "" : ",") + std::to_string(piv) + "/" + std::to_string(C.u);
            }
        const bool byWarp = mf_solve_by_warp(F);
        const int width = !byWarp ? 0 : (F.s <= 8 ? 8 : (F.s <= 16 ? 16 : 32));      // mf_bwd_warp_front
        printf("front %d depth %d s %d sp %d u %d fp %d nChild %d big %d why %s nChunk %d lastChunk %d warps %d cpiv %s solve %s width %d\n",
               k, F.depth, F.s, F.sp, F.u, F.fp(), F.nChild, F.isBig, why, F.nChunk, last.p1 - last.p0, F.isBig ? 0 : warpsAt[F.depth],
               cpiv.empty() ? "-" : cpiv.c_str(), byWarp ? "warp" : "cta", width);
    }
    for (int d = 0; d <= S.maxDepth; ++d)
        printf("depth %d nSmall %d nBig %d warps %d nSolveWarp %d nSolveCta %d threads %d\n", d, (int)S.byDepthSmall[d].size(),
               (int)S.byDepthBig[d].size(), warpsAt[d], nWarp[d], nCta[d], threadsAt[d]);
    return 0;
}
