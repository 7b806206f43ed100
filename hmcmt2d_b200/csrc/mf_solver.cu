// Host orchestration of the multifrontal solver (see mf_solver.cuh, mf_kernels.cuh).
#include "mf_solver.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "mf_kernels.cuh"

namespace hmcmt {
namespace mf {

namespace {
struct PerDeviceOnceMf {
    bool done[64] = {};
    bool need() {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};
constexpr size_t kMaxSmem = 227 * 1024;

template <int NW>
int launch_small(cudaStream_t st, const Tables& tb, const SmallDesc* list, int n, int nsys, size_t smem) {
    static PerDeviceOnceMf once;
    if (once.need()) HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_small_kernel<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    mf_small_kernel<NW><<<dim3(n, nsys), NW * 32, smem, st>>>(tb, list);
    return kOk;
}
int launch_stream(cudaStream_t st, const Tables& tb, const SmallDesc* list, int n, int nsys, size_t smem) {
    static PerDeviceOnceMf once;
    if (once.need()) HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_small_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    mf_small_stream_kernel<<<dim3(n, nsys), 16 * 32, smem, st>>>(tb, list);
    return kOk;
}
}  // namespace

template <typename Tp>
int Solver::upload(const std::vector<Tp>& h, Tp** d) {
    *d = nullptr;
    const size_t n = std::max<size_t>(h.size(), 1);
    if (cudaMalloc(d, n * sizeof(Tp)) != cudaSuccess) return kErrAlloc;
    owned.push_back(*d);
    bytes += n * sizeof(Tp);
    if (!h.empty() && cudaMemcpy(*d, h.data(), h.size() * sizeof(Tp), cudaMemcpyHostToDevice) != cudaSuccess) return kErrCuda;
    return kOk;
}

int Solver::upload_solve_descs(const std::vector<int>& fr, const SolveDesc** d) {
    std::vector<SolveDesc> v;
    v.reserve(fr.size());
    for (int k : fr) {
        const Front& F = S.fronts[k];
        SolveDesc sd{};
        sd.sp = F.sp; sd.up = F.up; sd.s = F.s; sd.u = F.u; sd.cbp = F.cbp; sd.rowPtr = F.rowPtr; sd.updOff = (int)F.updOff;
        sd.nChild = F.nChild;
        sd.gOff = S.chunks[F.chunkPtr].gOff; sd.mOff = S.chunks[F.chunkPtr].mOff;
        for (int c = 0; c < std::min(F.nChild, kDescChildren); ++c) {
            const Front& C = S.fronts[S.children[F.childPtr + c]];
            sd.cRel[c] = C.rowPtr; sd.cUpd[c] = (int)C.updOff; sd.cU[c] = C.u;
        }
        for (int i = 0; i < std::min(F.u, kDescRows); ++i) sd.rows[i] = S.rows[F.rowPtr + i];
        v.push_back(sd);
    }
    SolveDesc* p = nullptr;
    int rc = upload(v, &p);
    *d = p;
    return rc;
}

Solver* Solver::create(Symbolic&& S, int nsys, int maxRhs, int64_t valCount, int* rc) {
    Solver* s = new Solver();
    s->S = std::move(S);
    int r = s->build(nsys, maxRhs, valCount);
    if (rc) *rc = r;
    if (r != kOk) { delete s; return nullptr; }
    return s;
}

Solver::~Solver() {
    if (d_prof) {
        unsigned long long h[48] = {};
        cudaDeviceSynchronize();
        cudaMemcpy(h, d_prof, sizeof(h), cudaMemcpyDeviceToHost);
        for (int c = 0; c < 4; ++c) {
            const unsigned long long* q = h + 8 * c;
            if (q[6])
                fprintf(stderr, "[hmcmt_b200] mf_small_kernel<%d> cycles per front (%llu fronts, %.2f pivot blocks each): zero %.0f  orig %.0f  "
                        "children %.0f  mirror %.0f  sweep %.0f  output %.0f\n", 2 << c, q[6], (double)q[7] / q[6], (double)q[0] / q[6],
                        (double)q[1] / q[6], (double)q[2] / q[6], (double)q[3] / q[6], (double)q[4] / q[6], (double)q[5] / q[6]);
            const unsigned long long* w = h + 32 + 4 * c;
            if (q[7])
                fprintf(stderr, "[hmcmt_b200]     factorisation of the front, cycles per pivot block: 8x8 inversions %.0f  rest of the pivot-block sweep %.0f  M' = F21 (-G) %.0f  U += M' F21^T %.0f\n",
                        (double)w[0] / q[7], (double)w[1] / q[7], (double)w[2] / q[7], (double)w[3] / q[7]);
        }
    }
    for (void* p : owned) cudaFree(p);
}

int Solver::build(int nsys_, int maxRhs_, int64_t valCount_) {
    nsys = nsys_; maxRhs = std::max(1, maxRhs_); valCount = valCount_;
    int rc;
#define MF_TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    MF_TRY(upload(S.fronts, &d_fronts));
    MF_TRY(upload(S.rows, &d_rows));
    MF_TRY(upload(S.rel, &d_rel));
    MF_TRY(upload(S.children, &d_children));
    MF_TRY(upload(S.orig, &d_orig));
    MF_TRY(upload(S.chunks, &d_chunks));
    MF_TRY(upload(S.pos2orig, &d_pos2orig));
    auto dalloc = [&](void** p, size_t nbytes) {
        *p = nullptr;
        if (nbytes == 0) nbytes = 16;
        if (cudaMalloc(p, nbytes) != cudaSuccess) return (int)kErrAlloc;
        owned.push_back(*p);
        bytes += nbytes;
        return (int)kOk;
    };
    MF_TRY(dalloc((void**)&d_fac, (size_t)nsys * S.factorDoubles * sizeof(double)));
    for (int p = 0; p < 2; ++p) MF_TRY(dalloc((void**)&d_arena[p], (size_t)nsys * S.arenaDoubles[p] * sizeof(double)));
    MF_TRY(dalloc((void**)&d_vals, (size_t)nsys * valCount * sizeof(cplx)));
    MF_TRY(dalloc((void**)&d_v, (size_t)nsys * maxRhs * S.Np * sizeof(cplx)));
    MF_TRY(dalloc((void**)&d_upd, (size_t)nsys * maxRhs * S.updEntries * sizeof(cplx)));
    if (const char* e = std::getenv("HMCMT_MF_PROF"); e && std::atoi(e)) {
        MF_TRY(dalloc((void**)&d_prof, 48 * sizeof(unsigned long long)));
        cudaMemset(d_prof, 0, 48 * sizeof(unsigned long long));
    }

    // launch schedule
    std::vector<int> invMapsHost;
    const SchedKnobs knobs = SchedKnobs::from_env();
    sched.assign(S.maxDepth + 1, DepthSchedule());
    for (int d = 0; d <= S.maxDepth; ++d) {
        DepthSchedule& D = sched[d];
        const std::vector<int>& sm = S.byDepthSmall[d];
        const std::vector<int>& bg = S.byDepthBig[d];
        int* p = nullptr;
        D.nSmall = (int)sm.size();
        if (D.nSmall) {
            int mx = 0;
            for (int k : sm) mx = std::max(mx, S.fronts[k].fp());
            D.smallStream = mf_small_stream(S, sm);
            D.smallWarps = D.smallStream ? 16 : mf_small_warps(mx, knobs);
            D.smallSmem = 0;
            std::vector<SmallDesc> descs;
            for (int k : sm) {
                const Front& F = S.fronts[k];
                const int nb = F.fp() / 8, npb = F.sp / 8, rt = mf_rel_total(S, k);
                D.smallSmem = std::max(D.smallSmem, D.smallStream ? mf_stream_front_smem_bytes(nb, npb, rt, F.nChild)
                                                    : D.smallWarps >= 8 ? mf_mid_front_smem_bytes(nb, npb, rt, F.nChild)
                                                                        : mf_front_smem_bytes(nb, npb, rt));
                SmallDesc sd{};
                sd.sp = F.sp; sd.up = F.up; sd.s = F.s; sd.nChild = F.nChild; sd.nOrig = F.nOrig; sd.origPtr = F.origPtr;
                sd.par = F.depth & 1; sd.front = k;
                sd.gOff = S.chunks[F.chunkPtr].gOff; sd.mOff = S.chunks[F.chunkPtr].mOff; sd.uOff = F.frontOff;
                for (int c = 0; c < std::min(F.nChild, kDescChildren); ++c) {
                    const Front& C = S.fronts[S.children[F.childPtr + c]];
                    sd.cOff[c] = C.frontOff; sd.cLd[c] = C.ldU(); sd.cFirst[c] = C.offU(); sd.cU[c] = C.u; sd.cRel[c] = C.rowPtr;
                    int piv = 0;
                    while (piv < C.u && S.rel[C.rowPtr + piv] < F.sp) ++piv;
                    if (piv > 255) return kErrArg;
                    sd.cPiv[c] = (unsigned char)piv;
                }
                descs.push_back(sd);
            }
            SmallDesc* pd = nullptr;
            if (D.smallSmem > kMaxSmem) return kErrArg;
            MF_TRY(upload(descs, &pd));
            D.smallDescs = pd;
        }
        D.nBig = (int)bg.size();
        D.bigBytes = (size_t)S.bigDoublesAtDepth[d] * sizeof(double);
        // solves: one warp per front up to kSolveWarpMaxFp rows, one CTA per front above
        std::vector<int> sw, sc(bg);
        for (int k : sm) (mf_solve_by_warp(S.fronts[k]) ? sw : sc).push_back(k);
        D.nSolveWarp = (int)sw.size();
        D.nSolveCta = (int)sc.size();
        if (D.nSolveWarp) MF_TRY(upload_solve_descs(sw, &D.solveWarpList));
        if (D.nSolveCta) { MF_TRY(upload(sc, &p)); D.solveCtaList = p; }
        {
            int mxc = 0;
            for (int k : sc) mxc = std::max(mxc, S.fronts[k].fp());
            D.solveCtaThreads = mf_solve_cta_threads(mxc, knobs);
        }
        if (!D.nBig) continue;
        MF_TRY(upload(bg, &p));
        D.bigList = p;
        std::vector<int2> op;
        int maxChunk = 0;
        for (int k : bg) {
            const Front& F = S.fronts[k];
            for (int e = 0; e < F.nOrig; ++e) op.push_back(make_int2(k, F.origPtr + e));
            maxChunk = std::max(maxChunk, F.nChunk);
        }
        int2* p2 = nullptr;
        D.nOrigPairs = (int)op.size();
        if (D.nOrigPairs) { MF_TRY(upload(op, &p2)); D.origPairs = p2; }
        {
            std::vector<AsmTile> tiles;
            for (int k : bg) {
                const Front& F = S.fronts[k];
                const int fp = F.fp(), nt = (fp + 63) / 64;
                const int invPtr = (int)invMapsHost.size();
                for (int c = 0; c < F.nChild; ++c) {
                    const Front& C = S.fronts[S.children[F.childPtr + c]];
                    std::vector<int> inv(fp, -1);
                    for (int i = 0; i < C.u; ++i) inv[S.rel[C.rowPtr + i]] = i;
                    invMapsHost.insert(invMapsHost.end(), inv.begin(), inv.end());
                }
                for (int bi = 0; bi < nt; ++bi)
                    for (int bj = 0; bj <= bi; ++bj) tiles.push_back(AsmTile{k, bi, bj, invPtr});
            }
            AsmTile* pt = nullptr;
            MF_TRY(upload(tiles, &pt));
            D.asmTiles = pt;
            D.nAsmTiles = (int)tiles.size();
        }
        for (int c = 0; c < maxChunk; ++c) {
            DepthSchedule::ChunkStep cs;
            std::vector<int> inv;
            std::vector<GemmJob> jobs;
            std::vector<GemmTile> pt, st;
            int maxSc = 0;
            for (int k : bg) {
                const Front& F = S.fronts[k];
                if (F.nChunk <= c) continue;
                const Chunk& ch = S.chunks[F.chunkPtr + c];
                const int sc = ch.p1 - ch.p0, fp = F.fp(), mr = fp - ch.p1, par = F.depth & 1;
                inv.push_back(k);
                maxSc = std::max(maxSc, sc);
                if (mr <= 0) continue;
                GemmJob jp{};      // M = F21 G
                jp.aOff = F.frontOff; jp.aSp = par; jp.ldA = fp; jp.rA = ch.p1; jp.kA = ch.p0;
                jp.bOff = ch.gOff; jp.bSp = 2; jp.ldB = sc; jp.rB = 0; jp.kB = 0;
                jp.cOff = ch.mOff; jp.cSp = 2; jp.ldC = mr; jp.rC = 0; jp.cC = 0;
                jp.m = mr; jp.n = sc; jp.K = sc; jp.lower = 0; jp.beta = 0; jp.alpha = 1.0;
                const int jpi = (int)jobs.size();
                jobs.push_back(jp);
                for (int bi = 0; bi < (mr + 63) / 64; ++bi)
                    for (int bj = 0; bj < (sc + 63) / 64; ++bj) pt.push_back(GemmTile{jpi, bi, bj});
                GemmJob js{};      // F22 -= M F21^T (lower tiles)
                js.aOff = ch.mOff; js.aSp = 2; js.ldA = mr; js.rA = 0; js.kA = 0;
                js.bOff = F.frontOff; js.bSp = par; js.ldB = fp; js.rB = ch.p1; js.kB = ch.p0;
                js.cOff = F.frontOff; js.cSp = par; js.ldC = fp; js.rC = ch.p1; js.cC = ch.p1;
                js.m = mr; js.n = mr; js.K = sc; js.lower = 1; js.beta = 1; js.alpha = -1.0;
                const int jsi = (int)jobs.size();
                jobs.push_back(js);
                for (int bi = 0; bi < (mr + 63) / 64; ++bi)
                    for (int bj = 0; bj <= bi; ++bj) st.push_back(GemmTile{jsi, bi, bj});
            }
            MF_TRY(upload(inv, &p));
            cs.invList = p; cs.nInv = (int)inv.size();
            cs.invSmem = mf_front_smem_bytes(maxSc / 8, maxSc / 8);
            GemmJob* pj = nullptr;
            GemmTile* ptile = nullptr;
            MF_TRY(upload(jobs, &pj));
            cs.jobs = pj;
            MF_TRY(upload(pt, &ptile));
            cs.panelTiles = ptile; cs.nPanelTiles = (int)pt.size();
            MF_TRY(upload(st, &ptile));
            cs.schurTiles = ptile; cs.nSchurTiles = (int)st.size();
            D.chunkSteps.push_back(cs);
        }
    }
    MF_TRY(upload(invMapsHost, &d_invMaps));
    solveSmem = (size_t)(2 * S.maxFp + 16) * sizeof(cplx);
    if (solveSmem > kMaxSmem) return kErrArg;
    {
        int mx = 0;
        for (const Front& F : S.fronts) if (!mf_solve_by_warp(F)) mx = std::max(mx, F.fp() + F.sp);
        pairSmem = (size_t)2 * mx * sizeof(cplx);      // (checked by backward_pair, the only user)
    }
#undef MF_TRY
    return kOk;
}

int Solver::set_mt_values(cudaStream_t st, int N, const MtValSys* dSys, int sys0, int n) {
    if (valCount < 3 * (int64_t)N) return kErrArg;
    if (n < 0) n = nsys - sys0;
    if (sys0 < 0 || n < 1 || sys0 + n > nsys) return kErrArg;
    mf_mt_vals_kernel<<<dim3((3 * N + 255) / 256, n), 256, 0, st>>>(N, dSys + sys0, d_vals + (size_t)sys0 * valCount, valCount);
    HMCMT_CUDA_TRY(cudaGetLastError());
    return kOk;
}

int Solver::factor(cudaStream_t st, int* dStatus, int64_t* nLaunches, int sys0, int n) {
    if (n < 0) n = this->nsys - sys0;
    if (sys0 < 0 || n < 1 || sys0 + n > this->nsys) return kErrArg;
    const int nsys = n;      // systems of this call: the kernels index them 0..n-1 from the offset bases below
    Tables tb{};
    tb.fronts = d_fronts; tb.rows = d_rows; tb.rel = d_rel; tb.children = d_children; tb.orig = d_orig; tb.chunks = d_chunks;
    tb.pos2orig = d_pos2orig; tb.fac = d_fac + (size_t)sys0 * S.factorDoubles;
    tb.arena[0] = d_arena[0] + (size_t)sys0 * S.arenaDoubles[0]; tb.arena[1] = d_arena[1] + (size_t)sys0 * S.arenaDoubles[1];
    tb.facStride = S.factorDoubles; tb.arenaStride[0] = S.arenaDoubles[0]; tb.arenaStride[1] = S.arenaDoubles[1];
    tb.vals = d_vals + (size_t)sys0 * valCount; tb.valStride = valCount; tb.status = dStatus ? dStatus + sys0 : nullptr; tb.prof = d_prof;
    static PerDeviceOnceMf once;
    if (once.need()) {
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmemBytes));
    }
    int64_t nl = 0;
    for (int d = S.maxDepth; d >= 0; --d) {
        const DepthSchedule& D = sched[d];
        if (D.nSmall) {
            int rc = kOk;
            if (D.smallStream) rc = launch_stream(st, tb, D.smallDescs, D.nSmall, nsys, D.smallSmem);
            else if (D.smallWarps == 1) rc = launch_small<1>(st, tb, D.smallDescs, D.nSmall, nsys, D.smallSmem);
            else if (D.smallWarps == 2) rc = launch_small<2>(st, tb, D.smallDescs, D.nSmall, nsys, D.smallSmem);
            else if (D.smallWarps == 4) rc = launch_small<4>(st, tb, D.smallDescs, D.nSmall, nsys, D.smallSmem);
            else if (D.smallWarps == 8) rc = launch_small<8>(st, tb, D.smallDescs, D.nSmall, nsys, D.smallSmem);
            else rc = launch_small<16>(st, tb, D.smallDescs, D.nSmall, nsys, D.smallSmem);
            if (rc) return rc;
            ++nl;
        }
        if (!D.nBig) continue;
        if (D.nAsmTiles) {
            mf_asm_gather_kernel<<<dim3(D.nAsmTiles, nsys), 256, 0, st>>>(tb, (const AsmTile*)D.asmTiles, d_invMaps);
            ++nl;
        }
        if (D.nOrigPairs) {
            mf_asm_orig_kernel<<<dim3((D.nOrigPairs + 255) / 256, nsys), 256, 0, st>>>(tb, D.origPairs, D.nOrigPairs);
            ++nl;
        }
        for (size_t c = 0; c < D.chunkSteps.size(); ++c) {
            const DepthSchedule::ChunkStep& cs = D.chunkSteps[c];
            if (!cs.nInv) continue;
            mf_inv_kernel<<<dim3(cs.nInv, nsys), kInvWarps * 32, cs.invSmem, st>>>(tb, cs.invList, (int)c);
            ++nl;
            if (cs.nPanelTiles) {
                mf_gemm_kernel<<<dim3(cs.nPanelTiles, nsys), kGemmThreads, kGemmSmemBytes, st>>>(
                    tb, (const GemmJob*)cs.jobs, (const GemmTile*)cs.panelTiles);
                ++nl;
            }
            if (cs.nSchurTiles) {
                mf_gemm_kernel<<<dim3(cs.nSchurTiles, nsys), kGemmThreads, kGemmSmemBytes, st>>>(
                    tb, (const GemmJob*)cs.jobs, (const GemmTile*)cs.schurTiles);
                ++nl;
            }
        }
    }
    HMCMT_CUDA_TRY(cudaGetLastError());
    if (nLaunches) *nLaunches += nl;
    return kOk;
}

int Solver::add_rhs_pattern(const std::vector<unsigned char>& nz) {
    if ((int)nz.size() != S.N) return kErrArg;
    std::vector<char> active(S.K, 0);
    for (int k = 0; k < S.K; ++k) {          // elimination order: children before parents
        const Front& F = S.fronts[k];
        for (int i = 0; i < F.s && !active[k]; ++i) {
            const int o = S.pos2orig[F.cbp + i];
            if (o >= 0 && nz[o]) active[k] = 1;
        }
        if (active[k] && F.parent >= 0) active[F.parent] = 1;
    }
    PatternLists L;
    int rc;
#define MF_TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    for (int d = 0; d <= S.maxDepth; ++d) {
        std::vector<int> sw, sc, pw, pc;      // active set; all fronts, inactive first (backward_pair)
        for (int k : S.byDepthBig[d]) if (active[k]) sc.push_back(k);
        for (int k : S.byDepthSmall[d]) if (active[k]) (mf_solve_by_warp(S.fronts[k]) ? sw : sc).push_back(k);
        for (int k : S.byDepthBig[d]) if (!active[k]) pc.push_back(k);
        for (int k : S.byDepthSmall[d]) if (!active[k]) (mf_solve_by_warp(S.fronts[k]) ? pw : pc).push_back(k);
        L.nPairWarpBoth.push_back((int)pw.size());
        L.nPairCtaBoth.push_back((int)pc.size());
        pw.insert(pw.end(), sw.begin(), sw.end());
        pc.insert(pc.end(), sc.begin(), sc.end());
        const SolveDesc* pd = nullptr;
        if (!sw.empty()) MF_TRY(upload_solve_descs(sw, &pd));
        L.warpList.push_back(pd);
        L.nWarp.push_back((int)sw.size());
        int* p = nullptr;
        if (!sc.empty()) MF_TRY(upload(sc, &p));
        L.ctaList.push_back(sc.empty() ? nullptr : p);
        L.nCta.push_back((int)sc.size());
        L.nFronts += (int)(sw.size() + sc.size());
        pd = nullptr;
        if (!pw.empty()) MF_TRY(upload_solve_descs(pw, &pd));
        L.pairWarpList.push_back(pd);
        p = nullptr;
        if (!pc.empty()) MF_TRY(upload(pc, &p));
        L.pairCtaList.push_back(p);
    }
#undef MF_TRY
    patterns.push_back(std::move(L));
    return (int)patterns.size();
}

int Solver::fwd_fronts(int pattern) const {
    return pattern >= 1 && pattern <= (int)patterns.size() ? patterns[pattern - 1].nFronts : S.K;
}

Tables Solver::tables(int sys0) const {
    Tables tb{};
    tb.fronts = d_fronts; tb.rows = d_rows; tb.rel = d_rel; tb.children = d_children; tb.orig = d_orig; tb.chunks = d_chunks;
    tb.pos2orig = d_pos2orig; tb.fac = d_fac + (size_t)sys0 * S.factorDoubles;
    tb.arena[0] = d_arena[0] + (size_t)sys0 * S.arenaDoubles[0]; tb.arena[1] = d_arena[1] + (size_t)sys0 * S.arenaDoubles[1];
    tb.facStride = S.factorDoubles; tb.arenaStride[0] = S.arenaDoubles[0]; tb.arenaStride[1] = S.arenaDoubles[1];
    tb.vals = d_vals; tb.valStride = valCount; tb.status = nullptr; tb.prof = nullptr;
    return tb;
}

// vectors (sys0 + s, r) of a call: right-hand side / solution at B / X + (s*nrhs + r)*ld.  Workspace: from slot `slot` of
// system sys0 on, consecutive vectors of the call are one slot apart when nrhs > 1 (all calls that pass nrhs > 1 cover their
// systems' slots 0 .. nrhs-1) and one system apart when nrhs == 1 (slot `slot` of every system).
SolveArgs Solver::solve_args(const cplx* B, int64_t ldb, cplx* X, int64_t ldx, int sys0, int nrhs, int slot) const {
    const size_t vec0 = (size_t)sys0 * nrhs, ws0 = (size_t)sys0 * maxRhs + slot;
    const int64_t per = nrhs == 1 ? maxRhs : 1;
    return SolveArgs{B ? B + vec0 * ldb : nullptr, X ? X + vec0 * ldx : nullptr, ldb, ldx, d_v + ws0 * S.Np, d_upd + ws0 * S.updEntries,
                     per * S.Np, per * S.updEntries, nrhs};
}

int Solver::set_solve_attributes() {
    static PerDeviceOnceMf once;
    if (once.need()) {
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(mf_bwd_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    }
    return kOk;
}

// zero the workspace vectors of a call (sa: solve_args): the fronts a pruned forward elimination does not visit hold zero pivot
// parts and update vectors
int Solver::clear_ws(cudaStream_t st, const SolveArgs& sa, int nvec) {
    const struct { cplx* p; int64_t len, stride; } ws[2] = {{sa.v, (int64_t)S.Np, sa.vStride}, {sa.upd, S.updEntries, sa.uStride}};
    for (const auto& w : ws) {
        if (w.stride == w.len) HMCMT_CUDA_TRY(cudaMemsetAsync(w.p, 0, (size_t)nvec * w.len * sizeof(cplx), st));
        else HMCMT_CUDA_TRY(cudaMemset2DAsync(w.p, (size_t)w.stride * sizeof(cplx), 0, (size_t)w.len * sizeof(cplx), nvec, st));
    }
    return kOk;
}

int Solver::fwd_sweep(cudaStream_t st, const Tables& tb, const SolveArgs& sa, int nvec, int pattern, int64_t& nl) {
    const PatternLists* P = pattern ? &patterns[pattern - 1] : nullptr;
    for (int d = S.maxDepth; d >= 0; --d) {
        const DepthSchedule& D = sched[d];
        const int nW = P ? P->nWarp[d] : D.nSolveWarp, nC = P ? P->nCta[d] : D.nSolveCta;
        const SolveDesc* wl = P ? P->warpList[d] : D.solveWarpList;
        const int* cl = P ? P->ctaList[d] : D.solveCtaList;
        if (nW) {
            mf_fwd_warp_kernel<<<dim3((nW + kSolveWarpsPerCta - 1) / kSolveWarpsPerCta, nvec), kSolveWarpsPerCta * 32, 0, st>>>(tb, sa, wl, nW);
            ++nl;
        }
        if (nC) {
            mf_fwd_kernel<<<dim3(nC, nvec), D.solveCtaThreads, solveSmem, st>>>(tb, sa, cl);
            ++nl;
        }
    }
    return kOk;
}

int Solver::solve(cudaStream_t st, int nrhs, const cplx* B, int64_t ldb, cplx* X, int64_t ldx, int64_t* nLaunches, int sys0, int n,
                  int pattern) {
    if (nrhs < 1 || nrhs > maxRhs || pattern < 0 || pattern > (int)patterns.size()) return kErrArg;
    if (n < 0) n = this->nsys - sys0;
    if (sys0 < 0 || n < 1 || sys0 + n > this->nsys) return kErrArg;
    int rc = set_solve_attributes();
    if (rc) return rc;
    const Tables tb = tables(sys0);
    const SolveArgs sa = solve_args(B, ldb, X, ldx, sys0, nrhs, 0);
    const int nvec = n * nrhs;
    int64_t nl = 0;
    // fronts outside the pattern are not visited: their pivot parts and update vectors are zero
    if (pattern && (rc = clear_ws(st, sa, nvec))) return rc;
    fwd_sweep(st, tb, sa, nvec, pattern, nl);
    for (int d = 0; d <= S.maxDepth; ++d) {
        const DepthSchedule& D = sched[d];
        if (D.nSolveWarp) {
            mf_bwd_warp_kernel<<<dim3((D.nSolveWarp + kSolveWarpsPerCta - 1) / kSolveWarpsPerCta, nvec), kSolveWarpsPerCta * 32, 0, st>>>(
                tb, sa, D.solveWarpList, D.nSolveWarp);
            ++nl;
        }
        if (D.nSolveCta) {
            mf_bwd_kernel<<<dim3(D.nSolveCta, nvec), D.solveCtaThreads, solveSmem, st>>>(tb, sa, D.solveCtaList);
            ++nl;
        }
    }
    HMCMT_CUDA_TRY(cudaGetLastError());
    if (nLaunches) *nLaunches += nl;
    return kOk;
}

int Solver::forward_slot(cudaStream_t st, int slot, const cplx* B, int64_t ldb, int64_t* nLaunches, int sys0, int n, int pattern) {
    if (slot < 0 || slot >= maxRhs || pattern < 0 || pattern > (int)patterns.size()) return kErrArg;
    if (n < 0) n = this->nsys - sys0;
    if (sys0 < 0 || n < 1 || sys0 + n > this->nsys) return kErrArg;
    int rc = set_solve_attributes();
    if (rc) return rc;
    const SolveArgs sa = solve_args(B, ldb, nullptr, 0, sys0, 1, slot);
    int64_t nl = 0;
    if (pattern && (rc = clear_ws(st, sa, n))) return rc;
    fwd_sweep(st, tables(sys0), sa, n, pattern, nl);
    HMCMT_CUDA_TRY(cudaGetLastError());
    if (nLaunches) *nLaunches += nl;
    return kOk;
}

int Solver::backward_slot(cudaStream_t st, int slot, cplx* X, int64_t ldx, int64_t* nLaunches, int sys0, int n, int pattern) {
    if (slot < 0 || slot >= maxRhs || pattern < 1 || pattern > (int)patterns.size()) return kErrArg;
    if (n < 0) n = this->nsys - sys0;
    if (sys0 < 0 || n < 1 || sys0 + n > this->nsys) return kErrArg;
    int rc = set_solve_attributes();
    if (rc) return rc;
    const Tables tb = tables(sys0);
    const SolveArgs sa = solve_args(nullptr, 0, X, ldx, sys0, 1, slot);
    const PatternLists& P = patterns[pattern - 1];
    int64_t nl = 0;
    for (int d = 0; d <= S.maxDepth; ++d) {
        if (const int nW = P.nWarp[d]) {
            mf_bwd_warp_kernel<<<dim3((nW + kSolveWarpsPerCta - 1) / kSolveWarpsPerCta, n), kSolveWarpsPerCta * 32, 0, st>>>(
                tb, sa, P.warpList[d], nW);
            ++nl;
        }
        if (const int nC = P.nCta[d]) {
            mf_bwd_kernel<<<dim3(nC, n), sched[d].solveCtaThreads, solveSmem, st>>>(tb, sa, P.ctaList[d]);
            ++nl;
        }
    }
    HMCMT_CUDA_TRY(cudaGetLastError());
    if (nLaunches) *nLaunches += nl;
    return kOk;
}

int Solver::backward_pair(cudaStream_t st, cplx* Xa, cplx* Xb, int64_t ldx, int64_t* nLaunches, int sys0, int n, int done) {
    if (maxRhs < 2 || done < 1 || done > (int)patterns.size() || pairSmem > kMaxSmem) return kErrArg;
    if (n < 0) n = this->nsys - sys0;
    if (sys0 < 0 || n < 1 || sys0 + n > this->nsys) return kErrArg;
    int rc = set_solve_attributes();
    if (rc) return rc;
    const Tables tb = tables(sys0);
    const SolveArgs sa = solve_args(nullptr, 0, Xa, ldx, sys0, 1, 0), sb = solve_args(nullptr, 0, Xb, ldx, sys0, 1, 1);
    const PatternLists& P = patterns[done - 1];
    int64_t nl = 0;
    for (int d = 0; d <= S.maxDepth; ++d) {
        const DepthSchedule& D = sched[d];
        if (D.nSolveWarp) {
            mf_bwd_pair_warp_kernel<<<dim3((D.nSolveWarp + kSolveWarpsPerCta - 1) / kSolveWarpsPerCta, n), kSolveWarpsPerCta * 32, 0, st>>>(
                tb, sa, sb, P.pairWarpList[d], D.nSolveWarp, P.nPairWarpBoth[d]);
            ++nl;
        }
        if (D.nSolveCta) {
            mf_bwd_pair_kernel<<<dim3(D.nSolveCta, n), D.solveCtaThreads, pairSmem, st>>>(tb, sa, sb, P.pairCtaList[d], P.nPairCtaBoth[d]);
            ++nl;
        }
    }
    HMCMT_CUDA_TRY(cudaGetLastError());
    if (nLaunches) *nLaunches += nl;
    return kOk;
}

}  // namespace mf
}  // namespace hmcmt
