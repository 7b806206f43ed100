// libhmcmt_b200.so — plan, step orchestration and the Level-2 C ABI (include/hmcmt_b200.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "../../include/hmcmt_b200.h"
#include "band_factor.cuh"
#include "band_solve.cuh"
#include "mf_solver.cuh"
#include "mt_kernels.cuh"

using namespace hmcmt;

namespace {

template <typename Tp>
struct DevBuf {
    Tp* p = nullptr;
    size_t n = 0;
    int alloc(size_t count) {
        n = count;
        if (count == 0) return kOk;
        cudaError_t e = cudaMalloc(&p, count * sizeof(Tp));
        if (e != cudaSuccess) { p = nullptr; return kErrAlloc; }
        return kOk;
    }
    int upload(const Tp* h, size_t count) {
        int rc = alloc(count);
        if (rc) return rc;
        if (count) HMCMT_CUDA_TRY(cudaMemcpy(p, h, count * sizeof(Tp), cudaMemcpyHostToDevice));
        return kOk;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

}  // namespace

struct hmcmt_plan {
    // sizes
    int ny = 0, nz = 0, nFreq = 0, nRx = 0, nData = 0, nAC = 0, nChains = 1, nModes = 0, nComp = 0;
    int modeList[2] = {0, 1};
    int nSysPerChain = 0, nSys = 0, nFull = 0;      // nFull = nFreq*nRx*nComp per chain
    bool tipper = false;                            // an impedance plan with a TZY component (compMode 2)
    CompMap cm{};                                   // component <-> system of a tipper plan (k_rx_adjoint<false, true>)
    int T = 0, S = 0, b = 0, device = 0, conStaged = 0, numSMs = 148;
    BandDom dom{};
    int steps0 = 0, steps1 = 0;                     // macro-steps of half 0 (own lines + separator) / half 1 (0 when not split)
    double beta = 1.0, lo = 0.0, hi = 0.0;
    MeshDev M{};
    SysMap sm{};
    RxDev rx{};
    cudaStream_t stream = nullptr, side = nullptr;      // side: 1-D sensitivity scalars overlap the factorisation
    cudaEvent_t evFork = nullptr, evJoin = nullptr;
    cudaEvent_t evA = nullptr, evB = nullptr, evPre = nullptr, evRhs = nullptr;
    cudaGraphExec_t graphExec = nullptr;                // the gradient evaluation, captured on its second call (compute_step_graph)
    int graphState = 0;                                 // 0: not run yet, 1: warmed up, 2: graph ready, -1: disabled
    int64_t graphLaunches = 0;
    std::vector<cudaStream_t> groupStreams;             // >= 2: the systems of a step run as groups on these streams (compute_step_grouped)
    std::vector<cudaEvent_t> groupDone;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> factorEvents;
    std::vector<cudaEvent_t> factorMid;                 // between the factorisation and the forward solve of a timed evaluation
    size_t factorEventsUsed = 0;
    int64_t launches = 0, factorLaunches = 0;
    bool haveForward = false, haveSens = false, sigmaDirect = false, useMf = false, timeFactor = false;
    int respKind = 0;                               // 0 impedance, 1 apparent resistivity / phase (forward only)
    int dataKind = 0;                               // data of the plan: 0 impedance, 1 apparent resistivity / phase (rows real)
    // host copies
    std::vector<double> h_yLen, h_zLen, h_freqs;
    std::vector<int> h_packed2full;      // [nData] full index (without chain) of each packed datum; rho / phase plans: index into
                                         // the real view [nFull][2] (rho, phase) of the full arrays
    // device buffers
    DevBuf<double> yLen, zLen, zNode, freqs, fdy1, fdy2, wL, wR, twL, twR, bg, wmVal, wd, m, p, mref, sigma, meanSig, planes;
    DevBuf<double> wdPha;                           // phase weights of a rho / phase plan (wd holds the rho weights)
    DevBuf<double> driftPart;                       // block maxima of the drift (k_drift_max)
    DevBuf<double> xbuf, Gpart, phiPart, phi, gsig, gdata, gtotal, energies, panels, curM, curP, chainScal, zmom;
    DevBuf<int> fid, iL, iR, tjL, tjR, cell2act, act2cell, wmPtr, wmIdx, status, driftFlag, packed2full, full2packed, Lsteps;
    DevBuf<cplx> obs, bc, bcs, rhs, x, F, lam, Lam, srows, qrow, scratch, predFull, ainvz, zadj, vin, predPacked, wexp, conCols, respFull;
    // tangent mode (hmcmt_jvec / hmcmt_gn_hessvec), allocated on first use: dbc [nSys][nb], the full-layout tangent jvFull
    // [nChains][nFull], the conductivity direction dsigA [nChains][nAC] and the Gauss-Newton product's [v | 0 | gsig | gdata |
    // gtotal] (gnBuf, 5 [nChains][nAC]: k_reduce_grad writes there, so the plan's own gradient stays)
    DevBuf<cplx> dbc, jvFull;
    DevBuf<double> dsigA, gnBuf;
    // projected Gauss-Newton-CG (hmcmt_gauss_newton), allocated on first use: gnVec 6 [nChains][nAC] = [m_k | g_k | delta | r | p |
    // q], the active set gnAct [nChains][nAC], the p^T q block partials gnPart, the per-chain scalars / flags gnS / gnI (GnScalar /
    // GnFlag of mt_kernels.cuh) and gnE, k_energies' output for the trial points
    DevBuf<double> gnVec, gnPart, gnS, gnE;
    DevBuf<int> gnAct, gnI;
    DevBuf<BandSys> sysDesc;
    DevBuf<SolveJob> jobs, fwdJobs;                 // fwdJobs: back-substitution sweeps of the fused forward systems (split systems)
    // wide meshes (half-bandwidth > 104): nested-dissection multifrontal solver (mf_solver.cuh) instead of the band kernels
    mf::Solver* mfs = nullptr;
    DevBuf<mf::MtValSys> mfSys;
    int patRhs = 0, patAdj = 0;                     // sparsity patterns of the forward / adjoint right-hand sides (Solver::add_rhs_pattern)
    int patRx = 0;                                  // the receiver rows zid, zid + 1: its active set is the receiver path (gradient_range)
    // non-diagonal mass matrix M = Wm (setMassMatrix(invParam) HMCSampler.jl:478-489): invM p through a multifrontal
    // factorisation of Wm, sqrtM z through the banded Cholesky factor of Wm (natural ordering, as the reference's dense one)
    bool massOn = false;
    mf::Solver* massSolver = nullptr;
    DevBuf<double> gradK, Lband;
    DevBuf<cplx> massBuf;
    DevBuf<int> massStatus;
    int massBw = 0;
    // frequency-sharded steps: NCCL communicator over the ranks that share this chain (hmcmt_nccl_init)
    ncclComm_t comm = nullptr;
    int commWorld = 1;
    // pinned staging for the host-buffer entry points
    double* pin = nullptr;
    size_t pinBytes = 0;
};

namespace {

constexpr int kDefaultGroups = 3;              // groups of systems per evaluation on the multifrontal path (HMCMT_GROUPS)
constexpr size_t kMaxFactorEvents = 4096;      // CUDA-event pairs kept for hmcmt_kernel_time (opt-in, bounded)

#define LAUNCH_CHECK(pl)                                          \
    do {                                                          \
        ++(pl)->launches;                                         \
        cudaError_t _e = cudaGetLastError();                      \
        if (_e != cudaSuccess) {                                  \
            fprintf(stderr, "[hmcmt_b200] launch failed at %s:%d: %s\n", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return kErrCuda;                                      \
        }                                                         \
    } while (0)

// cudaFuncSetAttribute is per device: a process may hold plans on several GPUs (api.parallelHMCSampler without torchrun),
// so the "already configured" flags are kept per device.
struct PerDeviceOnce {
    bool done[64] = {};
    bool need() {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
        if (done[dev]) return false;
        done[dev] = true;
        return true;
    }
};

// A split system takes three launches in stream order: own lines of both halves, separator, back-substitution of both halves.
template <int T>
int launch_factor_T(cudaStream_t st, const BandSys* sys, int nsys, const BandDom& dom, const SolveJob* fwdJobs) {
    static PerDeviceOnce once;
    size_t smem = sizeof(FactorSmem<T>), smemSolve = sizeof(SolveSmem<T>);
    if (once.need()) {
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(band_factor_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(band_solve_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemSolve));
    }
    constexpr int NT = FactorCfg<T>::NTHREADS;
    if (!dom.split) {
        band_factor_kernel<T><<<nsys, NT, smem, st>>>(sys, dom, FM_FULL);
    } else {
        band_factor_kernel<T><<<2 * nsys, NT, smem, st>>>(sys, dom, FM_OWN);
        band_factor_kernel<T><<<nsys, NT, smem, st>>>(sys, dom, FM_SEP);
        // back-substitution of the two halves: the pipelined sweep of band_solve.cuh, z read from the factor stream
        if (fwdJobs) band_solve_kernel<T><<<2 * nsys, kSolveThreads, smemSolve, st>>>(fwdJobs, dom, SM_BACKZ_OWN);
        else band_factor_kernel<T><<<2 * nsys, NT, smem, st>>>(sys, dom, FM_BACK);
    }
    HMCMT_CUDA_TRY(cudaGetLastError());
    return kOk;
}
template <int T>
int launch_solve_T(cudaStream_t st, const SolveJob* jobs, int njobs, const BandDom& dom) {
    static PerDeviceOnce once;
    size_t smem = sizeof(SolveSmem<T>);
    if (once.need()) {
        HMCMT_CUDA_TRY(cudaFuncSetAttribute(band_solve_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (!dom.split) {
        band_solve_kernel<T><<<njobs, kSolveThreads, smem, st>>>(jobs, dom, FM_FULL);
    } else {
        band_solve_kernel<T><<<2 * njobs, kSolveThreads, smem, st>>>(jobs, dom, FM_OWN);
        band_solve_kernel<T><<<njobs, kSolveThreads, smem, st>>>(jobs, dom, FM_SEP);
        band_solve_kernel<T><<<2 * njobs, kSolveThreads, smem, st>>>(jobs, dom, FM_BACK);
    }
    HMCMT_CUDA_TRY(cudaGetLastError());
    return kOk;
}

}  // namespace

namespace hmcmt {
// shared with mumps_shim.cu
int round_T(int b) {
    if (b > 8 * 14 - 8) return 0;                 // too wide for the register window: multifrontal solver (mf_solver.cuh)
    int T = band_T_for(b);
    if (T < 2) T = 2;
    if (T & 1) ++T;
    return T;
}
// fwdJobs: back-substitution jobs of the fused forward systems (split systems: the pipelined sweep of band_solve.cuh).
// nLaunches (optional) receives the number of kernels launched.
int launch_factor(cudaStream_t st, int T, const BandSys* sys, int nsys, const BandDom& dom, const SolveJob* fwdJobs, int* nLaunches) {
    if (nLaunches) *nLaunches = dom.split ? 3 : 1;
    switch (T) {
        case 2: return launch_factor_T<2>(st, sys, nsys, dom, fwdJobs);
        case 4: return launch_factor_T<4>(st, sys, nsys, dom, fwdJobs);
        case 6: return launch_factor_T<6>(st, sys, nsys, dom, fwdJobs);
        case 8: return launch_factor_T<8>(st, sys, nsys, dom, fwdJobs);
        case 10: return launch_factor_T<10>(st, sys, nsys, dom, fwdJobs);
        case 12: return launch_factor_T<12>(st, sys, nsys, dom, fwdJobs);
        case 14: return launch_factor_T<14>(st, sys, nsys, dom, fwdJobs);
        default: return kErrArg;
    }
}
int launch_solve(cudaStream_t st, int T, const SolveJob* jobs, int njobs, const BandDom& dom) {
    switch (T) {
        case 2: return launch_solve_T<2>(st, jobs, njobs, dom);
        case 4: return launch_solve_T<4>(st, jobs, njobs, dom);
        case 6: return launch_solve_T<6>(st, jobs, njobs, dom);
        case 8: return launch_solve_T<8>(st, jobs, njobs, dom);
        case 10: return launch_solve_T<10>(st, jobs, njobs, dom);
        case 12: return launch_solve_T<12>(st, jobs, njobs, dom);
        case 14: return launch_solve_T<14>(st, jobs, njobs, dom);
        default: return kErrArg;
    }
}
// multifrontal tuning knobs (leaf boxes of the nested dissection; largest front handled by the single-CTA kernel)
int mf_leaf_size() {
    const char* e = std::getenv("HMCMT_MF_LEAF");
    const int v = e ? std::atoi(e) : 16;
    return v < 1 ? 1 : v;
}
int mf_cross_size() {
    const char* e = std::getenv("HMCMT_MF_CROSS");
    const int v = e ? std::atoi(e) : 0;
    return v < 0 ? 0 : v;
}
int mf_push_size() {
    const char* e = std::getenv("HMCMT_MF_PUSH");
    const int v = e ? std::atoi(e) : 2;      // measured at cfg2: 0 -> 4.85, 1 -> 4.82, 2 -> 4.73, 7 -> 4.78 ms per step
    return v < 0 ? 0 : (v > 7 ? 7 : v);
}
int mf_small_front() {
    const char* e = std::getenv("HMCMT_MF_FSMALL");
    int v = e ? std::atoi(e) : 256;
    return v < 0 ? 0 : (v > 256 ? 256 : v);
}
}  // namespace hmcmt

namespace {

// linearInterp sensUtils.jl:133-161 (0-based)
void linear_interp(double point, const std::vector<double>& x, int& iL, int& iR, double& wL, double& wR) {
    int n = (int)x.size(), ind = 0;
    double best = std::fabs(point - x[0]);
    for (int i = 1; i < n; ++i) {
        double d = std::fabs(point - x[i]);
        if (d < best) { best = d; ind = i; }
    }
    if (point - x[ind] > 0) { iL = ind; iR = ind + 1; } else { iL = ind - 1; iR = ind; }
    iL = std::max(std::min(iL, n - 1), 0);
    iR = std::max(std::min(iR, n - 1), 0);
    if (iL == iR) { wL = 0.5; wR = 0.5; return; }
    double len = x[iR] - x[iL];
    wL = 1 - (point - x[iL]) / len;
    wR = 1 - (x[iR] - point) / len;
}

// ---- kernels local to the HMC driver ----
__global__ void k_pack_pred(int nData, int nFull, const int* __restrict__ packed2full, const cplx* __restrict__ predFull,
                            cplx* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (i < nData) out[(size_t)ch * nData + i] = predFull[(size_t)ch * nFull + packed2full[i]];
}
// rho / phase plans: the packed real data from the (rho_a, phase) pairs of respFull, viewed as [nChains][2 nFull] doubles
__global__ void k_pack_pred_real(int nData, int nFull, const int* __restrict__ packed2full, const double* __restrict__ respFull,
                                 double* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (i < nData) out[(size_t)ch * nData + i] = respFull[(size_t)ch * 2 * nFull + packed2full[i]];
}
__global__ void k_kick_masked(int nAC, double dt, int kstep, const int* __restrict__ L, const double* __restrict__ grad,
                              double* __restrict__ p) {
    int ch = blockIdx.y, a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= nAC) return;
    int Lc = L[ch];
    double sc = (kstep == 0) ? 0.5 : (kstep < Lc) ? 1.0 : (kstep == Lc) ? 0.5 : 0.0;
    if (sc != 0.0) p[(size_t)ch * nAC + a] -= sc * dt * grad[(size_t)ch * nAC + a];
}
__global__ void k_fill(size_t n, double v, double* __restrict__ x) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = v;
}
__global__ void k_clip_momentum(int nAC, const double* __restrict__ z, double* __restrict__ p) {
    int ch = blockIdx.y, a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= nAC) return;
    double v = z[(size_t)ch * nAC + a];
    if (fabs(v) > 2.5) v = copysign(2.5, v);                     // getMomentumVector HMCSampler.jl:441-449
    p[(size_t)ch * nAC + a] = v;
}
// Metropolis accept on the device (HMCSampler.jl:149-186).  chainScal[ch] = {startD, startM, startK, startH}
// DT: element type of the packed data (cplx impedances, double for rho / phase plans)
template <typename DT>
__global__ void __launch_bounds__(kHmcThreads)
k_accept(int nAC, int nData, int it, int nsamples, const double* __restrict__ uacc, const double* __restrict__ phi,
         const double* __restrict__ energies, const double* __restrict__ znew, double* __restrict__ m, double* __restrict__ p,
         double* __restrict__ curM, double* __restrict__ chainScal, const DT* __restrict__ predPacked,
         double* __restrict__ hmcmodel, double* __restrict__ hmstats, int* __restrict__ accept, DT* __restrict__ hmcdata) {
    __shared__ double sh[32];
    __shared__ int accSh;
    const int ch = blockIdx.x;
    double* sc = chainScal + ch * 4;
    if (threadIdx.x == 0) {
        double finD = phi[ch], finK = energies[ch * 2], finM = energies[ch * 2 + 1];
        double finH = finD + finK + finM;
        double hdif = sc[3] - finH;
        int acc = (hdif > 0.0) || (uacc[(size_t)ch * nsamples + (it - 1)] < exp(hdif));
        if (acc) { sc[0] = finD; sc[1] = finM; }
        accSh = acc;
        accept[(size_t)ch * nsamples + (it - 1)] = acc;
    }
    __syncthreads();
    const int acc = accSh;
    double* mm = m + (size_t)ch * nAC;
    double* pp = p + (size_t)ch * nAC;
    double* cm = curM + (size_t)ch * nAC;
    const double* zn = znew + (size_t)ch * nAC;
    double* modelOut = hmcmodel + ((size_t)ch * nsamples + (it - 1)) * nAC;
    double k = 0.0;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) {
        double v = acc ? mm[a] : cm[a];
        mm[a] = v; cm[a] = v; modelOut[a] = v;
        double z = zn[a];
        if (fabs(z) > 2.5) z = copysign(2.5, z);
        pp[a] = z;
        k += z * z;
    }
    k = block_reduce(k, false, sh);
    DT* dout = hmcdata + ((size_t)ch * (nsamples + 1) + it) * nData;
    const DT* dprev = dout - nData;
    const DT* dnew = predPacked + (size_t)ch * nData;
    for (int i = threadIdx.x; i < nData; i += blockDim.x) dout[i] = acc ? dnew[i] : dprev[i];
    if (threadIdx.x == 0) {
        sc[2] = 0.5 * k;
        sc[3] = sc[0] + sc[1] + sc[2];
        double* st = hmstats + ((size_t)ch * (nsamples + 1) + it) * 4;
        st[0] = sc[0]; st[1] = sc[1]; st[2] = sc[2]; st[3] = sc[3];
    }
}

// Frequency-sharded evaluation (SURVEY.md 8e): every rank holds a subset of the frequencies.  The data gradient and the
// data misfit are sums over frequencies, so each rank packs its partial [gdata(nAC) | phi_d] per chain into one exchange
// buffer, the host all-reduces it (NCCL over NVLink), and the prior gradient — which must be counted once — is added after.
__global__ void k_pack_exchange(int nAC, const double* __restrict__ gdata, const double* __restrict__ phi, double* __restrict__ xbuf) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (a < nAC) xbuf[(size_t)ch * (nAC + 1) + a] = gdata[(size_t)ch * nAC + a];
    if (a == nAC) xbuf[(size_t)ch * (nAC + 1) + nAC] = phi[ch];
}
__global__ void k_unpack_exchange(int nAC, const double* __restrict__ xbuf, const double* __restrict__ m, const double* __restrict__ mref,
                                  const int* __restrict__ wmPtr, const int* __restrict__ wmIdx, const double* __restrict__ wmVal,
                                  double beta, double* __restrict__ gdata, double* __restrict__ gtotal, double* __restrict__ phi) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (a == nAC) phi[ch] = xbuf[(size_t)ch * (nAC + 1) + nAC];
    if (a >= nAC) return;
    const double* mm = m + (size_t)ch * nAC;
    const double* mr = mref + (size_t)ch * nAC;
    double pr = 0.0;
    for (int k = wmPtr[a]; k < wmPtr[a + 1]; ++k) { int j = wmIdx[k]; pr += wmVal[k] * (mm[j] - mr[j]); }
    const double gd = xbuf[(size_t)ch * (nAC + 1) + a];
    gdata[(size_t)ch * nAC + a] = gd;
    gtotal[(size_t)ch * nAC + a] = gd + beta * pr;
}

// Explicit Jacobian (compJacMat.jl:7-381 / compJacTMat.jl:9-406): one pass of the adjoint machinery per (receiver, real /
// imaginary part) yields, in every (frequency, mode) system, the row of that system's datum at this receiver.
//   v = e_d   -> real(J^T conj(v)) = Re J[d,:]  ;   v = i e_d -> Im J[d,:]
// Components that share a system (ZXY and TZY) need passes of their own: a pass covers the components of compMask, comp[mi] being
// the one of them that system mi holds (-1: none).
__global__ void k_jac_vin(int nFull, int nRx, int nComp, unsigned compMask, int r, cplx val, cplx* __restrict__ vin) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (i >= nFull) return;
    const int rx = (i / nComp) % nRx, c = i % nComp;
    vin[(size_t)ch * nFull + i] = (rx == r && ((compMask >> c) & 1u)) ? val : mk(0.0, 0.0);
}
__global__ void k_jac_rows(int nAC, int nCell, int nFreq, int nRx, int nModes, int nComp, int2 comp, int nData, int r, int part,
                           const int* __restrict__ act2cell, const int* __restrict__ full2packed, const double* __restrict__ Gpart,
                           double* __restrict__ J) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, sys = blockIdx.y;
    if (a >= nAC) return;
    const int f = sys % nFreq, t = sys / nFreq, mi = t % nModes, ch = t / nModes;
    const int c = mi == 0 ? comp.x : comp.y;
    if (c < 0) return;
    const int d = full2packed[(f * nRx + r) * nComp + c];
    if (d < 0) return;
    J[(((size_t)ch * nData + d) * nAC + a) * 2 + part] = Gpart[(size_t)sys * nCell + act2cell[a]];
}

// rho / phase plans: v = e_d carries v_rho = 1 (part 0) or v_phi = 1 (part 1), the real rows d rho_a / d sigma and
// d phase / d sigma of the datum, J [nChains][nData][nAC] doubles; full2packed indexes the real view [nFull][2]
__global__ void k_jac_rows_real(int nAC, int nCell, int nFreq, int nRx, int nModes, int nData, int r, int part,
                                const int* __restrict__ act2cell, const int* __restrict__ full2packed, const double* __restrict__ Gpart,
                                double* __restrict__ J) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, sys = blockIdx.y;
    if (a >= nAC) return;
    const int f = sys % nFreq, t = sys / nFreq, mi = t % nModes, ch = t / nModes;
    const int d = full2packed[2 * ((f * nRx + r) * nModes + mi) + part];
    if (d < 0) return;
    J[((size_t)ch * nData + d) * nAC + a] = Gpart[(size_t)sys * nCell + act2cell[a]];
}

int ensure_pin(hmcmt_plan* pl, size_t bytes) {
    if (pl->pinBytes >= bytes) return kOk;
    if (pl->pin) cudaFreeHost(pl->pin);
    pl->pin = nullptr;
    pl->pinBytes = 0;
    HMCMT_CUDA_TRY(cudaMallocHost(&pl->pin, bytes));
    pl->pinBytes = bytes;
    return kOk;
}

// layered-earth sensitivity scalars (depend on sigma only) on the side stream: they overlap the factorisation and are joined
// before the contraction
int launch_sens_side(hmcmt_plan* pl) {
    const MeshDev& M = pl->M;
    HMCMT_CUDA_TRY(cudaEventRecord(pl->evFork, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamWaitEvent(pl->side, pl->evFork, 0));
    k_row_mean<<<dim3(M.nz, pl->nChains), 128, 0, pl->side>>>(M.ny, M.nz, pl->sigma.p, pl->meanSig.p);
    LAUNCH_CHECK(pl);
    k_sens_scalars<<<(pl->nSys * 3 + 63) / 64, 64, 0, pl->side>>>(M, pl->sm, pl->nSys, pl->freqs.p, pl->sigma.p, pl->meanSig.p, pl->scratch.p, pl->bcs.p);
    LAUNCH_CHECK(pl);
    HMCMT_CUDA_TRY(cudaEventRecord(pl->evJoin, pl->side));
    pl->haveSens = true;
    return kOk;
}

// A contiguous range of systems [s0, s0 + n) and the stream its work is queued on.  One evaluation either runs the whole batch
// on the plan's stream, or (multifrontal solver, HMCMT_GROUPS >= 2) splits it into groups that run on their own streams: while
// one group is in the few-CTA top levels of its elimination tree, in the receiver functional or in the contraction, the
// thousands of small fronts of another group fill the SMs.  The systems of a step are independent (one per frequency x mode,
// MT2DFwdSolver.jl:163-191), so the groups never exchange anything before the final sums over systems.
struct SysRange {
    int s0, n;
    cudaStream_t st;
};

// sigma and stencil planes of all chains / modes: everything the factorisations need (plan stream)
int forward_model(hmcmt_plan* pl) {
    const MeshDev& M = pl->M;
    cudaStream_t st = pl->stream;
    const int nCh = pl->nChains;
    pl->haveForward = false;
    pl->haveSens = false;
    if (!pl->sigmaDirect) {
        k_model_transform<<<dim3((M.nCell + 255) / 256, nCh), 256, 0, st>>>(M.nCell, pl->nAC, pl->cell2act.p, pl->bg.p, pl->m.p, pl->sigma.p);
        LAUNCH_CHECK(pl);
    }
    k_stencil_planes<<<dim3((M.N + 255) / 256, nCh * pl->nModes), 256, 0, st>>>(M, pl->sm, pl->sigma.p, pl->planes.p);
    LAUNCH_CHECK(pl);
    return kOk;
}
// boundary values and right-hand sides of ALL systems (plan stream; the factorisations do not depend on them), then the
// layered-earth sensitivity scalars on the side stream
int forward_bc(hmcmt_plan* pl, bool wantAdjoint) {
    const MeshDev& M = pl->M;
    cudaStream_t st = pl->stream;
    const int nSys = pl->nSys, nCh = pl->nChains;
    {
        // as many profiles per block as shared memory allows: the serial phase keeps PB lanes of one warp busy and is bound by
        // FP64 issue slots, so fewer profiles per block (even when that avoids a second wave of blocks) measured slower
        const int PB = boundary_profiles_per_block(M.nz);
        k_boundary<<<dim3((M.ny + 1 + PB - 1) / PB, nCh * pl->sm.nFreq), kBcThreads, (size_t)PB * M.nz * 6 * sizeof(cplx), st>>>(
            M, pl->sm, pl->freqs.p, pl->sigma.p, pl->bc.p, PB);
    }
    LAUNCH_CHECK(pl);
    k_rhs<<<dim3((M.N + 255) / 256, nSys), 256, 0, st>>>(M, pl->sm, pl->sigma.p, pl->bc.p, pl->rhs.p);
    LAUNCH_CHECK(pl);
    if (wantAdjoint) {
        int rc = launch_sens_side(pl);
        if (rc) return rc;
    }
    return kOk;
}
int forward_pre(hmcmt_plan* pl, bool wantAdjoint) {
    int rc = forward_model(pl);
    return rc ? rc : forward_bc(pl, wantAdjoint);
}

// factorisation + forward solve of one range (the band kernels only take the whole batch and do both in forward_factor);
// rhsReady: event the forward solve waits for (the right-hand sides are produced on another stream), or null
int forward_factor(hmcmt_plan* pl, const SysRange& r) {
    const MeshDev& M = pl->M;
    if (pl->useMf) {
        int rc = pl->mfs->set_mt_values(r.st, M.N, pl->mfSys.p, r.s0, r.n);
        if (rc) return rc;
        ++pl->launches;
        return pl->mfs->factor(r.st, pl->status.p, &pl->launches, r.s0, r.n);
    }
    if (r.s0 != 0 || r.n != pl->nSys) return kErrArg;
    int nl = 0;
    int rc = launch_factor(r.st, pl->T, pl->sysDesc.p, pl->nSys, pl->dom, pl->fwdJobs.p, &nl);
    pl->launches += nl;
    return rc;
}
int forward_solve(hmcmt_plan* pl, const SysRange& r) {
    const MeshDev& M = pl->M;
    if (!pl->useMf) return kOk;      // fused into the band factorisation
    return pl->mfs->solve(r.st, 1, pl->rhs.p, M.N, pl->x.p, M.N, &pl->launches, r.s0, r.n, pl->patRhs);
}
int forward_fields(hmcmt_plan* pl, const SysRange& r) {
    const MeshDev& M = pl->M;
    k_node_field<<<dim3((M.nNode + 255) / 256, r.n), 256, 0, r.st>>>(M, pl->x.p, pl->bc.p, pl->F.p, r.s0, 0, M.nNode);
    LAUNCH_CHECK(pl);
    return kOk;
}

// forward part of the whole batch on the plan's stream, the factorisation + forward solve timed with CUDA events when the caller
// asked for it (hmcmt_kernel_time(reset=1))
int forward_phase(hmcmt_plan* pl, bool wantAdjoint) {
    cudaStream_t st = pl->stream;
    int rc = forward_pre(pl, wantAdjoint);
    if (rc) return rc;
    std::pair<cudaEvent_t, cudaEvent_t>* ev = nullptr;
    if (pl->timeFactor && pl->factorEventsUsed < kMaxFactorEvents) {
        if (pl->factorEventsUsed == pl->factorEvents.size()) {
            cudaEvent_t a, b;
            HMCMT_CUDA_TRY(cudaEventCreate(&a));
            HMCMT_CUDA_TRY(cudaEventCreate(&b));
            pl->factorEvents.emplace_back(a, b);
            cudaEvent_t c;
            HMCMT_CUDA_TRY(cudaEventCreate(&c));
            pl->factorMid.push_back(c);
        }
        ev = &pl->factorEvents[pl->factorEventsUsed++];
        HMCMT_CUDA_TRY(cudaEventRecord(ev->first, st));
    }
    const SysRange all{0, pl->nSys, st};
    rc = forward_factor(pl, all);
    if (rc == kOk && ev) HMCMT_CUDA_TRY(cudaEventRecord(pl->factorMid[pl->factorEventsUsed - 1], st));
    if (rc == kOk) rc = forward_solve(pl, all);
    if (rc) return rc;
    ++pl->factorLaunches;
    if (ev) HMCMT_CUDA_TRY(cudaEventRecord(ev->second, st));
    rc = forward_fields(pl, all);
    if (rc) return rc;
    pl->haveForward = true;
    return kOk;
}

// the receiver-functional instance of the plan's data (fixed when the plan is created)
decltype(&k_rx_adjoint<false, false>) rx_kernel(const hmcmt_plan* pl) {
    if (pl->dataKind) return k_rx_adjoint<true, false>;
    return pl->tipper ? k_rx_adjoint<false, true> : k_rx_adjoint<false, false>;
}
// receiver functional: responses, residual, misfit partial and (wantAdjoint) the adjoint sources for the data vector vin
// (null: v = Wd^2 (pred - obs))
int rx_range(hmcmt_plan* pl, const SysRange& r, bool wantAdjoint, const cplx* vin) {
    const MeshDev& M = pl->M;
    size_t rxSmem = (size_t)(6 * (M.ny + 1) + 3 * M.ny) * sizeof(cplx);
    if (wantAdjoint) HMCMT_CUDA_TRY(cudaMemsetAsync(pl->lam.p + (size_t)r.s0 * M.N, 0, sizeof(cplx) * (size_t)r.n * M.N, r.st));
    rx_kernel(pl)<<<r.n, kRxThreads, rxSmem, r.st>>>(M, pl->rx, pl->sm, pl->cm, pl->freqs.p, pl->sigma.p, pl->F.p, pl->obs.p, pl->wd.p,
                                                     pl->wdPha.p, vin, pl->predFull.p, pl->phiPart.p, pl->srows.p, pl->qrow.p, pl->lam.p,
                                                     wantAdjoint ? 1 : 0, pl->respKind, pl->respFull.p, r.s0);
    LAUNCH_CHECK(pl);
    return kOk;
}
int reduce_phi(hmcmt_plan* pl) {
    k_reduce_phi<<<pl->nChains, 32, 0, pl->stream>>>(pl->nSysPerChain, pl->phiPart.p, pl->phi.p);
    LAUNCH_CHECK(pl);
    return kOk;
}
int rx_phase(hmcmt_plan* pl, bool wantAdjoint, const cplx* vin) {
    int rc = rx_range(pl, SysRange{0, pl->nSys, pl->stream}, wantAdjoint, vin);
    return rc ? rc : reduce_phi(pl);
}

// adjoint field and contraction into the per-system gradient partials, once lam holds the adjoint solution
int adjoint_contract(hmcmt_plan* pl, const SysRange& r) {
    const MeshDev& M = pl->M;
    cudaStream_t st = r.st;
    k_node_field<<<dim3((M.nNode + 255) / 256, r.n), 256, 0, st>>>(M, pl->lam.p, nullptr, pl->Lam.p, r.s0, 0, M.nNode);
    LAUNCH_CHECK(pl);
    HMCMT_CUDA_TRY(cudaStreamWaitEvent(st, pl->evJoin, 0));
    k_contract_cols<<<r.n, kConThreads, contract_cols_smem(M.ny, M.nz, pl->conStaged), st>>>(M, pl->sm, pl->freqs.p, pl->sigma.p, pl->Lam.p,
                                                                                              pl->srows.p, pl->scratch.p, pl->conCols.p, pl->conStaged, r.s0);
    LAUNCH_CHECK(pl);
    k_contract_cells<<<dim3((M.nCell + 255) / 256, r.n), 256, 0, st>>>(M, pl->sm, pl->freqs.p, pl->sigma.p, pl->F.p, pl->Lam.p, pl->qrow.p,
                                                                       pl->bcs.p, pl->conCols.p, pl->Gpart.p, r.s0);
    LAUNCH_CHECK(pl);
    return kOk;
}
// adjoint part: one solve per system with the factors of the forward phase (A symmetric: no transposition,
// compJacTMatVec.jl:220-224), contraction into the per-system gradient partials
int adjoint_range(hmcmt_plan* pl, const SysRange& r) {
    const MeshDev& M = pl->M;
    cudaStream_t st = r.st;
    int rc;                                                            // lam <- A^{-1} s[ii]  (in place)
    if (pl->useMf) rc = pl->mfs->solve(st, 1, pl->lam.p, M.N, pl->lam.p, M.N, &pl->launches, r.s0, r.n, pl->patAdj);
    else {
        if (r.s0 != 0 || r.n != pl->nSys) return kErrArg;
        rc = launch_solve(st, pl->T, pl->jobs.p, pl->nSys, pl->dom);
        pl->launches += pl->dom.split ? 3 : 1;
    }
    return rc ? rc : adjoint_contract(pl, r);
}
// sum over the systems of a chain, chain rule to ln(sigma), prior gradient
int reduce_grad(hmcmt_plan* pl) {
    const MeshDev& M = pl->M;
    k_reduce_grad<<<dim3((pl->nAC + 255) / 256, pl->nChains), 256, 0, pl->stream>>>(pl->nAC, M.nCell, pl->nSysPerChain, pl->act2cell.p, pl->Gpart.p,
                                                                                    pl->m.p, pl->mref.p, pl->wmPtr.p, pl->wmIdx.p, pl->wmVal.p, pl->beta,
                                                                                    pl->sigma.p, pl->gsig.p, pl->gdata.p, pl->gtotal.p);
    LAUNCH_CHECK(pl);
    return kOk;
}
int adjoint_phase(hmcmt_plan* pl, bool reduce = true) {
    int rc = adjoint_range(pl, SysRange{0, pl->nSys, pl->stream});
    if (rc || !reduce) return rc;
    return reduce_grad(pl);
}

// Forward solve, receiver functional and adjoint solve of a range on the multifrontal path, once its factors and right-hand
// sides are ready.  The receiver functional reads the field on the node rows zid, zid + 1 only, so before it only the receiver
// path (the fronts holding those rows' unknowns and their ancestors: the active set of patRx) is back-substituted for x; the
// rest of x is back-substituted together with the adjoint lam, in one pass over the factor (Solver::backward_pair).  The
// backward substitutions read about 1.2 instead of 2 factors per gradient.  Every value is the one the complete solves give.
int gradient_range(hmcmt_plan* pl, const SysRange& r) {
    const MeshDev& M = pl->M;
    mf::Solver& S = *pl->mfs;
    int rc;
    if ((rc = S.forward_slot(r.st, 0, pl->rhs.p, M.N, &pl->launches, r.s0, r.n, pl->patRhs)) ||
        (rc = S.backward_slot(r.st, 0, pl->x.p, M.N, &pl->launches, r.s0, r.n, pl->patRx)))
        return rc;
    const int rx0 = M.zid * (M.ny + 1), rx1 = (M.zid + 2) * (M.ny + 1);
    k_node_field<<<dim3((rx1 - rx0 + 255) / 256, r.n), 256, 0, r.st>>>(M, pl->x.p, pl->bc.p, pl->F.p, r.s0, rx0, rx1);
    LAUNCH_CHECK(pl);
    if ((rc = rx_range(pl, r, true, nullptr)) ||
        (rc = S.forward_slot(r.st, 1, pl->lam.p, M.N, &pl->launches, r.s0, r.n, pl->patAdj)) ||
        (rc = S.backward_pair(r.st, pl->x.p, pl->lam.p, M.N, &pl->launches, r.s0, r.n, pl->patRx)) || (rc = forward_fields(pl, r)))
        return rc;
    return adjoint_contract(pl, r);
}

// forward + adjoint gradient of the whole batch with the systems split into groups on their own streams
int compute_step_grouped(hmcmt_plan* pl) {
    const int G = (int)pl->groupStreams.size();
    int rc = forward_model(pl);
    if (rc) return rc;
    HMCMT_CUDA_TRY(cudaEventRecord(pl->evPre, pl->stream));
    // the groups start factorising right away; boundary values / right-hand sides (plan stream) and the sensitivity scalars
    // (side stream) are produced meanwhile and joined where they are first needed
    std::vector<SysRange> rs;
    for (int g = 0; g < G; ++g) {
        const int s0 = (int)((int64_t)pl->nSys * g / G), s1 = (int)((int64_t)pl->nSys * (g + 1) / G);
        if (s1 <= s0) continue;
        rs.push_back(SysRange{s0, s1 - s0, pl->groupStreams[g]});
        HMCMT_CUDA_TRY(cudaStreamWaitEvent(rs.back().st, pl->evPre, 0));
        if ((rc = forward_factor(pl, rs.back()))) return rc;
    }
    if ((rc = forward_bc(pl, true))) return rc;
    HMCMT_CUDA_TRY(cudaEventRecord(pl->evRhs, pl->stream));
    for (size_t g = 0; g < rs.size(); ++g) {
        const SysRange& r = rs[g];
        HMCMT_CUDA_TRY(cudaStreamWaitEvent(r.st, pl->evRhs, 0));
        if ((rc = gradient_range(pl, r))) return rc;
        HMCMT_CUDA_TRY(cudaEventRecord(pl->groupDone[g], r.st));
        HMCMT_CUDA_TRY(cudaStreamWaitEvent(pl->stream, pl->groupDone[g], 0));
    }
    ++pl->factorLaunches;
    pl->haveForward = true;
    if ((rc = reduce_phi(pl))) return rc;
    return reduce_grad(pl);
}

// The gradient evaluation as a CUDA graph.  Its launches (a few hundred per evaluation on the multifrontal path: one per tree
// level, system group and phase) always have the same arguments — every buffer belongs to the plan — so the second evaluation
// of a plan is captured from the streams (the groups' and the side stream join the capture through their events) and replayed
// from then on: the host-buffer entry points no longer pay a launch per kernel before the device has work.  The first
// evaluation runs eagerly (it also sets the per-device kernel attributes, which must not happen under capture).
// HMCMT_GRAPH=0 switches it off.
int compute_step_eager(hmcmt_plan* pl) {
    if (pl->useMf && pl->groupStreams.size() >= 2) return compute_step_grouped(pl);
    if (pl->useMf) {
        const SysRange all{0, pl->nSys, pl->stream};
        int rc;
        if ((rc = forward_pre(pl, true)) || (rc = forward_factor(pl, all)) || (rc = gradient_range(pl, all))) return rc;
        ++pl->factorLaunches;
        pl->haveForward = true;
        return (rc = reduce_phi(pl)) ? rc : reduce_grad(pl);
    }
    int rc = forward_phase(pl, true);
    if (rc) return rc;
    rc = rx_phase(pl, true, nullptr);
    return rc ? rc : adjoint_phase(pl);
}
int compute_step_graph(hmcmt_plan* pl) {
    if (pl->graphState == 0) {
        pl->graphState = 1;
        return compute_step_eager(pl);
    }
    if (pl->graphState == 1) {
        const int64_t l0 = pl->launches, f0 = pl->factorLaunches;
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(pl->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            pl->graphState = -1;
            return compute_step_eager(pl);
        }
        const int rc = compute_step_eager(pl);
        const cudaError_t e = cudaStreamEndCapture(pl->stream, &graph);
        pl->graphLaunches = pl->launches - l0;
        pl->launches = l0;
        pl->factorLaunches = f0;
        if (rc != kOk || e != cudaSuccess || !graph || cudaGraphInstantiate(&pl->graphExec, graph, 0) != cudaSuccess) {
            cudaGetLastError();
            if (graph) cudaGraphDestroy(graph);
            pl->graphExec = nullptr;
            pl->graphState = -1;
            fprintf(stderr, "[hmcmt_b200] graph capture of the evaluation failed (%s): launching eagerly\n", cudaGetErrorString(e));
            return compute_step_eager(pl);
        }
        cudaGraphDestroy(graph);
        // evJoin was last recorded inside the capture and cannot be waited on outside it; the replays join the side stream
        // inside the graph, so an eager wait after them (hmcmt_jtvec, hmcmt_jvec, hmcmt_gn_hessvec) has nothing left to wait for
        HMCMT_CUDA_TRY(cudaEventRecord(pl->evJoin, pl->side));
        pl->graphState = 2;
    }
    HMCMT_CUDA_TRY(cudaGraphLaunch(pl->graphExec, pl->stream));
    pl->launches += pl->graphLaunches;
    ++pl->factorLaunches;
    pl->haveForward = true;
    pl->haveSens = true;
    return kOk;
}

// One evaluation of the hot path for the device-resident model pl->m:
//   forward (all chains x modes x freqs) [+ adjoint gradient + prior gradient].
int compute_step(hmcmt_plan* pl, bool wantAdjoint, const cplx* vin) {
    if (wantAdjoint && !vin && !pl->timeFactor) {
        // the graph holds the standard evaluation (sigma = exp(m), the plan's own data type); the forward-only response toggle and
        // direct conductivities are launched eagerly
        const bool standard = !pl->sigmaDirect && pl->respKind == 0;
        return pl->graphState >= 0 && standard ? compute_step_graph(pl) : compute_step_eager(pl);
    }
    int rc = forward_phase(pl, wantAdjoint);
    if (rc) return rc;
    rc = rx_phase(pl, wantAdjoint, vin);
    if (rc || !wantAdjoint) return rc;
    return adjoint_phase(pl);
}

// Device error flags of the work queued so far (synchronises).  The flags are cleared after reading, so a failure is reported
// once, by the call that caused it, and does not poison later evaluations of the (cached) plan.
int check_status(hmcmt_plan* pl) {
    std::vector<int> h(pl->nSys);
    int drift = 0;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(h.data(), pl->status.p, sizeof(int) * pl->nSys, cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaMemcpyAsync(&drift, pl->driftFlag.p, sizeof(int), cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    int rc = kOk;
    for (int v : h) if (v) { rc = v; break; }
    if (rc == kOk && drift) rc = kErrBounds;
    if (rc != kOk) {
        HMCMT_CUDA_TRY(cudaMemsetAsync(pl->status.p, 0, sizeof(int) * pl->nSys, pl->stream));
        HMCMT_CUDA_TRY(cudaMemsetAsync(pl->driftFlag.p, 0, sizeof(int), pl->stream));
    }
    return rc;
}

__global__ void k_real_to_cplx(size_t n, const double* __restrict__ x, cplx* __restrict__ y) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = mk(x[i], 0.0);
}
__global__ void k_cplx_to_real(size_t n, const cplx* __restrict__ x, double* __restrict__ y) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = x[i].x;
}
// p = L z with the banded lower Cholesky factor, Lband[i*(bw+1) + d] = L[i][i-d]   (getMomentumVector: mp = sqrtM * mp, :450)
__global__ void k_bandL_matvec(int n, int bw, const double* __restrict__ Lband, const double* __restrict__ z, double* __restrict__ p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (i >= n) return;
    const double* zz = z + (size_t)ch * n;
    const double* row = Lband + (size_t)i * (bw + 1);
    double acc = 0.0;
    for (int d = min(bw, i); d >= 0; --d) acc += row[d] * zz[i - d];
    p[(size_t)ch * n + i] = acc;
}

// gradK = invM p = Wm^{-1} p for every chain (one multifrontal solve with nChains right-hand sides)
int mass_apply(hmcmt_plan* pl) {
    if (!pl->massOn) return kOk;
    const size_t n = (size_t)pl->nChains * pl->nAC;
    k_real_to_cplx<<<(unsigned)((n + 255) / 256), 256, 0, pl->stream>>>(n, pl->p.p, pl->massBuf.p);
    LAUNCH_CHECK(pl);
    int rc = pl->massSolver->solve(pl->stream, pl->nChains, pl->massBuf.p, pl->nAC, pl->massBuf.p, pl->nAC, &pl->launches);
    if (rc) return rc;
    k_cplx_to_real<<<(unsigned)((n + 255) / 256), 256, 0, pl->stream>>>(n, pl->massBuf.p, pl->gradK.p);
    LAUNCH_CHECK(pl);
    return kOk;
}
// p <- sqrtM p in place (p holds the clipped normal draws)
int mass_sqrt_apply(hmcmt_plan* pl) {
    if (!pl->massOn) return kOk;
    k_bandL_matvec<<<dim3((pl->nAC + 255) / 256, pl->nChains), 256, 0, pl->stream>>>(pl->nAC, pl->massBw, pl->Lband.p, pl->p.p, pl->gradK.p);
    LAUNCH_CHECK(pl);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->p.p, pl->gradK.p, sizeof(double) * (size_t)pl->nChains * pl->nAC, cudaMemcpyDeviceToDevice, pl->stream));
    return kOk;
}

int energies(hmcmt_plan* pl) {
    int mrc = mass_apply(pl);
    if (mrc) return mrc;
    k_energies<<<pl->nChains, kHmcThreads, 0, pl->stream>>>(pl->nAC, pl->m.p, pl->mref.p, pl->p.p, pl->wmPtr.p, pl->wmIdx.p, pl->wmVal.p,
                                                            pl->beta, pl->energies.p, pl->massOn ? pl->gradK.p : nullptr);
    LAUNCH_CHECK(pl);
    return kOk;
}

inline int kDriftBlocks(int nAC) { return std::max(1, std::min(128, (nAC + kHmcThreads - 1) / kHmcThreads)); }
int drift(hmcmt_plan* pl, double dt) {
    int mrc = mass_apply(pl);
    if (mrc) return mrc;
    const double* gk = pl->massOn ? pl->gradK.p : nullptr;
    const dim3 grid(kDriftBlocks(pl->nAC), pl->nChains);
    k_drift_max<<<grid, kHmcThreads, 0, pl->stream>>>(pl->nAC, dt, pl->p.p, gk, pl->driftPart.p);
    LAUNCH_CHECK(pl);
    k_drift<<<grid, kHmcThreads, 0, pl->stream>>>(pl->nAC, dt, pl->lo, pl->hi, pl->m.p, pl->p.p, pl->driftFlag.p, gk, pl->driftPart.p);
    LAUNCH_CHECK(pl);
    return kOk;
}

}  // namespace

// ---- NCCL inside the library (SURVEY.md 8e): the sum over the ranks' frequency shards is one ncclAllReduce on the plan's own
// stream, between the contraction and the kick — no host round trip, no PyTorch on the data path.  libnccl is resolved at run
// time (dlopen by SONAME: a process that already loaded NCCL, e.g. through torch.distributed, shares that copy).
namespace {
struct NcclApi {
    void* handle = nullptr;
    decltype(&ncclGetUniqueId) getUniqueId = nullptr;
    decltype(&ncclCommInitRank) commInitRank = nullptr;
    decltype(&ncclAllReduce) allReduce = nullptr;
    decltype(&ncclCommDestroy) commDestroy = nullptr;
    decltype(&ncclGetErrorString) getErrorString = nullptr;
};
NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        api.handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (api.handle) {
            api.getUniqueId = (decltype(api.getUniqueId))dlsym(api.handle, "ncclGetUniqueId");
            api.commInitRank = (decltype(api.commInitRank))dlsym(api.handle, "ncclCommInitRank");
            api.allReduce = (decltype(api.allReduce))dlsym(api.handle, "ncclAllReduce");
            api.commDestroy = (decltype(api.commDestroy))dlsym(api.handle, "ncclCommDestroy");
            api.getErrorString = (decltype(api.getErrorString))dlsym(api.handle, "ncclGetErrorString");
        }
    }
    const bool ok = api.handle && api.getUniqueId && api.commInitRank && api.allReduce && api.commDestroy;
    if (!ok) fprintf(stderr, "[hmcmt_b200] libnccl.so.2 could not be loaded: %s\n", api.handle ? "missing symbols" : dlerror());
    return ok ? &api : nullptr;
}
}  // namespace

extern "C" {

const char* hmcmt_version(void) { return "hmcmt_b200 0.1 (sm_100a; DMMA.8x8x4 tile-window band LDL^T; no CPU fallback)"; }

// dataKind 0: impedance data (hmcmt_plan_create), 1: apparent resistivity / phase rows (hmcmt_plan_create_rho_phase)
static int plan_create(const hmcmt_problem* pr, hmcmt_plan** out, int dataKind) {
    if (!pr || !out) return kErrArg;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        fprintf(stderr, "[hmcmt_b200] no CUDA device: this library has no CPU fallback\n");
        return kErrNoDevice;
    }
    if (pr->ny < 3 || pr->nz < 3 || pr->nFreq < 1 || pr->nRx < 1 || pr->nComp < 1 || pr->nComp > 3 || pr->nChains < 1 || pr->nAC < 1)
        return kErrArg;
    // compMode 2 (TZY, the TE tipper): at most once, as the last component, impedance plans only; the impedance components before
    // it are one or two as without it
    const bool tipper = pr->compMode[pr->nComp - 1] == 2;
    const int nZ = pr->nComp - (tipper ? 1 : 0);
    if (nZ > 2 || (tipper && dataKind)) return kErrArg;
    for (int c = 0; c < nZ; ++c)
        if (pr->compMode[c] == 2) return kErrArg;
    int teSys = -1;                                  // the system the tipper shares (the first TE one), or a TE system of its own
    for (int c = 0; c < nZ && teSys < 0; ++c)
        if (pr->compMode[c] == 0) teSys = c;
    if (tipper && teSys < 0 && nZ == 2) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pr->device));
    hmcmt_plan* pl = new (std::nothrow) hmcmt_plan();
    if (!pl) return kErrAlloc;
    pl->device = pr->device;
    {
        int nsm = 0;
        if (cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, pr->device) == cudaSuccess && nsm > 0) pl->numSMs = nsm;
    }
    pl->ny = pr->ny; pl->nz = pr->nz; pl->nFreq = pr->nFreq; pl->nRx = pr->nRx; pl->nData = pr->nData; pl->nAC = pr->nAC;
    pl->nChains = pr->nChains; pl->nComp = pr->nComp; pl->nModes = nZ; pl->dataKind = dataKind; pl->tipper = tipper;
    for (int c = 0; c < nZ; ++c) pl->modeList[c] = pr->compMode[c];
    if (tipper) {
        if (teSys < 0) { teSys = nZ; pl->modeList[pl->nModes++] = 0; }
        pl->cm = CompMap{pl->nComp, {nZ > 0 ? 0 : -1, nZ > 1 ? 1 : -1}, pl->nComp - 1, teSys};
    }
    pl->beta = pr->regParam;
    pl->lo = std::log(pr->sigBounds[0]);
    pl->hi = std::log(pr->sigBounds[1]);
    const int ny = pr->ny, nz = pr->nz;
    MeshDev& M = pl->M;
    M.ny = ny; M.nz = nz; M.n1 = ny - 1; M.n2 = nz - 1; M.N = M.n1 * M.n2;
    M.fastZ = (M.n2 <= M.n1) ? 1 : 0;
    M.nf = M.fastZ ? M.n2 : M.n1; M.nl = M.fastZ ? M.n1 : M.n2;
    M.nCell = ny * nz; M.nNode = (ny + 1) * (nz + 1); M.nb = 2 * (ny + nz);
    pl->b = M.nf;
    pl->T = round_T(pl->b);
    if (M.nf < 2) { delete pl; return kErrArg; }
    {
        // "mf" / "band" force a solver (band only where the register window fits); default: see below
        const char* env = std::getenv("HMCMT_SOLVER");
        // measured on B200 (tools/dev/t_groups.py ... HMCMT_SOLVER band mf, ms per leapfrog step): the multifrontal solver wins
        // from ~1 000 unknowns per system upwards (20x16 cells: 0.25 vs 0.23; 30x24: 0.31 vs 0.32; 40x30: 0.37 vs 0.44; 48x40: 0.49 vs
        // 0.61; 96x56: 0.76 vs 1.52; 200x100: 4.04 vs 6.67), the band kernel below
        const bool wantMf = env ? !std::strcmp(env, "mf") : (M.N >= 1000);
        pl->useMf = pl->T == 0 || wantMf;
        if (pl->useMf) pl->T = 0;
    }
    {
        // two CTAs per system when there are enough lines: halves the sequential pivot chain
        const char* env = std::getenv("HMCMT_SPLIT");
        int want = env ? std::atoi(env) : 1;
        pl->dom = BandDom{M.N, M.nf, pl->b, M.nl, (!pl->useMf && want && M.nl >= 9) ? 1 : 0, M.nl / 2};
        if (!pl->useMf) {
            LocalDom L0 = LocalDom::make(pl->dom, 0);
            pl->steps0 = L0.sTot;
            pl->steps1 = pl->dom.split ? LocalDom::make(pl->dom, 1).sOwn : 0;
            pl->S = pl->steps0 + pl->steps1;
        }
    }
    pl->nSysPerChain = pl->nModes * pl->nFreq;
    pl->nSys = pl->nSysPerChain * pl->nChains;
    pl->nFull = pl->nFreq * pl->nRx * pl->nComp;
    pl->sm = SysMap{pl->nFreq, pl->nModes, pl->modeList[0], pl->modeList[1]};
    pl->h_yLen.assign(pr->yLen, pr->yLen + ny);
    pl->h_zLen.assign(pr->zLen, pr->zLen + nz);
    pl->h_freqs.assign(pr->freqs, pr->freqs + pr->nFreq);
    std::vector<double> yNode(ny + 1), zNode0(nz + 1), zNode(nz + 1);
    yNode[0] = 0; zNode0[0] = 0;
    for (int j = 0; j < ny; ++j) yNode[j + 1] = yNode[j] + pr->yLen[j];
    for (int k = 0; k < nz; ++k) zNode0[k + 1] = zNode0[k] + pr->zLen[k];
    for (auto& v : yNode) v -= pr->origin[0];
    for (int k = 0; k <= nz; ++k) zNode[k] = zNode0[k] - pr->origin[1];
    // receiver row (mt2DTE.jl:65-67)
    int zid = -1;
    for (int k = 0; k <= nz; ++k) if (std::fabs(zNode[k] - pr->rxLoc[1]) < 0.1) { zid = k; break; }
    if (zid < 0 || zid >= nz) { delete pl; return kErrArg; }
    M.zid = zid;
    std::vector<double> yCen(ny);
    for (int j = 0; j < ny; ++j) yCen[j] = 0.5 * (yNode[j] + yNode[j + 1]);
    std::vector<int> fid(pr->nRx), iL(pr->nRx), iR(pr->nRx), tjL(pr->nRx), tjR(pr->nRx);
    std::vector<double> d1(pr->nRx), d2(pr->nRx), wL(pr->nRx), wR(pr->nRx), twL(pr->nRx), twR(pr->nRx);
    for (int r = 0; r < pr->nRx; ++r) {
        double y = pr->rxLoc[2 * r];
        int id = -1;
        for (int j = 0; j <= ny; ++j) if (yNode[j] > y) { id = j; break; }
        if (id <= 0) { delete pl; return kErrArg; }       // "receiver location seems to be out of range"
        fid[r] = id; d1[r] = y - yNode[id - 1]; d2[r] = yNode[id] - y;
        linear_interp(y, yNode, iL[r], iR[r], wL[r], wR[r]);
        linear_interp(y, yCen, tjL[r], tjR[r], twL[r], twR[r]);
    }
    // data layout: full slot ((f*nRx + r)*nComp + c), one per DataComp entry, rows must be sorted (freq, rx, comp).  Rho / phase
    // plans (nComp = nModes): dtID = 2 mi + 1 (rho_a) or 2 mi + 2 (phase), real obsData; the slot keeps the observed pair and both
    // weights (0 where a row is absent) and a packed row maps to 2 slot + part of the real view of the full arrays
    std::vector<double> wdFull(pl->nFull, 0.0), wpFull(dataKind ? pl->nFull : 0, 0.0);
    std::vector<cplx> obsFull(pl->nFull, mk(0.0, 0.0));
    pl->h_packed2full.resize(pr->nData);
    const long nDt = dataKind ? 2 * pr->nComp : pr->nComp;
    long prev = -1;
    for (int i = 0; i < pr->nData; ++i) {
        long f = pr->freqID[i] - 1, r = pr->rxID[i] - 1, c = pr->dtID[i] - 1;
        if (f < 0 || f >= pr->nFreq || r < 0 || r >= pr->nRx || c < 0 || c >= nDt) { delete pl; return kErrArg; }
        const long ci = dataKind ? c / 2 : c, part = dataKind ? c % 2 : 0;     // DataComp entry (rho / phase: its mode)
        const long slot = (f * pr->nRx + r) * pl->nComp + ci;
        const long full = dataKind ? 2 * slot + part : slot;
        if (full <= prev) {
            fprintf(stderr, "[hmcmt_b200] data rows must be sorted by (freq, rx, comp) without duplicates\n");
            delete pl;
            return kErrArg;
        }
        prev = full;
        pl->h_packed2full[i] = (int)full;
        const double w = 1.0 / std::fabs(pr->dataErr[i]);
        if (!dataKind) {
            wdFull[slot] = w;
            obsFull[slot] = mk(pr->obsData[2 * i], pr->obsData[2 * i + 1]);
        } else if (part == 0) {
            wdFull[slot] = w;
            obsFull[slot].x = pr->obsData[i];
        } else {
            wpFull[slot] = w;
            obsFull[slot].y = pr->obsData[i];
        }
    }
    std::vector<int> cell2act(M.nCell, -1);
    for (int a = 0; a < pr->nAC; ++a) {
        int c = pr->activeIdx[a];
        if (c < 0 || c >= M.nCell) { delete pl; return kErrArg; }
        cell2act[c] = a;
    }
    int rc = kOk;
    auto ok = [&](int r) { if (r && !rc) rc = r; };
    ok(pl->yLen.upload(pr->yLen, ny)); ok(pl->zLen.upload(pr->zLen, nz)); ok(pl->zNode.upload(zNode0.data(), nz + 1));
    ok(pl->freqs.upload(pr->freqs, pr->nFreq));
    ok(pl->fid.upload(fid.data(), pr->nRx)); ok(pl->iL.upload(iL.data(), pr->nRx)); ok(pl->iR.upload(iR.data(), pr->nRx));
    ok(pl->fdy1.upload(d1.data(), pr->nRx)); ok(pl->fdy2.upload(d2.data(), pr->nRx));
    ok(pl->wL.upload(wL.data(), pr->nRx)); ok(pl->wR.upload(wR.data(), pr->nRx));
    ok(pl->tjL.upload(tjL.data(), pr->nRx)); ok(pl->tjR.upload(tjR.data(), pr->nRx));
    ok(pl->twL.upload(twL.data(), pr->nRx)); ok(pl->twR.upload(twR.data(), pr->nRx));
    ok(pl->cell2act.upload(cell2act.data(), M.nCell)); ok(pl->act2cell.upload(pr->activeIdx, pr->nAC));
    ok(pl->bg.upload(pr->bgModel, M.nCell));
    ok(pl->wmPtr.upload(pr->wmRowPtr, pr->nAC + 1));
    int nnzWm = pr->wmRowPtr[pr->nAC];
    ok(pl->wmIdx.upload(pr->wmColIdx, nnzWm)); ok(pl->wmVal.upload(pr->wmVal, nnzWm));
    ok(pl->wd.upload(wdFull.data(), pl->nFull)); ok(pl->obs.upload(obsFull.data(), pl->nFull));
    ok(pl->wdPha.upload(wpFull.data(), wpFull.size()));
    ok(pl->packed2full.upload(pl->h_packed2full.data(), pr->nData));
    {
        std::vector<int> f2p((dataKind ? 2 : 1) * (size_t)pl->nFull, -1);
        for (int i = 0; i < pr->nData; ++i) f2p[pl->h_packed2full[i]] = i;
        ok(pl->full2packed.upload(f2p.data(), f2p.size()));
    }
    const size_t nCh = pl->nChains, nSys = pl->nSys, N = M.N;
    ok(pl->m.alloc(nCh * pr->nAC)); ok(pl->p.alloc(nCh * pr->nAC)); ok(pl->mref.alloc(nCh * pr->nAC));
    ok(pl->curM.alloc(nCh * pr->nAC)); ok(pl->curP.alloc(nCh * pr->nAC)); ok(pl->zmom.alloc(nCh * pr->nAC)); ok(pl->driftPart.alloc(nCh * 128));
    ok(pl->sigma.alloc(nCh * M.nCell)); ok(pl->meanSig.alloc(nCh * nz));
    ok(pl->planes.alloc(nCh * pl->nModes * 4 * N));
    ok(pl->bc.alloc(nSys * M.nb)); ok(pl->bcs.alloc(nSys * M.nb));
    ok(pl->rhs.alloc(nSys * N)); ok(pl->x.alloc(nSys * N)); ok(pl->lam.alloc(nSys * N));
    ok(pl->F.alloc(nSys * M.nNode)); ok(pl->Lam.alloc(nSys * M.nNode));
    ok(pl->srows.alloc(nSys * 2 * (ny + 1))); ok(pl->qrow.alloc(nSys * ny));
    ok(pl->scratch.alloc(nSys * 3 * prof_stride(nz)));
    ok(pl->Gpart.alloc(nSys * M.nCell)); ok(pl->phiPart.alloc(nSys)); ok(pl->phi.alloc(nCh));
    ok(pl->gsig.alloc(nCh * pr->nAC)); ok(pl->gdata.alloc(nCh * pr->nAC)); ok(pl->gtotal.alloc(nCh * pr->nAC)); ok(pl->xbuf.alloc((size_t)nCh * (pl->nAC + 1))); ok(pl->energies.alloc(nCh * 2));
    ok(pl->chainScal.alloc(nCh * 4));
    ok(pl->predFull.alloc(nCh * pl->nFull)); ok(pl->respFull.alloc(nCh * pl->nFull)); ok(pl->vin.alloc(nCh * pl->nFull)); ok(pl->predPacked.alloc(nCh * pr->nData));
    ok(pl->panels.alloc(nSys * (size_t)pl->S * panel_doubles(pl->T)));
    ok(pl->ainvz.alloc(nSys * (size_t)pl->S * AZ)); ok(pl->zadj.alloc(nSys * (size_t)pl->S * 8));
    const size_t wexpN = split_scratch_entries(TS * pl->T);
    ok(pl->wexp.alloc(pl->dom.split ? nSys * wexpN : 0));
    ok(pl->conCols.alloc(nSys * contract_cols_out(ny, nz)));
    ok(pl->fwdJobs.alloc(nSys));
    ok(pl->status.alloc(nSys)); ok(pl->driftFlag.alloc(1)); ok(pl->Lsteps.alloc(nCh));
    ok(pl->sysDesc.alloc(nSys)); ok(pl->jobs.alloc(nSys));
    if (rc) { hmcmt_destroy(pl); return rc; }
    cudaMemset(pl->status.p, 0, sizeof(int) * nSys);
    cudaMemset(pl->driftFlag.p, 0, sizeof(int));
    cudaMemset(pl->m.p, 0, sizeof(double) * nCh * pr->nAC);
    cudaMemset(pl->p.p, 0, sizeof(double) * nCh * pr->nAC);
    cudaMemset(pl->mref.p, 0, sizeof(double) * nCh * pr->nAC);
    M.yLen = pl->yLen.p; M.zLen = pl->zLen.p; M.zNode = pl->zNode.p;
    pl->rx = RxDev{pr->nRx, pl->fid.p, pl->fdy1.p, pl->fdy2.p, pl->iL.p, pl->iR.p, pl->wL.p, pl->wR.p, pl->tjL.p, pl->tjR.p, pl->twL.p, pl->twR.p};
    // per-system descriptors
    std::vector<BandSys> sd(nSys);
    std::vector<SolveJob> jb(nSys), jfw(nSys);
    for (size_t s = 0; s < nSys; ++s) {
        int f = (int)(s % pl->nFreq);
        int t = (int)(s / pl->nFreq);
        int mi = t % pl->nModes, ch = t / pl->nModes;
        double* P = pl->planes.p + ((size_t)(ch * pl->nModes + mi) * 4) * N;
        BandSys& d = sd[s];
        d.dr = P; d.dm = P + N; d.e1 = P + 2 * N; d.e2 = P + 3 * N;
        d.omega = 2.0 * kPi * pr->freqs[f];
        d.band = nullptr;
        d.rhs = pl->rhs.p + s * N;
        d.panels[0] = pl->panels.p + s * (size_t)pl->S * panel_doubles(pl->T);
        d.panels[1] = d.panels[0] + (size_t)pl->steps0 * panel_doubles(pl->T);
        d.ainvz[0] = pl->ainvz.p + s * (size_t)pl->S * AZ;
        d.ainvz[1] = d.ainvz[0] + (size_t)pl->steps0 * AZ;
        d.wexp = pl->dom.split ? pl->wexp.p + s * wexpN : nullptr;
        d.x = pl->x.p + s * N;
        d.status = pl->status.p + s;
        SolveJob& j = jb[s];
        j.panels[0] = d.panels[0]; j.panels[1] = d.panels[1];
        j.ainvz[0] = d.ainvz[0]; j.ainvz[1] = d.ainvz[1];
        j.rhs = pl->lam.p + s * N; j.x = pl->lam.p + s * N;
        j.zbuf[0] = pl->zadj.p + s * (size_t)pl->S * 8;
        j.zbuf[1] = j.zbuf[0] + (size_t)pl->steps0 * 8;
        j.wexp = d.wexp;
        SolveJob& jf = jfw[s];
        jf = j;
        jf.rhs = nullptr; jf.x = d.x;
    }
    if (cudaMemcpy(pl->sysDesc.p, sd.data(), sizeof(BandSys) * nSys, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(pl->jobs.p, jb.data(), sizeof(SolveJob) * nSys, cudaMemcpyHostToDevice) != cudaSuccess ||
        (pl->fwdJobs.p && cudaMemcpy(pl->fwdJobs.p, jfw.data(), sizeof(SolveJob) * nSys, cudaMemcpyHostToDevice) != cudaSuccess)) {
        hmcmt_destroy(pl);
        return kErrCuda;
    }
    {
        // wide meshes: the receiver / contraction kernels stage whole node rows in shared memory
        const size_t rxSmem = (size_t)(6 * (M.ny + 1) + 3 * M.ny) * sizeof(cplx);
        // very deep meshes: one profile of the boundary kernel no longer fits the default 48 KB of dynamic shared memory
        const size_t bcSmem = (size_t)boundary_profiles_per_block(M.nz) * M.nz * 6 * sizeof(cplx);
        if (bcSmem > 227 * 1024) {
            fprintf(stderr, "[hmcmt_b200] nz = %d: the boundary kernel needs %zu bytes of shared memory per profile\n", M.nz, bcSmem);
            hmcmt_destroy(pl);
            return kErrArg;
        }
        if (bcSmem > 48 * 1024 && cudaFuncSetAttribute(k_boundary, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bcSmem) != cudaSuccess) {
            hmcmt_destroy(pl);
            return kErrCuda;
        }
        pl->conStaged = contract_cols_smem(M.ny, M.nz, 1) <= 200 * 1024 ? 1 : 0;
        const size_t cSmem = contract_cols_smem(M.ny, M.nz, pl->conStaged);
        if ((rxSmem > 48 * 1024 && cudaFuncSetAttribute(rx_kernel(pl), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rxSmem) != cudaSuccess) ||
            (cSmem > 48 * 1024 && cudaFuncSetAttribute(k_contract_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cSmem) != cudaSuccess)) {
            hmcmt_destroy(pl);
            return kErrArg;
        }
    }
    if (pl->useMf) {
        // nested-dissection multifrontal solver for all systems of the plan (one symbolic analysis, shared by every system)
        std::vector<std::vector<int>> sn;
        std::vector<mf::Entry> ent;
        mf::mf_order_grid(M.nl, M.nf, mf_leaf_size(), sn, mf_cross_size(), mf_push_size());
        mf::mf_grid_entries(M.nl, M.nf, ent);
        mf::Symbolic S;
        if (!mf::mf_symbolic(M.N, sn, ent, mf_small_front(), S)) { hmcmt_destroy(pl); return kErrArg; }
        int mrc = kOk;
        // two workspace slots per system: x and the adjoint lam of a gradient evaluation (gradient_range)
        pl->mfs = mf::Solver::create(std::move(S), pl->nSys, 2, 3 * (int64_t)M.N, &mrc);
        if (!pl->mfs) { hmcmt_destroy(pl); return mrc; }
        // rhs = -Aio bc (k_rhs) lives on the nodes next to the Dirichlet boundary, the adjoint sources (k_rx_adjoint) on the
        // two receiver node rows zid, zid + 1: with pruning the forward eliminations skip every subtree without such a node.
        // The receiver rows' pattern also gives the receiver path of gradient_range, so it exists with pruning off too.
        std::vector<unsigned char> nzR(M.N, 0), nzA(M.N, 0);
        for (int kn = 1; kn <= nz - 1; ++kn)
            for (int jn = 1; jn <= ny - 1; ++jn) {
                const int q = M.fastZ ? (jn - 1) * M.nf + (kn - 1) : (kn - 1) * M.nf + (jn - 1);
                if (jn == 1 || jn == ny - 1 || kn == 1 || kn == nz - 1) nzR[q] = 1;
                if (kn == M.zid || kn == M.zid + 1) nzA[q] = 1;
            }
        pl->patRx = pl->mfs->add_rhs_pattern(nzA);
        if (pl->patRx < 0) { hmcmt_destroy(pl); return kErrAlloc; }
        if (const char* e = std::getenv("HMCMT_MF_PRUNE"); !e || std::atoi(e)) {
            pl->patRhs = pl->mfs->add_rhs_pattern(nzR);
            pl->patAdj = pl->patRx;
            if (pl->patRhs < 0) { hmcmt_destroy(pl); return kErrAlloc; }
        }
        std::vector<mf::MtValSys> mv(nSys);
        for (size_t s = 0; s < nSys; ++s) { mv[s].planes = sd[s].dr; mv[s].omega = sd[s].omega; }
        if (pl->mfSys.upload(mv.data(), nSys) != kOk) { hmcmt_destroy(pl); return kErrAlloc; }
    }
    if (cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&pl->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&pl->evFork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&pl->evJoin, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&pl->evPre, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&pl->evRhs, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&pl->evA) != cudaSuccess || cudaEventCreate(&pl->evB) != cudaSuccess) {
        hmcmt_destroy(pl);
        return kErrCuda;
    }
    if (const char* e = std::getenv("HMCMT_GRAPH"); e && !std::atoi(e)) pl->graphState = -1;
    if (pl->useMf) {
        // groups of systems on their own streams (compute_step_grouped); HMCMT_GROUPS=1 keeps everything on the plan's stream
        const char* env = std::getenv("HMCMT_GROUPS");
        int G = env ? std::atoi(env) : kDefaultGroups;
        G = std::max(1, std::min(G, std::min(pl->nSys, 8)));
        for (int g = 0; G >= 2 && g < G; ++g) {
            cudaStream_t s = nullptr;
            cudaEvent_t e = nullptr;
            if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { hmcmt_destroy(pl); return kErrCuda; }
            pl->groupStreams.push_back(s);
            if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { hmcmt_destroy(pl); return kErrCuda; }
            pl->groupDone.push_back(e);
        }
    }
    *out = pl;
    return kOk;
}

int hmcmt_plan_create(const hmcmt_problem* pr, hmcmt_plan** out) { return plan_create(pr, out, 0); }
int hmcmt_plan_create_rho_phase(const hmcmt_problem* pr, hmcmt_plan** out) { return plan_create(pr, out, 1); }

void hmcmt_destroy(hmcmt_plan* pl) {
    if (!pl) return;
    cudaSetDevice(pl->device);
    if (pl->comm) {
        if (pl->stream) cudaStreamSynchronize(pl->stream);
        if (NcclApi* a = nccl_api()) a->commDestroy(pl->comm);
        pl->comm = nullptr;
    }
    if (pl->stream) { cudaStreamSynchronize(pl->stream); cudaStreamDestroy(pl->stream); }
    if (pl->side) { cudaStreamSynchronize(pl->side); cudaStreamDestroy(pl->side); }
    if (pl->graphExec) cudaGraphExecDestroy(pl->graphExec);
    for (cudaStream_t s : pl->groupStreams) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
    for (cudaEvent_t e : pl->groupDone) cudaEventDestroy(e);
    if (pl->evPre) cudaEventDestroy(pl->evPre);
    if (pl->evRhs) cudaEventDestroy(pl->evRhs);
    if (pl->evFork) cudaEventDestroy(pl->evFork);
    if (pl->evJoin) cudaEventDestroy(pl->evJoin);
    if (pl->evA) cudaEventDestroy(pl->evA);
    if (pl->evB) cudaEventDestroy(pl->evB);
    for (auto& e : pl->factorEvents) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    for (cudaEvent_t e : pl->factorMid) cudaEventDestroy(e);
    pl->yLen.release(); pl->zLen.release(); pl->zNode.release(); pl->freqs.release(); pl->fdy1.release(); pl->fdy2.release();
    pl->wL.release(); pl->wR.release(); pl->twL.release(); pl->twR.release(); pl->tjL.release(); pl->tjR.release(); pl->bg.release(); pl->wmVal.release(); pl->wd.release(); pl->wdPha.release(); pl->m.release(); pl->p.release();
    pl->mref.release(); pl->sigma.release(); pl->meanSig.release(); pl->planes.release(); pl->Gpart.release(); pl->phiPart.release();
    pl->phi.release(); pl->gsig.release(); pl->gdata.release(); pl->gtotal.release(); pl->energies.release(); pl->panels.release(); pl->curM.release();
    pl->curP.release(); pl->driftPart.release(); pl->chainScal.release(); pl->zmom.release(); pl->fid.release(); pl->iL.release(); pl->iR.release();
    pl->cell2act.release(); pl->act2cell.release(); pl->wmPtr.release(); pl->wmIdx.release(); pl->status.release();
    pl->driftFlag.release(); pl->packed2full.release(); pl->full2packed.release(); pl->Lsteps.release(); pl->obs.release(); pl->bc.release(); pl->bcs.release();
    pl->rhs.release(); pl->x.release(); pl->F.release(); pl->lam.release(); pl->Lam.release(); pl->srows.release(); pl->qrow.release();
    pl->scratch.release(); pl->predFull.release(); pl->ainvz.release(); pl->zadj.release(); pl->vin.release();
    pl->predPacked.release(); pl->conCols.release(); pl->dbc.release(); pl->jvFull.release(); pl->dsigA.release(); pl->gnBuf.release(); pl->gnVec.release(); pl->gnPart.release(); pl->gnS.release(); pl->gnE.release(); pl->gnAct.release(); pl->gnI.release(); pl->xbuf.release(); pl->wexp.release(); pl->respFull.release(); pl->gradK.release(); pl->Lband.release(); pl->massBuf.release(); pl->massStatus.release(); delete pl->massSolver; pl->massSolver = nullptr; pl->mfSys.release(); delete pl->mfs; pl->mfs = nullptr; pl->fwdJobs.release(); pl->sysDesc.release(); pl->jobs.release();
    if (pl->pin) cudaFreeHost(pl->pin);
    delete pl;
}

int64_t hmcmt_plan_info(const hmcmt_plan* pl, int what) {
    if (!pl) return -1;
    switch (what) {
        case 0: return pl->M.N;
        case 1: return pl->M.nNode;
        case 2: return pl->M.nCell;
        case 3: return pl->M.nb;
        case 4: return pl->b;
        case 5: return pl->T;                                      // 0: multifrontal solver
        case 6: return pl->S;
        case 7: return pl->nSysPerChain;
        case 8: return pl->M.zid;
        case 9: return pl->useMf ? pl->mfs->factor_doubles() * 8 : (int64_t)pl->S * (panel_doubles(pl->T) * 8 + AZ * 16);
        case 10: return pl->launches;
        case 11: return pl->useMf ? 1 : 0;
        case 12: return pl->useMf ? (int64_t)pl->mfs->factor_flops() : (int64_t)(4.0 * pl->M.N * (double)pl->b * pl->b);
        case 13: return pl->dom.split;
        default: return -1;
    }
}

int hmcmt_sync(hmcmt_plan* pl) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return kOk;
}
int hmcmt_set_mass_matrix(hmcmt_plan* pl, int32_t kind) {
    if (!pl || kind < 0 || kind > 1) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    if (kind == 0) { pl->massOn = false; return kOk; }
    if (pl->massSolver) { pl->massOn = true; return kOk; }
    const int n = pl->nAC;
    std::vector<int> ptr(n + 1), idx;
    std::vector<double> val;
    HMCMT_CUDA_TRY(cudaMemcpy(ptr.data(), pl->wmPtr.p, sizeof(int) * (n + 1), cudaMemcpyDeviceToHost));
    idx.resize(ptr[n]); val.resize(ptr[n]);
    HMCMT_CUDA_TRY(cudaMemcpy(idx.data(), pl->wmIdx.p, sizeof(int) * ptr[n], cudaMemcpyDeviceToHost));
    HMCMT_CUDA_TRY(cudaMemcpy(val.data(), pl->wmVal.p, sizeof(double) * ptr[n], cudaMemcpyDeviceToHost));
    // (1) invM p = Wm^{-1} p : multifrontal factorisation of the sparse SPD matrix, nested dissection of its graph
    std::vector<mf::Entry> ent;
    std::vector<int> aptr(n + 1, 0);
    int bw = 0;
    for (int a = 0; a < n; ++a)
        for (int q = ptr[a]; q < ptr[a + 1]; ++q) {
            const int j = idx[q];
            if (j > a) continue;
            ent.push_back(mf::Entry{a, j, q});
            bw = std::max(bw, a - j);
            if (j != a) { ++aptr[a + 1]; ++aptr[j + 1]; }
        }
    for (int a = 0; a < n; ++a) aptr[a + 1] += aptr[a];
    std::vector<int> adj(aptr[n]), at(aptr.begin(), aptr.end() - 1);
    for (const mf::Entry& e : ent)
        if (e.row != e.col) { adj[at[e.row]++] = e.col; adj[at[e.col]++] = e.row; }
    std::vector<std::vector<int>> sn;
    mf::mf_order_graph(n, aptr, adj, mf_leaf_size(), sn);
    mf::Symbolic S;
    if (!mf::mf_symbolic(n, sn, ent, mf_small_front(), S)) return kErrArg;
    int rc = kOk;
    pl->massSolver = mf::Solver::create(std::move(S), 1, pl->nChains, (int64_t)ptr[n], &rc);
    if (!pl->massSolver) return rc;
    {
        std::vector<cplx> cv(ptr[n]);
        for (int q = 0; q < ptr[n]; ++q) cv[q] = mk(val[q], 0.0);
        HMCMT_CUDA_TRY(cudaMemcpy(pl->massSolver->vals(), cv.data(), sizeof(cplx) * cv.size(), cudaMemcpyHostToDevice));
    }
    if ((rc = pl->massStatus.alloc(1)) != kOk) return rc;
    HMCMT_CUDA_TRY(cudaMemset(pl->massStatus.p, 0, sizeof(int)));
    rc = pl->massSolver->factor(pl->stream, pl->massStatus.p, &pl->launches);
    if (rc) return rc;
    int hst = 0;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(&hst, pl->massStatus.p, sizeof(int), cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    if (hst) return hst;
    // (2) sqrtM = the lower Cholesky factor of Wm in the NATURAL ordering (decomp.L of the reference's dense cholesky): Wm is
    //     banded there (half-bandwidth = cells per mesh row), so is L, and the band never fills outside itself
    std::vector<double> Lb((size_t)n * (bw + 1), 0.0);
    for (int a = 0; a < n; ++a)
        for (int q = ptr[a]; q < ptr[a + 1]; ++q)
            if (idx[q] <= a) Lb[(size_t)a * (bw + 1) + (a - idx[q])] = val[q];
    for (int j = 0; j < n; ++j) {
        double* rj = Lb.data() + (size_t)j * (bw + 1);
        double d = rj[0];
        for (int k = std::max(0, j - bw); k < j; ++k) d -= rj[j - k] * rj[j - k];
        if (!(d > 0.0)) return kErrNotPosDef;
        d = std::sqrt(d);
        rj[0] = d;
        for (int i = j + 1; i <= std::min(n - 1, j + bw); ++i) {
            double* ri = Lb.data() + (size_t)i * (bw + 1);
            double v = ri[i - j];
            for (int k = std::max(0, i - bw); k < j; ++k) v -= ri[i - k] * rj[j - k];
            ri[i - j] = v / d;
        }
    }
    if ((rc = pl->Lband.upload(Lb.data(), Lb.size())) != kOk) return rc;
    if ((rc = pl->gradK.alloc((size_t)pl->nChains * n)) != kOk) return rc;
    if ((rc = pl->massBuf.alloc((size_t)pl->nChains * n)) != kOk) return rc;
    pl->massBw = bw;
    pl->massOn = true;
    return kOk;
}

int hmcmt_status(hmcmt_plan* pl) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    return check_status(pl);
}
int hmcmt_set_response_kind(hmcmt_plan* pl, int32_t kind) {
    if (!pl || kind < 0 || kind > 1) return kErrArg;
    pl->respKind = kind;
    return kOk;
}
int hmcmt_get_responses(hmcmt_plan* pl, double* out) {
    if (!pl || !out || !pl->haveForward) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    const cplx* src = (pl->respKind == 1 || pl->dataKind == 1) ? pl->respFull.p : pl->predFull.p;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(out, src, sizeof(cplx) * (size_t)pl->nChains * pl->nFull, cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return kOk;
}
int hmcmt_timer_start(hmcmt_plan* pl) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaEventRecord(pl->evA, pl->stream));
    return kOk;
}
int hmcmt_timer_stop(hmcmt_plan* pl, float* ms) {
    if (!pl || !ms) return kErrArg;
    HMCMT_CUDA_TRY(cudaEventRecord(pl->evB, pl->stream));
    HMCMT_CUDA_TRY(cudaEventSynchronize(pl->evB));
    HMCMT_CUDA_TRY(cudaEventElapsedTime(ms, pl->evA, pl->evB));
    return kOk;
}
int hmcmt_kernel_time_split(hmcmt_plan* pl, float* factor_only_ms, float* forward_solve_ms) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    float a = 0.f, b = 0.f;
    for (size_t i = 0; i < pl->factorEventsUsed; ++i) {
        float ms = 0.f;
        HMCMT_CUDA_TRY(cudaEventElapsedTime(&ms, pl->factorEvents[i].first, pl->factorMid[i]));
        a += ms;
        HMCMT_CUDA_TRY(cudaEventElapsedTime(&ms, pl->factorMid[i], pl->factorEvents[i].second));
        b += ms;
    }
    if (factor_only_ms) *factor_only_ms = a;
    if (forward_solve_ms) *forward_solve_ms = b;
    return kOk;
}
int hmcmt_kernel_time(hmcmt_plan* pl, int reset, float* factor_ms, int64_t* factor_launches) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    float tot = 0.f;
    for (size_t i = 0; i < pl->factorEventsUsed; ++i) {
        float ms = 0.f;
        HMCMT_CUDA_TRY(cudaEventElapsedTime(&ms, pl->factorEvents[i].first, pl->factorEvents[i].second));
        tot += ms;
    }
    if (factor_ms) *factor_ms = tot;
    if (factor_launches) *factor_launches = (int64_t)pl->factorEventsUsed;
    // timing is opt-in: reset = 1 switches it on (the evaluations then run un-grouped on the plan's stream so that the events
    // bracket the factorisation alone), reset = -1 switches it off again
    if (reset) { pl->factorEventsUsed = 0; pl->timeFactor = reset > 0; }
    return kOk;
}

static int upload_model(hmcmt_plan* pl, const double* m) {
    size_t bytes = sizeof(double) * (size_t)pl->nChains * pl->nAC;
    int rc = ensure_pin(pl, std::max(bytes, (size_t)1 << 20));
    if (rc) return rc;
    std::memcpy(pl->pin, m, bytes);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->m.p, pl->pin, bytes, cudaMemcpyHostToDevice, pl->stream));
    return kOk;
}
// bytes of one packed datum: complex impedance, or one real rho_a / phase row
static size_t datum_bytes(const hmcmt_plan* pl) { return pl->dataKind ? sizeof(double) : sizeof(cplx); }
// predictions of the last evaluation into predPacked [nChains][nData] (complex, or real for rho / phase plans)
static int pack_pred(hmcmt_plan* pl) {
    const dim3 grid((pl->nData + 255) / 256, pl->nChains);
    if (pl->dataKind)
        k_pack_pred_real<<<grid, 256, 0, pl->stream>>>(pl->nData, pl->nFull, pl->packed2full.p, reinterpret_cast<const double*>(pl->respFull.p),
                                                       reinterpret_cast<double*>(pl->predPacked.p));
    else
        k_pack_pred<<<grid, 256, 0, pl->stream>>>(pl->nData, pl->nFull, pl->packed2full.p, pl->predFull.p, pl->predPacked.p);
    LAUNCH_CHECK(pl);
    return kOk;
}
static int download_pred(hmcmt_plan* pl, double* pred) {
    int rc = pack_pred(pl);
    if (rc) return rc;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pred, pl->predPacked.p, datum_bytes(pl) * (size_t)pl->nChains * pl->nData, cudaMemcpyDeviceToHost, pl->stream));
    return kOk;
}

static int forward_common(hmcmt_plan* pl, double* pred, double* exTE, double* hxTM);

int hmcmt_forward(hmcmt_plan* pl, const double* m, double* pred, double* exTE, double* hxTM) {
    if (!pl || !m) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    pl->sigmaDirect = false;
    int rc = upload_model(pl, m);
    if (rc) return rc;
    return forward_common(pl, pred, exTE, hxTM);
}

int hmcmt_forward_sigma(hmcmt_plan* pl, const double* sigma, double* pred, double* exTE, double* hxTM) {
    if (!pl || !sigma) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    pl->sigmaDirect = true;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->sigma.p, sigma, sizeof(double) * (size_t)pl->nChains * pl->M.nCell, cudaMemcpyHostToDevice, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return forward_common(pl, pred, exTE, hxTM);
}

static int forward_common(hmcmt_plan* pl, double* pred, double* exTE, double* hxTM) {
    int rc = compute_step(pl, false, nullptr);
    if (rc) return rc;
    if (pred) { rc = download_pred(pl, pred); if (rc) return rc; }
    const MeshDev& M = pl->M;
    for (int ch = 0; ch < pl->nChains; ++ch)
        for (int mi = 0; mi < pl->nModes; ++mi) {
            double* dst = pl->modeList[mi] == 0 ? exTE : hxTM;
            if (!dst) continue;
            size_t sys0 = ((size_t)ch * pl->nModes + mi) * pl->nFreq;
            HMCMT_CUDA_TRY(cudaMemcpyAsync(dst + 2 * (size_t)ch * pl->nFreq * M.nNode, pl->F.p + sys0 * M.nNode,
                                           sizeof(cplx) * (size_t)pl->nFreq * M.nNode, cudaMemcpyDeviceToHost, pl->stream));
        }
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return check_status(pl);
}

int hmcmt_jtvec(hmcmt_plan* pl, const double* v, double* gsig) {
    if (!pl || !v || !gsig) return kErrArg;
    if (!pl->haveForward) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    // scatter the packed data vector into the full layout (rho / phase plans: the real rows into the (v_rho, v_phi) pairs)
    std::vector<cplx> full((size_t)pl->nChains * pl->nFull, mk(0.0, 0.0));
    double* fullD = reinterpret_cast<double*>(full.data());
    for (int ch = 0; ch < pl->nChains; ++ch)
        for (int i = 0; i < pl->nData; ++i) {
            const size_t src = (size_t)ch * pl->nData + i;
            if (pl->dataKind) fullD[(size_t)ch * 2 * pl->nFull + pl->h_packed2full[i]] = v[src];
            else full[(size_t)ch * pl->nFull + pl->h_packed2full[i]] = mk(v[2 * src], v[2 * src + 1]);
        }
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->vin.p, full.data(), sizeof(cplx) * full.size(), cudaMemcpyHostToDevice, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    // the factors, fields and boundary values of the last forward evaluation are still on the device (the reference's AinvTE /
    // AinvTM, compJacTMatVec.jl:220-224): only the adjoint sources for v, one solve per system and the contraction run here
    int rc = kOk;
    if (!pl->haveSens) rc = launch_sens_side(pl);
    if (rc) return rc;
    rc = rx_phase(pl, true, pl->vin.p);
    if (rc) return rc;
    rc = adjoint_phase(pl);
    if (rc) return rc;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(gsig, pl->gsig.p, sizeof(double) * (size_t)pl->nChains * pl->nAC, cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return check_status(pl);
}

int hmcmt_jacobian(hmcmt_plan* pl, double* J) {
    if (!pl || !J || !pl->haveForward) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    const MeshDev& M = pl->M;
    cudaStream_t st = pl->stream;
    const size_t nJ = (size_t)pl->nChains * pl->nData * pl->nAC * (pl->dataKind ? 1 : 2);
    DevBuf<double> dJ;
    int rc = dJ.alloc(nJ);
    if (rc) return rc;
    HMCMT_CUDA_TRY(cudaMemsetAsync(dJ.p, 0, nJ * sizeof(double), st));
    if (!pl->haveSens) rc = launch_sens_side(pl);
    // groups of components that share no system, one set of 2 nRx passes each: all components, or (tipper plans) the impedance
    // components and then the tipper
    struct Group { unsigned mask; int2 comp; };
    std::vector<Group> groups;
    const CompMap& cm = pl->cm;
    if (!pl->tipper) groups.push_back(Group{(1u << pl->nComp) - 1u, make_int2(0, 1)});
    else if (cm.zc[0] >= 0 || cm.zc[1] >= 0)
        groups.push_back(Group{(cm.zc[0] >= 0 ? 1u << cm.zc[0] : 0u) | (cm.zc[1] >= 0 ? 1u << cm.zc[1] : 0u), make_int2(cm.zc[0], cm.zc[1])});
    if (pl->tipper) groups.push_back(Group{1u << cm.tc, make_int2(cm.tmi == 0 ? cm.tc : -1, cm.tmi == 1 ? cm.tc : -1)});
    for (const Group& grp : groups)
        for (int r = 0; r < pl->nRx && rc == kOk; ++r)
            for (int part = 0; part < 2 && rc == kOk; ++part) {
                k_jac_vin<<<dim3((pl->nFull + 255) / 256, pl->nChains), 256, 0, st>>>(pl->nFull, pl->nRx, pl->nComp, grp.mask, r,
                                                                                     part == 0 ? mk(1.0, 0.0) : mk(0.0, 1.0), pl->vin.p);
                ++pl->launches;
                rc = rx_phase(pl, true, pl->vin.p);
                if (rc == kOk) rc = adjoint_phase(pl, false);
                if (rc != kOk) break;
                const dim3 grid((pl->nAC + 255) / 256, pl->nSys);
                if (pl->dataKind)
                    k_jac_rows_real<<<grid, 256, 0, st>>>(pl->nAC, M.nCell, pl->nFreq, pl->nRx, pl->nModes, pl->nData, r, part, pl->act2cell.p,
                                                          pl->full2packed.p, pl->Gpart.p, dJ.p);
                else
                    k_jac_rows<<<grid, 256, 0, st>>>(pl->nAC, M.nCell, pl->nFreq, pl->nRx, pl->nModes, pl->nComp, grp.comp, pl->nData, r,
                                                     part, pl->act2cell.p, pl->full2packed.p, pl->Gpart.p, dJ.p);
                ++pl->launches;
            }
    if (rc == kOk && cudaGetLastError() != cudaSuccess) rc = kErrCuda;
    if (rc == kOk && cudaMemcpyAsync(J, dJ.p, nJ * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = kErrCuda;
    if (cudaStreamSynchronize(st) != cudaSuccess && rc == kOk) rc = kErrCuda;
    dJ.release();
    if (rc) return rc;
    // the adjoint passes overwrote the responses / misfit of the data residual: restore them for later calls
    rc = rx_phase(pl, false, nullptr);
    if (rc) return rc;
    return check_status(pl);
}

// the tangent buffers, allocated on first use so that plans that never ask for J v carry none of them
static int ensure_tangent(hmcmt_plan* pl) {
    if (pl->jvFull.p) return kOk;
    const MeshDev& M = pl->M;
    int rc;
    if ((rc = pl->dbc.alloc((size_t)pl->nSys * M.nb)) || (rc = pl->dsigA.alloc((size_t)pl->nChains * pl->nAC))) return rc;
    const size_t smem = (size_t)(6 * (M.ny + 1) + 2 * M.ny) * sizeof(cplx);
    auto k = pl->dataKind ? k_rx_tangent<true, false> : pl->tipper ? k_rx_tangent<false, true> : k_rx_tangent<false, false>;
    if (smem > 48 * 1024) HMCMT_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return pl->jvFull.alloc((size_t)pl->nChains * pl->nFull);
}

// jvFull <- J dsigA for the resident state: dbc = dBC dsig, the tangent right-hand side, one solve per system with the resident
// factors (the multifrontal path back-substitutes only the receiver path: only rows zid, zid + 1 are read), the tangent field
// on those rows and the tangent receiver functional.  Overwrites lam and the receiver rows of Lam.
static int jvec_device(hmcmt_plan* pl) {
    const MeshDev& M = pl->M;
    cudaStream_t st = pl->stream;
    const int nSys = pl->nSys;
    int rc = kOk;
    if (!pl->haveSens && (rc = launch_sens_side(pl))) return rc;
    HMCMT_CUDA_TRY(cudaStreamWaitEvent(st, pl->evJoin, 0));
    k_bc_tangent<<<dim3((M.ny + 1 + 127) / 128, nSys), 128, 0, st>>>(M, pl->sm, pl->freqs.p, pl->cell2act.p, pl->dsigA.p, pl->nAC,
                                                                     pl->scratch.p, pl->dbc.p);
    LAUNCH_CHECK(pl);
    k_tangent_rhs<<<dim3((M.N + 255) / 256, nSys), 256, 0, st>>>(M, pl->sm, pl->freqs.p, pl->sigma.p, pl->cell2act.p, pl->dsigA.p, pl->nAC,
                                                                 pl->F.p, pl->bcs.p, pl->dbc.p, pl->lam.p);
    LAUNCH_CHECK(pl);
    if (pl->useMf) {
        if ((rc = pl->mfs->forward_slot(st, 0, pl->lam.p, M.N, &pl->launches, 0, nSys, 0)) ||
            (rc = pl->mfs->backward_slot(st, 0, pl->lam.p, M.N, &pl->launches, 0, nSys, pl->patRx)))
            return rc;
    } else {
        if ((rc = launch_solve(st, pl->T, pl->jobs.p, nSys, pl->dom))) return rc;
        pl->launches += pl->dom.split ? 3 : 1;
    }
    const int rx0 = M.zid * (M.ny + 1), rx1 = (M.zid + 2) * (M.ny + 1);
    k_node_field<<<dim3((rx1 - rx0 + 255) / 256, nSys), 256, 0, st>>>(M, pl->lam.p, pl->dbc.p, pl->Lam.p, 0, rx0, rx1);
    LAUNCH_CHECK(pl);
    const size_t smem = (size_t)(6 * (M.ny + 1) + 2 * M.ny) * sizeof(cplx);
    auto k = pl->dataKind ? k_rx_tangent<true, false> : pl->tipper ? k_rx_tangent<false, true> : k_rx_tangent<false, false>;
    k<<<nSys, kRxThreads, smem, st>>>(M, pl->rx, pl->sm, pl->cm, pl->freqs.p, pl->sigma.p, pl->cell2act.p, pl->dsigA.p, pl->nAC, pl->F.p,
                                      pl->Lam.p, pl->jvFull.p);
    LAUNCH_CHECK(pl);
    return kOk;
}

int hmcmt_jvec(hmcmt_plan* pl, const double* dsig, double* jv) {
    if (!pl || !dsig || !jv || !pl->haveForward) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    int rc = ensure_tangent(pl);
    if (rc) return rc;
    cudaStream_t st = pl->stream;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->dsigA.p, dsig, sizeof(double) * (size_t)pl->nChains * pl->nAC, cudaMemcpyHostToDevice, st));
    if ((rc = jvec_device(pl))) return rc;
    // packed order through the prediction packers, staged in vin (adjoint scratch: the predictions stay as they are)
    const dim3 grid((pl->nData + 255) / 256, pl->nChains);
    if (pl->dataKind)
        k_pack_pred_real<<<grid, 256, 0, st>>>(pl->nData, pl->nFull, pl->packed2full.p, reinterpret_cast<const double*>(pl->jvFull.p),
                                               reinterpret_cast<double*>(pl->vin.p));
    else
        k_pack_pred<<<grid, 256, 0, st>>>(pl->nData, pl->nFull, pl->packed2full.p, pl->jvFull.p, pl->vin.p);
    LAUNCH_CHECK(pl);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(jv, pl->vin.p, datum_bytes(pl) * (size_t)pl->nChains * pl->nData, cudaMemcpyDeviceToHost, st));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(st));
    return check_status(pl);
}

// The Gauss-Newton product D Re(J^H Wd^2 J) D v for the resident state, v [nChains][nAC] in device memory, up to the per-system
// partials in Gpart: the caller reduces them over the systems (k_reduce_grad for hmcmt_gn_hessvec, k_reduce_gn for the CG of
// hmcmt_gauss_newton).  Needs ensure_tangent.
static int gn_partials(hmcmt_plan* pl, const double* v) {
    const MeshDev& M = pl->M;
    cudaStream_t st = pl->stream;
    k_sigma_scale<<<dim3((pl->nAC + 255) / 256, pl->nChains), 256, 0, st>>>(pl->nAC, M.nCell, pl->act2cell.p, pl->sigma.p, v, pl->dsigA.p);
    LAUNCH_CHECK(pl);
    int rc;
    if ((rc = jvec_device(pl))) return rc;
    k_gn_weight<<<dim3((pl->nFull + 255) / 256, pl->nChains), 256, 0, st>>>(pl->nFull, pl->dataKind, pl->wd.p, pl->wdPha.p, pl->jvFull.p,
                                                                            pl->vin.p);
    LAUNCH_CHECK(pl);
    // J^T of the weighted tangent through the adjoint machinery (the receiver functional recomputes the same predictions and
    // misfit from the unchanged fields)
    if ((rc = rx_phase(pl, true, pl->vin.p))) return rc;
    return adjoint_phase(pl, false);
}

int hmcmt_gn_hessvec(hmcmt_plan* pl, const double* v, int32_t with_prior, double* hv) {
    if (!pl || !v || !hv || !pl->haveForward) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    int rc = ensure_tangent(pl);
    if (rc) return rc;
    const MeshDev& M = pl->M;
    cudaStream_t st = pl->stream;
    const size_t nA = (size_t)pl->nChains * pl->nAC;
    if (!pl->gnBuf.p) {
        if ((rc = pl->gnBuf.alloc(5 * nA))) return rc;
        HMCMT_CUDA_TRY(cudaMemsetAsync(pl->gnBuf.p + nA, 0, sizeof(double) * nA, st));      // m_ref = 0 of the prior term
    }
    double *vD = pl->gnBuf.p, *zero = vD + nA, *gs = zero + nA, *gd = gs + nA, *gt = gd + nA;
    HMCMT_CUDA_TRY(cudaMemcpyAsync(vD, v, sizeof(double) * nA, cudaMemcpyHostToDevice, st));
    if ((rc = gn_partials(pl, vD))) return rc;
    // the chain rule and prior term of the gradient's reduction with (m, m_ref) = (v, 0)
    k_reduce_grad<<<dim3((pl->nAC + 255) / 256, pl->nChains), 256, 0, st>>>(pl->nAC, M.nCell, pl->nSysPerChain, pl->act2cell.p, pl->Gpart.p,
                                                                            vD, zero, pl->wmPtr.p, pl->wmIdx.p, pl->wmVal.p, pl->beta,
                                                                            pl->sigma.p, gs, gd, gt);
    LAUNCH_CHECK(pl);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(hv, with_prior ? gt : gd, sizeof(double) * nA, cudaMemcpyDeviceToHost, st));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(st));
    return check_status(pl);
}

static int forward_gradient_impl(hmcmt_plan* pl, const double* m, double* pred, double* phid, double* grad, bool withPrior);
int hmcmt_forward_gradient(hmcmt_plan* pl, const double* m, double* pred, double* phid, double* grad) {
    return forward_gradient_impl(pl, m, pred, phid, grad, false);
}
int hmcmt_forward_gradient_total(hmcmt_plan* pl, const double* m, double* pred, double* phid, double* grad) {
    return forward_gradient_impl(pl, m, pred, phid, grad, true);
}
static int forward_gradient_impl(hmcmt_plan* pl, const double* m, double* pred, double* phid, double* grad, bool withPrior) {
    if (!pl || !m) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    pl->sigmaDirect = false;
    // One pinned staging buffer for everything that crosses the bus: [model up | pred | phi | gradient | error flags down], one
    // stream synchronisation per call (device-to-host copies into pageable caller memory would be staged by the driver one by one).
    const size_t nM = sizeof(double) * (size_t)pl->nChains * pl->nAC, nP = datum_bytes(pl) * (size_t)pl->nChains * pl->nData;
    const size_t nPhi = sizeof(double) * pl->nChains, nS = sizeof(int) * ((size_t)pl->nSys + 1);
    const size_t oP = (nM + 255) & ~(size_t)255, oPhi = oP + ((nP + 255) & ~(size_t)255), oG = oPhi + ((nPhi + 255) & ~(size_t)255);
    const size_t oS = oG + ((nM + 255) & ~(size_t)255), total = oS + nS;
    int rc = ensure_pin(pl, std::max(total, (size_t)1 << 20));
    if (rc) return rc;
    unsigned char* pin = reinterpret_cast<unsigned char*>(pl->pin);
    std::memcpy(pin, m, nM);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->m.p, pin, nM, cudaMemcpyHostToDevice, pl->stream));
    rc = compute_step(pl, true, nullptr);
    if (rc) return rc;
    if (pred) {
        if ((rc = pack_pred(pl))) return rc;
        HMCMT_CUDA_TRY(cudaMemcpyAsync(pin + oP, pl->predPacked.p, nP, cudaMemcpyDeviceToHost, pl->stream));
    }
    if (phid) HMCMT_CUDA_TRY(cudaMemcpyAsync(pin + oPhi, pl->phi.p, nPhi, cudaMemcpyDeviceToHost, pl->stream));
    if (grad) HMCMT_CUDA_TRY(cudaMemcpyAsync(pin + oG, withPrior ? pl->gtotal.p : pl->gdata.p, nM, cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pin + oS, pl->status.p, sizeof(int) * pl->nSys, cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pin + oS + sizeof(int) * pl->nSys, pl->driftFlag.p, sizeof(int), cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    if (pred) std::memcpy(pred, pin + oP, nP);
    if (phid) std::memcpy(phid, pin + oPhi, nPhi);
    if (grad) std::memcpy(grad, pin + oG, nM);
    // error flags of this call (same meaning as check_status; cleared when set so that they do not poison later evaluations)
    const int* st = reinterpret_cast<const int*>(pin + oS);
    rc = kOk;
    for (int i = 0; i < pl->nSys; ++i) if (st[i]) { rc = st[i]; break; }
    if (rc == kOk && st[pl->nSys]) rc = kErrBounds;
    if (rc != kOk) {
        HMCMT_CUDA_TRY(cudaMemsetAsync(pl->status.p, 0, sizeof(int) * pl->nSys, pl->stream));
        HMCMT_CUDA_TRY(cudaMemsetAsync(pl->driftFlag.p, 0, sizeof(int), pl->stream));
    }
    return rc;
}

int hmcmt_set_state(hmcmt_plan* pl, const double* m, const double* p, const double* mref) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    size_t bytes = sizeof(double) * (size_t)pl->nChains * pl->nAC;
    pl->sigmaDirect = false;
    if (m) HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->m.p, m, bytes, cudaMemcpyHostToDevice, pl->stream));
    if (p) HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->p.p, p, bytes, cudaMemcpyHostToDevice, pl->stream));
    if (mref) HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->mref.p, mref, bytes, cudaMemcpyHostToDevice, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return kOk;
}
int hmcmt_get_state(hmcmt_plan* pl, double* m, double* p) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    size_t bytes = sizeof(double) * (size_t)pl->nChains * pl->nAC;
    if (m) HMCMT_CUDA_TRY(cudaMemcpyAsync(m, pl->m.p, bytes, cudaMemcpyDeviceToHost, pl->stream));
    if (p) HMCMT_CUDA_TRY(cudaMemcpyAsync(p, pl->p.p, bytes, cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return kOk;
}

// the Gauss-Newton buffers, allocated on first use (and the tangent ones the CG's products need)
static int ensure_gn(hmcmt_plan* pl) {
    int rc = ensure_tangent(pl);
    if (rc || pl->gnI.p) return rc;
    const size_t nA = (size_t)pl->nChains * pl->nAC, nPart = (size_t)pl->nChains * ((pl->nAC + kGnReduceThreads - 1) / kGnReduceThreads);
    if ((rc = pl->gnVec.alloc(6 * nA)) || (rc = pl->gnAct.alloc(nA)) || (rc = pl->gnPart.alloc(nPart)) ||
        (rc = pl->gnS.alloc((size_t)pl->nChains * kGnS)) || (rc = pl->gnE.alloc(2 * (size_t)pl->nChains)))
        return rc;
    return pl->gnI.alloc((size_t)pl->nChains * kGnI);
}

// the per-chain flags into the pinned staging buffer, the device error flags, one synchronisation
static int gn_read_flags(hmcmt_plan* pl) {
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->pin, pl->gnI.p, sizeof(int) * pl->gnI.n, cudaMemcpyDeviceToHost, pl->stream));
    return check_status(pl);
}

// Projected Gauss-Newton-CG, every chain on its own (include/hmcmt_b200.h, DESIGN.md 4.8).  The host drives the outer iteration
// and the line search; every per-chain decision is taken on the device, from values that do not depend on the other chains.
int hmcmt_gauss_newton(hmcmt_plan* pl, const double* m0, int32_t maxIter, int32_t maxCG, double cgTol, int32_t maxLS, double maxStep,
                       double tolRel, double* m_out, double* history, int32_t* info) {
    if (!pl || !m_out || !history || !info || maxIter < 0 || maxCG < 1 || maxLS < 1 || !(maxStep > 0.0) || !(cgTol >= 0.0) ||
        !std::isfinite(cgTol) || !(tolRel >= 0.0) || !std::isfinite(tolRel))
        return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    int rc = ensure_gn(pl);
    if (rc) return rc;
    cudaStream_t st = pl->stream;
    const int nCh = pl->nChains, nAC = pl->nAC;
    const size_t nA = (size_t)nCh * nAC, nHist = (size_t)nCh * (maxIter + 1) * kGnHist;
    const size_t bytes = std::max(sizeof(double) * (nA + nHist) + sizeof(int) * pl->gnI.n, (size_t)1 << 20);
    if ((rc = ensure_pin(pl, bytes))) return rc;
    DevBuf<double> hist;
    if ((rc = hist.alloc(nHist))) return rc;
    double *mk = pl->gnVec.p, *gk = mk + nA, *delta = gk + nA, *r = delta + nA, *p = r + nA, *q = p + nA;
    const int nPart = (nAC + kGnReduceThreads - 1) / kGnReduceThreads;
    const int* flags = reinterpret_cast<const int*>(pl->pin);
    auto any = [&](int slot, int value) {
        for (int ch = 0; ch < nCh; ++ch)
            if (flags[(size_t)ch * kGnI + slot] == value) return true;
        return false;
    };
    // evaluation of the current model, then phi_m of it (k_energies' prior reduction; its kinetic half is not used)
    auto evaluate = [&]() -> int {
        int e = compute_step(pl, true, nullptr);
        if (e) return e;
        k_energies<<<nCh, kHmcThreads, 0, st>>>(nAC, pl->m.p, pl->mref.p, pl->p.p, pl->wmPtr.p, pl->wmIdx.p, pl->wmVal.p, pl->beta,
                                                pl->gnE.p, nullptr);
        LAUNCH_CHECK(pl);
        return kOk;
    };
    auto linearise = [&](int first) -> int {
        k_gn_linearise<<<nCh, kHmcThreads, 0, st>>>(nAC, first, maxIter, tolRel, pl->lo, pl->hi, pl->m.p, pl->gtotal.p, pl->phi.p,
                                                    pl->gnE.p, mk, gk, pl->gnAct.p, r, p, delta, pl->gnS.p, pl->gnI.p, hist.p);
        LAUNCH_CHECK(pl);
        return kOk;
    };
    auto run = [&]() -> int {
        int e;
        pl->sigmaDirect = false;
        if (m0) {
            std::memcpy(pl->pin, m0, sizeof(double) * nA);
            HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->m.p, pl->pin, sizeof(double) * nA, cudaMemcpyHostToDevice, st));
        }
        HMCMT_CUDA_TRY(cudaMemsetAsync(hist.p, 0, sizeof(double) * nHist, st));
        HMCMT_CUDA_TRY(cudaMemsetAsync(pl->gnI.p, 0, sizeof(int) * pl->gnI.n, st));
        k_gn_project<<<dim3((nAC + 255) / 256, nCh), 256, 0, st>>>(nAC, pl->lo, pl->hi, pl->m.p);
        LAUNCH_CHECK(pl);
        if ((e = evaluate()) || (e = linearise(1)) || (e = gn_read_flags(pl))) return e;
        for (int it = 0; it < maxIter && any(kGnActive, 1); ++it) {
            // CG on P H P delta = -P g: maxCG products of all chains, no host round trip (a chain whose CG stopped is masked)
            for (int j = 0; j < maxCG; ++j) {
                if ((e = gn_partials(pl, p))) return e;
                k_reduce_gn<<<dim3(nPart, nCh), kGnReduceThreads, 0, st>>>(nAC, pl->M.nCell, pl->nSysPerChain, pl->act2cell.p, pl->Gpart.p,
                                                                           p, pl->wmPtr.p, pl->wmIdx.p, pl->wmVal.p, pl->beta, pl->sigma.p,
                                                                           pl->gnAct.p, q, pl->gnPart.p);
                LAUNCH_CHECK(pl);
                k_gn_cg_update<<<nCh, kHmcThreads, 0, st>>>(nAC, nPart, cgTol, pl->gnPart.p, q, r, p, delta, pl->gnS.p, pl->gnI.p);
                LAUNCH_CHECK(pl);
            }
            k_gn_direction<<<nCh, kHmcThreads, 0, st>>>(nAC, maxStep, delta, pl->gnI.p);
            LAUNCH_CHECK(pl);
            // Armijo backtracking on the projected path: one evaluation of all chains per trial; a chain that accepted keeps its
            // model, so its evaluation (deterministic) stays that of its accepted trial
            for (int t = 0; t < maxLS; ++t) {
                k_gn_trial<<<nCh, kHmcThreads, 0, st>>>(nAC, t, pl->lo, pl->hi, mk, gk, delta, pl->m.p, pl->gnS.p, pl->gnI.p);
                LAUNCH_CHECK(pl);
                if ((e = evaluate())) return e;
                k_gn_armijo<<<(nCh + 127) / 128, 128, 0, st>>>(nCh, t, maxLS, pl->phi.p, pl->gnE.p, pl->gnS.p, pl->gnI.p);
                LAUNCH_CHECK(pl);
                if ((e = gn_read_flags(pl))) return e;
                if (!any(kGnLs, kLsSearch)) break;
            }
            if (any(kGnLs, kLsFailed)) {
                // the chains whose search failed keep m_k; one more evaluation makes the resident state that of the models kept
                k_gn_revert<<<nCh, kHmcThreads, 0, st>>>(nAC, mk, pl->m.p, pl->gnI.p);
                LAUNCH_CHECK(pl);
                if ((e = compute_step(pl, true, nullptr))) return e;
            }
            if ((e = linearise(0)) || (e = gn_read_flags(pl))) return e;
        }
        return kOk;
    };
    rc = run();
    if (rc == kOk) {
        unsigned char* pin = reinterpret_cast<unsigned char*>(pl->pin);
        const size_t oH = sizeof(double) * nA, oI = oH + sizeof(double) * nHist;
        if (cudaMemcpyAsync(pin, pl->m.p, oH, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaMemcpyAsync(pin + oH, hist.p, sizeof(double) * nHist, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaMemcpyAsync(pin + oI, pl->gnI.p, sizeof(int) * pl->gnI.n, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            rc = kErrCuda;
        if (rc == kOk) {
            std::memcpy(m_out, pin, oH);
            std::memcpy(history, pin + oH, sizeof(double) * nHist);
            const int* f = reinterpret_cast<const int*>(pin + oI);
            for (int ch = 0; ch < nCh; ++ch) {
                info[2 * ch] = f[(size_t)ch * kGnI + kGnAcc];
                info[2 * ch + 1] = f[(size_t)ch * kGnI + kGnReason];
            }
        }
    }
    cudaStreamSynchronize(st);
    hist.release();
    return rc;
}

static int trajectory_device(hmcmt_plan* pl, double dt, int Lmax, const int* dL) {
    // proposeLeapfrog HMCSampler.jl:206-269 (per-chain step counts in dL, device memory)
    dim3 g((pl->nAC + 255) / 256, pl->nChains);
    int rc = compute_step(pl, true, nullptr);
    if (rc) return rc;
    k_kick_masked<<<g, 256, 0, pl->stream>>>(pl->nAC, dt, 0, dL, pl->gtotal.p, pl->p.p);
    LAUNCH_CHECK(pl);
    for (int k = 1; k <= Lmax; ++k) {
        // chains that already finished (k > L) are frozen by a zero drift: handled through dt masking below
        rc = drift(pl, dt);
        if (rc) return rc;
        rc = compute_step(pl, true, nullptr);
        if (rc) return rc;
        k_kick_masked<<<g, 256, 0, pl->stream>>>(pl->nAC, dt, k, dL, pl->gtotal.p, pl->p.p);
        LAUNCH_CHECK(pl);
    }
    return kOk;
}

int hmcmt_leapfrog_trajectory(hmcmt_plan* pl, double dt, const int32_t* intstep, double* stats, double* pred) {
    if (!pl || !intstep) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    int Lmax = 0;
    for (int ch = 0; ch < pl->nChains; ++ch) {
        if (intstep[ch] != intstep[0]) {
            fprintf(stderr, "[hmcmt_b200] chains batched on one device must share the leapfrog step count\n");
            return kErrArg;
        }
        Lmax = std::max(Lmax, (int)intstep[ch]);
    }
    std::vector<int> L(intstep, intstep + pl->nChains);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(pl->Lsteps.p, L.data(), sizeof(int) * pl->nChains, cudaMemcpyHostToDevice, pl->stream));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    int rc = trajectory_device(pl, dt, Lmax, pl->Lsteps.p);
    if (rc) return rc;
    rc = energies(pl);
    if (rc) return rc;
    std::vector<double> e(2 * pl->nChains), ph(pl->nChains);
    HMCMT_CUDA_TRY(cudaMemcpyAsync(e.data(), pl->energies.p, sizeof(double) * e.size(), cudaMemcpyDeviceToHost, pl->stream));
    HMCMT_CUDA_TRY(cudaMemcpyAsync(ph.data(), pl->phi.p, sizeof(double) * ph.size(), cudaMemcpyDeviceToHost, pl->stream));
    if (pred) { rc = download_pred(pl, pred); if (rc) return rc; }
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    if (stats)
        for (int ch = 0; ch < pl->nChains; ++ch) {
            stats[4 * ch + 0] = ph[ch];
            stats[4 * ch + 1] = e[2 * ch + 1];
            stats[4 * ch + 2] = e[2 * ch];
            stats[4 * ch + 3] = ph[ch] + e[2 * ch] + e[2 * ch + 1];     // hmp = dataMisfit + kp + mnorm (:393)
        }
    return check_status(pl);
}

int hmcmt_leapfrog_steps_device(hmcmt_plan* pl, double dt, int32_t nsteps) {
    if (!pl || nsteps < 0) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    dim3 g((pl->nAC + 255) / 256, pl->nChains);
    for (int k = 0; k < nsteps; ++k) {
        int rc = drift(pl, dt);
        if (rc) return rc;
        rc = compute_step(pl, true, nullptr);
        if (rc) return rc;
        k_kick<<<dim3((pl->nAC + 255) / 256, pl->nChains), 256, 0, pl->stream>>>(pl->nAC, dt, pl->gtotal.p, pl->p.p);
        LAUNCH_CHECK(pl);
    }
    return kOk;
}

int hmcmt_nccl_unique_id(char* out128) {
    NcclApi* a = nccl_api();
    if (!a || !out128) return kErrArg;
    ncclUniqueId id;
    if (a->getUniqueId(&id) != ncclSuccess) return kErrCuda;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    std::memcpy(out128, &id, 128);
    return kOk;
}

int hmcmt_nccl_init(hmcmt_plan* pl, const char* id128, int32_t rank, int32_t world) {
    NcclApi* a = nccl_api();
    if (!a || !pl || !id128 || world < 1 || rank < 0 || rank >= world) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    if (pl->comm) { a->commDestroy(pl->comm); pl->comm = nullptr; }
    ncclUniqueId id;
    std::memcpy(&id, id128, 128);
    ncclResult_t r = a->commInitRank(&pl->comm, world, id, rank);
    if (r != ncclSuccess) {
        fprintf(stderr, "[hmcmt_b200] ncclCommInitRank failed: %s\n", a->getErrorString ? a->getErrorString(r) : "?");
        pl->comm = nullptr;
        return kErrCuda;
    }
    pl->commWorld = world;
    return kOk;
}

// nsteps leapfrog steps of a frequency-sharded chain, entirely enqueued on the plan's stream:
//   drift + reflect, forward + adjoint over THIS rank's systems, [gdata | phi_d] packed, ncclAllReduce(SUM), prior gradient, kick.
int hmcmt_leapfrog_steps_sharded(hmcmt_plan* pl, double dt, int32_t nsteps) {
    if (!pl || nsteps < 0) return kErrArg;
    NcclApi* a = pl->comm ? nccl_api() : nullptr;
    if (!a) {
        fprintf(stderr, "[hmcmt_b200] hmcmt_leapfrog_steps_sharded needs hmcmt_nccl_init first\n");
        return kErrArg;
    }
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    const size_t count = (size_t)pl->nChains * (pl->nAC + 1);
    for (int k = 0; k < nsteps; ++k) {
        int rc = hmcmt_step_partial(pl, dt);
        if (rc) return rc;
        if (a->allReduce(pl->xbuf.p, pl->xbuf.p, count, ncclFloat64, ncclSum, pl->comm, pl->stream) != ncclSuccess) return kErrCuda;
        ++pl->launches;
        rc = hmcmt_step_finish(pl, dt);
        if (rc) return rc;
    }
    return kOk;
}

int hmcmt_step_partial(hmcmt_plan* pl, double dt) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    int rc = drift(pl, dt);
    if (rc) return rc;
    rc = compute_step(pl, true, nullptr);
    if (rc) return rc;
    k_pack_exchange<<<dim3((pl->nAC + 1 + 255) / 256, pl->nChains), 256, 0, pl->stream>>>(pl->nAC, pl->gdata.p, pl->phi.p, pl->xbuf.p);
    LAUNCH_CHECK(pl);
    return kOk;
}

int hmcmt_exchange_buffer(hmcmt_plan* pl, void** dptr, int64_t* count) {
    if (!pl || !dptr || !count) return kErrArg;
    *dptr = pl->xbuf.p;
    *count = (int64_t)pl->nChains * (pl->nAC + 1);
    return kOk;
}

int hmcmt_step_finish(hmcmt_plan* pl, double dt) {
    if (!pl) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    k_unpack_exchange<<<dim3((pl->nAC + 1 + 255) / 256, pl->nChains), 256, 0, pl->stream>>>(
        pl->nAC, pl->xbuf.p, pl->m.p, pl->mref.p, pl->wmPtr.p, pl->wmIdx.p, pl->wmVal.p, pl->beta, pl->gdata.p, pl->gtotal.p, pl->phi.p);
    LAUNCH_CHECK(pl);
    k_kick<<<dim3((pl->nAC + 255) / 256, pl->nChains), 256, 0, pl->stream>>>(pl->nAC, dt, pl->gtotal.p, pl->p.p);
    LAUNCH_CHECK(pl);
    return kOk;
}

int hmcmt_run_chain(hmcmt_plan* pl, double dt, int32_t nsamples, double rhoref, const double* m_start, const double* z_init,
                    const int32_t* intsteps, const double* u_accept, const double* z_mom, int32_t reuse_last_forward, double* hmcmodel,
                    double* hmstats, int32_t* accept, double* hmcdata) {
    // rhoref = round(unirandDouble(0.5 rho0, 1.5 rho0)), rho0 = 1/exp(strModel[1]) (HMCSampler.jl:100-105), drawn by the caller.
    if (!pl || nsamples < 1 || !z_init || !intsteps || !u_accept || !z_mom) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    const int nCh = pl->nChains, nAC = pl->nAC, nData = pl->nData;
    const size_t nState = (size_t)nCh * nAC;
    cudaStream_t st = pl->stream;
    pl->sigmaDirect = false;
    // momentum draws travel in chunks through a two-slot device ring filled by a copy stream, so the sampling loop never
    // synchronises the compute stream with the host; everything else is uploaded once
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)nsamples, ((size_t)64 << 20) / (nState * sizeof(double))));
    DevBuf<double> dModel, dStats, dUacc, dZ;
    DevBuf<int> dAcc, dL;
    DevBuf<unsigned char> dData;                     // [nChains][nsamples+1][nData] packed data (complex, or real for rho / phase plans)
    const size_t dsz = datum_bytes(pl);
    cudaStream_t copy = nullptr;
    cudaEvent_t evCopied[2] = {nullptr, nullptr}, evFree[2] = {nullptr, nullptr};
    int rc = kOk;
    auto ok = [&](int r) { if (r && !rc) rc = r; };
    ok(dModel.alloc((size_t)nCh * nsamples * nAC)); ok(dStats.alloc((size_t)nCh * (nsamples + 1) * 4));
    ok(dUacc.upload(u_accept, (size_t)nCh * nsamples)); ok(dAcc.alloc((size_t)nCh * nsamples));
    ok(dData.alloc((size_t)nCh * (nsamples + 1) * nData * dsz));
    ok(dZ.alloc(2 * (size_t)chunk * nState));
    {
        std::vector<int> Lall((size_t)nsamples * nCh);
        for (int it = 0; it < nsamples; ++it)
            for (int ch = 0; ch < nCh; ++ch) Lall[(size_t)it * nCh + ch] = intsteps[it];
        ok(dL.upload(Lall.data(), Lall.size()));
    }
    auto cleanup = [&]() {
        cudaStreamSynchronize(st);
        if (copy) { cudaStreamSynchronize(copy); cudaStreamDestroy(copy); }
        for (int q = 0; q < 2; ++q) { if (evCopied[q]) cudaEventDestroy(evCopied[q]); if (evFree[q]) cudaEventDestroy(evFree[q]); }
        dModel.release(); dStats.release(); dUacc.release(); dAcc.release(); dData.release(); dZ.release(); dL.release();
    };
    if (rc) { cleanup(); return rc; }
    dim3 g((nAC + 255) / 256, nCh);
#define RC_TRY(x) do { int _r = (x); if (_r) { cleanup(); return _r; } } while (0)
#define RC_CUDA(x) do { if ((x) != cudaSuccess) { cleanup(); return kErrCuda; } } while (0)
    RC_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    for (int q = 0; q < 2; ++q) {
        RC_CUDA(cudaEventCreateWithFlags(&evCopied[q], cudaEventDisableTiming));
        RC_CUDA(cudaEventCreateWithFlags(&evFree[q], cudaEventDisableTiming));
    }
    // homogeneous rhoref model (HMCSampler.jl:100-109): invParam.strModel = invParam.refModel = log(1/rhoref)
    double mstart = std::log(1.0 / rhoref);
    k_fill<<<(unsigned)((nState + 255) / 256), 256, 0, st>>>(nState, mstart, pl->m.p);
    k_fill<<<(unsigned)((nState + 255) / 256), 256, 0, st>>>(nState, mstart, pl->mref.p);
    RC_CUDA(cudaMemcpyAsync(pl->zmom.p, z_init, sizeof(double) * nState, cudaMemcpyHostToDevice, st));
    k_clip_momentum<<<g, 256, 0, st>>>(nAC, pl->zmom.p, pl->p.p);
    pl->launches += 3;
    RC_TRY(mass_sqrt_apply(pl));
    // Hamiltonian at the start (getHamiltonian HMCSampler.jl:113-115): forward for the homogeneous model, mnorm = 0
    RC_TRY(compute_step(pl, false, nullptr));
    RC_TRY(energies(pl));
    RC_TRY(pack_pred(pl));
    {
        std::vector<double> e(2 * nCh), ph(nCh), sc(4 * nCh);
        RC_CUDA(cudaMemcpyAsync(e.data(), pl->energies.p, sizeof(double) * e.size(), cudaMemcpyDeviceToHost, st));
        RC_CUDA(cudaMemcpyAsync(ph.data(), pl->phi.p, sizeof(double) * ph.size(), cudaMemcpyDeviceToHost, st));
        RC_CUDA(cudaStreamSynchronize(st));
        for (int ch = 0; ch < nCh; ++ch) {
            sc[4 * ch + 0] = ph[ch]; sc[4 * ch + 1] = e[2 * ch + 1]; sc[4 * ch + 2] = e[2 * ch];
            sc[4 * ch + 3] = ph[ch] + e[2 * ch] + e[2 * ch + 1];
            RC_CUDA(cudaMemcpyAsync(dStats.p + (size_t)ch * (nsamples + 1) * 4, &sc[4 * ch], sizeof(double) * 4, cudaMemcpyHostToDevice, st));
            RC_CUDA(cudaMemcpyAsync(dData.p + (size_t)ch * (nsamples + 1) * nData * dsz,
                                    reinterpret_cast<const unsigned char*>(pl->predPacked.p) + (size_t)ch * nData * dsz, dsz * nData,
                                    cudaMemcpyDeviceToDevice, st));
        }
        RC_CUDA(cudaMemcpyAsync(pl->chainScal.p, sc.data(), sizeof(double) * sc.size(), cudaMemcpyHostToDevice, st));
        // the first trajectory starts from hmcParamCurrent.rhomodel = the model-file strModel, copied BEFORE strModel / refModel
        // were replaced by the homogeneous model (HMCSampler.jl:87 vs :100-109); m_start == NULL keeps the homogeneous model
        if (m_start) RC_CUDA(cudaMemcpyAsync(pl->m.p, m_start, sizeof(double) * nState, cudaMemcpyHostToDevice, st));
        RC_CUDA(cudaMemcpyAsync(pl->curM.p, pl->m.p, sizeof(double) * nState, cudaMemcpyDeviceToDevice, st));
        RC_CUDA(cudaStreamSynchronize(st));
    }
    auto stage_chunk = [&](int c) -> int {           // z_mom layout: [sample][chain][nAC]
        const int slot = c & 1, first = c * chunk, cnt = std::min(chunk, nsamples - first);
        if (c >= 2 && cudaStreamWaitEvent(copy, evFree[slot], 0) != cudaSuccess) return kErrCuda;
        if (cudaMemcpyAsync(dZ.p + (size_t)slot * chunk * nState, z_mom + (size_t)first * nState, sizeof(double) * (size_t)cnt * nState,
                            cudaMemcpyHostToDevice, copy) != cudaSuccess || cudaEventRecord(evCopied[slot], copy) != cudaSuccess)
            return kErrCuda;
        return kOk;
    };
    const int nChunks = (nsamples + chunk - 1) / chunk;
    RC_TRY(stage_chunk(0));
    for (int it = 1; it <= nsamples; ++it) {
        const int c = (it - 1) / chunk, slot = c & 1, inChunk = (it - 1) % chunk;
        if (inChunk == 0) {
            RC_CUDA(cudaStreamWaitEvent(st, evCopied[slot], 0));
            if (c + 1 < nChunks) RC_TRY(stage_chunk(c + 1));          // the next chunk travels while this one is sampled
        }
        const int L = intsteps[it - 1];
        RC_TRY(trajectory_device(pl, dt, L, dL.p + (size_t)(it - 1) * nCh));
        if (!reuse_last_forward) RC_TRY(compute_step(pl, false, nullptr));       // the reference's redundant forward sweep
        RC_TRY(energies(pl));
        RC_TRY(pack_pred(pl));
        const double* zsrc = dZ.p + ((size_t)slot * chunk + inChunk) * nState;
        if (pl->dataKind)
            k_accept<double><<<nCh, kHmcThreads, 0, st>>>(nAC, nData, it, nsamples, dUacc.p, pl->phi.p, pl->energies.p, zsrc, pl->m.p, pl->p.p,
                                                          pl->curM.p, pl->chainScal.p, reinterpret_cast<const double*>(pl->predPacked.p),
                                                          dModel.p, dStats.p, dAcc.p, reinterpret_cast<double*>(dData.p));
        else
            k_accept<cplx><<<nCh, kHmcThreads, 0, st>>>(nAC, nData, it, nsamples, dUacc.p, pl->phi.p, pl->energies.p, zsrc, pl->m.p, pl->p.p,
                                                        pl->curM.p, pl->chainScal.p, pl->predPacked.p, dModel.p, dStats.p, dAcc.p,
                                                        reinterpret_cast<cplx*>(dData.p));
        pl->launches += 1;
        if (cudaGetLastError() != cudaSuccess) { cleanup(); return kErrCuda; }
        RC_TRY(mass_sqrt_apply(pl));             // p = sqrtM clip(z); k_accept's kinetic energy 1/2 z^T z equals 1/2 p^T invM p
        if (inChunk == chunk - 1 || it == nsamples) RC_CUDA(cudaEventRecord(evFree[slot], st));
    }
    RC_CUDA(cudaMemcpyAsync(hmcmodel, dModel.p, sizeof(double) * dModel.n, cudaMemcpyDeviceToHost, st));
    RC_CUDA(cudaMemcpyAsync(hmstats, dStats.p, sizeof(double) * dStats.n, cudaMemcpyDeviceToHost, st));
    RC_CUDA(cudaMemcpyAsync(accept, dAcc.p, sizeof(int) * dAcc.n, cudaMemcpyDeviceToHost, st));
    RC_CUDA(cudaMemcpyAsync(hmcdata, dData.p, dData.n, cudaMemcpyDeviceToHost, st));
    RC_CUDA(cudaStreamSynchronize(st));
    cleanup();
#undef RC_TRY
#undef RC_CUDA
    return check_status(pl);
}

int hmcmt_export_system(hmcmt_plan* pl, int32_t chain, int32_t mode, int32_t freq, int64_t* colptr, int64_t* rowval, double* nzval,
                        double* rhs, double* bc) {
    if (!pl || chain < 0 || chain >= pl->nChains || freq < 0 || freq >= pl->nFreq) return kErrArg;
    int mi = -1;
    for (int c = 0; c < pl->nModes; ++c) if (pl->modeList[c] == mode) mi = c;
    if (mi < 0 || !pl->haveForward) return kErrArg;
    HMCMT_CUDA_TRY(cudaSetDevice(pl->device));
    HMCMT_CUDA_TRY(cudaStreamSynchronize(pl->stream));
    const MeshDev& M = pl->M;
    const size_t N = M.N;
    std::vector<double> P(4 * N);
    HMCMT_CUDA_TRY(cudaMemcpy(P.data(), pl->planes.p + ((size_t)(chain * pl->nModes + mi) * 4) * N, sizeof(double) * 4 * N, cudaMemcpyDeviceToHost));
    const size_t sys = ((size_t)chain * pl->nModes + mi) * pl->nFreq + freq;
    std::vector<cplx> r(N), b(M.nb);
    HMCMT_CUDA_TRY(cudaMemcpy(r.data(), pl->rhs.p + sys * N, sizeof(cplx) * N, cudaMemcpyDeviceToHost));
    HMCMT_CUDA_TRY(cudaMemcpy(b.data(), pl->bc.p + sys * M.nb, sizeof(cplx) * M.nb, cudaMemcpyDeviceToHost));
    const double omega = 2.0 * kPi * pl->h_freqs[freq];
    const int n1 = M.n1, n2 = M.n2;
    auto qof = [&](int jn, int kn) { return M.fastZ ? (size_t)(jn - 1) * M.nf + (kn - 1) : (size_t)(kn - 1) * M.nf + (jn - 1); };
    // coupling between (jn,kn) and its -y / -z neighbour, from the internal planes
    auto cy = [&](int jn, int kn) { size_t q = qof(jn, kn); return M.fastZ ? P[3 * N + q] : P[2 * N + q]; };   // to (jn-1,kn)
    auto cz = [&](int jn, int kn) { size_t q = qof(jn, kn); return M.fastZ ? P[2 * N + q] : P[3 * N + q]; };   // to (jn,kn-1)
    int64_t nnz = 0;
    for (int kn = 1; kn <= n2; ++kn)
        for (int jn = 1; jn <= n1; ++jn) {
            int64_t pcol = (int64_t)(kn - 1) * n1 + (jn - 1);      // reference interior numbering, y fastest (0-based)
            colptr[pcol] = nnz + 1;
            size_t q = qof(jn, kn);
            if (kn > 1) { rowval[nnz] = pcol - n1 + 1; nzval[2 * nnz] = cz(jn, kn); nzval[2 * nnz + 1] = 0.0; ++nnz; }
            if (jn > 1) { rowval[nnz] = pcol - 1 + 1; nzval[2 * nnz] = cy(jn, kn); nzval[2 * nnz + 1] = 0.0; ++nnz; }
            rowval[nnz] = pcol + 1; nzval[2 * nnz] = P[q]; nzval[2 * nnz + 1] = omega * P[N + q]; ++nnz;
            if (jn < n1) { rowval[nnz] = pcol + 1 + 1; nzval[2 * nnz] = cy(jn + 1, kn); nzval[2 * nnz + 1] = 0.0; ++nnz; }
            if (kn < n2) { rowval[nnz] = pcol + n1 + 1; nzval[2 * nnz] = cz(jn, kn + 1); nzval[2 * nnz + 1] = 0.0; ++nnz; }
            if (rhs) { rhs[2 * pcol] = r[q].x; rhs[2 * pcol + 1] = r[q].y; }
        }
    colptr[N] = nnz + 1;
    if (bc) for (int i = 0; i < M.nb; ++i) { bc[2 * i] = b[i].x; bc[2 * i + 1] = b[i].y; }
    return kOk;
}

}  // extern "C"
