// Physics kernels of the MT2D forward + adjoint hot path (everything except the band solver).
// Each kernel cites the reference routine it replaces (paths relative to HMCMT/src/).
//
// Index conventions (0-based): cell (jc,kc) -> kc*ny+jc ; node (jn,kn) -> kn*(ny+1)+jn ;
// interior node (jn in 1..ny-1, kn in 1..nz-1) -> internal index q = l*nf+f with (l,f) =
// (jn-1,kn-1) when the fast axis is z (fastZ), else (kn-1,jn-1).  Arrays crossing the C ABI use the
// reference numbering (SURVEY.md A.2); the internal ordering never leaves the library.
#pragma once
#include "common.cuh"

namespace hmcmt {

struct MeshDev {
    int ny, nz;            // cells incl. air
    int n1, n2, N;         // interior nodes per axis, unknowns
    int nf, nl, fastZ;     // internal ordering
    int nCell, nNode, nb;
    int zid;               // receiver node row
    const double* yLen;    // [ny]
    const double* zLen;    // [nz]
    const double* zNode;   // [nz+1] cumulative from 0
};

__device__ __forceinline__ int q_of(const MeshDev& M, int jn, int kn) {
    return M.fastZ ? (jn - 1) * M.nf + (kn - 1) : (kn - 1) * M.nf + (jn - 1);
}
__device__ __forceinline__ void jk_of(const MeshDev& M, int q, int& jn, int& kn) {
    int l = q / M.nf, f = q - l * M.nf;
    if (M.fastZ) { jn = l + 1; kn = f + 1; } else { kn = l + 1; jn = f + 1; }
}

// system index: sys = (ch*nModes + mi)*nFreq + f ; mode = 0 (TE, ZXY) or 1 (TM, ZYX)
struct SysMap {
    int nFreq, nModes, mode0, mode1;
};
__device__ __forceinline__ void sys_decode(const SysMap& sm, int sys, int& ch, int& mi, int& mode, int& f) {
    f = sys % sm.nFreq;
    int t = sys / sm.nFreq;
    mi = t % sm.nModes;
    ch = t / sm.nModes;
    mode = mi == 0 ? sm.mode0 : sm.mode1;
}

// ---------------------------------------------------------------------------------------------
// K1: sigma = activeCell*exp(m) + bgModel     (HMCSampler.jl:290-294, HMCUtility.jl:69-77)
// grid: (ceil(nCell/256), nChains)
__global__ void k_model_transform(int nCell, int nAC, const int* __restrict__ cell2act,
                                  const double* __restrict__ bg, const double* __restrict__ m,
                                  double* __restrict__ sigma) {
    int c = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (c >= nCell) return;
    int a = cell2act[c];
    sigma[(size_t)ch * nCell + c] = (a >= 0) ? exp(m[(size_t)ch * nAC + a]) : bg[c];
}

// ---------------------------------------------------------------------------------------------
// K2: 5-point stencil planes in internal ordering (SURVEY.md A.3; MT2DFwdSolver.jl:123-135,149-161)
//   TE: v = 1/mu0, w = sigma ;  TM: v = 1/sigma, w = mu0.
// planes layout: [chain][mi][4][N]  (dr, dm, e1, e2).  grid: (ceil(N/256), nChains*nModes)
struct StencilW {
    double wyL, wyR, wzU, wzD, mass;
};
__device__ __forceinline__ StencilW stencil_at(const MeshDev& M, const double* __restrict__ sig, int mode, int jn, int kn) {
    const int ny = M.ny;
    const double dyl = M.yLen[jn - 1], dyr = M.yLen[jn], dzu = M.zLen[kn - 1], dzd = M.zLen[kn];
    const double s00 = sig[(kn - 1) * ny + jn - 1], s10 = sig[(kn - 1) * ny + jn];
    const double s01 = sig[kn * ny + jn - 1], s11 = sig[kn * ny + jn];
    double v00, v10, v01, v11, w00, w10, w01, w11;
    if (mode == 0) {
        v00 = v10 = v01 = v11 = 1.0 / kMu0;
        w00 = s00; w10 = s10; w01 = s01; w11 = s11;
    } else {
        v00 = 1.0 / s00; v10 = 1.0 / s10; v01 = 1.0 / s01; v11 = 1.0 / s11;
        w00 = w10 = w01 = w11 = kMu0;
    }
    StencilW r;
    // Wy(jn',kn) = 1/2 (dz_{kn-1} v_{jn',kn-1} + dz_kn v_{jn',kn}) / dy_{jn'}   (edge to the +y neighbour of node jn')
    r.wyL = 0.5 * (dzu * v00 + dzd * v01) / dyl;     // edge (jn-1,kn)-(jn,kn), cells jc = jn-1
    r.wyR = 0.5 * (dzu * v10 + dzd * v11) / dyr;     // edge (jn,kn)-(jn+1,kn), cells jc = jn
    r.wzU = 0.5 * (dyl * v00 + dyr * v10) / dzu;     // edge (jn,kn-1)-(jn,kn), cells kc = kn-1
    r.wzD = 0.5 * (dyl * v01 + dyr * v11) / dzd;     // edge (jn,kn)-(jn,kn+1), cells kc = kn
    r.mass = 0.25 * (dyl * dzu * w00) + 0.25 * (dyr * dzu * w10) + 0.25 * (dyl * dzd * w01) + 0.25 * (dyr * dzd * w11);
    return r;
}
__global__ void k_stencil_planes(MeshDev M, SysMap sm, const double* __restrict__ sigma, double* __restrict__ planes) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= M.N) return;
    int ch = blockIdx.y / sm.nModes, mi = blockIdx.y % sm.nModes, mode = mi == 0 ? sm.mode0 : sm.mode1;
    int jn, kn;
    jk_of(M, q, jn, kn);
    StencilW w = stencil_at(M, sigma + (size_t)ch * M.nCell, mode, jn, kn);
    double* P = planes + ((size_t)(ch * sm.nModes + mi) * 4) * M.N;
    P[q] = w.wyL + w.wyR + w.wzU + w.wzD;
    P[M.N + q] = w.mass;
    double e1, e2;
    if (M.fastZ) { e1 = (kn > 1) ? -w.wzU : 0.0; e2 = (jn > 1) ? -w.wyL : 0.0; }
    else         { e1 = (jn > 1) ? -w.wyL : 0.0; e2 = (kn > 1) ? -w.wzU : 0.0; }
    P[2 * (size_t)M.N + q] = e1;
    P[3 * (size_t)M.N + q] = e2;
}

// ---------------------------------------------------------------------------------------------
// K3: Dirichlet boundary values from 1-D layered-earth solutions
//   (getBoundaryMT2DTE mt2DTE.jl:100-134, getBoundaryMT2DTM mt2DTM.jl:100-134, mt1DAnalyticField mt1DField.jl:23-98)
// One thread per profile: p=0 left column, p=1 right column, p=2.. bottom node jn=p-1 (jn=1..ny-1).
// bc layout (reference `io` order): [top ny+1 | left nz | right nz | bottom ny-1].
__device__ __forceinline__ double prof_sigma(const MeshDev& M, const double* __restrict__ sig, int p, int k) {
    const int ny = M.ny;
    if (p == 0) return sig[k * ny];
    if (p == 1) return sig[k * ny + ny - 1];
    int jn = p - 1;
    double y1 = M.yLen[jn - 1], y2 = M.yLen[jn];
    return (sig[k * ny + jn - 1] * y1 + sig[k * ny + jn] * y2) / (y1 + y2);
}
__device__ __forceinline__ cplx wavenumber(double omega, double s) {
    return csqrt_(mk(kMu0 * kEps0 * omega * omega, -kMu0 * s * omega));
}
// The layered-earth recursion depends on (chain, frequency, profile) only: it is computed once and written to every mode
// (TE: E = eu+ed, TM: H = (ed-eu) k / (omega mu)).  The expensive per-layer terms (wavenumber, tanh, exponentials, ratios)
// do not depend on the recursion state: phase A evaluates them for all layers of the block's PB profiles in parallel into
// shared memory, phase B runs the two serial recursions (a few complex multiplies / divisions per layer) one thread per profile.
// systems: sys = (ch*nModes+mi)*nFreq + f.   grid: (ceil((ny+1)/PB), nChains*nFreq), block kBcThreads, smem PB*nz*6 complex
constexpr int kBcThreads = 128;
__host__ __device__ inline int boundary_profiles_per_block(int nz) {
    int pb = (int)((44 * 1024) / (6 * sizeof(cplx) * (size_t)nz));
    return pb < 1 ? 1 : (pb > 8 ? 8 : pb);      // the serial phase keeps PB lanes of one warp busy: as many as shared memory allows
}
__global__ void __launch_bounds__(kBcThreads)
k_boundary(MeshDev M, SysMap sm, const double* __restrict__ freqs, const double* __restrict__ sigma, cplx* __restrict__ bc, int PB) {
    extern __shared__ __align__(16) unsigned char bcraw[];
    cplx* const sh = reinterpret_cast<cplx*>(bcraw);          // [PB][6][nz]: k, tanh(ikh), exp(ikh), exp(-ikh), omu/k, k_j/k_{j+1}
    const int ch = blockIdx.y / sm.nFreq, f = blockIdx.y - ch * sm.nFreq;
    const int ny = M.ny, nz = M.nz, p0 = blockIdx.x * PB;
    const double* sig = sigma + (size_t)ch * M.nCell;
    const double omega = 2.0 * kPi * freqs[f], omu = omega * kMu0;
    auto A = [&](int pl, int which) { return sh + ((size_t)pl * 6 + which) * nz; };
    for (int item = threadIdx.x; item < PB * nz; item += kBcThreads) {
        const int pl = item / nz, j = item - pl * nz, p = p0 + pl;
        if (p > ny) continue;
        const cplx k = wavenumber(omega, prof_sigma(M, sig, p, j));
        const cplx kh = k * M.zLen[j];
        A(pl, 0)[j] = k;
        A(pl, 1)[j] = ctanh_(mk(-kh.y, kh.x));          // tanh(i k h)
        A(pl, 2)[j] = cexp_(mk(-kh.y, kh.x));
        A(pl, 3)[j] = cexp_(mk(kh.y, -kh.x));
        A(pl, 4)[j] = omu / k;
    }
    __syncthreads();
    for (int item = threadIdx.x; item < PB * nz; item += kBcThreads) {
        const int pl = item / nz, j = item - pl * nz;
        if (p0 + pl > ny) continue;
        A(pl, 5)[j] = A(pl, 0)[j] / A(pl, 0)[(j + 1 < nz) ? j + 1 : nz - 1];
    }
    __syncthreads();
    const int p = p0 + threadIdx.x;
    const bool active = (int)threadIdx.x < PB && p <= ny;        // ny+1 profiles (2 + ny-1) and ny+1 top-row entries
    const int nM = sm.nModes;
    cplx* out[2];
    int modes[2];
    for (int mi = 0; mi < nM; ++mi) {
        out[mi] = bc + (size_t)((ch * sm.nModes + mi) * sm.nFreq + f) * M.nb;
        modes[mi] = mi == 0 ? sm.mode0 : sm.mode1;
    }
    auto field_of = [&](int mode, cplx eu, cplx ed, cplx kk) { return (mode == 0) ? eu + ed : (ed * kk - eu * kk) / omu; };   // E or H
    if (active) {
        const cplx *K = A(threadIdx.x, 0), *TH = A(threadIdx.x, 1), *EP = A(threadIdx.x, 2), *EM = A(threadIdx.x, 3),
                   *ZP = A(threadIdx.x, 4), *KR = A(threadIdx.x, 5);
        for (int mi = 0; mi < nM; ++mi) out[mi][p] = mk(1.0, 0.0);      // top row
        // bottom-up impedance recursion
        cplx zt = ZP[nz - 1];
        for (int j = nz - 1; j >= 0; --j) {
            const cplx zp = ZP[j], th = TH[j];
            zt = zp * (zt + zp * th) / (zp + zt * th);
        }
        const cplx k = K[0];
        cplx r0 = omu / (zt * k);
        cplx eu = 0.5 * (mk(1.0, 0.0) - r0), ed = 0.5 * (mk(1.0, 0.0) + r0);
        const cplx eu0 = eu, ed0 = ed;
        // the two edge columns (p = 0, 1) need every row: their amplitudes are parked in shared memory (the tanh / impedance
        // arrays are dead by now) and turned into normalised fields by the whole block below; a bottom profile only needs its
        // last row
        const bool edge = p < 2;
        cplx* EU = A(threadIdx.x, 1);
        cplx* ED = A(threadIdx.x, 4);
        bool dead = false, live = false;
        double e1 = cabs_(eu + ed);                    // |E| of the previous row: the guard compares consecutive rows
        for (int i = 0; i < nz; ++i) {
            live = false;
            if (!dead) {
                const cplx kr = KR[i], ep = EP[i], em = EM[i];
                cplx one = mk(1.0, 0.0);
                cplx a = 0.5 * (one + kr), bq = 0.5 * (one - kr);
                cplx nu = (a * ep) * eu + (bq * em) * ed;
                cplx nd = (bq * ep) * eu + (a * em) * ed;
                double e2 = cabs_(nu + nd);
                if (e2 - e1 > 0.0 || isnan(e2)) {
                    dead = true;                       // mt1DField.jl:77-81: zero all deeper entries
                } else {
                    eu = nu; ed = nd; e1 = e2;
                    live = true;
                }
            }
            if (edge) { EU[i] = live ? eu : mk(0.0, 0.0); ED[i] = live ? ed : mk(0.0, 0.0); }
        }
        if (edge) {
            A(threadIdx.x, 5)[0] = eu0;                // (the ratio array is dead as well)
            A(threadIdx.x, 5)[1] = ed0;
        } else {
            const cplx ki = K[nz - 1];
            for (int mi = 0; mi < nM; ++mi) {
                const cplx last = live ? field_of(modes[mi], eu, ed, ki) : mk(0.0, 0.0);
                out[mi][ny + 1 + 2 * nz + (p - 2)] = last / field_of(modes[mi], eu0, ed0, k);
            }
        }
    }
    if (p0 >= 2) return;                               // only the first block(s) of a (chain, frequency) hold the edge columns p = 0, 1
    __syncthreads();
    for (int item = threadIdx.x; item < 2 * nM * nz; item += kBcThreads) {
        const int pl = item / (nM * nz), rem = item - pl * nM * nz, mi = rem / nz, i = rem - mi * nz;
        const int pg = p0 + pl;                        // global profile of local profile pl
        if (pl >= PB || pg >= 2) continue;
        const cplx* K = A(pl, 0);
        const cplx top = field_of(modes[mi], A(pl, 5)[0], A(pl, 5)[1], K[0]);
        const cplx val = field_of(modes[mi], A(pl, 1)[i], A(pl, 4)[i], K[(i + 1 < nz) ? i + 1 : nz - 1]);
        out[mi][ny + 1 + pg * nz + i] = val / top;
    }
}

// rhs = -Aio*bc in internal ordering (mt2DTE.jl:44).  grid: (ceil(N/256), nSys)
__global__ void k_rhs(MeshDev M, SysMap sm, const double* __restrict__ sigma, const cplx* __restrict__ bc,
                      cplx* __restrict__ rhs) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= M.N) return;
    const int sys = blockIdx.y;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    int jn, kn;
    jk_of(M, q, jn, kn);
    cplx r = mk(0.0, 0.0);
    const int ny = M.ny, nz = M.nz;
    if (jn == 1 || jn == ny - 1 || kn == 1 || kn == nz - 1) {
        StencilW w = stencil_at(M, sigma + (size_t)ch * M.nCell, mode, jn, kn);
        const cplx* b = bc + (size_t)sys * M.nb;
        if (kn == 1) r += w.wzU * b[jn];                                   // top
        if (jn == 1) r += w.wyL * b[ny + 1 + (kn - 1)];                    // left  (kn = 1..nz)
        if (jn == ny - 1) r += w.wyR * b[ny + 1 + nz + (kn - 1)];          // right
        if (kn == nz - 1) r += w.wzD * b[ny + 1 + 2 * nz + (jn - 1)];      // bottom (jn = 1..ny-1)
    }
    rhs[(size_t)sys * M.N + q] = r;
}

// full node-ordered field from the interior solution + boundary values (mt2DTE.jl:57-62), nodes [n0, n1) of it.
// grid: (ceil((n1 - n0)/256), nSys).  If bc == nullptr the boundary is zero (adjoint field).
// (sys0: first system of the group this launch covers; the groups of a step run on different streams, hmcmt_b200.cu)
__global__ void k_node_field(MeshDev M, const cplx* __restrict__ x, const cplx* __restrict__ bc, cplx* __restrict__ F, int sys0, int n0,
                             int n1) {
    int n = n0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= n1) return;
    const int sys = blockIdx.y + sys0, ny = M.ny, nz = M.nz;
    int kn = n / (ny + 1), jn = n - kn * (ny + 1);
    cplx v = mk(0.0, 0.0);
    if (jn >= 1 && jn <= ny - 1 && kn >= 1 && kn <= nz - 1) {
        v = x[(size_t)sys * M.N + q_of(M, jn, kn)];
    } else if (bc) {
        const cplx* b = bc + (size_t)sys * M.nb;
        if (kn == 0) v = b[jn];
        else if (jn == 0) v = b[ny + 1 + (kn - 1)];
        else if (jn == ny) v = b[ny + 1 + nz + (kn - 1)];
        else v = b[ny + 1 + 2 * nz + (jn - 1)];
    }
    F[(size_t)sys * M.nNode + n] = v;
}

// ---------------------------------------------------------------------------------------------
// K6+K7: receiver functional, residual, misfit partial and adjoint source, one CTA per system.
//   forward  : compFieldsAtRxTE mt2DTE.jl:153-210 / compFieldsAtRxTM mt2DTM.jl:152-210, Z = num/den
//   adjoint  : closed-form reverse mode of getDataFuncSensTE/TM (dataFuncSens.jl:21-176,197-344),
//              s = L^T conj(v), q = Q^T conj(v)  (compJacTMatVec.jl:183-214, 254-285)
struct RxDev {
    int nRx;
    const int* fid;        // forward interpolation: first node with yNode > y_rx
    const double* fdy1;    // y_rx - yNode[id-1]
    const double* fdy2;    // yNode[id] - y_rx
    const int* iL;         // normalised weights of sensUtils.jl:133-161
    const int* iR;
    const double* wL;
    const double* wR;
    const int* tjL;        // the same weights on the cell centres (linRxMap2, sensUtils.jl:17-52): Hz of the tipper
    const int* tjR;
    const double* twL;
    const double* twR;
};
// Data components of an impedance plan with a tipper (kTipper): system mi holds the impedance component zc[mi] (-1: none, a
// [TZY]-only plan) and system tmi also the tipper component tc.  Without a tipper nComp = nModes and component = system.
struct CompMap {
    int nComp, zc[2], tc, tmi;
};
// data arrays are "full": index ((ch*nFreq+f)*nRx + r)*nComp + c ; wd = 0 where the datum is absent.
// vin: optional externally supplied data vector (hmcmt_jtvec); if null v = wd^2 (Z - obs).
// kRhoPhase (plans of hmcmt_plan_create_rho_phase): the data of a slot are rho_a = |Z|^2/(omega mu0) and phase
// phi = atan2(Im Z, Re Z) 180/pi; obs holds the pair (rho, phi), wd / wdPha their weights, resp receives the predicted pair.
// With v_rho = w_rho^2 (rho - rho_obs), v_phi = w_phi^2 (phi - phi_obs) (or the real pair (v_rho, v_phi) carried by vin) the
// slot's adjoint weight on Z is V = v_rho 2/(omega mu0) Z + v_phi 180/pi i Z/|Z|^2: Re(J^T conj(V)) is the misfit gradient
// (d rho/d sigma = 2/(omega mu0) Re(conj(Z) J), d phi/d sigma = 180/pi Im(J/Z)), and everything after it is the impedance path.
// kTipper (impedance plans with a TZY component): the TE system tmi also forms, per receiver, the tipper
//   Hz0_j = (F0_{j+1} - F0_j)/(yLen_j i omega mu0) at the cell centres, Hzr = twL Hz0_{tjL} + twR Hz0_{tjR},
//   Hyr = wL Hy0_{iL} + wR Hy0_{iR} (G0, the normalised node weights), T = Hzr/Hyr,
// and with d = conj(v_T) adds the reverse mode d/Hyr (onto F0 through the two-point difference of each cell) and -d T/Hyr (onto
// G0 with the node weights) to the impedance adjoints; everything after that is the impedance path.
constexpr int kRxThreads = 256;
template <bool kRhoPhase, bool kTipper>
__global__ void __launch_bounds__(kRxThreads)
k_rx_adjoint(MeshDev M, RxDev rx, SysMap sm, CompMap cm, const double* __restrict__ freqs, const double* __restrict__ sigma,
             const cplx* __restrict__ F, const cplx* __restrict__ obs, const double* __restrict__ wd,
             const double* __restrict__ wdPha, const cplx* __restrict__ vin, cplx* __restrict__ pred,
             double* __restrict__ phiPart, cplx* __restrict__ srows, cplx* __restrict__ qrow, cplx* __restrict__ adjrhs,
             int wantAdjoint, int respKind, cplx* __restrict__ resp, int sys0) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int ny = M.ny;
    cplx* F0 = reinterpret_cast<cplx*>(smraw);        // ny+1
    cplx* F1 = F0 + (ny + 1);
    cplx* G0 = F1 + (ny + 1);                          // Hy0 / Ey0 (ny+1)
    cplx* aF0 = G0 + (ny + 1);                         // adjoints
    cplx* aF1 = aF0 + (ny + 1);
    cplx* aG0 = aF1 + (ny + 1);
    cplx* Qc = aG0 + (ny + 1);                         // HzQ / EzQ  (ny)
    cplx* aQc = Qc + ny;                               // adjoint of HzQ / EzQ (ny)
    cplx* qv = aQc + ny;                               // q on the receiver cell row (ny)
    const int sys = blockIdx.x + sys0;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    const int nFreq = sm.nFreq;
    const int tid = threadIdx.x;
    const double omega = 2.0 * kPi * freqs[f];
    const double h = M.zLen[M.zid];
    const double* sig1 = sigma + (size_t)ch * M.nCell + (size_t)M.zid * ny;
    const cplx* Fs = F + (size_t)sys * M.nNode;
    const cplx iw = mk(0.0, omega), iwmu = mk(0.0, omega * kMu0);
    for (int j = tid; j <= ny; j += kRxThreads) {
        F0[j] = Fs[(size_t)M.zid * (ny + 1) + j];
        F1[j] = Fs[(size_t)(M.zid + 1) * (ny + 1) + j];
        aF0[j] = aF1[j] = aG0[j] = mk(0.0, 0.0);
    }
    __syncthreads();
    for (int j = tid; j < ny; j += kRxThreads) {
        if (mode == 0) {
            cplx bz0 = (F0[j + 1] - F0[j]) / M.yLen[j] / iw;
            cplx bz1 = (F1[j + 1] - F1[j]) / M.yLen[j] / iw;
            Qc[j] = (0.75 * bz0 + 0.25 * bz1) / kMu0;
        } else {
            cplx jz0 = -((F0[j + 1] - F0[j]) / M.yLen[j]);
            cplx jz1 = -((F1[j + 1] - F1[j]) / M.yLen[j]);
            Qc[j] = (0.75 * jz0 + 0.25 * jz1) / sig1[j];
        }
        aQc[j] = mk(0.0, 0.0);
        qv[j] = mk(0.0, 0.0);
    }
    __syncthreads();
    for (int i = tid + 1; i < ny; i += kRxThreads) {
        const double yb = 0.5 * M.yLen[i - 1] + 0.5 * M.yLen[i];
        if (mode == 0) {
            cplx HyH = -((F1[i] - F0[i]) / h / iwmu);
            cplx ExQ = 0.75 * F0[i] + 0.25 * F1[i];
            double sv = (0.5 * (sig1[i - 1] * M.yLen[i - 1]) + 0.5 * (sig1[i] * M.yLen[i])) / yb;
            cplx dHz = (Qc[i] - Qc[i - 1]) / yb;
            G0[i] = HyH - (dHz - sv * ExQ) * (0.5 * h);
        } else {
            cplx JyH = (F1[i] - F0[i]) / h;
            double rv = (0.5 * ((1.0 / sig1[i - 1]) * M.yLen[i - 1]) + 0.5 * ((1.0 / sig1[i]) * M.yLen[i])) / yb;
            cplx HxQ = 0.75 * F0[i] + 0.25 * F1[i];
            cplx dEz = (Qc[i] - Qc[i - 1]) / yb;
            G0[i] = JyH * rv - (dEz + iwmu * HxQ) * (0.5 * h);
        }
    }
    __syncthreads();
    if (tid == 0) { G0[0] = G0[1]; G0[ny] = G0[ny - 1]; }
    __syncthreads();
    // ---- responses, residual, misfit, receiver adjoints (serial over receivers: deterministic) ----
    __shared__ double phiSh;
    const int nC = kTipper ? cm.nComp : sm.nModes;                 // data slots per (frequency, receiver)
    const int zc = kTipper ? (mi == 0 ? cm.zc[0] : cm.zc[1]) : mi;    // this system's impedance component
    if (tid == 0) {
        double phi = 0.0;
        const int nRxZ = (kTipper && zc < 0) ? 0 : rx.nRx;
        for (int r = 0; r < nRxZ; ++r) {
            const int id = rx.fid[r];
            const double d1 = rx.fdy1[r], d2 = rx.fdy2[r];
            cplx numF, denF;     // un-normalised interpolation used by the forward (mt2DTE.jl:196-207)
            if (mode == 0) { numF = F0[id - 1] * d2 + F0[id] * d1; denF = G0[id - 1] * d2 + G0[id] * d1; }
            else           { numF = G0[id - 1] * d2 + G0[id] * d1; denF = F0[id - 1] * d2 + F0[id] * d1; }
            cplx Z = numF / denF;
            size_t di = (((size_t)ch * nFreq + f) * rx.nRx + r) * nC + zc;
            pred[di] = Z;
            size_t dob = ((size_t)f * rx.nRx + r) * nC + zc;     // obs / weights are shared by all chains
            cplx d;
            if constexpr (kRhoPhase) {
                // apparent resistivity and phase (compMTRespTE mt2DTE.jl:253-256, compMTRespTM mt2DTM.jl:236-239)
                const double rhoA = cabs2(Z) / (omega * kMu0), phs = atan2(Z.y, Z.x) * 180.0 / kPi;
                resp[di] = mk(rhoA, phs);
                const double wr = wd[dob], wp = wdPha[dob];
                const double rr = wr * (rhoA - obs[dob].x), rp = wp * (phs - obs[dob].y);     // no phase wrapping
                phi += 0.5 * (rr * rr + rp * rp);
                if (!wantAdjoint) continue;
                if (wr == 0.0 && wp == 0.0 && !vin) continue;
                const double vr = vin ? vin[di].x : wr * rr, vp = vin ? vin[di].y : wp * rp;
                const cplx V = (vr * 2.0 / (omega * kMu0)) * Z + (vp * 180.0 / kPi / cabs2(Z)) * mk(-Z.y, Z.x);
                d = cconj(V);
            } else {
                // apparent resistivity and phase (compMTRespTE mt2DTE.jl:253-256, compMTRespTM mt2DTM.jl:236-239): forward only
                if (respKind == 1) resp[di] = mk(cabs2(Z) / (omega * kMu0), atan2(Z.y, Z.x) * 180.0 / kPi);
                double w = wd[dob];
                cplx res = w * (Z - obs[dob]);
                phi += 0.5 * cabs2(res);
                if (!wantAdjoint) continue;
                cplx v = vin ? vin[di] : w * res;
                if (w == 0.0 && !vin) continue;
                d = cconj(v);
            }
            const int iL = rx.iL[r], iR = rx.iR[r];
            const double wl = rx.wL[r], wr = rx.wR[r];
            cplx numS, denS;     // normalised interpolation used by the sensitivities (dataFuncSens.jl:89-91)
            if (mode == 0) { numS = wl * F0[iL] + wr * F0[iR]; denS = wl * G0[iL] + wr * G0[iR]; }
            else           { numS = wl * G0[iL] + wr * G0[iR]; denS = wl * F0[iL] + wr * F0[iR]; }
            cplx nbar = d / denS;
            cplx dbar = -(d * numS / (denS * denS));
            if (mode == 0) {     // num <- F0, den <- Hy0
                aF0[iL] += wl * nbar; aF0[iR] += wr * nbar;
                aG0[iL] += wl * dbar; aG0[iR] += wr * dbar;
            } else {             // num <- Ey0, den <- F0
                aG0[iL] += wl * nbar; aG0[iR] += wr * nbar;
                aF0[iL] += wl * dbar; aF0[iR] += wr * dbar;
            }
        }
        if constexpr (kTipper) {
            const int tc = mi == cm.tmi ? cm.tc : -1;
            for (int r = 0; tc >= 0 && r < rx.nRx; ++r) {
                const int jL = rx.tjL[r], jR = rx.tjR[r], iL = rx.iL[r], iR = rx.iR[r];
                const double vl = rx.twL[r], vr = rx.twR[r], wl = rx.wL[r], wr = rx.wR[r];
                const cplx hzr = vl * ((F0[jL + 1] - F0[jL]) / M.yLen[jL] / iwmu) + vr * ((F0[jR + 1] - F0[jR]) / M.yLen[jR] / iwmu);
                const cplx hyr = wl * G0[iL] + wr * G0[iR];
                const cplx T = hzr / hyr;
                const size_t di = (((size_t)ch * nFreq + f) * rx.nRx + r) * nC + tc;
                pred[di] = T;
                if (respKind == 1) resp[di] = T;                  // the response toggle keeps the tipper complex
                const size_t dob = ((size_t)f * rx.nRx + r) * nC + tc;
                const double w = wd[dob];
                const cplx res = w * (T - obs[dob]);
                phi += 0.5 * cabs2(res);
                if (!wantAdjoint) continue;
                if (w == 0.0 && !vin) continue;
                const cplx d = cconj(vin ? vin[di] : w * res);
                const cplx hzbar = d / hyr / iwmu;
                const cplx aL = (vl / M.yLen[jL]) * hzbar, aR = (vr / M.yLen[jR]) * hzbar;
                aF0[jL + 1] += aL; aF0[jL] -= aL;
                aF0[jR + 1] += aR; aF0[jR] -= aR;
                const cplx hybar = -(d * T / hyr);
                aG0[iL] += wl * hybar; aG0[iR] += wr * hybar;
            }
        }
        phiSh = phi;
        aG0[1] += aG0[0];             // copied ends fold back onto their sources
        aG0[ny - 1] += aG0[ny];
    }
    __syncthreads();
    if (tid == 0) phiPart[sys] = phiSh;
    if (!wantAdjoint) return;
    // ---- push the Hy0/Ey0 adjoint through the half-cell correction (interior nodes) ----
    for (int i = tid + 1; i < ny; i += kRxThreads) {
        const double yb = 0.5 * M.yLen[i - 1] + 0.5 * M.yLen[i];
        const cplx u = aG0[i];
        if (mode == 0) {
            cplx a = u / h / iwmu;                       // HyH = -(F1-F0)/h/(i w mu0)
            aF1[i] -= a; aF0[i] += a;
            double sv = (0.5 * (sig1[i - 1] * M.yLen[i - 1]) + 0.5 * (sig1[i] * M.yLen[i])) / yb;
            cplx e = (sv * (0.5 * h)) * u;               // + sigma1v*ExQ*h/2
            aF0[i] += 0.75 * e; aF1[i] += 0.25 * e;
            cplx ExQ = 0.75 * F0[i] + 0.25 * F1[i];
            cplx svbar = ExQ * (0.5 * h) * u;            // d/d sigma1v
            // two-cell writes: resolved after the loop through per-node storage (no races)
            G0[i] = svbar;                               // reuse G0 as scratch: sigma1v-bar at node i
        } else {
            double rv = (0.5 * ((1.0 / sig1[i - 1]) * M.yLen[i - 1]) + 0.5 * ((1.0 / sig1[i]) * M.yLen[i])) / yb;
            cplx a = (rv * u) / h;                       // EyH = JyH*rho1v, JyH = (F1-F0)/h
            aF1[i] += a; aF0[i] -= a;
            cplx JyH = (F1[i] - F0[i]) / h;
            cplx e = -(iwmu * (0.5 * h)) * u;            // - i w mu0 HxQ h/2
            aF0[i] += 0.75 * e; aF1[i] += 0.25 * e;
            G0[i] = JyH * u;                             // rho1v-bar at node i
        }
    }
    __syncthreads();
    // gather the two-point stencils per cell j (no atomics):  adjoint of dQ = (Q[i]-Q[i-1])/yb_i * (-h/2)
    for (int j = tid; j < ny; j += kRxThreads) {
        cplx acc = mk(0.0, 0.0), qa = mk(0.0, 0.0);
        if (j >= 1) {           // node i = j uses Q[j] with +
            const int i = j;
            const double yb = 0.5 * M.yLen[i - 1] + 0.5 * M.yLen[i];
            acc += (-(0.5 * h) / yb) * aG0[i];
            double wgt = 0.5 * M.yLen[j] / yb;          // d sigma1v_i / d sigma_j  (or rho1v with 1/sigma)
            qa += (mode == 0) ? wgt * G0[i] : (-wgt / (sig1[j] * sig1[j])) * G0[i];
        }
        if (j + 1 <= ny - 1) {  // node i = j+1 uses Q[j] with -
            const int i = j + 1;
            const double yb = 0.5 * M.yLen[i - 1] + 0.5 * M.yLen[i];
            acc -= (-(0.5 * h) / yb) * aG0[i];
            double wgt = 0.5 * M.yLen[j] / yb;
            qa += (mode == 0) ? wgt * G0[i] : (-wgt / (sig1[j] * sig1[j])) * G0[i];
        }
        aQc[j] = acc;
        if (mode == 1) {        // EzQ = (0.75 Jz0 + 0.25 Jz1)/sigma1 : sigma adjoint  (dataFuncSens.jl:229)
            cplx jzq = Qc[j] * sig1[j];
            qa += acc * (-(jzq / (sig1[j] * sig1[j])));
        }
        qv[j] = qa;
    }
    __syncthreads();
    // HzQ / EzQ adjoint onto the node rows through the forward difference
    for (int n = tid; n <= ny; n += kRxThreads) {
        cplx a0 = mk(0.0, 0.0), a1 = mk(0.0, 0.0);
        // cell j = n-1 contributes +, cell j = n contributes -
        for (int s = 0; s < 2; ++s) {
            int j = n - 1 + s;
            if (j < 0 || j >= ny) continue;
            double sgn = (s == 0) ? 1.0 : -1.0;
            cplx wq;
            if (mode == 0) wq = aQc[j] / kMu0 / M.yLen[j] / iw;             // Bz = dF/yLen/(iw); HzQ = (.)/mu0
            else wq = -(aQc[j] / sig1[j] / M.yLen[j]);                        // Jz = -dF/yLen; EzQ = (.)/sigma1
            a0 += sgn * 0.75 * wq;
            a1 += sgn * 0.25 * wq;
        }
        aF0[n] += a0;
        aF1[n] += a1;
    }
    __syncthreads();
    cplx* so = srows + (size_t)sys * 2 * (ny + 1);
    for (int n = tid; n <= ny; n += kRxThreads) { so[n] = aF0[n]; so[ny + 1 + n] = aF1[n]; }
    cplx* qo = qrow + (size_t)sys * ny;
    for (int j = tid; j < ny; j += kRxThreads) qo[j] = qv[j];
    // adjoint right-hand side s[ii] in internal ordering (dense, zero elsewhere: the caller has cleared the vector — a memset
    // of the whole range instead of N stores by this one CTA)
    cplx* ar = adjrhs + (size_t)sys * M.N;
    for (int n = tid; n < 2 * (ny + 1); n += kRxThreads) {
        int row = n / (ny + 1), jn = n - row * (ny + 1), kn = M.zid + row;
        if (jn >= 1 && jn <= ny - 1 && kn >= 1 && kn <= M.nz - 1) ar[q_of(M, jn, kn)] = row ? aF1[jn] : aF0[jn];
    }
}

// ---------------------------------------------------------------------------------------------
// K9: 1-D sensitivity profiles needed by the matrix-free dBC^T t
//   (mt1DFieldSensMatrix MT1DSensitivity.jl:25-176, compImpJacMatrix :188-243, getBCDerivMatrix :253-333)
// One CTA per (system, profile) with profile 0 = left column, 1 = right column, 2 = row-mean.
// Outputs: bcs (the derivative routine's own boundary field: nb entries, used by the TM term),
//          and nothing else is stored: the (nz+1) x nz derivative blocks are contracted with t on the fly
//          in k_bc_contract below, which re-runs the per-column recursion from the scalars saved here.
struct ProfScalars {         // per (system, profile), arrays of length nz+1 (layers incl. half-space)
    cplx* ka;                // wavenumbers (no eps0 term, MT1DSensitivity.jl:59)
    cplx* dka;               // d ka / d sigma
    cplx* eu;                // up-going amplitude at the top of each layer
    cplx* ed;
    cplx* dz1;               // d Z_top / d sigma_layer   (zimpDeri)
    cplx* z1;                // [1]
    int* jbreak;             // [1] index j at which the overflow guard fired (nz if never)
    cplx* kr;                // [nz] ka[j]/ka[j+1]            } layer transfer factors of the top-down propagation, shared by
    cplx* expt;              // [nz] exp(i ka[j] h_j)          } every column of the sensitivity recursion (sens_column)
    cplx* expr;              // [nz] 1/expt
    cplx* m11;               // [nz] (1+kr) expt   } the 2x2 layer transfer matrix
    cplx* m12;               // [nz] (1-kr) expr   }
    cplx* m21;               // [nz] (1-kr) expt   }
    cplx* m22;               // [nz] (1+kr) expr   }
    cplx* kao;               // [nz] ka[j+1] / (omega mu)
    cplx* dS;                // [4*nz] d(layer matrix j)/d sigma_j     (d11,d12,d21,d22)
    cplx* dN;                // [4*nz] d(layer matrix j)/d sigma_{j+1}
};
__device__ __forceinline__ double sens_sigma(const MeshDev& M, const double* __restrict__ sig, int prof, int k, const double* meanSig) {
    if (prof == 0) return sig[k * M.ny];
    if (prof == 1) return sig[k * M.ny + M.ny - 1];
    return meanSig[k];
}
// row means of sigma: mean(sig2D, dims=2) (MT1DSensitivity.jl:313).  grid (nz, nChains), block 128
__global__ void k_row_mean(int ny, int nz, const double* __restrict__ sigma, double* __restrict__ meanSig) {
    __shared__ double sh[128];
    const int k = blockIdx.x, ch = blockIdx.y;
    const double* s = sigma + (size_t)ch * ny * nz + (size_t)k * ny;
    // pairwise-ish: fixed order so the result is deterministic
    double acc = 0.0;
    for (int j = threadIdx.x; j < ny; j += 128) acc += s[j];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) meanSig[(size_t)ch * nz + k] = sh[0] / ny;
}

// scratch layout per (sys,prof): 5*(nz+1) cplx + 1 cplx + pad + 16*nz cplx ; see prof_ptrs
__host__ __device__ inline size_t prof_stride(int nz) { return 5 * (size_t)(nz + 1) + 2 + 16 * (size_t)nz; }
__device__ __forceinline__ ProfScalars prof_ptrs(cplx* base, int nz) {
    ProfScalars P;
    P.ka = base; P.dka = base + (nz + 1); P.eu = base + 2 * (nz + 1); P.ed = base + 3 * (nz + 1);
    P.dz1 = base + 4 * (nz + 1); P.z1 = base + 5 * (nz + 1);
    P.jbreak = reinterpret_cast<int*>(base + 5 * (nz + 1) + 1);
    P.kr = base + 5 * (nz + 1) + 2; P.expt = P.kr + nz; P.expr = P.expt + nz;
    P.m11 = P.expr + nz; P.m12 = P.m11 + nz; P.m21 = P.m12 + nz; P.m22 = P.m21 + nz; P.kao = P.m22 + nz;
    P.dS = P.kao + nz; P.dN = P.dS + 4 * nz;
    return P;
}
// serial part: one thread per (sys, prof).  grid: ceil(nSys*3/64), block 64
__global__ void k_sens_scalars(MeshDev M, SysMap sm, int nSys, const double* __restrict__ freqs,
                               const double* __restrict__ sigma, const double* __restrict__ meanSig,
                               cplx* __restrict__ scratch, cplx* __restrict__ bcs) {
    int id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= nSys * 3) return;
    const int sys = id / 3, prof = id - sys * 3;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    const int nz = M.nz, ny = M.ny, nL = nz + 1;
    const double* sig = sigma + (size_t)ch * M.nCell;
    const double* ms = meanSig + (size_t)ch * nz;
    ProfScalars P = prof_ptrs(scratch + (size_t)id * prof_stride(nz), nz);
    const double omega = 2.0 * kPi * freqs[f], omu = omega * kMu0;
    auto sg = [&](int j) { return sens_sigma(M, sig, prof, j < nz ? j : nz - 1, ms); };
    // ---- compImpJacMatrix: bottom-up, storing dZ_ZP1 in P.eu and dZ_sigma in P.dz1 temporarily ----
    cplx Z = mk(0.0, 0.0);
    for (int j = nL - 1; j >= 0; --j) {
        double s = sg(j);
        cplx k = csqrt_(mk(0.0, -omu * s));
        P.ka[j] = k;
        P.dka[j] = mk(0.0, -omu / 2.0) / k;
        cplx Zt = omu / k;
        cplx k3 = k * k * k;
        cplx dZt = mk(0.0, omu * omu) / (2.0 * k3);
        if (j == nL - 1) { Z = Zt; P.dz1[j] = dZt; P.eu[j] = mk(0.0, 0.0); continue; }
        cplx RI = (Zt - Z) / (Zt + Z);
        cplx kh2 = k * (2.0 * M.zLen[j]);
        cplx ex = cexp_(mk(kh2.y, -kh2.x));                 // exp(-2i k h)
        cplx L = RI * ex;
        cplx one = mk(1.0, 0.0);
        cplx Ztmp = Zt * (one - L) / (one + L);
        cplx zs = Zt + Z;
        cplx dL = 2.0 * Z / (zs * zs) * ex * dZt + (mk(0.0, -2.0 * M.zLen[j]) * L) * (mk(0.0, -omu) / 2.0 / k);
        cplx den = (one + L) * zs;
        P.eu[j] = 4.0 * Zt * Zt * ex / (den * den);         // dZ_ZP1[j]
        P.dz1[j] = dZt * (one - L) / (one + L) + Zt * (-2.0) / ((one + L) * (one + L)) * dL;   // dZ_sigma[j]
        Z = Ztmp;
    }
    // chain rule (MT1DSensitivity.jl:232-240): zimpDeri[i] = prod_{j<i} dZ_ZP1[j] * dZ_sigma[i]
    {
        cplx prod = mk(1.0, 0.0);
        for (int i = 1; i < nL; ++i) {
            prod = prod * P.eu[i - 1];
            P.dz1[i] = prod * P.dz1[i];
        }
    }
    *P.z1 = Z;
    // ---- top amplitudes and top-down propagation of the amplitudes ----
    const cplx z1 = Z, k1 = P.ka[0];
    cplx eu, ed;
    if (mode == 0) {
        cplx r = omu / (z1 * k1);
        eu = 0.5 * (mk(1.0, 0.0) - r); ed = 0.5 * (mk(1.0, 0.0) + r);
    } else {
        cplx r = z1 * k1 / omu;
        cplx hu = 0.5 * (mk(1.0, 0.0) - r), hd = 0.5 * (mk(1.0, 0.0) + r);
        eu = -(omu / k1) * hu; ed = (omu / k1) * hd;
    }
    P.eu[0] = eu; P.ed[0] = ed;
    int jb = nz;
    for (int j = 0; j < nz; ++j) {
        cplx kr = P.ka[j] / P.ka[j + 1];
        cplx kh = P.ka[j] * M.zLen[j];
        cplx expt = cexp_(mk(-kh.y, kh.x));
        cplx expr = 1.0 / expt;
        cplx one = mk(1.0, 0.0);
        // per-layer factors reused (bit-identical) by every column of the sensitivity recursion (sens_column)
        P.kr[j] = kr; P.expt[j] = expt; P.expr[j] = expr;
        P.m11[j] = (one + kr) * expt; P.m12[j] = (one - kr) * expr; P.m21[j] = (one - kr) * expt; P.m22[j] = (one + kr) * expr;
        P.kao[j] = P.ka[j + 1] / omu;
        {   // derivatives of the layer matrix w.r.t. its own layer (kp == j) and the next one (kp == j+1), MT1DSensitivity.jl:100-118
            const cplx kaj = P.ka[j], kaj1 = P.ka[j + 1];
            const cplx dexpt = mk(0.0, M.zLen[j]) * expt * P.dka[j];
            const cplx dexpr = mk(0.0, -M.zLen[j]) * expr * P.dka[j];
            cplx dkr = P.dka[j] / kaj1;
            P.dS[4 * j + 0] = (one + kr) * dexpt + expt * dkr; P.dS[4 * j + 1] = (one - kr) * dexpr - expr * dkr;
            P.dS[4 * j + 2] = (one - kr) * dexpt - expt * dkr; P.dS[4 * j + 3] = (one + kr) * dexpr + expr * dkr;
            const cplx zero = mk(0.0, 0.0);
            dkr = zero - kaj / (kaj1 * kaj1) * P.dka[j + 1];
            P.dN[4 * j + 0] = (one + kr) * zero + expt * dkr; P.dN[4 * j + 1] = (one - kr) * zero - expr * dkr;
            P.dN[4 * j + 2] = (one - kr) * zero - expt * dkr; P.dN[4 * j + 3] = (one + kr) * zero + expr * dkr;
        }
        cplx nu = (0.5 * (one + kr) * expt) * eu + (0.5 * (one - kr) * expr) * ed;
        cplx nd = (0.5 * (one - kr) * expt) * eu + (0.5 * (one + kr) * expr) * ed;
        double e2 = cabs_(nu + nd), e1 = cabs_(eu + ed);
        if (e2 - e1 > 0.0 || isnan(e2)) {
            jb = j;
            for (int r = j + 1; r <= nz; ++r) { P.eu[r] = mk(0.0, 0.0); P.ed[r] = mk(0.0, 0.0); }
            break;
        }
        eu = nu; ed = nd;
        P.eu[j + 1] = eu; P.ed[j + 1] = ed;
    }
    *P.jbreak = jb;
    // ---- the derivative routine's own boundary field (MT1DSensitivity.jl:276,283,325) ----
    cplx* b = bcs + (size_t)sys * M.nb;
    auto fieldAt = [&](int r) {
        cplx a = P.eu[r], c = P.ed[r];
        return (mode == 0) ? a + c : (c * P.ka[r] - a * P.ka[r]) / omu;
    };
    if (prof == 0) for (int r = 1; r <= nz; ++r) b[ny + 1 + (r - 1)] = fieldAt(r);
    else if (prof == 1) for (int r = 1; r <= nz; ++r) b[ny + 1 + nz + (r - 1)] = fieldAt(r);
    else {
        cplx v = fieldAt(nz);
        for (int j = 0; j < ny - 1; ++j) b[ny + 1 + 2 * nz + j] = v;
        for (int j = 0; j <= ny; ++j) b[j] = mk(1.0, 0.0);
    }
}

// per-column recursion: thread kp (derivative w.r.t. layer kp) returns sum_r dF[r][kp]*t[r] for rows r=1..nz
// (profiles 0,1) or dF[nz][kp] (profile 2).  Follows MT1DSensitivity.jl:66-157 entry by entry.
__device__ inline cplx sens_column(const MeshDev& M, const ProfScalars& P, int mode, double omu, int kp,
                                   const cplx* __restrict__ tvec, bool lastRowOnly) {
    const int nz = M.nz;
    const cplx z1 = *P.z1, k1 = P.ka[0];
    const int jb = *P.jbreak;
    const cplx zero = mk(0.0, 0.0), one = mk(1.0, 0.0);
    const cplx dz = P.dz1[kp];
    const cplx dk0 = (kp == 0) ? P.dka[0] : zero;
    cplx dEu, dEd, dHu, dHd;
    if (mode == 0) {
        dEu = 0.5 * omu / (z1 * k1) * (one / z1 * dz + one / k1 * dk0);
        dEd = -dEu;
        dHu = -(P.eu[0] / omu) * dk0 - P.ka[0] / omu * dEu;
        dHd = (P.ed[0] / omu) * dk0 + P.ka[0] / omu * dEd;
    } else {
        dHu = (-0.5 / omu) * (z1 * dk0 + k1 * dz);
        dHd = -dHu;
        cplx a = (omu / (k1 * k1)) * dk0;
        dEu = 0.5 * (dz + a);
        dEd = 0.5 * (dz - a);
    }
    cplx acc = zero;
    for (int j = 0; j < nz; ++j) {
        // row j+1 from row j
        if (j > jb) { dEu = dEd = dHu = dHd = zero; if (lastRowOnly) continue; else continue; }
        const cplx eu = P.eu[j], ed = P.ed[j];
        // (d11 d12; d21 d22) = d/dsigma_kp of the layer matrix: non-zero only for kp == j or kp == j+1
        cplx nEu, nEd;
        if (kp == j || kp == j + 1) {
            const cplx* D = (kp == j) ? P.dS + 4 * j : P.dN + 4 * j;      // precomputed once per layer in k_sens_scalars
            nEu = 0.5 * (D[0] * eu + P.m11[j] * dEu + D[1] * ed + P.m12[j] * dEd);
            nEd = 0.5 * (D[2] * eu + P.m21[j] * dEu + D[3] * ed + P.m22[j] * dEd);
        } else {                                      // the derivative terms are exact zeros: same sums without them
            nEu = 0.5 * (P.m11[j] * dEu + P.m12[j] * dEd);
            nEd = 0.5 * (P.m21[j] * dEu + P.m22[j] * dEd);
        }
        // NB at j == jb the reference computes row j+1 from the *pre-guard* amplitudes and then zeroes
        // columns >= j+1 of that row (MT1DSensitivity.jl:131-151); P.eu/ed[j+1] are already zero there, but
        // dHu/dHd use epu/epd = the freshly propagated (non-zeroed) amplitudes, so recompute them.
        const cplx kao = P.kao[j];
        cplx nHu, nHd;
        if (kp == j + 1) {
            cplx epu = P.eu[j + 1], epd = P.ed[j + 1];
            if (j == jb) {
                const cplx kr = P.kr[j], expt = P.expt[j], expr = P.expr[j];
                epu = (0.5 * (one + kr) * expt) * eu + (0.5 * (one - kr) * expr) * ed;
                epd = (0.5 * (one - kr) * expt) * eu + (0.5 * (one + kr) * expr) * ed;
            }
            const cplx dk1 = P.dka[j + 1];
            nHu = -(epu / omu) * dk1 - kao * nEu;
            nHd = (epd / omu) * dk1 + kao * nEd;
        } else {
            nHu = -(kao * nEu);
            nHd = kao * nEd;
        }
        if (j == jb && kp >= j + 1) { nEu = nEd = nHu = nHd = zero; }
        dEu = nEu; dEd = nEd; dHu = nHu; dHd = nHd;
        cplx dF = (mode == 0) ? dEu + dEd : dHu + dHd;
        if (lastRowOnly) { if (j == nz - 1) acc = dF; }
        else acc += dF * tvec[j];                       // tvec[j] <-> node row j+1
    }
    if (lastRowOnly && jb < nz - 1) acc = zero;           // rows beyond the guard stay zero
    return acc;
}

// ---------------------------------------------------------------------------------------------
// K10: gradient contraction -> Gpart[sys][nCell] (real part of the cell gradient), two kernels:
//   k_contract_cols   one CTA per system: t = -Aio^T lambda + s[io], then the boundary-derivative columns dBC^T t by per-column
//                     recursions over the three 1-D profiles (their per-layer factors are staged in shared memory first: the
//                     recursion is a chain of dependent steps and must not wait on global loads);
//   k_contract_cells  fully parallel over cells.
//   TE: compJacTMatVec.jl:235-244 ; TM: :306-318 ; Q term :198-214, :269-285 ; final real() :325-327
constexpr int kConThreads = 320;      // >= 3*nz columns of the per-column recursions at nz = 100: one round
__host__ __device__ inline size_t contract_cols_out(int ny, int nz) { return 3 * (size_t)nz + ny; }      // oL | oR | oM | colw
// shared memory of k_contract_cols: the t vectors, plus the staged profile scalars when they fit (staged = 1)
__host__ __device__ inline size_t contract_cols_smem(int ny, int nz, int staged) {
    return ((size_t)(2 * nz + (ny - 1)) + (staged ? 3 * prof_stride(nz) : 0)) * sizeof(cplx);
}
__global__ void __launch_bounds__(kConThreads)
k_contract_cols(MeshDev M, SysMap sm, const double* __restrict__ freqs, const double* __restrict__ sigma,
                const cplx* __restrict__ Lam, const cplx* __restrict__ srows, cplx* __restrict__ scratch,
                cplx* __restrict__ cols, int staged, int sys0) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int ny = M.ny, nz = M.nz;
    cplx* tL = reinterpret_cast<cplx*>(smraw);   // nz   (node rows 1..nz)
    cplx* tR = tL + nz;                            // nz
    cplx* tB = tR + nz;                            // ny-1 (nodes jn = 1..ny-1)
    cplx* prof = staged ? tB + (ny - 1)            // 3 * prof_stride(nz): the three profiles' scalars, staged
                        : scratch + (size_t)(blockIdx.x + sys0) * 3 * prof_stride(nz);       // (too deep a mesh: read them in place)
    const int sys = blockIdx.x + sys0;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    const int tid = threadIdx.x;
    const double omega = 2.0 * kPi * freqs[f], omu = omega * kMu0;
    const double* sig = sigma + (size_t)ch * M.nCell;
    const cplx* Ls = Lam + (size_t)sys * M.nNode;
    const cplx* so = srows + (size_t)sys * 2 * (ny + 1);
    cplx* out = cols + (size_t)sys * contract_cols_out(ny, nz);
    cplx *oL = out, *oR = out + nz, *oM = out + 2 * nz, *colw = out + 3 * nz;
    auto node = [&](int jn, int kn) { return (size_t)kn * (ny + 1) + jn; };
    auto sAt = [&](int jn, int kn) {       // s on boundary nodes: only node rows zid, zid+1 are non-zero
        int row = kn - M.zid;
        return (row == 0 || row == 1) ? so[row * (ny + 1) + jn] : mk(0.0, 0.0);
    };
    if (staged) {
        const cplx* src = scratch + (size_t)sys * 3 * prof_stride(nz);
        for (size_t i = tid; i < 3 * prof_stride(nz); i += kConThreads) prof[i] = src[i];
    }
    // t = -Aio^T lambda + s[io]  (Aio[n,b] = -W(edge n-b)):  t_b = W * lambda_n + s_b
    for (int kn = tid + 1; kn <= nz; kn += kConThreads) {
        cplx l = mk(0.0, 0.0), r = mk(0.0, 0.0);
        if (kn <= nz - 1) {
            StencilW w1 = stencil_at(M, sig, mode, 1, kn);
            l = w1.wyL * Ls[node(1, kn)];
            StencilW w2 = stencil_at(M, sig, mode, ny - 1, kn);
            r = w2.wyR * Ls[node(ny - 1, kn)];
        }
        tL[kn - 1] = l + sAt(0, kn);
        tR[kn - 1] = r + sAt(ny, kn);
    }
    for (int jn = tid + 1; jn <= ny - 1; jn += kConThreads) {
        StencilW w = stencil_at(M, sig, mode, jn, nz - 1);
        tB[jn - 1] = w.wzD * Ls[node(jn, nz - 1)] + sAt(jn, nz);
    }
    __syncthreads();
    // dBC^T t: per-column recursions (MT1DSensitivity.jl), three profiles
    for (int w = tid; w < 3 * nz; w += kConThreads) {
        int pr = w / nz, kp = w - pr * nz;
        ProfScalars P = prof_ptrs(prof + (size_t)pr * prof_stride(nz), nz);
        if (pr == 0) oL[kp] = sens_column(M, P, mode, omu, kp, tL, false);
        else if (pr == 1) oR[kp] = sens_column(M, P, mode, omu, kp, tR, false);
        else oM[kp] = sens_column(M, P, mode, omu, kp, nullptr, true);
    }
    for (int jc = tid; jc < ny; jc += kConThreads) {
        cplx a = mk(0.0, 0.0);
        if (jc + 1 <= ny - 1) {       // bottom node jn = jc+1 : this cell is its left cell (weight dy[jn-1])
            int jn = jc + 1;
            a += (M.yLen[jn - 1] / (M.yLen[jn - 1] + M.yLen[jn])) * tB[jn - 1];
        }
        if (jc >= 1) {                // bottom node jn = jc : this cell is its right cell (weight dy[jn])
            int jn = jc;
            a += (M.yLen[jn] / (M.yLen[jn - 1] + M.yLen[jn])) * tB[jn - 1];
        }
        colw[jc] = a;
    }
}

// grid (ceil(nCell/256), nSys), block 256
__global__ void __launch_bounds__(256)
k_contract_cells(MeshDev M, SysMap sm, const double* __restrict__ freqs, const double* __restrict__ sigma,
                 const cplx* __restrict__ F, const cplx* __restrict__ Lam, const cplx* __restrict__ qrow,
                 const cplx* __restrict__ bcs, const cplx* __restrict__ cols, double* __restrict__ Gpart, int sys0) {
    const int ny = M.ny, nz = M.nz;
    const int sys = blockIdx.y + sys0;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= M.nCell) return;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    const double omega = 2.0 * kPi * freqs[f];
    const double* sig = sigma + (size_t)ch * M.nCell;
    const cplx* Fs = F + (size_t)sys * M.nNode;
    const cplx* Ls = Lam + (size_t)sys * M.nNode;
    const cplx* bs = bcs + (size_t)sys * M.nb;
    const cplx* in = cols + (size_t)sys * contract_cols_out(ny, nz);
    const cplx *oL = in, *oR = in + nz, *oM = in + 2 * nz, *colw = in + 3 * nz;
    const cplx* qo = qrow + (size_t)sys * ny;
    auto node = [&](int jn, int kn) { return (size_t)kn * (ny + 1) + jn; };
    // field with the derivative routine's boundary values (TM term, compJacTMatVec.jl:309,315)
    auto Hf = [&](int jn, int kn) -> cplx {
        if (jn >= 1 && jn <= ny - 1 && kn >= 1 && kn <= nz - 1) return Fs[node(jn, kn)];
        if (kn == 0) return bs[jn];
        if (jn == 0) return bs[ny + 1 + (kn - 1)];
        if (jn == ny) return bs[ny + 1 + nz + (kn - 1)];
        return bs[ny + 1 + 2 * nz + (jn - 1)];
    };
    const int kc = c / ny, jc = c - kc * ny;
    const double dy = M.yLen[jc], dz = M.zLen[kc], area = dy * dz;
    cplx g = mk(0.0, 0.0);
    if (mode == 0) {
        cplx sum = mk(0.0, 0.0);
#pragma unroll
        for (int dk = 0; dk < 2; ++dk)
#pragma unroll
            for (int dj = 0; dj < 2; ++dj) {
                int jn = jc + dj, kn = kc + dk;
                if (jn >= 1 && jn <= ny - 1 && kn >= 1 && kn <= nz - 1) sum += 0.25 * (Fs[node(jn, kn)] * Ls[node(jn, kn)]);
            }
        g = mk(0.0, -omega) * (area * sum);
    } else {
        // four edges of the cell: gradient of H (with bcs boundary) times -(gradient of lambda), weight 1/2
        cplx sum = mk(0.0, 0.0);
#pragma unroll
        for (int dk = 0; dk < 2; ++dk) {     // y-edges on node rows kc, kc+1
            int kn = kc + dk;
            cplx gh = (Hf(jc + 1, kn) - Hf(jc, kn)) / dy;
            cplx gl = (Ls[node(jc + 1, kn)] - Ls[node(jc, kn)]) / dy;
            sum += 0.5 * (gh * (-gl));
        }
#pragma unroll
        for (int dj = 0; dj < 2; ++dj) {     // z-edges on node columns jc, jc+1
            int jn = jc + dj;
            cplx gh = (Hf(jn, kc + 1) - Hf(jn, kc)) / dz;
            cplx gl = (Ls[node(jn, kc + 1)] - Ls[node(jn, kc)]) / dz;
            sum += 0.5 * (gh * (-gl));
        }
        const double s = sig[c];
        g = (area * (-1.0 / (s * s))) * sum;
    }
    if (jc == 0) g += oL[kc];
    if (jc == ny - 1) g += oR[kc];
    g += oM[kc] * colw[jc];
    if (kc == M.zid) g += qo[jc];
    Gpart[(size_t)sys * M.nCell + c] = g.x;
}

// ---------------------------------------------------------------------------------------------
// K12: tangent (forward) mode J dsig, the transpose of K9 / K10 / the adjoint of K6+K7 term by term (hmcmt_jvec, DESIGN 4.7).
// dsig [nChains][nAC] is the conductivity perturbation of the active cells; an inactive cell has none.
__device__ __forceinline__ double dsig_cell(const int* __restrict__ cell2act, const double* __restrict__ dsig, int c) {
    const int a = cell2act[c];
    return a >= 0 ? dsig[a] : 0.0;
}
// sum_kp ds(kp) dF[row][kp] of the columns sens_column computes, rows 1..nz into out[0..nz-1] (or null: the last row only,
// returned).  The columns share one recursion over the layers; only their starting values (through Z_top) and the two layer
// matrices a column's own layer enters differ, so the sum runs that recursion once with the weighted sums of those terms.
// The overflow guard of sens_column: rows past jb+1 are zero and row jb+1 keeps the columns kp <= jb only — a second state
// `lo` carries the part of the sum from those columns (the deeper ones enter rows <= jb only through Z_top).
template <typename DS>
__device__ cplx sens_tangent(const MeshDev& M, const ProfScalars& P, int mode, double omu, DS ds, cplx* __restrict__ out) {
    const int nz = M.nz, jb = *P.jbreak;
    const cplx z1 = *P.z1, k1 = P.ka[0], zero = mk(0.0, 0.0), one = mk(1.0, 0.0);
    cplx dz = zero, dzLo = zero;
    for (int kp = 0; kp < nz; ++kp) {
        const cplx t = ds(kp) * P.dz1[kp];
        dz += t;
        if (kp <= jb) dzLo += t;
    }
    const cplx dk0 = ds(0) * P.dka[0];
    auto start = [&](cplx d, cplx& eu, cplx& ed) {
        if (mode == 0) {
            eu = 0.5 * omu / (z1 * k1) * (one / z1 * d + one / k1 * dk0);
            ed = -eu;
        } else {
            const cplx a = (omu / (k1 * k1)) * dk0;
            eu = 0.5 * (d + a);
            ed = 0.5 * (d - a);
        }
    };
    cplx Eu, Ed, Lu, Ld;
    start(dz, Eu, Ed);
    start(dzLo, Lu, Ld);
    cplx last = zero;
    for (int j = 0; j < nz; ++j) {
        cplx dF = zero;
        if (j <= jb) {
            const cplx eu = P.eu[j], ed = P.ed[j];
            const double sj = ds(j), sn = (j + 1 < nz && j < jb) ? ds(j + 1) : 0.0;   // columns kp = j, j+1 (kp = jb+1 is cut)
            const cplx* S = P.dS + 4 * j;
            const cplx* N = P.dN + 4 * j;
            const cplx iu = sj * (S[0] * eu + S[1] * ed) + sn * (N[0] * eu + N[1] * ed);
            const cplx id = sj * (S[2] * eu + S[3] * ed) + sn * (N[2] * eu + N[3] * ed);
            const cplx bu = (j == jb) ? Lu : Eu, bd = (j == jb) ? Ld : Ed;
            const cplx nEu = 0.5 * (P.m11[j] * bu + P.m12[j] * bd + iu);
            const cplx nEd = 0.5 * (P.m21[j] * bu + P.m22[j] * bd + id);
            if (j < jb) {
                const cplx lu = 0.5 * (P.m11[j] * Lu + P.m12[j] * Ld + iu);
                Ld = 0.5 * (P.m21[j] * Lu + P.m22[j] * Ld + id);
                Lu = lu;
            }
            Eu = nEu; Ed = nEd;
            if (mode == 0) dF = nEu + nEd;
            else {
                const cplx kao = P.kao[j], dk1 = sn * P.dka[j + 1];
                dF = (kao * nEd - kao * nEu) + (P.ed[j + 1] / omu) * dk1 - (P.eu[j + 1] / omu) * dk1;
            }
        }
        if (out) out[j] = dF;
        last = dF;
    }
    return last;
}
// dbc = dBC dsig: one thread per profile p of a system (p = 0 left, 1 right column, p >= 2 bottom node jn = p - 1), each
// O(nz); the top row has no derivative.  grid (ceil((ny+1)/128), nSys), block 128
__global__ void __launch_bounds__(128)
k_bc_tangent(MeshDev M, SysMap sm, const double* __restrict__ freqs, const int* __restrict__ cell2act, const double* __restrict__ dsig,
             int nAC, const cplx* __restrict__ scratch, cplx* __restrict__ dbc) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x, sys = blockIdx.y, ny = M.ny, nz = M.nz;
    if (p > ny) return;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    const double omu = 2.0 * kPi * freqs[f] * kMu0;
    const double* ds = dsig + (size_t)ch * nAC;
    cplx* b = dbc + (size_t)sys * M.nb;
    b[p] = mk(0.0, 0.0);                                                  // top row (ny + 1 entries, one per thread)
    const int pr = p < 2 ? p : 2;
    const ProfScalars P = prof_ptrs(const_cast<cplx*>(scratch) + ((size_t)sys * 3 + pr) * prof_stride(nz), nz);
    if (pr < 2) {
        const int jc = pr == 0 ? 0 : ny - 1;
        sens_tangent(M, P, mode, omu, [&](int k) { return dsig_cell(cell2act, ds, k * ny + jc); }, b + ny + 1 + pr * nz);
    } else {
        const int jn = p - 1;
        const double yl = M.yLen[jn - 1], yr = M.yLen[jn], wl = yl / (yl + yr), wr = yr / (yl + yr);     // the colw weights
        b[ny + 1 + 2 * nz + (jn - 1)] = sens_tangent(
            M, P, mode, omu, [&](int k) { return wl * dsig_cell(cell2act, ds, k * ny + jn - 1) + wr * dsig_cell(cell2act, ds, k * ny + jn); },
            nullptr);
    }
}

// tangent right-hand side on the interior unknowns (internal ordering): the coefficient of Lambda_n in k_contract_cells applied
// to dsig, plus W dbc of the t = W lambda + s step of k_contract_cols.  grid (ceil(N/256), nSys)
__global__ void __launch_bounds__(256)
k_tangent_rhs(MeshDev M, SysMap sm, const double* __restrict__ freqs, const double* __restrict__ sigma, const int* __restrict__ cell2act,
              const double* __restrict__ dsig, int nAC, const cplx* __restrict__ F, const cplx* __restrict__ bcs,
              const cplx* __restrict__ dbc, cplx* __restrict__ rhs) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= M.N) return;
    const int sys = blockIdx.y, ny = M.ny, nz = M.nz;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    int jn, kn;
    jk_of(M, q, jn, kn);
    const double omega = 2.0 * kPi * freqs[f];
    const double* sig = sigma + (size_t)ch * M.nCell;
    const double* ds = dsig + (size_t)ch * nAC;
    const cplx* Fs = F + (size_t)sys * M.nNode;
    const cplx* bs = bcs + (size_t)sys * M.nb;
    auto node = [&](int j, int k) { return (size_t)k * (ny + 1) + j; };
    auto Hf = [&](int j, int k) -> cplx {
        if (j >= 1 && j <= ny - 1 && k >= 1 && k <= nz - 1) return Fs[node(j, k)];
        if (k == 0) return bs[j];
        if (j == 0) return bs[ny + 1 + (k - 1)];
        if (j == ny) return bs[ny + 1 + nz + (k - 1)];
        return bs[ny + 1 + 2 * nz + (j - 1)];
    };
    cplx r = mk(0.0, 0.0);
#pragma unroll
    for (int dk = 0; dk < 2; ++dk)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj) {
            const int jc = jn - 1 + dj, kc = kn - 1 + dk, c = kc * ny + jc;
            const double d = dsig_cell(cell2act, ds, c);
            if (d == 0.0) continue;
            const double dy = M.yLen[jc], dz = M.zLen[kc], area = dy * dz;
            if (mode == 0) {
                r += (d * area) * (mk(0.0, -omega) * (0.25 * Fs[node(jn, kn)]));
            } else {
                const double s = sig[c], pre = area * (-1.0 / (s * s)) * 0.5;
                const cplx ghy = (Hf(jc + 1, kn) - Hf(jc, kn)) / dy;          // the cell's y-edge on node row kn
                const cplx ghz = (Hf(jn, kc + 1) - Hf(jn, kc)) / dz;          // its z-edge on node column jn
                const double sy = (jn == jc + 1) ? 1.0 : -1.0, sz = (kn == kc + 1) ? 1.0 : -1.0;
                r += (d * pre) * (ghy * (-sy / dy) + ghz * (-sz / dz));
            }
        }
    if (jn == 1 || jn == ny - 1 || kn == nz - 1) {
        const StencilW w = stencil_at(M, sig, mode, jn, kn);
        const cplx* b = dbc + (size_t)sys * M.nb;
        if (jn == 1) r += w.wyL * b[ny + 1 + (kn - 1)];
        if (jn == ny - 1) r += w.wyR * b[ny + 1 + nz + (kn - 1)];
        if (kn == nz - 1) r += w.wzD * b[ny + 1 + 2 * nz + (jn - 1)];
    }
    rhs[(size_t)sys * M.N + q] = r;
}

// Tangent receiver functional: the forward mode of k_rx_adjoint's reverse recipe (its normalised sensitivity weights), from the
// field tangent dF on node rows zid, zid+1 (interior: the tangent solve, boundary: dbc) and dsig on cell row zid, into the full
// data layout jv (rho / phase plans: the real pair (d rho_a, d phase)).  One CTA per system; the receivers are independent.
template <bool kRhoPhase, bool kTipper>
__global__ void __launch_bounds__(kRxThreads)
k_rx_tangent(MeshDev M, RxDev rx, SysMap sm, CompMap cm, const double* __restrict__ freqs, const double* __restrict__ sigma,
             const int* __restrict__ cell2act, const double* __restrict__ dsig, int nAC, const cplx* __restrict__ F,
             const cplx* __restrict__ dF, cplx* __restrict__ jv) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int ny = M.ny;
    cplx* F0 = reinterpret_cast<cplx*>(smraw);        // ny+1
    cplx* F1 = F0 + (ny + 1);
    cplx* G0 = F1 + (ny + 1);
    cplx* dF0 = G0 + (ny + 1);
    cplx* dF1 = dF0 + (ny + 1);
    cplx* dG0 = dF1 + (ny + 1);
    cplx* Qc = dG0 + (ny + 1);                         // ny
    cplx* dQc = Qc + ny;                               // ny
    const int sys = blockIdx.x;
    int ch, mi, mode, f;
    sys_decode(sm, sys, ch, mi, mode, f);
    const int tid = threadIdx.x;
    const double omega = 2.0 * kPi * freqs[f];
    const double h = M.zLen[M.zid];
    const double* sig1 = sigma + (size_t)ch * M.nCell + (size_t)M.zid * ny;
    const double* ds = dsig + (size_t)ch * nAC;
    const int* c2a = cell2act + (size_t)M.zid * ny;
    const cplx* Fs = F + (size_t)sys * M.nNode;
    const cplx* dFs = dF + (size_t)sys * M.nNode;
    const cplx iw = mk(0.0, omega), iwmu = mk(0.0, omega * kMu0);
    for (int j = tid; j <= ny; j += kRxThreads) {
        F0[j] = Fs[(size_t)M.zid * (ny + 1) + j];
        F1[j] = Fs[(size_t)(M.zid + 1) * (ny + 1) + j];
        dF0[j] = dFs[(size_t)M.zid * (ny + 1) + j];
        dF1[j] = dFs[(size_t)(M.zid + 1) * (ny + 1) + j];
    }
    __syncthreads();
    for (int j = tid; j < ny; j += kRxThreads) {
        if (mode == 0) {
            Qc[j] = (0.75 * ((F0[j + 1] - F0[j]) / M.yLen[j] / iw) + 0.25 * ((F1[j + 1] - F1[j]) / M.yLen[j] / iw)) / kMu0;
            dQc[j] = (0.75 * ((dF0[j + 1] - dF0[j]) / M.yLen[j] / iw) + 0.25 * ((dF1[j + 1] - dF1[j]) / M.yLen[j] / iw)) / kMu0;
        } else {
            const cplx jzq = 0.75 * (-((F0[j + 1] - F0[j]) / M.yLen[j])) + 0.25 * (-((F1[j + 1] - F1[j]) / M.yLen[j]));
            const cplx djzq = 0.75 * (-((dF0[j + 1] - dF0[j]) / M.yLen[j])) + 0.25 * (-((dF1[j + 1] - dF1[j]) / M.yLen[j]));
            Qc[j] = jzq / sig1[j];
            dQc[j] = djzq / sig1[j] - jzq * (dsig_cell(c2a, ds, j) / (sig1[j] * sig1[j]));
        }
    }
    __syncthreads();
    for (int i = tid + 1; i < ny; i += kRxThreads) {
        const double yb = 0.5 * M.yLen[i - 1] + 0.5 * M.yLen[i];
        const double d0 = dsig_cell(c2a, ds, i - 1), d1 = dsig_cell(c2a, ds, i);
        const cplx Q = 0.75 * F0[i] + 0.25 * F1[i], dQ = 0.75 * dF0[i] + 0.25 * dF1[i];
        const cplx dEz = (Qc[i] - Qc[i - 1]) / yb, ddEz = (dQc[i] - dQc[i - 1]) / yb;
        if (mode == 0) {
            const double sv = (0.5 * (sig1[i - 1] * M.yLen[i - 1]) + 0.5 * (sig1[i] * M.yLen[i])) / yb;
            const double dsv = (0.5 * (d0 * M.yLen[i - 1]) + 0.5 * (d1 * M.yLen[i])) / yb;
            G0[i] = -((F1[i] - F0[i]) / h / iwmu) - (dEz - sv * Q) * (0.5 * h);
            dG0[i] = -((dF1[i] - dF0[i]) / h / iwmu) - (ddEz - sv * dQ - dsv * Q) * (0.5 * h);
        } else {
            const double rv = (0.5 * ((1.0 / sig1[i - 1]) * M.yLen[i - 1]) + 0.5 * ((1.0 / sig1[i]) * M.yLen[i])) / yb;
            const double drv = (0.5 * ((-d0 / (sig1[i - 1] * sig1[i - 1])) * M.yLen[i - 1]) + 0.5 * ((-d1 / (sig1[i] * sig1[i])) * M.yLen[i])) / yb;
            const cplx JyH = (F1[i] - F0[i]) / h, dJyH = (dF1[i] - dF0[i]) / h;
            G0[i] = JyH * rv - (dEz + iwmu * Q) * (0.5 * h);
            dG0[i] = dJyH * rv + JyH * drv - (ddEz + iwmu * dQ) * (0.5 * h);
        }
    }
    __syncthreads();
    if (tid == 0) { G0[0] = G0[1]; G0[ny] = G0[ny - 1]; dG0[0] = dG0[1]; dG0[ny] = dG0[ny - 1]; }
    __syncthreads();
    const int nC = kTipper ? cm.nComp : sm.nModes;
    const int zc = kTipper ? (mi == 0 ? cm.zc[0] : cm.zc[1]) : mi;
    const size_t row0 = ((size_t)ch * sm.nFreq + f) * rx.nRx;
    for (int r = tid; r < rx.nRx; r += kRxThreads) {
        const int iL = rx.iL[r], iR = rx.iR[r];
        const double wl = rx.wL[r], wr = rx.wR[r];
        if (!(kTipper && zc < 0)) {
            cplx numS, denS, dnum, dden;
            if (mode == 0) {
                numS = wl * F0[iL] + wr * F0[iR]; denS = wl * G0[iL] + wr * G0[iR];
                dnum = wl * dF0[iL] + wr * dF0[iR]; dden = wl * dG0[iL] + wr * dG0[iR];
            } else {
                numS = wl * G0[iL] + wr * G0[iR]; denS = wl * F0[iL] + wr * F0[iR];
                dnum = wl * dG0[iL] + wr * dG0[iR]; dden = wl * dF0[iL] + wr * dF0[iR];
            }
            const cplx dZ = dnum / denS - numS * dden / (denS * denS);
            const size_t di = (row0 + r) * nC + zc;
            if constexpr (kRhoPhase) {
                const int id = rx.fid[r];           // the forward (un-normalised) Z, as the adjoint weight V uses it
                const double d1 = rx.fdy1[r], d2 = rx.fdy2[r];
                const cplx Z = (mode == 0) ? (F0[id - 1] * d2 + F0[id] * d1) / (G0[id - 1] * d2 + G0[id] * d1)
                                           : (G0[id - 1] * d2 + G0[id] * d1) / (F0[id - 1] * d2 + F0[id] * d1);
                const cplx zd = cconj(Z) * dZ;
                jv[di] = mk(2.0 / (omega * kMu0) * zd.x, 180.0 / kPi * zd.y / cabs2(Z));
            } else {
                jv[di] = dZ;
            }
        }
        if constexpr (kTipper) {
            if (mi == cm.tmi) {
                const int jL = rx.tjL[r], jR = rx.tjR[r];
                const double vl = rx.twL[r], vr = rx.twR[r];
                const cplx hzr = vl * ((F0[jL + 1] - F0[jL]) / M.yLen[jL] / iwmu) + vr * ((F0[jR + 1] - F0[jR]) / M.yLen[jR] / iwmu);
                const cplx dhzr = vl * ((dF0[jL + 1] - dF0[jL]) / M.yLen[jL] / iwmu) + vr * ((dF0[jR + 1] - dF0[jR]) / M.yLen[jR] / iwmu);
                const cplx hyr = wl * G0[iL] + wr * G0[iR], dhyr = wl * dG0[iL] + wr * dG0[iR];
                jv[(row0 + r) * nC + cm.tc] = (dhzr - (hzr / hyr) * dhyr) / hyr;
            }
        }
    }
}

// Gauss-Newton data weights on a tangent in the full layout: vin = Wd^2 jv (rho / phase plans: (w_rho^2 d rho, w_phi^2 d phi)).
// grid (ceil(nFull/256), nChains)
__global__ void k_gn_weight(int nFull, int rhoPhase, const double* __restrict__ wd, const double* __restrict__ wdPha,
                            const cplx* __restrict__ jv, cplx* __restrict__ vin) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (i >= nFull) return;
    const cplx t = jv[(size_t)ch * nFull + i];
    const double w = wd[i], wp = rhoPhase ? wdPha[i] : w;
    vin[(size_t)ch * nFull + i] = mk(w * w * t.x, (rhoPhase ? wp * wp : w * w) * t.y);
}
// dsig = sigma_active * v: the ln(sigma) direction v as a conductivity perturbation.  grid (ceil(nAC/256), nChains)
__global__ void k_sigma_scale(int nAC, int nCell, const int* __restrict__ act2cell, const double* __restrict__ sigma,
                              const double* __restrict__ v, double* __restrict__ dsig) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (a < nAC) dsig[(size_t)ch * nAC + a] = sigma[(size_t)ch * nCell + act2cell[a]] * v[(size_t)ch * nAC + a];
}

// ---------------------------------------------------------------------------------------------
// Reduction over systems + chain rule + prior gradient (HMCSampler.jl:306, :223-224, :255-256):
//   grad[a] = sigma_a * sum_sys Gpart[sys][cell(a)] + beta * (Wm (m - mref))[a]     (fixed summation order)
// grid: (ceil(nAC/256), nChains)
__global__ void k_reduce_grad(int nAC, int nCell, int nSysPerChain, const int* __restrict__ act2cell,
                              const double* __restrict__ Gpart, const double* __restrict__ m, const double* __restrict__ mref,
                              const int* __restrict__ wmPtr, const int* __restrict__ wmIdx, const double* __restrict__ wmVal,
                              double beta, const double* __restrict__ sigma, double* __restrict__ gsig,
                              double* __restrict__ gdata, double* __restrict__ gtotal) {
    int a = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (a >= nAC) return;
    const int c = act2cell[a];
    const double* G = Gpart + (size_t)ch * nSysPerChain * nCell;
    double acc = 0.0;
    for (int s = 0; s < nSysPerChain; ++s) acc += G[(size_t)s * nCell + c];
    const double* mm = m + (size_t)ch * nAC;
    const double* mr = mref + (size_t)ch * nAC;
    gsig[(size_t)ch * nAC + a] = acc;                               // real(J^T v) w.r.t. conductivity
    double gd = sigma[(size_t)ch * nCell + c] * acc;                // dsigma' * dataGrad, sigma_a = exp(m_a)
    double pr = 0.0;
    for (int k = wmPtr[a]; k < wmPtr[a + 1]; ++k) { int j = wmIdx[k]; pr += wmVal[k] * (mm[j] - mr[j]); }
    gdata[(size_t)ch * nAC + a] = gd;
    gtotal[(size_t)ch * nAC + a] = gd + beta * pr;
}

// phi_d per chain: fixed-order sum of the per-system partials.  grid nChains, block 32
__global__ void k_reduce_phi(int nSysPerChain, const double* __restrict__ phiPart, double* __restrict__ phi) {
    if (threadIdx.x == 0) {
        double acc = 0.0;
        for (int s = 0; s < nSysPerChain; ++s) acc += phiPart[(size_t)blockIdx.x * nSysPerChain + s];
        phi[blockIdx.x] = acc;
    }
}

// ---------------------------------------------------------------------------------------------
// K11: leapfrog pieces (HMCSampler.jl:206-269, 515-559), one CTA per chain, identity mass matrix.
constexpr int kHmcThreads = 1024;
__device__ inline double block_reduce(double v, bool isMax, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o > 0; o >>= 1) {
        double u = __shfl_xor_sync(0xffffffffu, v, o);
        v = isMax ? fmax(v, u) : v + u;
    }
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    if (warp == 0) {
        v = (lane < (int)(blockDim.x >> 5)) ? sh[lane] : (isMax ? 0.0 : 0.0);
        for (int o = 16; o > 0; o >>= 1) {
            double u = __shfl_xor_sync(0xffffffffu, v, o);
            v = isMax ? fmax(v, u) : v + u;
        }
        if (lane == 0) sh[0] = v;
    }
    __syncthreads();
    double r = sh[0];
    __syncthreads();
    return r;
}
// p -= scale*dt*grad
// grid (ceil(nAC / blockDim), nChains)
__global__ void k_kick(int nAC, double dtScaled, const double* __restrict__ grad, double* __restrict__ p) {
    const int ch = blockIdx.y, a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a < nAC) p[(size_t)ch * nAC + a] -= dtScaled * grad[(size_t)ch * nAC + a];
}
// drift with max-step clip 3.0 and reflection at the log-conductivity bounds (HMCSampler.jl:235-250, checkParameterBound! :515-559),
// two launches of grid (nBlocks, nChains): the largest |dt gradK| of every block, then the update (every block first folds the
// block maxima: a maximum does not depend on the order, so the result is the one a single block would produce)
__global__ void __launch_bounds__(kHmcThreads)
k_drift_max(int nAC, double dt, const double* __restrict__ p, const double* __restrict__ gradK, double* __restrict__ part) {
    // gradK = invM p (getKineticGradient HMCSampler.jl:424-431); null: identity mass matrix, gradK = p
    __shared__ double sh[32];
    const int ch = blockIdx.y;
    const double* gk = (gradK ? gradK : p) + (size_t)ch * nAC;
    double mx = 0.0;
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < nAC; a += gridDim.x * blockDim.x) mx = fmax(mx, fabs(dt * gk[a]));
    mx = block_reduce(mx, true, sh);
    if (threadIdx.x == 0) part[(size_t)ch * gridDim.x + blockIdx.x] = mx;
}
__global__ void __launch_bounds__(kHmcThreads)
k_drift(int nAC, double dt, double lo, double hi, double* __restrict__ m, double* __restrict__ p, int* __restrict__ flag,
        const double* __restrict__ gradK, const double* __restrict__ part) {
    __shared__ double sh[32];
    const int ch = blockIdx.y;
    double* mm = m + (size_t)ch * nAC;
    double* pp = p + (size_t)ch * nAC;
    const double* gk = gradK ? gradK + (size_t)ch * nAC : pp;
    double mx = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) mx = fmax(mx, part[(size_t)ch * gridDim.x + b]);
    mx = block_reduce(mx, true, sh);
    for (int a = blockIdx.x * blockDim.x + threadIdx.x; a < nAC; a += gridDim.x * blockDim.x) {
        double dm = dt * gk[a];
        if (mx > 3.0) dm = dm / mx * 3.0;
        double v = mm[a] + dm, mom = pp[a];
        if (!(v <= hi && v >= lo)) {
            int it = 0;
            while (true) {
                ++it;
                if (v < lo) { v = 2.0 * lo - v; mom = -mom; }
                if (v > hi) { v = 2.0 * hi - v; mom = -mom; }
                if (v <= hi && v >= lo) break;
                if (it >= 500) { if (flag) atomicExch(flag, 1); break; }   // reference loops forever here
            }
        }
        mm[a] = v;
        pp[a] = mom;
    }
}
__global__ void __launch_bounds__(kHmcThreads)
k_energies(int nAC, const double* __restrict__ m, const double* __restrict__ mref, const double* __restrict__ p,
           const int* __restrict__ wmPtr, const int* __restrict__ wmIdx, const double* __restrict__ wmVal, double beta,
           double* __restrict__ out /* [ch][2] = K, phi_m */, const double* __restrict__ gradK) {
    // K = 1/2 p^T invM p (getKineticEnergy HMCSampler.jl:407-415): gradK = invM p, null for the identity mass matrix
    __shared__ double sh[32];
    const int ch = blockIdx.x;
    const double* mm = m + (size_t)ch * nAC;
    const double* mr = mref + (size_t)ch * nAC;
    const double* pp = p + (size_t)ch * nAC;
    const double* gk = gradK ? gradK + (size_t)ch * nAC : pp;
    double k = 0.0, pm = 0.0;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) {
        k += pp[a] * gk[a];
        double row = 0.0;
        for (int q = wmPtr[a]; q < wmPtr[a + 1]; ++q) { int j = wmIdx[q]; row += wmVal[q] * (mm[j] - mr[j]); }
        pm += (mm[a] - mr[a]) * row;
    }
    k = block_reduce(k, false, sh);
    pm = block_reduce(pm, false, sh);
    if (threadIdx.x == 0) { out[ch * 2] = 0.5 * k; out[ch * 2 + 1] = 0.5 * pm * beta; }
}

// ---------------------------------------------------------------------------------------------
// Projected Gauss-Newton-CG (hmcmt_gauss_newton).  Every chain runs its own iteration; the per-chain scalars and flags live on
// the device (S [nChains][kGnS], I [nChains][kGnI]) so that the CG loop needs no host round trip.  Every reduction is either one
// CTA per chain (block_reduce over a fixed blockDim) or fixed-size block partials folded by one CTA in block order: the results
// do not depend on timing, on the other chains or on how the launches were issued.
enum GnScalar { kGnU, kGnPhid, kGnPhim, kGnRR, kGnRR0, kGnGtd, kGnAlpha, kGnS };
enum GnFlag { kGnActive, kGnReason, kGnAcc, kGnCgRun, kGnCgIt, kGnLs, kGnTrials, kGnI };
enum GnLs { kLsSearch, kLsAccepted, kLsFailed, kLsIdle };
constexpr int kGnHist = 6;            // history row: phi_d, phi_m, |P g|, CG iterations, alpha, line-search trials
constexpr int kGnReduceThreads = 256;

// m <- clip(m, lo, hi).  grid (ceil(nAC/256), nChains)
__global__ void k_gn_project(int nAC, double lo, double hi, double* __restrict__ m) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (a < nAC) m[(size_t)ch * nAC + a] = fmin(fmax(m[(size_t)ch * nAC + a], lo), hi);
}

// New linearisation point of every chain that accepted a step (first: of every chain, iteration 0): U = phi_d + phi_m, the
// active set A = {m <= lo, g > 0} u {m >= hi, g < 0}, r = p = -P g, delta = 0, the history row and the stopping tests
// (decrease below tolRel U_k, or P g = 0).  en: k_energies output ([ch][1] = phi_m).  grid nChains, block kHmcThreads
__global__ void __launch_bounds__(kHmcThreads)
k_gn_linearise(int nAC, int first, int maxIter, double tolRel, double lo, double hi, const double* __restrict__ m,
               const double* __restrict__ g, const double* __restrict__ phi, const double* __restrict__ en, double* __restrict__ mk,
               double* __restrict__ gk, int* __restrict__ act, double* __restrict__ r, double* __restrict__ p, double* __restrict__ delta,
               double* __restrict__ S, int* __restrict__ I, double* __restrict__ hist) {
    __shared__ double sh[32];
    const int ch = blockIdx.x;
    double* s = S + (size_t)ch * kGnS;
    int* f = I + (size_t)ch * kGnI;
    if (!first && !(f[kGnActive] && f[kGnLs] == kLsAccepted)) return;
    const size_t o = (size_t)ch * nAC;
    double rr = 0.0;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) {
        const double mi = m[o + a], gi = g[o + a];
        const int A = (mi <= lo && gi > 0.0) || (mi >= hi && gi < 0.0);
        const double ri = A ? 0.0 : -gi;
        mk[o + a] = mi;
        gk[o + a] = gi;
        act[o + a] = A;
        r[o + a] = ri;
        p[o + a] = ri;
        delta[o + a] = 0.0;
        rr += ri * ri;
    }
    rr = block_reduce(rr, false, sh);
    if (threadIdx.x == 0) {
        const double phid = phi[ch], phim = en[2 * ch + 1], U = phid + phim;
        const int acc = first ? 0 : f[kGnAcc] + 1;
        bool stop = rr == 0.0;
        if (!first && s[kGnU] - U <= tolRel * s[kGnU]) stop = true;
        double* h = hist + ((size_t)ch * (maxIter + 1) + acc) * kGnHist;
        h[0] = phid;
        h[1] = phim;
        h[2] = sqrt(rr);
        h[3] = first ? 0.0 : (double)f[kGnCgIt];
        h[4] = first ? 0.0 : s[kGnAlpha];
        h[5] = first ? 0.0 : (double)f[kGnTrials];
        s[kGnU] = U;
        s[kGnPhid] = phid;
        s[kGnPhim] = phim;
        s[kGnRR] = rr;
        s[kGnRR0] = rr;
        f[kGnAcc] = acc;
        f[kGnActive] = stop ? 0 : 1;
        f[kGnReason] = stop ? 1 : 0;
        f[kGnCgRun] = stop ? 0 : 1;
        f[kGnCgIt] = 0;
    }
}

// The reduction over systems of the Gauss-Newton product (k_reduce_grad with (m, m_ref) = (p, 0)), masked: q = P (H p), and the
// per-block partials of p^T q.  grid (ceil(nAC/kGnReduceThreads), nChains), block kGnReduceThreads
__global__ void __launch_bounds__(kGnReduceThreads)
k_reduce_gn(int nAC, int nCell, int nSysPerChain, const int* __restrict__ act2cell, const double* __restrict__ Gpart,
            const double* __restrict__ p, const int* __restrict__ wmPtr, const int* __restrict__ wmIdx, const double* __restrict__ wmVal,
            double beta, const double* __restrict__ sigma, const int* __restrict__ act, double* __restrict__ q, double* __restrict__ part) {
    __shared__ double sh[32];
    const int a = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    double pq = 0.0;
    if (a < nAC) {
        const int c = act2cell[a];
        const double* G = Gpart + (size_t)ch * nSysPerChain * nCell;
        double acc = 0.0;
        for (int s = 0; s < nSysPerChain; ++s) acc += G[(size_t)s * nCell + c];
        const double* pp = p + (size_t)ch * nAC;
        double pr = 0.0;
        for (int k = wmPtr[a]; k < wmPtr[a + 1]; ++k) pr += wmVal[k] * pp[wmIdx[k]];
        const double gd = sigma[(size_t)ch * nCell + c] * acc;
        const double qa = act[(size_t)ch * nAC + a] ? 0.0 : gd + beta * pr;
        q[(size_t)ch * nAC + a] = qa;
        pq = pp[a] * qa;
    }
    pq = block_reduce(pq, false, sh);
    if (threadIdx.x == 0) part[(size_t)ch * gridDim.x + blockIdx.x] = pq;
}

// One CG update of every chain whose CG still runs: p^T q from the partials (in block order), alpha = r^T r / p^T q,
// delta += alpha p, r -= alpha q, stop at |r| <= cgTol |r_0|, else p = r + (r_new^T r_new / r^T r) p.  p^T q <= 0 stops the
// chain's CG (delta = r_0 if that happens at its first iteration).  grid nChains, block kHmcThreads
__global__ void __launch_bounds__(kHmcThreads)
k_gn_cg_update(int nAC, int nPart, double cgTol, const double* __restrict__ part, const double* __restrict__ q, double* __restrict__ r,
               double* __restrict__ p, double* __restrict__ delta, double* __restrict__ S, int* __restrict__ I) {
    __shared__ double sh[32];
    const int ch = blockIdx.x;
    double* s = S + (size_t)ch * kGnS;
    int* f = I + (size_t)ch * kGnI;
    if (!f[kGnCgRun]) return;
    const size_t o = (size_t)ch * nAC;
    const double rr = s[kGnRR], rr0 = s[kGnRR0];
    const int it = f[kGnCgIt];
    double pq = 0.0;
    for (int b = threadIdx.x; b < nPart; b += blockDim.x) pq += part[(size_t)ch * nPart + b];
    pq = block_reduce(pq, false, sh);
    if (!(pq > 0.0)) {
        if (it == 0)
            for (int a = threadIdx.x; a < nAC; a += blockDim.x) delta[o + a] = r[o + a];
        if (threadIdx.x == 0) f[kGnCgRun] = 0;
        return;
    }
    const double alpha = rr / pq;
    double rn = 0.0;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) {
        delta[o + a] += alpha * p[o + a];
        const double ri = r[o + a] - alpha * q[o + a];
        r[o + a] = ri;
        rn += ri * ri;
    }
    rn = block_reduce(rn, false, sh);
    const bool done = sqrt(rn) <= cgTol * sqrt(rr0);
    if (!done) {
        const double b = rn / rr;
        for (int a = threadIdx.x; a < nAC; a += blockDim.x) p[o + a] = r[o + a] + b * p[o + a];
    }
    if (threadIdx.x == 0) {
        s[kGnRR] = rn;
        f[kGnCgIt] = it + 1;
        if (done) f[kGnCgRun] = 0;
    }
}

// Step length of every running chain: delta scaled so that max|delta_i| <= maxStep, the line search armed; stopped chains sit it
// out.  grid nChains, block kHmcThreads
__global__ void __launch_bounds__(kHmcThreads)
k_gn_direction(int nAC, double maxStep, double* __restrict__ delta, int* __restrict__ I) {
    __shared__ double sh[32];
    const int ch = blockIdx.x;
    int* f = I + (size_t)ch * kGnI;
    if (!f[kGnActive]) {
        if (threadIdx.x == 0) f[kGnLs] = kLsIdle;
        return;
    }
    double* d = delta + (size_t)ch * nAC;
    double mx = 0.0;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) mx = fmax(mx, fabs(d[a]));
    mx = block_reduce(mx, true, sh);
    if (mx > maxStep)
        for (int a = threadIdx.x; a < nAC; a += blockDim.x) d[a] = d[a] / mx * maxStep;
    if (threadIdx.x == 0) {
        f[kGnLs] = kLsSearch;
        f[kGnTrials] = 0;
    }
}

// Trial t of the line search of every chain still searching: m = clip(m_k + 2^-t delta, lo, hi) and g_k^T (m - m_k).
// grid nChains, block kHmcThreads
__global__ void __launch_bounds__(kHmcThreads)
k_gn_trial(int nAC, int t, double lo, double hi, const double* __restrict__ mk, const double* __restrict__ gk,
           const double* __restrict__ delta, double* __restrict__ m, double* __restrict__ S, const int* __restrict__ I) {
    __shared__ double sh[32];
    const int ch = blockIdx.x;
    if (I[(size_t)ch * kGnI + kGnLs] != kLsSearch) return;
    const size_t o = (size_t)ch * nAC;
    const double al = ldexp(1.0, -t);
    double gtd = 0.0;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) {
        const double v = fmin(fmax(mk[o + a] + al * delta[o + a], lo), hi);
        m[o + a] = v;
        gtd += gk[o + a] * (v - mk[o + a]);
    }
    gtd = block_reduce(gtd, false, sh);
    if (threadIdx.x == 0) {
        S[(size_t)ch * kGnS + kGnGtd] = gtd;
        S[(size_t)ch * kGnS + kGnAlpha] = al;
    }
}

// Armijo test of trial t: accept when U(m) <= U_k + 1e-4 g_k^T (m - m_k); the last trial (maxLS) fails the search.
// grid ceil(nChains/128), block 128
__global__ void k_gn_armijo(int nChains, int t, int maxLS, const double* __restrict__ phi, const double* __restrict__ en,
                            const double* __restrict__ S, int* __restrict__ I) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= nChains) return;
    int* f = I + (size_t)ch * kGnI;
    if (f[kGnLs] != kLsSearch) return;
    const double* s = S + (size_t)ch * kGnS;
    const double U = phi[ch] + en[2 * ch + 1];
    if (U <= s[kGnU] + 1e-4 * s[kGnGtd]) {
        f[kGnLs] = kLsAccepted;
        f[kGnTrials] = t + 1;
    } else if (t + 1 >= maxLS) {
        f[kGnLs] = kLsFailed;
        f[kGnTrials] = t + 1;
    }
}

// A chain whose line search failed goes back to m_k and stops.  grid nChains, block kHmcThreads
__global__ void __launch_bounds__(kHmcThreads)
k_gn_revert(int nAC, const double* __restrict__ mk, double* __restrict__ m, int* __restrict__ I) {
    const int ch = blockIdx.x;
    int* f = I + (size_t)ch * kGnI;
    if (f[kGnLs] != kLsFailed) return;
    for (int a = threadIdx.x; a < nAC; a += blockDim.x) m[(size_t)ch * nAC + a] = mk[(size_t)ch * nAC + a];
    if (threadIdx.x == 0) {
        f[kGnActive] = 0;
        f[kGnReason] = 2;
    }
}

}  // namespace hmcmt
