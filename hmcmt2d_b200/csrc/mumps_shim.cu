// Level-1 ABI: the Fortran-style symbols the reference's Julia wrapper ccalls in
// MUMPS/src/MUMPSfuncs.jl (factor :32-35/:49-52, solve :105-107/:128-130, sparse rhs :115-118/:139-143,
// destroy :155-156/:170-171).  Matrices must be structurally symmetric (sym = 1 or 2; the hot path passes sym = 1 for the
// complex-symmetric Aii).  Like MUMPS, the library chooses its own elimination order: matrices whose half-bandwidth in the
// CALLER's numbering is <= 104 go to the register-window band kernel (band_factor.cuh); everything else — e.g. the
// reference's y-fastest Aii (b = ny-1, MT2DFwdSolver.jl:232-234) or the 3-D div-grad matrices of MUMPS/test — is ordered by
// nested dissection (breadth-first level-set bisection, mf_symbolic.h) and factorised by the multifrontal kernels
// (mf_kernels.cuh).  The symbolic analysis is cached per sparsity pattern, so the per-frequency factorMUMPS calls of the
// unmodified reference (mt2DTE.jl:50-53 inside the frequency loop) analyse the pattern once.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/hmcmt_b200.h"
#include "band_factor.cuh"
#include "band_solve.cuh"
#include "mf_solver.cuh"

namespace hmcmt {
int round_T(int b);
int launch_factor(cudaStream_t st, int T, const BandSys* sys, int nsys, const BandDom& dom, const SolveJob* fwdJobs, int* nLaunches);
int launch_solve(cudaStream_t st, int T, const SolveJob* jobs, int njobs, const BandDom& dom);
int mf_leaf_size();
int mf_small_front();
}  // namespace hmcmt
using namespace hmcmt;

namespace {

constexpr int kShimMaxRhs = 16;       // right-hand sides per multifrontal solve launch

struct Factor {
    int n = 0, b = 0, T = 0, S = 0;
    bool isReal = false;
    double* panels = nullptr;
    cplx* ainvz = nullptr;
    mf::Solver* mfs = nullptr;          // multifrontal factor (general ordering); else the band factor above
    const void* pattern = nullptr;      // identity of the cached symbolic analysis the solver was built from
    int64_t epoch = 0;                  // generation of the symbolic cache it belongs to
};
std::mutex g_mu;
std::unordered_map<int64_t, Factor*> g_factors;
int64_t g_next = 1;

// Solvers (device tables, launch schedule, factor / update arenas) of destroyed factors are kept per pattern and handed to the next
// factorisation of the same pattern: the unmodified reference factorises one matrix per frequency and mode with an identical
// pattern, destroys the handles after the gradient and starts over in the next step (MT2DFwdSolver.jl:119-120, HMCSampler.jl:316-321)
std::unordered_map<const void*, std::vector<mf::Solver*>> g_pool;
constexpr size_t kPoolMax = 256;
int64_t g_epoch = 0;                    // bumped whenever the symbolic cache is dropped (pattern pointers may be reused afterwards)

void free_factor(Factor* f) {
    if (!f) return;
    if (f->panels) cudaFree(f->panels);
    if (f->ainvz) cudaFree(f->ainvz);
    if (f->mfs) {
        std::lock_guard<std::mutex> lk(g_mu);
        std::vector<mf::Solver*>& v = g_pool[f->pattern];
        if (f->pattern && f->epoch == g_epoch && v.size() < kPoolMax) v.push_back(f->mfs);
        else delete f->mfs;
    }
    delete f;
}

// ---- multifrontal path ----------------------------------------------------------------------------------------------
// symbolic analysis cached per sparsity pattern (key: n, nnz and an FNV hash of colptr / rowval and of every knob the analysis or
// the solver's launch schedule reads: a pooled solver of the same key is reused as it was built)
struct PatternKey {
    int64_t n, nnz;
    uint64_t h;
    bool operator==(const PatternKey& o) const { return n == o.n && nnz == o.nnz && h == o.h; }
};
struct PatternHash {
    size_t operator()(const PatternKey& k) const { return (size_t)(k.h ^ (uint64_t)k.n * 0x9e3779b97f4a7c15ull); }
};
std::unordered_map<PatternKey, mf::Symbolic*, PatternHash> g_symbolic;

uint64_t fnv(const int64_t* p, int64_t n, uint64_t h) {
    for (int64_t i = 0; i < n; ++i) { h ^= (uint64_t)p[i]; h *= 0x100000001b3ull; }
    return h;
}

const mf::Symbolic* symbolic_for(int64_t n, const int64_t* rowval, const int64_t* colptr) {
    const int64_t nnz = colptr[n] - 1;
    const mf::SchedKnobs sk = mf::SchedKnobs::from_env();
    const int64_t knobs[7] = {mf_leaf_size(), mf_small_front(), sk.fp1, sk.fp2, sk.fp4, sk.fp8, sk.solveThreads};
    PatternKey key{n, nnz, fnv(knobs, 7, fnv(rowval, nnz, fnv(colptr, n + 1, 0xcbf29ce484222325ull)))};
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_symbolic.find(key);
        if (it != g_symbolic.end()) return it->second;
    }
    mf::Symbolic* S = new mf::Symbolic();
    if (!mf::mf_analyse_csc(n, rowval, colptr, mf_leaf_size(), mf_small_front(), *S)) { delete S; return nullptr; }
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_symbolic.size() >= 8) {                         // a handful of patterns at most (TE / TM, real / complex tests)
        for (auto& kv : g_pool)
            for (mf::Solver* sv : kv.second) delete sv;
        g_pool.clear();
        ++g_epoch;
        for (auto& kv : g_symbolic) delete kv.second;
        g_symbolic.clear();
    }
    g_symbolic[key] = S;
    return S;
}

int64_t factor_mf(int64_t n, const double* nzval, const int64_t* rowval, const int64_t* colptr, bool isReal, int64_t* status) {
    auto fail = [&](int code) { if (status) *status = code; return (int64_t)0; };
    const mf::Symbolic* S0 = symbolic_for(n, rowval, colptr);
    if (!S0) return fail(kErrArg);
    const int64_t nnz = colptr[n] - 1;
    int rc = kOk;
    mf::Solver* sv = nullptr;
    int64_t epoch = 0;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        epoch = g_epoch;
        auto it = g_pool.find(S0);
        if (it != g_pool.end() && !it->second.empty()) { sv = it->second.back(); it->second.pop_back(); }
    }
    if (!sv) {
        mf::Symbolic copy = *S0;
        sv = mf::Solver::create(std::move(copy), 1, kShimMaxRhs, nnz, &rc);
    }
    if (!sv) return fail(rc);
    std::vector<cplx> hv((size_t)nnz);
    for (int64_t k = 0; k < nnz; ++k) hv[k] = isReal ? mk(nzval[k], 0.0) : mk(nzval[2 * k], nzval[2 * k + 1]);
    int* dstatus = nullptr;
    if (cudaMalloc(&dstatus, sizeof(int)) != cudaSuccess) { delete sv; return fail(kErrAlloc); }
    cudaMemset(dstatus, 0, sizeof(int));
    cudaMemcpy(sv->vals(), hv.data(), hv.size() * sizeof(cplx), cudaMemcpyHostToDevice);
    rc = sv->factor(nullptr, dstatus);
    int hst = 0;
    if (rc == kOk && cudaDeviceSynchronize() != cudaSuccess) rc = kErrCuda;
    if (rc == kOk) cudaMemcpy(&hst, dstatus, sizeof(int), cudaMemcpyDeviceToHost);
    cudaFree(dstatus);
    if (rc != kOk || hst != 0) { delete sv; return fail(rc != kOk ? rc : hst); }
    Factor* f = new Factor();
    f->n = (int)n; f->isReal = isReal; f->mfs = sv; f->pattern = S0; f->epoch = epoch;
    std::lock_guard<std::mutex> lk(g_mu);
    int64_t h = g_next++;
    g_factors[h] = f;
    return h;
}

// common factor path; vals are complex (re,im) or real depending on isReal
int64_t factor_common(int64_t n, int64_t sym, const double* nzval, const int64_t* rowval, const int64_t* colptr, bool isReal,
                      int64_t* status) {
    auto fail = [&](int code) { if (status) *status = code; return (int64_t)0; };
    if (status) *status = 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        fprintf(stderr, "[hmcmt_b200] no CUDA device: this library has no CPU fallback\n");
        return fail(kErrNoDevice);
    }
    if (n < 1 || !nzval || !rowval || !colptr) return fail(kErrArg);
    if (sym != 1 && sym != 2) {
        fprintf(stderr, "[hmcmt_b200] factor_mumps: only symmetric matrices (sym=1,2) are supported\n");
        return fail(kErrArg);
    }
    // half-bandwidth from the pattern (1-based CSC, MUMPSfuncs.jl:32-35)
    int64_t b = 0;
    for (int64_t j = 0; j < n; ++j)
        for (int64_t k = colptr[j] - 1; k < colptr[j + 1] - 1; ++k) b = std::max<int64_t>(b, std::llabs(rowval[k] - 1 - j));
    if (b < 1) b = 1;
    int T = round_T((int)b);
    {
        const char* env = std::getenv("HMCMT_SHIM_SOLVER");      // "mf": multifrontal for every matrix; "band": refuse wide matrices
        const bool forceMf = env && !std::strcmp(env, "mf"), forceBand = env && !std::strcmp(env, "band");
        if ((T == 0 && !forceBand) || forceMf) return factor_mf(n, nzval, rowval, colptr, isReal, status);
        if (T == 0) return fail(kErrArg);
    }
    // lower band image: band[g*(b+1)+d] = A[g][g-d]   (the lower triangle is what LDL^T reads)
    std::vector<cplx> band((size_t)n * (b + 1), mk(0.0, 0.0));
    for (int64_t j = 0; j < n; ++j)
        for (int64_t k = colptr[j] - 1; k < colptr[j + 1] - 1; ++k) {
            int64_t i = rowval[k] - 1;
            if (i < j) continue;
            cplx v = isReal ? mk(nzval[k], 0.0) : mk(nzval[2 * k], nzval[2 * k + 1]);
            band[(size_t)i * (b + 1) + (i - j)] = v;
        }
    Factor* f = new Factor();
    f->n = (int)n; f->b = (int)b; f->T = T; f->S = (int)((n + TS - 1) / TS); f->isReal = isReal;
    cplx* dband = nullptr;
    BandSys* dsys = nullptr;
    int* dstatus = nullptr;
    auto cleanup = [&]() { if (dband) cudaFree(dband); if (dsys) cudaFree(dsys); if (dstatus) cudaFree(dstatus); };
    if (cudaMalloc(&dband, band.size() * sizeof(cplx)) != cudaSuccess ||
        cudaMalloc(&f->panels, (size_t)f->S * panel_doubles(T) * sizeof(double)) != cudaSuccess ||
        cudaMalloc(&f->ainvz, (size_t)f->S * AZ * sizeof(cplx)) != cudaSuccess || cudaMalloc(&dsys, sizeof(BandSys)) != cudaSuccess ||
        cudaMalloc(&dstatus, sizeof(int)) != cudaSuccess) {
        cleanup(); free_factor(f);
        return fail(kErrAlloc);
    }
    cudaMemcpy(dband, band.data(), band.size() * sizeof(cplx), cudaMemcpyHostToDevice);
    cudaMemset(dstatus, 0, sizeof(int));
    BandSys s{};
    s.band = dband; s.omega = 0.0; s.rhs = nullptr; s.panels[0] = f->panels; s.panels[1] = nullptr; s.ainvz[0] = f->ainvz; s.ainvz[1] = nullptr; s.wexp = nullptr; s.x = nullptr; s.status = dstatus;
    cudaMemcpy(dsys, &s, sizeof(BandSys), cudaMemcpyHostToDevice);
    BandDom dom{(int)n, (int)b, (int)b, 0, 0, 0};
    int rc = launch_factor(nullptr, T, dsys, 1, dom, nullptr, nullptr);
    int hst = 0;
    if (rc == kOk && cudaDeviceSynchronize() != cudaSuccess) rc = kErrCuda;
    if (rc == kOk) cudaMemcpy(&hst, dstatus, sizeof(int), cudaMemcpyDeviceToHost);
    cleanup();
    if (rc != kOk || hst != 0) { free_factor(f); return fail(rc != kOk ? rc : hst); }
    std::lock_guard<std::mutex> lk(g_mu);
    int64_t h = g_next++;
    g_factors[h] = f;
    return h;
}

Factor* lookup(int64_t h) {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_factors.find(h);
    return it == g_factors.end() ? nullptr : it->second;
}

// dense rhs (complex interleaved or real), n x nrhs column-major
int64_t solve_common(int64_t h, int64_t nrhs, const double* rhs, double* x, bool isRealIO) {
    Factor* f = lookup(h);
    if (!f || nrhs < 1 || !rhs || !x) return kErrArg;
    const size_t n = f->n;
    std::vector<cplx> hb(n * nrhs);
    for (size_t i = 0; i < n * (size_t)nrhs; ++i) hb[i] = isRealIO ? mk(rhs[i], 0.0) : mk(rhs[2 * i], rhs[2 * i + 1]);
    if (f->mfs) {
        cplx* db = nullptr;
        if (cudaMalloc(&db, hb.size() * sizeof(cplx)) != cudaSuccess) return kErrAlloc;
        cudaMemcpy(db, hb.data(), hb.size() * sizeof(cplx), cudaMemcpyHostToDevice);
        int rc = kOk;
        for (int64_t r0 = 0; r0 < nrhs && rc == kOk; r0 += kShimMaxRhs) {
            const int nr = (int)std::min<int64_t>(kShimMaxRhs, nrhs - r0);
            rc = f->mfs->solve(nullptr, nr, db + r0 * n, (int64_t)n, db + r0 * n, (int64_t)n);
        }
        if (rc == kOk && cudaDeviceSynchronize() != cudaSuccess) rc = kErrCuda;
        if (rc == kOk) {
            cudaMemcpy(hb.data(), db, hb.size() * sizeof(cplx), cudaMemcpyDeviceToHost);
            for (size_t i = 0; i < hb.size(); ++i) {
                if (isRealIO) x[i] = hb[i].x;
                else { x[2 * i] = hb[i].x; x[2 * i + 1] = hb[i].y; }
            }
        }
        cudaFree(db);
        return rc;
    }
    cplx *dx = nullptr, *dz = nullptr;
    SolveJob* djobs = nullptr;
    auto cleanup = [&]() { if (dx) cudaFree(dx); if (dz) cudaFree(dz); if (djobs) cudaFree(djobs); };
    if (cudaMalloc(&dx, hb.size() * sizeof(cplx)) != cudaSuccess || cudaMalloc(&dz, (size_t)nrhs * f->S * 8 * sizeof(cplx)) != cudaSuccess ||
        cudaMalloc(&djobs, sizeof(SolveJob) * nrhs) != cudaSuccess) {
        cleanup();
        return kErrAlloc;
    }
    cudaMemcpy(dx, hb.data(), hb.size() * sizeof(cplx), cudaMemcpyHostToDevice);
    std::vector<SolveJob> jobs(nrhs);
    for (int64_t r = 0; r < nrhs; ++r) {
        jobs[r].panels[0] = f->panels; jobs[r].panels[1] = nullptr; jobs[r].ainvz[0] = f->ainvz; jobs[r].ainvz[1] = nullptr;
        jobs[r].rhs = dx + r * n; jobs[r].x = dx + r * n; jobs[r].zbuf[0] = dz + (size_t)r * f->S * 8; jobs[r].zbuf[1] = nullptr;
        jobs[r].wexp = nullptr;
    }
    cudaMemcpy(djobs, jobs.data(), sizeof(SolveJob) * nrhs, cudaMemcpyHostToDevice);
    BandDom dom{f->n, f->b, f->b, 0, 0, 0};
    int rc = launch_solve(nullptr, f->T, djobs, (int)nrhs, dom);
    if (rc == kOk && cudaDeviceSynchronize() != cudaSuccess) rc = kErrCuda;
    if (rc == kOk) {
        cudaMemcpy(hb.data(), dx, hb.size() * sizeof(cplx), cudaMemcpyDeviceToHost);
        for (size_t i = 0; i < hb.size(); ++i) {
            if (isRealIO) x[i] = hb[i].x;
            else { x[2 * i] = hb[i].x; x[2 * i + 1] = hb[i].y; }
        }
    }
    cleanup();
    return rc;
}

void solve_sparse_common(int64_t h, int64_t nrhs, const double* nzval, const int64_t* rowval, const int64_t* colptr, double* x,
                         bool isRealIO) {
    Factor* f = lookup(h);
    if (!f || nrhs < 1) return;
    const size_t n = f->n, w = isRealIO ? 1 : 2;
    std::vector<double> dense(n * nrhs * w, 0.0);
    for (int64_t j = 0; j < nrhs; ++j)
        for (int64_t k = colptr[j] - 1; k < colptr[j + 1] - 1; ++k) {
            size_t i = (size_t)(rowval[k] - 1) + (size_t)j * n;
            if (isRealIO) dense[i] = nzval[k];
            else { dense[2 * i] = nzval[2 * k]; dense[2 * i + 1] = nzval[2 * k + 1]; }
        }
    solve_common(h, nrhs, dense.data(), x, isRealIO);
}

int64_t destroy_common(int64_t h) {
    Factor* f = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_factors.find(h);
        if (it == g_factors.end()) return kErrArg;
        f = it->second;
        g_factors.erase(it);
    }
    free_factor(f);
    return kOk;
}

}  // namespace

extern "C" {

int64_t factor_mumps_cmplx_(const int64_t* n, const int64_t* sym, const int64_t* ooc, const double* nzval, const int64_t* rowval,
                            const int64_t* colptr, int64_t* status) {
    (void)ooc;
    if (!n || !sym) { if (status) *status = kErrArg; return 0; }
    return factor_common(*n, *sym, nzval, rowval, colptr, false, status);
}
int64_t factor_mumps_(const int64_t* n, const int64_t* sym, const int64_t* ooc, const double* nzval, const int64_t* rowval,
                      const int64_t* colptr, int64_t* status) {
    (void)ooc;
    if (!n || !sym) { if (status) *status = kErrArg; return 0; }
    return factor_common(*n, *sym, nzval, rowval, colptr, true, status);
}
int64_t solve_mumps_cmplx_(const int64_t* handle, const int64_t* nrhs, const double* rhs, double* x, const int64_t* transpose) {
    (void)transpose;      // A is symmetric: A^T x = b is the same system (compJacTMatVec.jl:221-224)
    if (!handle || !nrhs) return kErrArg;
    return solve_common(*handle, *nrhs, rhs, x, false);
}
int64_t solve_mumps_(const int64_t* handle, const int64_t* nrhs, const double* rhs, double* x, const int64_t* transpose) {
    (void)transpose;
    if (!handle || !nrhs) return kErrArg;
    return solve_common(*handle, *nrhs, rhs, x, true);
}
void solve_mumps_sparse_rhs_(const int64_t* handle, const int64_t* nzrhs, const int64_t* nrhs, const double* nzval,
                             const int64_t* rowval, const int64_t* colptr, double* x, const int64_t* transpose) {
    (void)nzrhs; (void)transpose;
    if (!handle || !nrhs) return;
    solve_sparse_common(*handle, *nrhs, nzval, rowval, colptr, x, true);
}
void solve_mumps_cmplx_sparse_rhs_(const int64_t* handle, const int64_t* nzrhs, const int64_t* nrhs, const double* nzval,
                                   const int64_t* rowval, const int64_t* colptr, double* x, const int64_t* transpose) {
    (void)nzrhs; (void)transpose;
    if (!handle || !nrhs) return;
    solve_sparse_common(*handle, *nrhs, nzval, rowval, colptr, x, false);
}
// debug: copy the raw factor (panel images, pivot-block inverses) back to the host
int64_t hmcmt_debug_get_factor(int64_t handle, double* panels, double* ainv, int64_t* dims) {
    Factor* f = lookup(handle);
    if (!f || f->mfs) return kErrArg;
    if (dims) { dims[0] = f->n; dims[1] = f->b; dims[2] = f->T; dims[3] = f->S; }
    if (panels) cudaMemcpy(panels, f->panels, (size_t)f->S * panel_doubles(f->T) * sizeof(double), cudaMemcpyDeviceToHost);
    if (ainv) cudaMemcpy(ainv, f->ainvz, (size_t)f->S * AZ * sizeof(cplx), cudaMemcpyDeviceToHost);
    return kOk;
}
int64_t hmcmt_factor_inverse_diag(const int64_t* handle, double* out) {
    if (!handle || !out) return kErrArg;
    Factor* f = lookup(*handle);
    if (!f || !f->mfs) return kErrArg;
    const size_t n = f->n;
    cplx* d = nullptr;
    if (cudaMalloc(&d, n * sizeof(cplx)) != cudaSuccess) return kErrAlloc;
    int rc = f->mfs->inverse_diag(nullptr, d, (int64_t)n);
    if (rc == kOk && cudaDeviceSynchronize() != cudaSuccess) rc = kErrCuda;
    if (rc == kOk) {
        std::vector<cplx> h(n);
        if (cudaMemcpy(h.data(), d, n * sizeof(cplx), cudaMemcpyDeviceToHost) != cudaSuccess) rc = kErrCuda;
        for (size_t i = 0; rc == kOk && i < n; ++i) {
            if (f->isReal) out[i] = h[i].x;
            else { out[2 * i] = h[i].x; out[2 * i + 1] = h[i].y; }
        }
    }
    cudaFree(d);
    return rc;
}
int64_t hmcmt_debug_factor_flops(const int64_t* handle, double* flops) {
    if (!handle || !flops) return kErrArg;
    Factor* f = lookup(*handle);
    if (!f || !f->mfs) return kErrArg;
    flops[0] = f->mfs->factor_flops();
    flops[1] = f->mfs->selinv_flops();
    return kOk;
}
int64_t destroy_mumps_(const int64_t* handle) { return handle ? destroy_common(*handle) : kErrArg; }
int64_t destroy_mumps_cmplx_(const int64_t* handle) { return handle ? destroy_common(*handle) : kErrArg; }

}  // extern "C"
