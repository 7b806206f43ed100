/* hmcmt_b200.h — C ABI of libhmcmt_b200.so: the B200-native drop-in for the direct-solver hot path
 * of CUG-EMI/HMCMT2D (forward response + adjoint gradient per leapfrog step).
 *
 * Two levels (SURVEY.md section 8b):
 *
 *  Level 1 — the eight Fortran-style symbols the reference's Julia wrapper `ccall`s in
 *            MUMPS/src/MUMPSfuncs.jl (library path MUMPS/src/MUMPS.jl:14).  Every argument is
 *            passed by pointer, integers are int64, matrices are full 1-based CSC.  With this
 *            library symlinked to MUMPS/lib/MUMPS the unmodified reference runs on the GPU solver
 *            (symmetric matrices only: sym = 1 or 2, which is all the hot path passes).
 *
 *  Level 2 — fused entry points mirroring the reference's sampler-facing functions
 *            (MT2DFwdSolver, compJacTMatVec, compDataGradient, proposeLeapfrog, runHMCSampler).
 *            Plain C, status-code returns with the MUMPS negative-code convention
 *            (MUMPSfuncs.jl:59-73): 0 ok, -10 singular, -13 allocation, -3 bad argument,
 *            -98 no CUDA device, -99 CUDA error.  There is NO CPU fallback.
 *
 * All complex arrays are interleaved (re,im) doubles (ComplexF64 / numpy complex128).
 * Index arrays named *ID are 1-based exactly as in the reference's data files; every other
 * index array is 0-based.
 */
#ifndef HMCMT_B200_H
#define HMCMT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ----------------------------------------------------------------------------------------------
 * Level 1: MUMPS shim (replaces the binary MUMPS/lib/MUMPS, .MISSING_LARGE_BLOBS)
 * ---------------------------------------------------------------------------------------------- */

/* factorMUMPS(A::SparseMatrixCSC{ComplexF64},sym,ooc)  MUMPSfuncs.jl:24-39 (ccall :32-35).
 * sym: 0 unsymmetric, 1 "SPD", 2 general symmetric (:25-26).  Only symmetric matrices are
 * supported (the hot path passes sym=1 for a complex-symmetric matrix, mt2DTE.jl:51); the
 * matrix is factorised pivot-free without conjugation.  Like MUMPS the library picks its own elimination order: a
 * half-bandwidth <= 104 in the caller's numbering goes to the register-window band kernel, everything else (e.g. the
 * reference's y-fastest Aii, the 3-D div-grad matrices of MUMPS/test) is ordered by nested dissection and factorised by
 * the multifrontal kernels; the analysis is cached per sparsity pattern.  Returns an opaque handle; *status < 0 on error. */
int64_t factor_mumps_cmplx_(const int64_t* n, const int64_t* sym, const int64_t* ooc, const double* nzval,
                            const int64_t* rowval, const int64_t* colptr, int64_t* status);
/* factorMUMPS(A::SparseMatrixCSC{Float64},...)  MUMPSfuncs.jl:41-56 (ccall :49-52) */
int64_t factor_mumps_(const int64_t* n, const int64_t* sym, const int64_t* ooc, const double* nzval,
                      const int64_t* rowval, const int64_t* colptr, int64_t* status);
/* applyMUMPS!(factor{ComplexF64}, rhs, x, tr)  MUMPSfuncs.jl:123-132.  rhs, x: n x nrhs column-major
 * (the reference mis-declares x as Ptr{ComplexF32} but passes complex128 memory). */
int64_t solve_mumps_cmplx_(const int64_t* handle, const int64_t* nrhs, const double* rhs, double* x,
                           const int64_t* transpose);
/* applyMUMPS!(factor{Float64}, rhs, x, tr)  MUMPSfuncs.jl:100-109 */
int64_t solve_mumps_(const int64_t* handle, const int64_t* nrhs, const double* rhs, double* x,
                     const int64_t* transpose);
/* sparse right-hand sides  MUMPSfuncs.jl:111-121, 134-145 (unused by the hot path) */
void solve_mumps_sparse_rhs_(const int64_t* handle, const int64_t* nzrhs, const int64_t* nrhs, const double* nzval,
                             const int64_t* rowval, const int64_t* colptr, double* x, const int64_t* transpose);
void solve_mumps_cmplx_sparse_rhs_(const int64_t* handle, const int64_t* nzrhs, const int64_t* nrhs,
                                   const double* nzval, const int64_t* rowval, const int64_t* colptr, double* x,
                                   const int64_t* transpose);
/* destroyMUMPS  MUMPSfuncs.jl:148-176 */
int64_t destroy_mumps_(const int64_t* handle);
int64_t destroy_mumps_cmplx_(const int64_t* handle);

/* ----------------------------------------------------------------------------------------------
 * Level 2: fused MT2D forward + adjoint + HMC entry points
 * ---------------------------------------------------------------------------------------------- */

typedef struct hmcmt_plan hmcmt_plan;

/* Problem description = the reference's (TensorMesh2D, MTData, InvDataModel, HMCPrior) quadruple
 * returned by readstartupFile (readstartupFile.jl:4-103). */
typedef struct hmcmt_problem {
    /* TensorMesh2D  HMCFileIO.jl:46-60 — sizes include the air layers (air first, z downward) */
    int32_t ny, nz;
    const double* yLen;       /* [ny] */
    const double* zLen;       /* [nz] */
    double origin[2];         /* mesh origin after the air shift (readEMModel2D.jl:139) */
    /* MTData  HMCFileIO.jl:26-41 */
    int32_t nFreq;
    const double* freqs;      /* [nFreq] Hz */
    int32_t nRx;
    const double* rxLoc;      /* [nRx][2] row-major (y, z) */
    int32_t nComp;            /* number of DataComp entries (1 to 3) */
    const int32_t* compMode;  /* [nComp] 0 = ZXY (TE), 1 = ZYX (TM), 2 = TZY (TE tipper, below); reference order is [ZXY, ZYX].
                                 2 may appear once, as the last entry, after at most two impedance entries, and only in a plan of
                                 hmcmt_plan_create; anything else returns -3 */
    int32_t nData;
    const int64_t* freqID;    /* [nData] 1-based, rows sorted by (freq, rx, comp) as the reference requires */
    const int64_t* rxID;      /* [nData] 1-based */
    const int64_t* dtID;      /* [nData] 1-based index into DataComp */
    /* InvDataModel  HMCStruct.jl:75-91 */
    const double* obsData;    /* [nData] complex */
    const double* dataErr;    /* [nData]; Wd = 1/|err| (HMCUtility.jl:168-190) */
    int32_t nAC;              /* number of active (free) cells */
    const int32_t* activeIdx; /* [nAC] 0-based cell index (y fastest), increasing */
    const double* bgModel;    /* [ny*nz] background conductivity (0 on active cells) */
    const int32_t* wmRowPtr;  /* Wm = (G P)^T (G P) as 0-based CSR, [nAC+1] */
    const int32_t* wmColIdx;
    const double* wmVal;
    /* HMCPrior  HMCStruct.jl:18-38 */
    double regParam;          /* beta */
    double sigBounds[2];      /* [sigma_min, sigma_max] (linear conductivity) */
    int32_t nChains;          /* independent chains batched on this device (>= 1) */
    int32_t device;           /* CUDA device ordinal */
} hmcmt_problem;

int hmcmt_plan_create(const hmcmt_problem* prob, hmcmt_plan** out);
/* compMode 2 (TZY) is the vertical magnetic transfer function of the TE system, T = Hz/Hy, with the reference's conventions
 * (e^{+i omega t}, z down, the Faraday sign of its Bz and Hy).  For frequency f and receiver r, with F0 = Ex on the receiver node
 * row (the air/earth interface), yc_j the cell-centre y coordinates and Hy0 the surface field the impedance ZXY is formed from
 * (compFieldsAtRxTE mt2DTE.jl:153-210, copied end values):
 *   Hz0_j = (F0_{j+1} - F0_j) / (yLen_j i omega mu0)                  j = 0..ny-1, at yc_j    (Bz_0/mu0 of mt2DTE.jl)
 *   Hzr   = wzL Hz0_{jL} + wzR Hz0_{jR},  (jL, jR, wzL, wzR) = linearInterp(y_r, yc)          (sensUtils.jl:133-161)
 *   Hyr   = wL Hy0_{iL} + wR Hy0_{iR},    (iL, iR, wL, wR) = linearInterp(y_r, yNode)        (the normalised weights of the
 *                                                                                             impedance sensitivities)
 *   T     = Hzr / Hyr.
 * ZXY and ZYX are computed exactly as without it.  A tipper row is a complex datum like an impedance: its misfit
 * 1/2 |(T - T_obs)/|err||^2 is summed into phi_d, and its gradient is the derivative through the same adjoint solve, with the same
 * boundary-condition approximations as the impedance gradient.  Every packed data array keeps its complex rows in place; the
 * explicit Jacobian takes 2 nRx adjoint passes for the impedance components and 2 nRx more for the tipper (they share the TE
 * system).  [TZY] alone or [ZYX, TZY] still solve the TE system, which then carries no impedance datum. */
/* The same plan for apparent resistivity / phase data ("DataType: Rho_Pha", readMT2DData.jl:87), the same struct read with:
 *   obsData  [nData] real: rho_a = |Z|^2/(omega mu0) in Ohm m, or phase = atan2(Im Z, Re Z) in degrees;
 *   dataErr  [nData], weights 1/|err| per row;
 *   nComp / compMode the modes as above; dtID = 2 (mode index) + 1 for rho_a, 2 (mode index) + 2 for phase, i.e. the reference's
 *            DataComp order [RhoXY, PhsXY, RhoYX, PhsYX] (or the two rows of one mode).
 * The misfit is phi_d = 1/2 sum_i ((pred_i - obs_i)/|err_i|)^2 over the rows present, the phase difference taken literally (no
 * wrapping), and the gradients are its exact derivatives.  For such a plan every packed data array of the entry points below is
 * [..][nData] REAL (doubles): pred of hmcmt_forward / _sigma / _forward_gradient / _total / hmcmt_leapfrog_trajectory, v of
 * hmcmt_jtvec (gsig = sum_i v_i d pred_i / d sigma), J of hmcmt_jacobian ([nChains][nData][nAC]: d rho_a / d sigma and
 * d phase / d sigma rows) and hmcdata of hmcmt_run_chain.  hmcmt_get_responses returns the (rho_a, phase) pairs. */
int hmcmt_plan_create_rho_phase(const hmcmt_problem* prob, hmcmt_plan** out);      /* compMode 2 (complex tipper rows): -3 */
void hmcmt_destroy(hmcmt_plan* plan);
/* sizes derived by the plan: n=0 N (unknowns/system), 1 nNode, 2 nCell, 3 nb, 4 half-bandwidth,
 * 5 tile-window T, 6 macro-steps S, 7 systems per chain, 8 receiver node row zid (0-based),
 * 9 factor bytes per system, 10 kernel launches issued so far (of this library), 11 solver of the plan (0 register-window
 * band kernel, 1 nested-dissection multifrontal), 12 real flops of one factorisation of one system in the implemented
 * ordering, 13 two CTAs per system (band kernel only) */
int64_t hmcmt_plan_info(const hmcmt_plan* plan, int what);

/* MT2DFwdSolver(mtMesh, mtData)  MT2DFwdSolver.jl:74-216 with sigma = activeCell*exp(m)+bg
 * (HMCSampler.jl:290-294).  m: [nChains][nAC]; pred: [nChains][nData] complex (dataID-masked order);
 * exTE / hxTM (optional, may be NULL): [nChains][nFreq][nNode] complex, node numbering of SURVEY.md A.2.
 * Keeps the factors alive on the device for hmcmt_jtvec (the reference's AinvTE/AinvTM). */
int hmcmt_forward(hmcmt_plan* plan, const double* m, double* pred, double* exTE, double* hxTM);
/* Same, but with the cell conductivities given directly (mtMesh.sigma, [nChains][ny*nz]) — the literal
 * MT2DFwdSolver(mtMesh, mtData) call without the log-conductivity transform. */
int hmcmt_forward_sigma(hmcmt_plan* plan, const double* sigma, double* pred, double* exTE, double* hxTM);

/* compJacTMatVec(exTE,hxTM,datVec,...)  compJacTMatVec.jl:8-329 for the state left by the last
 * hmcmt_forward: v [nChains][nData] complex -> gsig [nChains][nAC] = real(J^T v) w.r.t. conductivity.
 * Reuses the factors, fields and boundary values still resident from that forward evaluation (the reference's AinvTE /
 * AinvTM, compJacTMatVec.jl:220-224, 291-295): only the adjoint sources, one solve per system and the contraction run. */
int hmcmt_jtvec(hmcmt_plan* plan, const double* v, double* gsig);

/* Explicit Jacobian of the predicted impedances with respect to the active-cell conductivities for the state left by the
 * last forward evaluation — compJacMat.jl:7-381 (equivalently the transpose compJacTMat.jl:9-406 builds) with the same boundary-
 * condition approximations as compJacTMatVec: J [nChains][nData][nAC] complex, rows in the packed data order.  One adjoint
 * pass (adjoint sources, one solve per system with the resident factors, contraction) per receiver and per real / imaginary
 * part fills that receiver's row in every (frequency, mode) system at once: 2 nRx passes instead of nData. */
int hmcmt_jacobian(hmcmt_plan* plan, double* J);

/* J·dsig for the state of the last forward evaluation (forward-mode directional derivative, no explicit Jacobian).
 *   dsig [nChains][nAC]: conductivity perturbation of the active cells.
 *   jv   [nChains][nData] in the packed order: complex, or real (d rho_a, d phase rows) for Rho_Pha plans.
 * The result is hmcmt_jacobian's J times dsig: the exact transpose of the adjoint hmcmt_jtvec runs, with the same boundary-
 * condition approximations.  One tangent boundary recursion, one solve per system with the resident factors and the tangent
 * receiver functional; runs on the plan's stream and leaves the fields, factors, predictions, misfit and chain state as they
 * were.  -3 without a prior forward evaluation or on NULL arguments. */
int hmcmt_jvec(hmcmt_plan* plan, const double* dsig, double* jv);
/* Gauss-Newton Hessian of the data misfit in the sampler's coordinates m = ln sigma:
 *   hv = D Re(J^H Wd^2 J) D v,  D = diag(sigma_active);  Wd = 1/|err| per row (wd / wdPha for rho / phase rows).
 * with_prior != 0 adds beta Wm v.  v, hv: [nChains][nAC].  One hmcmt_jvec and one hmcmt_jtvec pass; the plan's gradient of the
 * last evaluation is kept.  -3 without a prior forward evaluation or on NULL arguments. */
int hmcmt_gn_hessvec(hmcmt_plan* plan, const double* v, int32_t with_prior, double* hv);
/* Projected Gauss-Newton-CG for the posterior mode, every chain on its own: minimises
 *   U(m) = phi_d(m) + 1/2 beta (m - m_ref)^T Wm (m - m_ref)   over  ln sigma_min <= m_i <= ln sigma_max
 * (the sampler's potential energy, with the plan's m_ref of hmcmt_set_state and the plan's bounds).  Iteration k:
 *   - evaluate U(m_k) and g_k (the plan's gradient evaluation, prior included);
 *   - active set A = {m_i <= lo and g_i > 0} u {m_i >= hi and g_i < 0}, P the mask that zeroes A;
 *   - CG from delta = 0 on P H P delta = -P g, H = D Re(J^H Wd^2 J) D + beta Wm (hmcmt_gn_hessvec with the prior): at most maxCG
 *     iterations, stop at |r| <= cgTol |r_0|; p^T H p <= 0 stops the CG (delta = r_0 if that happens at its first iteration);
 *   - delta scaled so that max |delta_i| <= maxStep;
 *   - Armijo backtracking on m(alpha) = clip(m_k + alpha delta, lo, hi), alpha = 1, 1/2, ..., at most maxLS trials: accept when
 *     U(m(alpha)) <= U(m_k) + 1e-4 g_k^T (m(alpha) - m_k);
 *   - the chain stops when U_k - U_{k+1} <= tolRel U_k or P g = 0 (stop reason 1), or when its line search fails: it then keeps
 *     m_k (stop reason 2).  maxIter outer iterations at most (stop reason 0).
 * m0: [nChains][nAC] start model, or NULL for the plan's current model; it is projected onto the bounds first.
 * m_out: [nChains][nAC].  history: [nChains][maxIter + 1][6], one row per accepted step, row 0 the start: (phi_d, phi_m, |P g|_2,
 * CG iterations, alpha, line-search trials); rows after a chain stopped are zero.  info: [nChains][2] = (accepted steps, stop
 * reason).  A chain's results do not depend on the other chains of the plan or on how the launches were issued.
 * Afterwards the plan's model, fields, factors, predictions, misfit and gradient are those of m_out, as after
 * hmcmt_forward_gradient_total(m_out); the momentum, m_ref and the mass matrix are untouched.
 * -3 on NULL m_out / history / info, maxIter < 0, maxCG < 1, maxLS < 1, maxStep <= 0, or a negative or non-finite cgTol / tolRel;
 * the device error flags (as hmcmt_status reports them) are checked once per outer iteration. */
int hmcmt_gauss_newton(hmcmt_plan* plan, const double* m0, int32_t maxIter, int32_t maxCG, double cgTol, int32_t maxLS,
                       double maxStep, double tolRel, double* m_out, double* history, int32_t* info);

/* compDataGradient(mtMesh,mtData,invParam,hmcprior)  HMCSampler.jl:277-330:
 * m -> pred [nChains][nData] complex, phi_d [nChains], grad [nChains][nAC] (w.r.t. log conductivity,
 * data part only, as the reference returns it). Host buffers; H2D/D2H inside. */
int hmcmt_forward_gradient(hmcmt_plan* plan, const double* m, double* pred, double* phid, double* grad);
/* The same evaluation, but grad = data part + model-norm part beta Wm (m - m_ref): the quantity proposeLeapfrog forms on the host
 * right after compDataGradient (HMCSampler.jl:240-262, getModelNormGradient).  m_ref is the reference model of the device-resident
 * chain state (hmcmt_set_state); the library computes that sum on the device in every evaluation anyway. */
int hmcmt_forward_gradient_total(hmcmt_plan* plan, const double* m, double* pred, double* phid, double* grad);

/* Device-resident chain state (hmcParamCurrent: rhomodel, momentum; invParam.refModel). */
int hmcmt_set_state(hmcmt_plan* plan, const double* m, const double* p, const double* mref);
int hmcmt_get_state(hmcmt_plan* plan, double* m, double* p);

/* proposeLeapfrog + getHamiltonian  HMCSampler.jl:206-269, 358-397, entirely on the device:
 * half kick, L x {drift (step clip 3.0), reflect at bounds, gradient, kick}, last kick halved.
 * intstep: [nChains] number of leapfrog steps (the reference's rand(t1:t2), injected).
 * stats out: [nChains][4] = (dataMisfit, mnorm, kinetic, H) at the proposal; pred (optional): [nChains][nData].
 * The proposal replaces the device state (m,p); use hmcmt_get_state / hmcmt_set_state to accept or reject. */
int hmcmt_leapfrog_trajectory(hmcmt_plan* plan, double dt, const int32_t* intstep, double* stats, double* pred);

/* `nsteps` leapfrog steps (drift, reflect, forward+adjoint gradient, prior gradient, kick) with no host
 * transfer at all — the timed region of bench.py's `value`. */
int hmcmt_leapfrog_steps_device(hmcmt_plan* plan, double dt, int32_t nsteps);

/* Frequency-sharded leapfrog step (SURVEY.md 8e; BASELINE.json configs[3]): every rank's plan holds a subset of the
 * frequencies and the full model.  compDataGradient is a sum over frequencies (the loop of MT2DFwdSolver.jl:163-191 and
 * compJacTMatVec.jl:200-324), so one step is
 *   hmcmt_step_partial   drift + reflect, forward + adjoint over THIS rank's frequencies, partial [gdata | phi_d] per chain
 *                        packed into the exchange buffer (device memory, nChains*(nAC+1) doubles);
 *   <caller>             sum-all-reduce of the exchange buffer across ranks (ncclAllReduce / torch.distributed);
 *   hmcmt_step_finish    prior gradient beta*Wm*(m-m_ref) added once, kick (HMCSampler.jl:255-265).
 * All of it is enqueued on the plan's stream: call hmcmt_sync before the caller's collective reads the buffer. */
int hmcmt_step_partial(hmcmt_plan* plan, double dt);
int hmcmt_exchange_buffer(hmcmt_plan* plan, void** device_ptr, int64_t* count);
int hmcmt_step_finish(hmcmt_plan* plan, double dt);
/* The same step with the exchange inside the library: NCCL over NVLink / NVSwitch on the plan's own stream (no host round
 * trip, no framework on the data path).  libnccl.so.2 is resolved at run time (dlopen by SONAME, so a process that already
 * loaded NCCL shares that copy).
 *   hmcmt_nccl_unique_id          rank 0: 128-byte ncclUniqueId, to be broadcast to the other ranks by the caller's own means
 *   hmcmt_nccl_init               every rank: communicator of `world` ranks bound to this plan's device
 *   hmcmt_leapfrog_steps_sharded  nsteps x { drift, forward + adjoint over this rank's systems, ncclAllReduce(SUM) of
 *                                 [gdata | phi_d], prior gradient, kick }, enqueued without synchronisation */
int hmcmt_nccl_unique_id(char* out128);
int hmcmt_nccl_init(hmcmt_plan* plan, const char* id128, int32_t rank, int32_t world);
int hmcmt_leapfrog_steps_sharded(hmcmt_plan* plan, double dt, int32_t nsteps);
/* blocks until all work queued on the plan's stream has finished */
int hmcmt_sync(hmcmt_plan* plan);
/* Device error flags of everything queued so far (synchronises): 0, or -10 (a singular / non-finite pivot block in some
 * system), or -21 (checkParameterBound!: a bound could not be met within 500 reflections, HMCSampler.jl:546-548, where the
 * reference prints a message and loops forever).  Reading clears the flags.  The asynchronous entry points
 * (hmcmt_leapfrog_steps_device, hmcmt_step_partial / _finish) do not check: call this after them. */
int hmcmt_status(hmcmt_plan* plan);
/* Mass matrix of the sampler (hmcprior.massType, HMCSampler.jl:81-86): kind 0 = "diagonal" (identity, the default), 1 =
 * non-diagonal M = Wm (setMassMatrix(invParam) HMCSampler.jl:478-489: dense Cholesky of Wm in the reference).  Here invM p is one
 * multifrontal solve with the sparse factor of Wm and sqrtM z the product with Wm's banded Cholesky factor (natural ordering,
 * identical to the reference's dense L).  Affects drift (getKineticGradient), kinetic energy and the momentum draws of
 * hmcmt_run_chain.  -40 if Wm is not positive definite. */
int hmcmt_set_mass_matrix(hmcmt_plan* plan, int32_t kind);
/* Response type of the forward evaluation of an impedance plan (compMTRespTE mt2DTE.jl:240-259, compMTRespTM mt2DTM.jl:224-242):
 * kind 0 = impedance, 1 = apparent resistivity rho_a = |Z|^2/(omega mu0) and phase atan2(Im Z, Re Z) in degrees (tipper slots keep
 * (Re T, Im T)).  A forward-only
 * toggle: the misfit and gradients of such a plan stay those of its impedance data (evaluations with kind 1 are launched eagerly,
 * outside the captured graph).  Gradients of rho / phase data come from a plan made by hmcmt_plan_create_rho_phase.
 * hmcmt_get_responses copies the responses of the last forward evaluation, unmasked:
 * out [nChains][nFreq][nRx][nComp][2] doubles = (Re Z, Im Z) or (rho_a, phase). */
int hmcmt_set_response_kind(hmcmt_plan* plan, int32_t kind);
int hmcmt_get_responses(hmcmt_plan* plan, double* out);
/* CUDA-event bracket on the plan's stream: start / stop (returns elapsed ms through *ms) */
int hmcmt_timer_start(hmcmt_plan* plan);
int hmcmt_timer_stop(hmcmt_plan* plan, float* ms);
/* accumulated CUDA-event time of the factorisation + forward solve since the last reset, and how many were timed.
 * reset = 1: clear and switch the timing on — evaluations then run un-grouped on the plan's stream so that the events bracket
 * the factorisation alone; reset = -1: clear and switch it off again (the default: groups of systems on their own streams
 * overlap each other, HMCMT_GROUPS); reset = 0: read only. */
int hmcmt_kernel_time(hmcmt_plan* plan, int reset, float* factor_ms, int64_t* factor_launches);
/* the same accumulated time split at the end of the factorisation: factorisation alone / forward solve alone (on the band path both
 * are one fused group of launches: everything is reported in the first part).  Read before a reset. */
int hmcmt_kernel_time_split(hmcmt_plan* plan, float* factor_only_ms, float* forward_solve_ms);

/* runHMCSampler(mtMesh,mtData,invParam,hmcprior)  HMCSampler.jl:72-196 for all chains of the plan with injected
 * random draws in the reference's draw order (SURVEY.md A.7):
 *   rhoref = round(unirandDouble(0.5 rho0, 1.5 rho0)) with rho0 = 1/exp(strModel[1]) (HMCSampler.jl:100-105,
 *   the homogeneous model that becomes invParam.strModel / refModel and defines the start Hamiltonian, drawn by the caller),
 *   m_start [nChains][nAC] = the model-file strModel: the reference copies it into hmcParamCurrent.rhomodel BEFORE replacing
 *   strModel (HMCSampler.jl:87 vs :100-109), so the first trajectory starts there (NULL: start from the homogeneous model),
 *   z_init [nChains][nAC], then per sample
 *   intsteps[i] (shared by the chains of this plan), u_accept [nChains][nsamples], z_mom [nsamples][nChains][nAC].
 * Outputs (leading dimension nChains): hmcmodel [nsamples][nAC] (sample-major = Julia's column-major
 *          nparam x nsamples), hmstats [nsamples+1][4] (Julia 4 x (nsamples+1)), accept [nsamples] (0/1),
 *          hmcdata [nsamples+1][nData] complex.  The Metropolis test and the sample bookkeeping run on the device; all
 *          random draws are uploaded once before the loop, which then enqueues without any host synchronisation.
 * reuse_last_forward != 0 drops the reference's redundant getHamiltonian forward sweep (the proposal's
 * misfit equals the last leapfrog step's); 0 re-runs the forward exactly as the reference does. */
int hmcmt_run_chain(hmcmt_plan* plan, double dt, int32_t nsamples, double rhoref, const double* m_start, const double* z_init,
                    const int32_t* intsteps, const double* u_accept, const double* z_mom, int32_t reuse_last_forward,
                    double* hmcmodel, double* hmstats, int32_t* accept, double* hmcdata);

/* Debug / parity: emit Aii of system (chain, mode, freq) in the reference's 1-based CSC numbering, its
 * right-hand side and boundary values, so sparsity pattern and DOF indexing can be compared bit-exactly
 * (SURVEY.md A.2).  colptr [N+1], rowval/nzval sized for nnz = 5N - 2(ny-1) - 2(nz-1); bc [2(ny+nz)] complex. */
int hmcmt_export_system(hmcmt_plan* plan, int32_t chain, int32_t mode, int32_t freq, int64_t* colptr, int64_t* rowval,
                        double* nzval, double* rhs, double* bc);

/* library build info: returns "sm_100a" etc. */
const char* hmcmt_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HMCMT_B200_H */
