// Batched complex-symmetric banded block-LDL^T factorisation for sm_100a.
//
// Replaces the per-frequency sparse direct factorisation the reference obtains from
// `factorMUMPS(Aii,1)` / `lu(Aii)` (mt2DTE.jl:47-55, mt2DTM.jl:46-54, MUMPSfuncs.jl:24-39).
//
// Algorithm (validated in tools/proto/tile_band_proto.py): the matrix is kept in the internal
// "fast-axis" ordering with half-bandwidth b.  A sliding window of T x T tiles of 8x8 complex
// entries (8T >= b+8) lives entirely in REGISTERS as FP64 tensor-core accumulator fragments:
// tile slots are addressed circularly (global tile-block beta -> slot beta mod T) and the
// unordered slot pair {I,J} always holds exactly one live lower-triangle tile, so T(T+1)/2
// register tiles are 100 % occupied and nothing ever moves.  One macro-step eliminates an
// 8-column panel:
//     S  <-  S - raw * A11^{-1} * raw^T            (pivot-free block elimination)
//   * the tile warps form M' = raw * (-A11^{-1}) and apply the rank-8 update with
//     mma.sync.m8n8k4.f64 (DMMA.8x8x4, measured full-rate 37.1 TF/s on B200); the next pivot
//     column is updated first and published to shared memory;
//   * the "factor warp" runs one panel AHEAD of them: it applies the current panel's update to the
//     next 8x8 pivot block itself (16 DMMAs), inverts it in registers (fraction-free Gauss-Jordan
//     through warp shuffles, pivot-free) and forms z = A11^{-1} y_p for the fused right-hand side;
//   * recycled slots are refilled from the 5-point stencil planes (assembly is fused: the matrix is
//     never written to memory); those rows are prefetched into a shared-memory ring two steps ahead.
//
// Two CTAs per system (`split`): the mesh lines are cut at a separator line; CTA 0 eliminates the
// lines before it, CTA 1 the lines after it in reverse order, both towards the separator (launch
// FM_OWN, 2 CTAs per system).  Each exports its window — its share of the separator's Schur
// complement — to global scratch; a second launch (FM_SEP, 1 CTA per system) sums the two images,
// eliminates the separator and back-substitutes it; a third launch (2 CTAs per system) back-substitutes
// the two halves — the pipelined sweep of band_solve.cuh in SM_BACKZ_OWN mode when the caller provides
// solve jobs, else this kernel in FM_BACK mode.  Stream order is the only synchronisation between the
// CTAs of a system.  This halves the sequential pivot chain and doubles the SMs a single chain can use.
//
// The stored factor is { raw_s (8T x 8), [A11_s^{-1} (8x8) | z_s (8)] } per macro-step and rank; it
// serves the forward solve (back-substitution fused below for unsplit systems and the separator) and
// the adjoint solve (band_solve.cuh).
#pragma once
#include <type_traits>
#ifndef HMCMT_GATE_ALL
#define HMCMT_GATE_ALL 0      // 1: every tile warp waits for the inversion before pass 2 (measured slower: 141.6 vs 144.9 steps/s at cfg2)
#endif

#include "common.cuh"

namespace hmcmt {

constexpr int TS = 8;         // tile size == DMMA m,n
constexpr int AZ = 72;        // complex entries per macro-step in the ainv stream: A11^{-1} (64) + z (8)

// Per-system description for a batched launch (one CTA, or two CTAs, per system).
struct BandSys {
    // stencil provider (internal ordering q = line*nf + f, see mt_kernels.cuh): A[q][q] = dr[q] + i*omega*dm[q],
    // A[q][q-1] = e1[q] (0 at line starts), A[q][q-nf] = e2[q] (0 on the first line)
    const double* dr;
    const double* dm;
    const double* e1;
    const double* e2;
    double omega;
    // dense lower-band provider (generic matrices through the MUMPS-shim ABI): band[g*(b+1)+d] = A[g][g-d]
    const cplx* band;
    const cplx* rhs;     // fused forward right-hand side (internal ordering, length N) or nullptr
    cplx* x;             // [N] solution of the fused system — only if rhs != nullptr
    double* panels[2];   // per half (rank): [steps][16*R] doubles: re/im x kk x R x 4 (exactly the smem operand layout)
    cplx* ainvz[2];      // per half (rank): [steps][72]: A11^{-1} row-major, then z = A11^{-1} * (forward-eliminated rhs block)
    cplx* wexp;          // split only: hand-over scratch [2][R*R] window images, [2][R] rhs windows, [R] separator solution
    int* status;         // 0 ok, -10 zero/NaN pivot block
};

// Geometry of the elimination order (uniform over the batch).
struct BandDom {
    int N;        // unknowns of the full system
    int nf;       // line length == half-bandwidth of the stencil systems
    int b;        // half-bandwidth
    int nl;       // number of lines (stencil systems); unused for the band provider
    int split;    // 1: two CTAs per system (FM_OWN / FM_SEP / FM_BACK launches)
    int lineSep;  // separator line (split only)
};

// Local ordering of one half (rank): [head padding | own lines | separator line | tail padding]; the padding makes
// the separator start on a tile boundary so that both ranks' windows can be merged tile by tile.
struct LocalDom {
    int rank, split, nf, nl, lineSep, N;
    int pad, nOwn, lineStart, lineStep, sOwn, sTot, nLoc;
    __host__ __device__ static LocalDom make(const BandDom& d, int rank) {
        LocalDom L;
        L.rank = rank; L.split = d.split; L.nf = d.nf; L.nl = d.nl; L.lineSep = d.lineSep; L.N = d.N;
        if (!d.split) {
            L.pad = 0; L.nOwn = d.N; L.lineStart = 0; L.lineStep = 1; L.nLoc = d.N;
            L.sOwn = L.sTot = (d.N + TS - 1) / TS;
        } else {
            int lines = rank == 0 ? d.lineSep : d.nl - 1 - d.lineSep;
            L.nOwn = lines * d.nf;
            L.lineStart = rank == 0 ? 0 : d.nl - 1;
            L.lineStep = rank == 0 ? 1 : -1;
            L.pad = (TS - L.nOwn % TS) % TS;
            L.nLoc = L.pad + L.nOwn + d.nf;
            L.sOwn = (L.pad + L.nOwn) / TS;
            L.sTot = rank == 0 ? (L.nLoc + TS - 1) / TS : L.sOwn;
        }
        return L;
    }
    // local row -> global internal index; -1 head padding, -2 tail padding.  kind: 0 own row, 1 separator row.
    __host__ __device__ int map(int g, int& kind, int& lrel) const {
        kind = 0; lrel = 0;
        if (!split) return g < N ? g : -2;
        if (g < pad) return -1;
        int u = g - pad;
        if (u >= nOwn) {
            u -= nOwn;
            if (u >= nf) return -2;
            kind = 1;
            return lineSep * nf + u;
        }
        lrel = u / nf;
        int f = u - lrel * nf;
        return (lineStart + lineStep * lrel) * nf + f;
    }
};

__host__ __device__ constexpr int band_T_for(int b) { return (b + 7) / 8 + 1; }
__host__ __device__ constexpr int panel_doubles(int T) { return 16 * TS * T; }

template <int T>
struct FactorCfg {
    static constexpr int NT = T * (T + 1) / 2;
    // tile {X,Y} belongs to warp (X+Y) mod (T+1): every warp owns exactly T/2 tiles and at most ONE tile of any
    // pivot column, so recycle / look-ahead / trailing-update roles are balanced and found by one table lookup
    static_assert(T % 2 == 0, "even tile windows only");
    static constexpr int NW = T + 1;
    static constexpr int TPW = T / 2;
    static constexpr int R = TS * T;
    static constexpr int NTHREADS = (NW + 1) * 32;
};

constexpr int kRing = 4;       // prefetch ring depth (recycle rows / rhs), filled kPre steps ahead
constexpr int kPre = 2;

template <int T>
struct FactorSmem {
    static constexpr int R = TS * T;
    static constexpr int kBackStages = 5;
    // [buf][re/im][kk][r][t]  — raw[buf] is one contiguous panel image (16*R doubles)
    double raw[2][2][2][R][4];
    double m[2][2][2][R][4];
    double nainv[2][2][2][8][4];   // -A11^{-1} in B-fragment layout [buf][re/im][kk][n][t]
    double mscr[2][2][8][4];       // factor warp: M' of the next pivot block (A-fragment layout)
    double dnext[2][2][8][8];      // [buf][re/im][row][col]: next-next pivot block, updated through the current panel
    cplx ainvz[2][AZ];             // plain A11^{-1} (row-major) + z, staged for the store
    cplx y[R];                     // circular window of the forward-eliminated rhs / back-substituted x
    double ringRow[kRing][4][8];   // stencil planes (dr, dm, e1, e2) of the rows entering the window
    cplx ringRhs[kRing][8];
    cplx part[16][8];              // back-substitution partial sums
    double stage[kBackStages][2][2][R][4];   // TMA landing buffers of the fused back-substitution
    cplx stageAZ[kBackStages][AZ];
    unsigned char tI[FactorCfg<T>::NT], tJ[FactorCfg<T>::NT];    // [warp*TPW + i]
    signed char li[FactorCfg<T>::NW][T];                          // local index of the tile of warp w touching block b (-1: none)
    uint64_t mbar[kBackStages];
    int fail;
};

enum { BAR_RAW = 1, BAR_INV = 2, BAR_M = 3, BAR_GJ = 4 /* and 5: alternates with the step parity */ };
// what one launch does: the whole system / own lines of both halves / separator (+ its back-substitution) / back-substitution of the halves
enum FactorMode { FM_FULL = 0, FM_OWN = 1, FM_SEP = 2, FM_BACK = 3 };
__host__ __device__ constexpr size_t split_scratch_entries(int R) { return 2 * (size_t)R * R + 3 * (size_t)R; }

// Matrix entries in the LOCAL ordering of a half (rank).
struct EntryProvider {
    const double *dr, *dm, *e1, *e2;
    const cplx* band;
    double omega;
    int b;
    LocalDom L;
    // one stencil plane (0 dr, 1 dm, 2 e1, 3 e2) of local row g
    __device__ __forceinline__ double plane(int g, int pl) const {
        int kind, lrel;
        const int q = L.map(g, kind, lrel);
        if (q == -1) return pl == 0 ? 1.0 : 0.0;                              // head padding: identity rows
        if (q == -2) return (pl == 0 && L.rank == 0) ? 1.0 : 0.0;             // tail padding: identity, counted once
        if (kind == 1 && L.rank == 1) return pl == 3 ? e2[q + L.nf] : 0.0;    // separator seen from behind: coupling only
        if (pl == 0) return dr[q];
        if (pl == 1) return dm[q];
        if (pl == 2) return e1[q];
        if (L.lineStep > 0 || kind == 1) return e2[q];
        return lrel > 0 ? e2[q + L.nf] : 0.0;                                 // reversed lines: the previous local line is line+1
    }
    // direct (global-memory) evaluation, local indices hi >= lo
    __device__ __forceinline__ cplx get(int hi, int lo) const {
        const int d = hi - lo;
        if (band) {
            if (hi >= L.N) return mk(d == 0 ? 1.0 : 0.0, 0.0);               // identity padding past the end
            return d <= b ? band[(size_t)hi * (b + 1) + d] : mk(0.0, 0.0);
        }
        if (d == 0) return mk(plane(hi, 0), omega * plane(hi, 1));
        if (d == 1) return mk(plane(hi, 2), 0.0);
        if (d == L.nf) return mk(plane(hi, 3), 0.0);
        return mk(0.0, 0.0);
    }
    // rows of one 8-row block staged in shared memory: row[plane][hi & 7]
    __device__ __forceinline__ cplx get_staged(const double (*row)[8], int hi, int lo) const {
        const int d = hi - lo, r = hi & 7;
        if (d == 0) return mk(row[0][r], omega * row[1][r]);
        if (d == 1) return mk(row[2][r], 0.0);
        if (d == L.nf) return mk(row[3][r], 0.0);
        return mk(0.0, 0.0);
    }
    __device__ __forceinline__ cplx rhs_at(const cplx* rhs, int g) const {
        int kind, lrel;
        const int q = L.map(g, kind, lrel);
        if (q < 0 || (kind == 1 && L.rank == 1)) return mk(0.0, 0.0);
        return rhs[q];
    }
    __device__ __forceinline__ void x_store(cplx* x, int g, cplx v) const {
        int kind, lrel;
        const int q = L.map(g, kind, lrel);
        if (q >= 0 && !(kind == 1 && L.rank == 1)) x[q] = v;
    }
};

// In-register inversion of an 8x8 complex-symmetric block by one warp, pivot-free.  Lane 4*i + t holds A[i][2t], A[i][2t+1]
// on entry and A^{-1}[i][2t], A^{-1}[i][2t+1] on return.
// Fraction-free Gauss-Jordan (validated in numpy, DESIGN.md): rows i != k take  row_i <- (p row_i - a_ik row_k) 2^-e
// with an exact power-of-two rescale, so no reciprocal sits on the 8-pivot dependency chain; every row carries
// its accumulated scale q_i and the true inverse is  a_ij / q_i, formed with one reciprocal per row at the end.
// UNROLL: the fully unrolled form has the shorter dependency chain (2 000 vs ~3 000 cycles alone) and suits kernels whose other
// warps wait for it (mf_kernels.cuh); inside band_factor_kernel, where ~800 more instructions per macro-step compete for the
// instruction cache with the tile warps' code, the rolled loop measured 5 % faster end to end.
// nsteps < 8: rows / columns nsteps..7 are identity padding (multifrontal fronts pad their pivot counts to the tile size): their
// pivot steps would change nothing and are skipped.
template <bool UNROLL>
__device__ __forceinline__ void gj_invert8(cplx& a0, cplx& a1, bool& bad, const int i, const int t, const int nsteps = 8) {
    const int j0 = 2 * t;
    cplx q = mk(1.0, 0.0);
    auto pivot_step = [&](const int k) {
        const int srcRow = 4 * k + t, srcCol = 4 * i + (k >> 1), srcPiv = 4 * k + (k >> 1);
        const cplx mine = (k & 1) ? a1 : a0;
        const cplx pk = mk(__shfl_sync(0xffffffffu, mine.x, srcPiv), __shfl_sync(0xffffffffu, mine.y, srcPiv));
        const cplx f = mk(__shfl_sync(0xffffffffu, mine.x, srcCol), __shfl_sync(0xffffffffu, mine.y, srcCol));
        const cplx ck = mk(__shfl_sync(0xffffffffu, q.x, 4 * k), __shfl_sync(0xffffffffu, q.y, 4 * k));
        cplx r0 = mk(__shfl_sync(0xffffffffu, a0.x, srcRow), __shfl_sync(0xffffffffu, a0.y, srcRow));
        cplx r1 = mk(__shfl_sync(0xffffffffu, a1.x, srcRow), __shfl_sync(0xffffffffu, a1.y, srcRow));
        if (j0 == k) r0 = ck;                       // slot (k,k) switches to the right-hand block: value c_k
        if (j0 + 1 == k) r1 = ck;
        const double mag = fmax(fabs(pk.x), fabs(pk.y));
        if (!(mag > 1e-290) || !(mag < 1e290)) bad = true;
        const int eb = (__double2hiint(mag) >> 20) & 0x7ff;
        const double sc = __hiloint2double((2046 - eb) << 20, 0);          // 2^-(exponent of the pivot), exact
        const cplx ps = mk(pk.x * sc, pk.y * sc), fs = mk(f.x * sc, f.y * sc);
        if (i == k) {
            a0 = r0; a1 = r1; q = pk;
        } else {
            const cplx b0 = (j0 == k) ? mk(0.0, 0.0) : a0, b1 = (j0 + 1 == k) ? mk(0.0, 0.0) : a1;
            cplx n0 = ps * b0, n1 = ps * b1;
            cfma(n0, -fs, r0);
            cfma(n1, -fs, r1);
            a0 = n0; a1 = n1;
            q = ps * q;
        }
    };
    if constexpr (UNROLL) {
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < nsteps) pivot_step(k);
    } else {
#pragma unroll 1
        for (int k = 0; k < nsteps; ++k) pivot_step(k);
    }
    // 1/q = s conj(qs) / |qs|^2 with qs = s q, s = 2^-(exponent of q) exact: |qs|^2 lies in [1, 8) whatever the scale of the
    // matrix, so neither overflows nor turns subnormal where |q|^2 would (|q| beyond ~2^511 or below ~2^-511); for every other q
    // the result is bit-identical to conj(q) / |q|^2
    const int eq = (__double2hiint(fmax(fabs(q.x), fabs(q.y))) >> 20) & 0x7ff;
    const double sq = __hiloint2double((2046 - eq) << 20, 0);
    const cplx qs = mk(q.x * sq, q.y * sq);
    const double den = fma(qs.x, qs.x, qs.y * qs.y);
    const double iden = __drcp_rn(den) * sq;
    if (!(den > 0.0) || isinf(den) || isinf(iden)) bad = true;
    const cplx qi = mk(qs.x * iden, -qs.y * iden);
    a0 = a0 * qi;
    a1 = a1 * qi;
}

// grid = nsys CTAs (FM_FULL, FM_SEP) or 2*nsys CTAs (FM_OWN, FM_BACK: CTA = 2*system + rank), block = FactorCfg<T>::NTHREADS,
// dynamic smem = sizeof(FactorSmem<T>)
template <int T>
__global__ void __launch_bounds__(FactorCfg<T>::NTHREADS, 1)
band_factor_kernel(const BandSys* __restrict__ systems, BandDom dom, int mode) {
    using Cfg = FactorCfg<T>;
    constexpr int NW = Cfg::NW, TPW = Cfg::TPW, R = Cfg::R, NTHR = Cfg::NTHREADS;
    constexpr bool kGateAll = HMCMT_GATE_ALL;
    constexpr int kGateThreads = kGateAll ? NTHR : 32 * (NW / 4 + 1);      // warps w <= NW with w % 4 == NW % 4 (the factor warp's scheduler)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FactorSmem<T>& sm = *reinterpret_cast<FactorSmem<T>*>(smem_raw);

    const bool paired = (mode == FM_OWN || mode == FM_BACK);
    const int rank = paired ? (int)(blockIdx.x & 1) : 0;
    const BandSys sys = systems[paired ? (blockIdx.x >> 1) : blockIdx.x];
    const LocalDom L = LocalDom::make(dom, rank);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);      // tells the compiler the role branches are warp-uniform
    const int g = lane >> 2, t = lane & 3;
    const int nf = dom.nf;
    EntryProvider prov{sys.dr, sys.dm, sys.e1, sys.e2, sys.band, sys.omega, dom.b, L};
    const bool staged = (sys.band == nullptr);      // stencil rows come through the smem ring
    double* const panels = sys.panels[rank];
    cplx* const ainvz = sys.ainvz[rank];
    const int nLoc = L.nLoc;
    // macro-steps [sBeg, sEnd) of this launch (local numbering of this rank)
    const int sBeg = (mode == FM_SEP) ? L.sOwn : 0;
    const int sEnd = (mode == FM_FULL || mode == FM_SEP) ? L.sTot : (mode == FM_OWN ? L.sOwn : 0);
    // hand-over scratch of a split system; window images / rhs windows are indexed relative to the separator start
    cplx* const wimg0 = sys.wexp;
    cplx* const wimg1 = sys.wexp + (size_t)R * R;
    cplx* const yimg0 = sys.wexp + 2 * (size_t)R * R;
    cplx* const yimg1 = yimg0 + R;
    cplx* const xsep = yimg0 + 2 * R;
    // window slot block -> position relative to local block `base`
    auto rel = [&](int slot, int base) { int a = slot - base % T; return a < 0 ? a + T : a; };

  if (mode != FM_BACK) {
    // tile tables: warp w owns the unordered slot pairs {X,Y}, X <= Y, with (X+Y) mod NW == w
    for (int w_b = 0; w_b < NW; w_b += NTHR) if (const int w = w_b + tid; w < NW) {
        int cnt = 0;
        for (int bb = 0; bb < T; ++bb) sm.li[w][bb] = -1;
        for (int X = 0; X < T; ++X) {
            int Y = w - X; if (Y < 0) Y += NW;
            if (Y >= T || Y < X) continue;
            sm.tI[w * TPW + cnt] = (unsigned char)X;
            sm.tJ[w * TPW + cnt] = (unsigned char)Y;
            sm.li[w][X] = (signed char)cnt;
            sm.li[w][Y] = (signed char)cnt;
            ++cnt;
        }
    }
    // rhs window: slot block X holds local block sBeg + rel(X)
    for (int i_b = 0; i_b < R; i_b += NTHR) if (const int i = i_b + tid; i < R) {
        cplx v = mk(0.0, 0.0);
        if (sys.rhs) {
            if (mode == FM_SEP) {
                const int a = rel(i >> 3, sBeg) * TS + (i & 7);
                v = yimg0[a] + yimg1[a];
            } else if (i < nLoc) v = prov.rhs_at(sys.rhs, i);
        }
        sm.y[i] = v;
    }
    if (warp == 0) {        // ring entries of steps sBeg..sBeg+kPre-1: blocks sBeg+T .. sBeg+T+kPre-1
        for (int q = 0; q < kPre; ++q) {
            const int gr = (sBeg + T + q) * TS + (lane & 7);
            sm.ringRow[(sBeg + q) % kRing][lane >> 3][lane & 7] = staged ? prov.plane(gr, lane >> 3) : 0.0;
            if (lane < 8) sm.ringRhs[(sBeg + q) % kRing][lane] = (sys.rhs && gr < nLoc) ? prov.rhs_at(sys.rhs, gr) : mk(0.0, 0.0);
        }
    }
    if (tid == 0) sm.fail = 0;
    cta_sync();

    if (warp < NW) {
        // =============================== tile warps ===============================
        double cre[TPW][2], cim[TPW][2];
        int tI[TPW], tJ[TPW];
#pragma unroll
        for (int i = 0; i < TPW; ++i) {
            tI[i] = sm.tI[warp * TPW + i];
            tJ[i] = sm.tJ[warp * TPW + i];
            if (mode == FM_SEP) {
                // window = sum of the two Schur-complement images exported by the FM_OWN launch
                const int row = rel(tI[i], sBeg) * TS + g, col = rel(tJ[i], sBeg) * TS + 2 * t;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const cplx v = wimg0[(size_t)row * R + col + e] + wimg1[(size_t)row * R + col + e];
                    cre[i][e] = v.x;
                    cim[i][e] = v.y;
                }
            } else {
                // initial window: slot block X holds local block X
                const int gi = tI[i] * TS + g;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int gj = tJ[i] * TS + 2 * t + e;
                    cplx v = prov.get(max(gi, gj), min(gi, gj));
                    cre[i][e] = v.x;
                    cim[i][e] = v.y;
                }
            }
        }
        // dump of the tiles touching slot block `q` into raw[nb] (panel columns = block q)
        auto dump = [&](int i, int q, int nb) {
            if (tJ[i] == q) {   // rows <-> I, cols <-> pivot  (also the diagonal tile)
                int r = tI[i] * TS + g;
                *reinterpret_cast<double2*>(&sm.raw[nb][0][t >> 1][r][(t & 1) * 2]) = make_double2(cre[i][0], cre[i][1]);
                *reinterpret_cast<double2*>(&sm.raw[nb][1][t >> 1][r][(t & 1) * 2]) = make_double2(cim[i][0], cim[i][1]);
            } else {            // tI == q: rows <-> pivot, cols <-> J : transposed
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    int r = tJ[i] * TS + 2 * t + e;
                    sm.raw[nb][0][g >> 2][r][g & 3] = cre[i][e];
                    sm.raw[nb][1][g >> 2][r][g & 3] = cim[i][e];
                }
            }
        };
        auto dump_diag = [&](int i, int nb) {      // plain 8x8 image of a diagonal tile for the factor warp
            *reinterpret_cast<double2*>(&sm.dnext[nb][0][g][2 * t]) = make_double2(cre[i][0], cre[i][1]);
            *reinterpret_cast<double2*>(&sm.dnext[nb][1][g][2 * t]) = make_double2(cim[i][0], cim[i][1]);
        };
        // DMMA latency on B200 is ~138 cycles (tools/ubench): 4 independent 2-link accumulation chains per tile
        auto update = [&](int i, int buf) {
            const int ra = tI[i] * TS + g, rb = tJ[i] * TS + g;
            double t1[2] = {0.0, 0.0}, t2[2] = {0.0, 0.0};
            double are[2], aim[2], bre[2], bim[2];
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                are[kk] = sm.m[buf][0][kk][ra][t]; aim[kk] = sm.m[buf][1][kk][ra][t];
                bre[kk] = sm.raw[buf][0][kk][rb][t]; bim[kk] = sm.raw[buf][1][kk][rb][t];
            }
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                dmma884(cre[i], are[kk], bre[kk]);
                dmma884(cim[i], are[kk], bim[kk]);
                dmma884(t1, -aim[kk], bim[kk]);
                dmma884(t2, aim[kk], bre[kk]);
            }
            cre[i][0] += t1[0]; cre[i][1] += t1[1];
            cim[i][0] += t2[0]; cim[i][1] += t2[1];
        };
        // fused forward elimination of the rhs for block X: y_X -= raw_X z   (z = A11^{-1} y_p from the factor warp)
        auto y_update = [&](int X, int buf) {
            if (lane < 8) {
                const int ry = X * TS + lane;
                cplx acc = sm.y[ry];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    cplx rv = mk(sm.raw[buf][0][k >> 2][ry][k & 3], sm.raw[buf][1][k >> 2][ry][k & 3]);
                    cfma(acc, -rv, sm.ainvz[buf][64 + k]);
                }
                sm.y[ry] = acc;
            }
        };

        {
            const int s0 = sBeg, s1 = sEnd;
            // prologue: publish panel s0 (tiles touching its slot) and the pivot block of panel s0+1
            {
                const int q0 = s0 % T, q1 = (s0 + 1) % T;
                const int i0 = sm.li[warp][q0];
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    if (i == i0) dump(i, q0, s0 & 1);
                    if (tI[i] == q1 && tJ[i] == q1) dump_diag(i, (s0 + 1) & 1);
                }
                bar_arrive(BAR_RAW, NTHR);
            }
            for (int s = s0; s < s1; ++s) {
                const int p = s % T, p1 = (s + 1) % T, p2 = (s + 2) % T, buf = s & 1;
                // roles of this warp's tiles in this step (at most one tile per pivot column)
                const int ip = sm.li[warp][p];
                int ip1 = -1, idg = -1;                         // look-ahead tile / pivot block of panel s+2 (if owned)
                if (s + 1 < s1) {
                    ip1 = sm.li[warp][p1];
                    int c = sm.li[warp][p2];
                    if (c >= 0 && 2 * p2 == ((2 * p2 >= NW) ? warp + NW : warp)) idg = c;
                }
                bar_sync(BAR_INV, NTHR);                       // raw(s) complete, -A11^{-1}(s) and z(s) published
                if (__any_sync(0xffffffffu, sm.fail != 0)) break;
                // M'_X = raw_X * (-A11^{-1}) for slot block X != p (one block per warp)
                int myX = -1;
                if (warp < T - 1) {
                    int X = p + 1 + warp; if (X >= T) X -= T;
                    myX = X;
                    double mre[2] = {0.0, 0.0}, mim[2] = {0.0, 0.0}, mr2[2] = {0.0, 0.0}, mi2[2] = {0.0, 0.0};
                    const int r = X * TS + g;
#pragma unroll
                    for (int kk = 0; kk < 2; ++kk) {
                        double are = sm.raw[buf][0][kk][r][t], aim = sm.raw[buf][1][kk][r][t];
                        double bre = sm.nainv[buf][0][kk][g][t], bim = sm.nainv[buf][1][kk][g][t];
                        dmma884(mre, are, bre);
                        dmma884(mim, are, bim);
                        dmma884(mr2, -aim, bim);
                        dmma884(mi2, aim, bre);
                    }
                    mre[0] += mr2[0]; mre[1] += mr2[1]; mim[0] += mi2[0]; mim[1] += mi2[1];
                    *reinterpret_cast<double2*>(&sm.m[buf][0][t >> 1][r][(t & 1) * 2]) = make_double2(mre[0], mre[1]);
                    *reinterpret_cast<double2*>(&sm.m[buf][1][t >> 1][r][(t & 1) * 2]) = make_double2(mim[0], mim[1]);
                    if (sys.rhs && warp == 0) y_update(X, buf);     // X == p1: the factor warp needs y_{p1} for z(s+1)
                }
                if (sys.rhs && warp == NW - 1 && lane >= 8 && lane < 16)      // recycle the rhs window slot p: local block s+T
                    sm.y[p * TS + lane - 8] = sm.ringRhs[s % kRing][lane - 8];
                if (warp == T - 1) {
                    // this warp has no M' block: it streams the finished panel s and [A11^{-1} | z] to HBM (coalesced 16-byte stores)
                    const double2* src = reinterpret_cast<const double2*>(&sm.raw[buf][0][0][0][0]);
                    double2* dst = reinterpret_cast<double2*>(panels + (size_t)s * panel_doubles(T));
                    constexpr int NQ = panel_doubles(T) / 2 / 32;      // 16-byte chunks per lane
                    constexpr int HQ = (NQ + 1) / 2;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        double2 tmp[HQ];
#pragma unroll
                        for (int qq = 0; qq < HQ; ++qq) if (h * HQ + qq < NQ) tmp[qq] = src[lane + 32 * (h * HQ + qq)];
#pragma unroll
                        for (int qq = 0; qq < HQ; ++qq) if (h * HQ + qq < NQ) dst[lane + 32 * (h * HQ + qq)] = tmp[qq];
                    }
                    cplx* dz = ainvz + (size_t)s * AZ;
                    for (int qq = lane; qq < AZ; qq += 32) dz[qq] = sm.ainvz[buf][qq];
                }
                bar_sync(BAR_M, NW * 32);
                // recycle the tile touching slot block p: its panel (raw(s)) is already published, and it now holds
                // entries of local block s+T, whose untouched stencil couplings may already reach the next pivot block.
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    if (i != ip) continue;
                    int dI = tI[i] - p1; if (dI < 0) dI += T;      // position inside the window [s+1, s+T]
                    int dJ = tJ[i] - p1; if (dJ < 0) dJ += T;
                    // row/column distance between the entering block (position T-1) and the other block of the tile
                    const int delta = TS * (T - 1 - min(dI, dJ));
                    const bool cand = !staged || delta <= TS || (delta + 7 >= nf && delta - 7 <= nf);   // warp-uniform
                    cre[i][0] = cre[i][1] = cim[i][0] = cim[i][1] = 0.0;
                    if (cand) {
                        int gi = (s + 1 + dI) * TS + g;
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            int gj = (s + 1 + dJ) * TS + 2 * t + e;
                            int hi = max(gi, gj), lo = min(gi, gj);    // hi always lies in the entering block s+T
                            cplx v = staged ? prov.get_staged(sm.ringRow[s % kRing], hi, lo) : prov.get(hi, lo);
                            cre[i][e] = v.x;
                            cim[i][e] = v.y;
                        }
                    }
                }
                // pass 1: the tile of the next pivot column (and the pivot block after it) first, then publish
                if (s + 1 < s1) {
#pragma unroll
                    for (int i = 0; i < TPW; ++i) {
                        if (i == ip1) {
                            if (i != ip) update(i, buf);            // the recycled {p,p1} tile is fresh: no update
                            dump(i, p1, buf ^ 1);
                        } else if (i == idg) {
                            if (i != ip) update(i, buf);            // (T == 2: p2 == p, already recycled)
                            dump_diag(i, buf);                      // pivot block of panel s+2, updated through panel s
                        }
                    }
                    bar_arrive(BAR_RAW, NTHR);
                }
                if (sys.rhs && myX >= 0 && warp != 0) y_update(myX, buf);
                // The tile warps that share a scheduler (and its FP64 / DMMA pipe) with the factor warp hold their bulk of
                // DMMAs back until it has inverted the next pivot block: that inversion is the serial chain of the loop and
                // ran 1.5x slower when it had to compete for the pipe.
                // Two barrier ids alternating with the step parity: the factor warp only arrives, so with a single id it
                // could arrive for step s+1 before a slow tile warp has waited for step s (it is held back by BAR_RAW one
                // step later, which makes the alternating pair safe).
                if (kGateAll || (warp & 3) == (NW & 3)) bar_sync(BAR_GJ + (s & 1), kGateThreads);
                // pass 2: the rest of the trailing window
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    if (i == ip || i == ip1 || i == idg) continue;
                    update(i, buf);
                }
            }
            if (mode == FM_OWN) {
                // end of the own lines: export the window (positions relative to the separator start), both triangles
                cplx* const img = rank == 0 ? wimg0 : wimg1;
#pragma unroll
                for (int i = 0; i < TPW; ++i) {
                    const int aI = rel(tI[i], s1), aJ = rel(tJ[i], s1);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const cplx v = mk(cre[i][e], cim[i][e]);
                        img[(size_t)(aI * TS + g) * R + aJ * TS + 2 * t + e] = v;
                        if (aI != aJ) img[(size_t)(aJ * TS + 2 * t + e) * R + aI * TS + g] = v;
                    }
                }
            }
        }
    } else {
        // =============================== factor warp ===============================
        const int i = g, j0 = 2 * t;
        cplx a0, a1;                                        // A11^{-1}[i][j0], [i][j0+1] of the CURRENT panel
        bool bad = false;
        auto invert = [&]() { gj_invert8<false>(a0, a1, bad, g, t); };
        auto publish = [&](int buf) {      // -A11^{-1} as B-fragments, plain A11^{-1} for the store
            // B-fragment layout wants plane[kk][n][tt] = -Ainv[4kk+tt][n]; Ainv is symmetric, so write -Ainv[i][j] at [j>>2][i][j&3]
            *reinterpret_cast<double2*>(&sm.nainv[buf][0][j0 >> 2][i][j0 & 3]) = make_double2(-a0.x, -a1.x);
            *reinterpret_cast<double2*>(&sm.nainv[buf][1][j0 >> 2][i][j0 & 3]) = make_double2(-a0.y, -a1.y);
            sm.ainvz[buf][i * 8 + j0] = a0;
            sm.ainvz[buf][i * 8 + j0 + 1] = a1;
        };
        {
            const int s0 = sBeg, s1 = sEnd;
            // prologue: invert the pivot block of panel s0
            bar_sync(BAR_RAW, NTHR);
            {
                const int rp0 = (s0 % T) * TS;
                double2 lre = *reinterpret_cast<const double2*>(&sm.raw[s0 & 1][0][j0 >> 2][rp0 + i][j0 & 3]);
                double2 lim = *reinterpret_cast<const double2*>(&sm.raw[s0 & 1][1][j0 >> 2][rp0 + i][j0 & 3]);
                a0 = mk(lre.x, lim.x); a1 = mk(lre.y, lim.y);
                invert();
                publish(s0 & 1);
            }
            for (int s = s0; s < s1; ++s) {
                const int p = s % T, p1 = (s + 1) % T, buf = s & 1;
                const int rp = p * TS;
                bad = __any_sync(0xffffffffu, bad);
                if (bad && lane == 0) { sm.fail = 1; if (sys.status) *sys.status = kErrSingular; }
                if (sys.rhs) {
                    // z_i = sum_j Ainv[i][j] y_p[j] : two terms per lane, reduced over the 4 lanes of a row
                    cplx acc = a0 * sm.y[rp + j0] + a1 * sm.y[rp + j0 + 1];
#pragma unroll
                    for (int off = 1; off <= 2; off <<= 1) {
                        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off);
                        acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
                    }
                    if (t == 0) sm.ainvz[buf][64 + i] = acc;
                } else if (t == 0) sm.ainvz[buf][64 + i] = mk(0.0, 0.0);
                bar_arrive(BAR_INV, NTHR);                      // panel s may be applied (bar.arrive orders the prior smem writes)
                if (bad) break;
                // ring prefetch for the block entering the window kPre steps from now (loads stay in flight over the inversion)
                const int gr = (s + kPre + T) * TS + (lane & 7);
                const double rowv = staged ? prov.plane(gr, lane >> 3) : 0.0;
                const cplx rhsv = (sys.rhs && lane < 8 && gr < nLoc) ? prov.rhs_at(sys.rhs, gr) : mk(0.0, 0.0);
                if (s + 1 < s1) {
                    // ---- early inversion of the next pivot block:  A11(s+1) = D(s+1; through s-1) + M'_{p1} raw_{p1}^T ----
                    double dre[2], dim_[2];
                    {
                        double2 vre = *reinterpret_cast<const double2*>(&sm.dnext[buf ^ 1][0][i][j0]);
                        double2 vim = *reinterpret_cast<const double2*>(&sm.dnext[buf ^ 1][1][i][j0]);
                        dre[0] = vre.x; dre[1] = vre.y; dim_[0] = vim.x; dim_[1] = vim.y;
                    }
                    const int r1 = p1 * TS + g;
                    double mre[2] = {0.0, 0.0}, mim[2] = {0.0, 0.0}, mr2[2] = {0.0, 0.0}, mi2[2] = {0.0, 0.0};
                    double bre[2], bim[2];
#pragma unroll
                    for (int kk = 0; kk < 2; ++kk) {
                        bre[kk] = sm.raw[buf][0][kk][r1][t]; bim[kk] = sm.raw[buf][1][kk][r1][t];
                        double nre = sm.nainv[buf][0][kk][g][t], nim = sm.nainv[buf][1][kk][g][t];
                        dmma884(mre, bre[kk], nre);
                        dmma884(mim, bre[kk], nim);
                        dmma884(mr2, -bim[kk], nim);
                        dmma884(mi2, bim[kk], nre);
                    }
                    mre[0] += mr2[0]; mre[1] += mr2[1]; mim[0] += mi2[0]; mim[1] += mi2[1];
                    *reinterpret_cast<double2*>(&sm.mscr[0][t >> 1][g][(t & 1) * 2]) = make_double2(mre[0], mre[1]);
                    *reinterpret_cast<double2*>(&sm.mscr[1][t >> 1][g][(t & 1) * 2]) = make_double2(mim[0], mim[1]);
                    __syncwarp();
                    double dr2[2] = {0.0, 0.0}, di2[2] = {0.0, 0.0};
#pragma unroll
                    for (int kk = 0; kk < 2; ++kk) {
                        double are = sm.mscr[0][kk][g][t], aim = sm.mscr[1][kk][g][t];
                        dmma884(dre, are, bre[kk]);
                        dmma884(dim_, are, bim[kk]);
                        dmma884(dr2, -aim, bim[kk]);
                        dmma884(di2, aim, bre[kk]);
                    }
                    a0 = mk(dre[0] + dr2[0], dim_[0] + di2[0]); a1 = mk(dre[1] + dr2[1], dim_[1] + di2[1]);
                    invert();
                    publish(buf ^ 1);
                }
                bar_arrive(BAR_GJ + (s & 1), kGateThreads);    // releases the tile warps on this warp's scheduler into pass 2
                // ring slot of step s+kPre: its previous content (step s+kPre-kRing) was consumed before BAR_M(s+kPre-kRing)
                sm.ringRow[(s + kPre) % kRing][lane >> 3][lane & 7] = rowv;
                if (lane < 8) sm.ringRhs[(s + kPre) % kRing][lane] = rhsv;
                if (s + 1 < s1) bar_sync(BAR_RAW, NTHR);        // raw(s+1) complete (y_p(s+1) final as well)
            }
        }
    }
  }   // mode != FM_BACK
    fence_proxy_async_all();                                // the panels are read back below through the async proxy (TMA)
    __threadfence();
    cta_sync();
    if (!sys.rhs) return;
    if (mode == FM_OWN) {
        // forward-eliminated rhs window, relative to the separator start
        cplx* const yimg = rank == 0 ? yimg0 : yimg1;
        for (int r_b = 0; r_b < R; r_b += NTHR) if (const int r = r_b + tid; r < R) yimg[rel(r >> 3, sEnd) * TS + (r & 7)] = sm.y[r];
        return;
    }
    // NB on a singular pivot block (sm.fail) the status is set; the substitution below then runs on garbage but terminates.

    // =============================== fused back-substitution ===============================
    //   x_p = z_s - A11_s^{-1} (raw_s^T x_rest),  s = last .. first   (x window circular in smem: reuse sm.y)
    // The factor is streamed back with TMA bulk loads, kBackStages-1 panels in flight.  With a split system FM_SEP
    // solves the separator steps and publishes the separator solution, FM_BACK finishes the own steps of both halves.
    constexpr int NST = FactorSmem<T>::kBackStages;
    for (int i_b = 0; i_b < R; i_b += NTHR) if (const int i = i_b + tid; i < R)
        sm.y[i] = (mode == FM_BACK) ? xsep[rel(i >> 3, L.sOwn) * TS + (i & 7)] : mk(0.0, 0.0);
    if (tid == 0) {
        for (int q = 0; q < NST; ++q) mbar_init(&sm.mbar[q], 1);
        fence_mbar_init();
    }
    cta_sync();
    constexpr uint32_t PBYTES = panel_doubles(T) * 8;
    constexpr int NRG = NTHR / 8;        // row groups
    int itBase = 0;                      // running count of panel visits: stage = visit % NST, parity = (visit / NST) & 1
    auto back_range = [&](int sHi, int sLo) {        // steps sHi-1 .. sLo
        const int n = sHi - sLo;
        auto issue = [&](int k) {        // k-th visit of this range -> panel sHi-1-k
            const int s = sHi - 1 - k, st = (itBase + k) % NST;
            mbar_arrive_expect_tx(&sm.mbar[st], PBYTES + AZ * 16);
            bulk_g2s(&sm.stage[st][0][0][0][0], panels + (size_t)s * panel_doubles(T), PBYTES, &sm.mbar[st]);
            bulk_g2s(&sm.stageAZ[st][0], ainvz + (size_t)s * AZ, AZ * 16, &sm.mbar[st]);
        };
        if (tid == 0) {
            fence_proxy_async();
            for (int k = 0; k < NST - 1 && k < n; ++k) issue(k);
        }
        for (int k = 0; k < n; ++k) {
            const int s = sHi - 1 - k, p = s % T, it = itBase + k, st = it % NST;
            if (tid == 0 && k + NST - 1 < n) issue(k + NST - 1);       // stage freed at the end of the previous step
            mbar_wait(&sm.mbar[st], (uint32_t)((it / NST) & 1));
            const int c = tid & 7, rg = tid >> 3;
            cplx acc = mk(0.0, 0.0);
            for (int r = rg; r < R; r += NRG) {
                if ((r >> 3) == p) continue;
                cplx rv = mk(sm.stage[st][0][c >> 2][r][c & 3], sm.stage[st][1][c >> 2][r][c & 3]);
                cfma(acc, rv, sm.y[r]);
            }
            // reduce the 4 row groups inside a warp (lanes differing in bits 3,4)
#pragma unroll
            for (int off = 8; off <= 16; off <<= 1) {
                acc.x += __shfl_xor_sync(0xffffffffu, acc.x, off);
                acc.y += __shfl_xor_sync(0xffffffffu, acc.y, off);
            }
            if (lane < 8) sm.part[warp][lane] = acc;
            cta_sync();
            if (warp == 0) {
                // d_k = sum_w part[w][k] (lanes k + 8j hold partial sums), then x_i = z_i - sum_k Ainv[i][k] d_k
                cplx d = mk(0.0, 0.0);
                for (int w = (lane >> 3); w < NW + 1; w += 4) d += sm.part[w][lane & 7];
#pragma unroll
                for (int off = 8; off <= 16; off <<= 1) {
                    d.x += __shfl_xor_sync(0xffffffffu, d.x, off);
                    d.y += __shfl_xor_sync(0xffffffffu, d.y, off);
                }
                const int ii = lane >> 2, tt = lane & 3;     // lane handles k = 2tt, 2tt+1 of row ii
                cplx d0 = mk(__shfl_sync(0xffffffffu, d.x, 2 * tt), __shfl_sync(0xffffffffu, d.y, 2 * tt));
                cplx d1 = mk(__shfl_sync(0xffffffffu, d.x, 2 * tt + 1), __shfl_sync(0xffffffffu, d.y, 2 * tt + 1));
                cplx xv = sm.stageAZ[st][ii * 8 + 2 * tt] * d0 + sm.stageAZ[st][ii * 8 + 2 * tt + 1] * d1;
#pragma unroll
                for (int off = 1; off <= 2; off <<= 1) {
                    xv.x += __shfl_xor_sync(0xffffffffu, xv.x, off);
                    xv.y += __shfl_xor_sync(0xffffffffu, xv.y, off);
                }
                if (tt == 0) {
                    cplx xo = sm.stageAZ[st][64 + ii] - xv;
                    sm.y[p * TS + ii] = xo;
                    prov.x_store(sys.x, s * TS + ii, xo);
                }
            }
            cta_sync();
        }
        itBase += n;
    };
    if (mode == FM_FULL) {
        back_range(L.sTot, 0);
    } else if (mode == FM_SEP) {
        back_range(L.sTot, L.sOwn);
        for (int r_b = 0; r_b < R; r_b += NTHR) if (const int r = r_b + tid; r < R) xsep[rel(r >> 3, L.sOwn) * TS + (r & 7)] = sm.y[r];
    } else {
        back_range(L.sOwn, 0);
    }
}

}  // namespace hmcmt
