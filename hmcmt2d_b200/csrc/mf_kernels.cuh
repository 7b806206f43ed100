// Numeric phase of the nested-dissection multifrontal solver: batched dense partial factorisations of the fronts on the
// FP64 tensor cores (DMMA.8x8x4) and the level-by-level triangular solves.  Replaces `factorMUMPS(Aii,1)` / `applyMUMPS`
// (mt2DTE.jl:50-53, compJacTMatVec.jl:220-224, MUMPSfuncs.jl:24-39,75-132) for the MT systems of 1 000 unknowns and more (below
// that the register-window band kernel, band_factor.cuh, is faster) and for arbitrary symmetric matrices handed to the Level-1 shim.
//
// Front arithmetic (pivot-free, complex symmetric, no conjugation; prototype tools/proto/mf_proto.py), front = [pivots | update]:
//     G = F11^{-1},   M = F21 G,   U = F22 - M F21^T          (the block "sweep" of the pivots; 8x8 pivot blocks inverted in
//                                                               registers by gj_invert8)
//     forward  w2 -= M w1 ;   backward  x1 = G w1 - M^T x2       — no triangular solves: every step is a dense product.
//   * small fronts (fp <= fSmall): ONE CTA (1 ... 16 warps) assembles the front in shared memory (original entries + extend-add
//     of the children's update matrices), sweeps the pivot block, forms M and U as two tile products and writes G, M (factor
//     arena) and U (update arena);
//   * large fronts live in global memory: gather assembly (mf_asm_gather_kernel, mf_asm_orig_kernel), then per chunk of <= 96
//     pivots: mf_inv_kernel (G of the diagonal block, shared memory), mf_gemm_kernel (M = F21 G), mf_gemm_kernel (trailing update
//     U -= M F21^T) — cp.async-staged 64x64x16 tiles, 8 warps, DMMA.
//
// Matrix storage ("k-grouped"): element (i,j) of a matrix with ld rows sits at ((j/4*2 + plane)*ld + i)*4 + j%4 doubles
// (plane 0 = real, 1 = imaginary).  A block of rows of four consecutive columns is contiguous — exactly the DMMA A/B operand
// image (lane (g,t) reads [row g][k t]) — so operand tiles are copied global -> shared with 16-byte cp.async and no transposition,
// and C fragments (lane holds [g][2t], [g][2t+1]) are read / written as 16-byte pairs.
#pragma once
#include "band_factor.cuh"
#include "mf_solver.cuh"

namespace hmcmt {
namespace mf {

__host__ __device__ __forceinline__ size_t kg_off(int ld, int i, int j, int plane) {
    return ((size_t)((j >> 2) * 2 + plane) * ld + i) * 4 + (j & 3);
}

// device view of the symbolic tables + per-batch arenas
struct Tables {
    const Front* fronts;
    const int* rows;
    const int* rel;
    const int* children;
    const OrigEntry* orig;
    const Chunk* chunks;
    const int* pos2orig;
    double* fac;            // [nsys][facStride]
    double* arena[2];       // [nsys][arenaStride[p]]
    int64_t facStride, arenaStride[2];
    const cplx* vals;       // [nsys][valStride]
    int64_t valStride;
    int* status;            // [nsys]
    unsigned long long* prof;   // optional (HMCMT_MF_PROF=1): per-phase cycle totals of mf_small_kernel, thread 0 of every CTA
};
#define MF_PROF_MARK(slot) do { if (tb.prof && threadIdx.x == 0) { const long long _t = clock64(); atomicAdd(tb.prof + _pc * 8 + (slot), (unsigned long long)(_t - _t0)); _t0 = _t; } } while (0)

// ------------------------------------------------------------------------------------------------------------------------
// Fronts in shared memory: lower-triangle 8x8 tiles, tile (I,J), I >= J, at tiles + (I(I+1)/2 + J) * 128 doubles.  Inside a tile the
// layout is the k-grouped one of the global matrices, element (r,c) of plane pl at pl*64 + (c/4)*32 + r*4 + c%4:
//   * the DMMA A / B operand of a k-half (lane (g,t) reads [row g][k 4kk+t]) is 32 consecutive doubles: conflict-free, so the tiles
//     themselves serve as operands and no operand panels are copied;
//   * the C fragment (lane holds [g][2t], [g][2t+1]) is two runs of 32 consecutive doubles read / written as 16-byte pairs;
//   * a (plane, column group) chunk of a tile is 32 consecutive doubles in shared AND in global memory (kg_off): outputs are
//     straight vector copies.
// Of a diagonal tile the assembly maintains the lower triangle only; the pivot-block sweep replaces the pivot diagonal tiles by
// full symmetric ones.
__device__ __forceinline__ int tl_off(int r, int c) { return ((c >> 2) << 5) | (r << 2) | (c & 3); }
__device__ __forceinline__ double* mf_tile(double* tiles, int I, int J) { return tiles + (size_t)(I * (I + 1) / 2 + J) * 128; }
// Mid-size fronts (the 8- and 16-warp instantiations) keep the pivot columns only, tiles (I, J) with J < npb: the pivot triangle
// as above, then the nub x npb block of F21 row by row.  The update block F22 never enters shared memory (see mf_small_kernel).
__device__ __forceinline__ int mf_pc_row(int I, int npb) { return I < npb ? I * (I + 1) / 2 : npb * (npb + 1) / 2 + (I - npb) * npb; }
template <bool PC>
__device__ __forceinline__ double* mf_tile(double* tiles, int npb, int I, int J) {
    return PC ? tiles + (size_t)(mf_pc_row(I, npb) + J) * 128 : mf_tile(tiles, I, J);
}

struct TileFrag {      // A or B operand of one 8x8 complex tile (both k-halves), or its C fragment
    double re[2], im[2];
};
// operand [row g][k 4kk+t] of the tile as stored / of its transpose
__device__ __forceinline__ void frag_load(TileFrag& f, const double* T, int lane) {
    f.re[0] = T[lane]; f.re[1] = T[32 + lane]; f.im[0] = T[64 + lane]; f.im[1] = T[96 + lane];
}
__device__ __forceinline__ void frag_load_t(TileFrag& f, const double* T, int g, int t) {
    const int o0 = tl_off(t, g), o1 = tl_off(4 + t, g);
    f.re[0] = T[o0]; f.re[1] = T[o1]; f.im[0] = T[64 + o0]; f.im[1] = T[64 + o1];
}
__device__ __forceinline__ void frag_store(const TileFrag& f, double* T, int lane) {
    T[lane] = f.re[0]; T[32 + lane] = f.re[1]; T[64 + lane] = f.im[0]; T[96 + lane] = f.im[1];
}
// C fragment: elements (g, 2t), (g, 2t+1)
__device__ __forceinline__ void cfrag_load(TileFrag& c, const double* T, int g, int t) {
    const int o = tl_off(g, 2 * t);
    const double2 r = *reinterpret_cast<const double2*>(T + o), i = *reinterpret_cast<const double2*>(T + 64 + o);
    c.re[0] = r.x; c.re[1] = r.y; c.im[0] = i.x; c.im[1] = i.y;
}
__device__ __forceinline__ void cfrag_store(const TileFrag& c, double* T, int g, int t, double sign = 1.0) {
    const int o = tl_off(g, 2 * t);
    *reinterpret_cast<double2*>(T + o) = make_double2(sign * c.re[0], sign * c.re[1]);
    *reinterpret_cast<double2*>(T + 64 + o) = make_double2(sign * c.im[0], sign * c.im[1]);
}
// c += a b^T (complex, no conjugation), x accumulates the -Im Im / Im Re parts separately: two independent DMMA chains per plane
__device__ __forceinline__ void frag_mma(TileFrag& c, TileFrag& x, const TileFrag& a, const TileFrag& b) {
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
        dmma884(c.re, a.re[kk], b.re[kk]);
        dmma884(c.im, a.re[kk], b.im[kk]);
        dmma884(x.re, -a.im[kk], b.im[kk]);
        dmma884(x.im, a.im[kk], b.re[kk]);
    }
}
__device__ __forceinline__ void frag_zero(TileFrag& c) { c.re[0] = c.re[1] = c.im[0] = c.im[1] = 0.0; }
__device__ __forceinline__ void frag_add(TileFrag& c, const TileFrag& x) {
    c.re[0] += x.re[0]; c.re[1] += x.re[1]; c.im[0] += x.im[0]; c.im[1] += x.im[1];
}

// Partial factorisation of an nb x nb tile matrix whose first npb tile rows / columns are the pivots (sReal of the 8 npb pivot
// unknowns are real, the rest identity padding):
//   B  block sweep of the pivot x pivot tiles alone (8x8 pivot blocks inverted in registers)         -> pivot tiles = -G (full)
//   C  M' = F21 (-G)      into mbuf (tile (I - npb, kb) at mbuf + ((I - npb) npb + kb) 128)          -> mbuf = -M
//   D  U  = F22 + M' F21^T  accumulated over all pivots in registers                                  -> update tiles = U
// The update rows never enter the latency-bound sweep: they see two perfectly parallel products with K = all pivots.
// PC: the tiles hold the pivot columns only (mf_tile<true>); phase D is then the caller's (it gathers F22 from the children).
// STREAM (PC only): phase C writes -M' = M straight from the registers to the factor arena (mglob, k-grouped, ldm rows) instead
// of mbuf.
// scratch: 2 npb tiles (column operands of the sweep; may alias mbuf).  All NW warps call; ends with a CTA barrier.
template <int NW, bool PC = false, bool STREAM = false>
__device__ __forceinline__ void mf_front_factor(double* __restrict__ tiles, double* __restrict__ scratch, double* __restrict__ mbuf,
                                                double* __restrict__ nainv, int* __restrict__ fail, const int nb, const int npb,
                                                const int sReal, unsigned long long* __restrict__ prof = nullptr,
                                                double* mglob = nullptr, const int ldm = 0) {
    const int tid = threadIdx.x, lane = tid & 31;
    long long _s0 = prof ? clock64() : 0;
#define MF_SWEEP_MARK(slot) do { if (prof && tid == 0) { const long long _t = clock64(); atomicAdd(prof + (slot), (unsigned long long)(_t - _s0)); _s0 = _t; } } while (0)
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int g = lane >> 2, t = lane & 3;
    double* const rawb = scratch;                         // raw_I = A[I][kb] of the current sweep step, I in the pivot range
    double* const mmb = scratch + (size_t)npb * 128;      // m_I = raw_I (-P)
    // ---- B: sweep of the pivot block ----
    for (int kb = 0; kb < npb; ++kb) {
        if (warp == 0) {
            // P = A[kb][kb]^{-1} in registers (mirrored read of the lower triangle), -P published as an operand tile
            const double* D = mf_tile(tiles, kb, kb);
            auto sym = [&](int r, int c, int pl) { return r >= c ? D[pl * 64 + tl_off(r, c)] : D[pl * 64 + tl_off(c, r)]; };
            cplx a0 = mk(sym(g, 2 * t, 0), sym(g, 2 * t, 1)), a1 = mk(sym(g, 2 * t + 1, 0), sym(g, 2 * t + 1, 1));
            bool bad = false;
            const int left = sReal - 8 * kb;
            gj_invert8<(NW > 4)>(a0, a1, bad, g, t, left < 8 ? (left < 0 ? 0 : left) : 8);
            if (__any_sync(0xffffffffu, bad) && lane == 0) *fail = 1;
            TileFrag p;
            p.re[0] = -a0.x; p.re[1] = -a1.x; p.im[0] = -a0.y; p.im[1] = -a1.y;
            cfrag_store(p, nainv, g, t);
            __syncwarp();
            // the diagonal tile itself takes -P (nobody else reads it during this step)
            double* Dw = mf_tile(tiles, kb, kb);
            cfrag_store(p, Dw, g, t);
        }
        if (npb == 1) break;
        __syncthreads();
        MF_SWEEP_MARK(0);      // slot 0: 8x8 inversions
        // m_I = raw_I (-P) for the other pivot block rows; raw_I kept as an operand tile for the update below
        for (int I = warp; I < npb; I += NW) {
            if (I == kb) continue;
            TileFrag a, b, c, x;
            if (I > kb) frag_load(a, mf_tile(tiles, I, kb), lane);
            else frag_load_t(a, mf_tile(tiles, kb, I), g, t);
            frag_load(b, nainv, lane);
            frag_zero(c); frag_zero(x);
            frag_mma(c, x, a, b);
            frag_add(c, x);
            frag_store(a, rawb + (size_t)I * 128, lane);
            cfrag_store(c, mmb + (size_t)I * 128, g, t);
        }
        __syncthreads();
        MF_SWEEP_MARK(1);      // slot 1: rest of the pivot-block sweep
        // A[I][J] += m_I raw_J^T (I, J != kb), column / row kb <- -m
        {
            int I = 0, J = warp;
            while (J > I) { J -= I + 1; ++I; }
            for (int L = warp; L < npb * (npb + 1) / 2; L += NW) {
                double* T = mf_tile(tiles, I, J);
                if (I == kb && J == kb) {
                } else if (J == kb) {
                    TileFrag c;
                    cfrag_load(c, mmb + (size_t)I * 128, g, t);
                    cfrag_store(c, T, g, t, -1.0);
                } else if (I == kb) {              // J < kb: tile (kb, J) = -(m_J)^T
                    const double* Ms = mmb + (size_t)J * 128;
                    TileFrag c;
                    c.re[0] = Ms[tl_off(2 * t, g)]; c.re[1] = Ms[tl_off(2 * t + 1, g)];
                    c.im[0] = Ms[64 + tl_off(2 * t, g)]; c.im[1] = Ms[64 + tl_off(2 * t + 1, g)];
                    cfrag_store(c, T, g, t, -1.0);
                } else {
                    TileFrag a, b, c, x;
                    frag_load(a, mmb + (size_t)I * 128, lane);
                    frag_load(b, rawb + (size_t)J * 128, lane);
                    cfrag_load(c, T, g, t);
                    frag_zero(x);
                    frag_mma(c, x, a, b);
                    frag_add(c, x);
                    cfrag_store(c, T, g, t);
                }
                J += NW;
                while (J > I) { J -= I + 1; ++I; }
            }
        }
        __syncthreads();
        MF_SWEEP_MARK(1);
    }
    const int nub = nb - npb;
    if (nub == 0) { __syncthreads(); return; }
    __syncthreads();
    if (npb == 1) MF_SWEEP_MARK(0);
    // ---- C: M'(I, kb) = sum_j F21(I, j) (-G)(j, kb) ----
    for (int Iu = warp; Iu < nub; Iu += NW) {
        const int I = npb + Iu;
        for (int kb = 0; kb < npb; ++kb) {
            TileFrag c, x;
            frag_zero(c); frag_zero(x);
            for (int j = 0; j < npb; ++j) {
                TileFrag a, b;
                frag_load(a, mf_tile<PC>(tiles, npb, I, j), lane);
                if (kb >= j) frag_load(b, mf_tile(tiles, kb, j), lane);       // B[n][k] = (-G)(kb n, j k)
                else frag_load_t(b, mf_tile(tiles, j, kb), g, t);
                frag_mma(c, x, a, b);
            }
            frag_add(c, x);
            if (STREAM) {
                double* o = mglob + kg_off(ldm, 8 * Iu + g, 8 * kb + 2 * t, 0);
                *reinterpret_cast<double2*>(o) = make_double2(-c.re[0], -c.re[1]);
                *reinterpret_cast<double2*>(o + 4 * ldm) = make_double2(-c.im[0], -c.im[1]);
            } else {
                cfrag_store(c, mbuf + (size_t)(Iu * npb + kb) * 128, g, t);
            }
        }
    }
    __syncthreads();
    MF_SWEEP_MARK(2);      // slot 2: M' = F21 (-G)
    if (PC) return;
    // ---- D: U(I, J) += sum_kb M'(I, kb) F21(J, kb)^T, lower tiles, two tiles per trip (independent DMMA chains) ----
    {
        const int nU = nub * (nub + 1) / 2;
        int I = 0, J = warp;
        while (J > I) { J -= I + 1; ++I; }
        constexpr bool kPair = NW > 4;      // few warps: the fronts resident on the SM hide the DMMA latency, registers are scarce
        for (int L = warp; L < nU; L += (kPair ? 2 : 1) * NW) {
            const int I0 = I, J0 = J;
            J += NW;
            while (J > I) { J -= I + 1; ++I; }
            const bool two = kPair && L + NW < nU;
            const int I1 = I, J1 = J;
            if (kPair) {
                J += NW;
                while (J > I) { J -= I + 1; ++I; }
            }
            double* T0 = mf_tile(tiles, npb + I0, npb + J0);
            double* T1 = mf_tile(tiles, npb + I1, npb + J1);
            TileFrag c0, x0, c1, x1;
            cfrag_load(c0, T0, g, t);
            frag_zero(x0);
            if (two) { cfrag_load(c1, T1, g, t); frag_zero(x1); }
            for (int kb = 0; kb < npb; ++kb) {
                TileFrag a, b;
                frag_load(a, mbuf + (size_t)(I0 * npb + kb) * 128, lane);
                frag_load(b, mf_tile(tiles, npb + J0, kb), lane);
                frag_mma(c0, x0, a, b);
                if (two) {
                    frag_load(a, mbuf + (size_t)(I1 * npb + kb) * 128, lane);
                    frag_load(b, mf_tile(tiles, npb + J1, kb), lane);
                    frag_mma(c1, x1, a, b);
                }
            }
            frag_add(c0, x0);
            cfrag_store(c0, T0, g, t);
            if (two) { frag_add(c1, x1); cfrag_store(c1, T1, g, t); }
        }
    }
    __syncthreads();
    MF_SWEEP_MARK(3);
#undef MF_SWEEP_MARK
}

// one 8x8 tile (shared memory) -> k-grouped global matrix with ld rows at (row0, col0), executed by one warp: the four (plane,
// column group) chunks are 32 consecutive doubles on both sides.  TRANSPOSED: the tile holds the transposed block (gather).
template <bool TRANSPOSED>
__device__ __forceinline__ void mf_store_tile(const double* __restrict__ T, double* __restrict__ dst, int ld, int row0, int col0,
                                              double sign, int lane) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int idx = lane + 32 * h;               // 16-byte pair index: chunk = idx / 16, (row, column pair) inside
        const int chunk = idx >> 4, w = idx & 15, pl = chunk >> 1, cg = chunk & 1, r = w >> 1, c2 = (w & 1) * 2;
        double2 v;
        if (!TRANSPOSED) v = *reinterpret_cast<const double2*>(T + chunk * 32 + w * 2);
        else v = make_double2(T[pl * 64 + tl_off(cg * 4 + c2, r)], T[pl * 64 + tl_off(cg * 4 + c2 + 1, r)]);
        double* out = dst + kg_off(ld, row0 + r, col0 + cg * 4, pl) + c2;
        *reinterpret_cast<double2*>(out) = make_double2(sign * v.x, sign * v.y);
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// small fronts: one CTA per (front, system).  list[blockIdx.x] = front id.
// (register budget: the two- and four-warp instantiations serve the thousands of tiny fronts at the bottom of the tree, where the
// number of fronts resident per SM hides the latency of the 8x8 inversions: 64 registers per thread -> 16 / 8 CTAs per SM.
// The 8- and 16-warp instantiations (kMid) keep only the pivot columns in shared memory, so that 4 / 2 of them fit on an SM
// beside each other: 64 registers per thread as well.  STREAM: mf_small_stream_kernel, see there.)
template <int NW, bool STREAM>
__device__ __forceinline__ void mf_small_front(const Tables& tb, const SmallDesc* __restrict__ descs) {
    constexpr int NT = NW * 32;
    constexpr bool kMid = NW >= 8;
    static_assert(!STREAM || kMid, "streamed M' exists in the pivot-column layout only");
    extern __shared__ __align__(16) unsigned char mf_smem[];
    SmallDesc& F = *reinterpret_cast<SmallDesc*>(mf_smem);      // the first kFrontDescBytes of the dynamic block
    const int sys = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    constexpr int _pc = NW <= 2 ? 0 : (NW == 4 ? 1 : (NW == 8 ? 2 : 3));      // profiler class (streamed: with the 16 warps)
    long long _t0 = clock64();
    // the front's record: one coalesced read
    static_assert(sizeof(SmallDesc) % 4 == 0 && sizeof(SmallDesc) <= kFrontDescBytes, "SmallDesc is copied word by word into the head of the dynamic shared memory");
    for (int i = tid; i < (int)(sizeof(SmallDesc) / 4); i += NT)
        reinterpret_cast<int*>(&F)[i] = reinterpret_cast<const int*>(descs + blockIdx.x)[i];
    __syncthreads();
    const int fp = F.sp + F.up, nb = fp >> 3, npb = F.sp >> 3, nub = nb - npb;
    const int nT = kMid ? mf_pc_row(nb, npb) : nb * (nb + 1) / 2;      // tiles kept in shared memory
    double* tiles = reinterpret_cast<double*>(mf_smem + kFrontDescBytes);
    double* mbuf = tiles + (size_t)nT * 128;                                   // sweep scratch, then M' (unless streamed)
    double* nainv = mbuf + (size_t)(STREAM || 2 * npb > nub * npb ? 2 * npb : nub * npb) * 128;
    int* fail = reinterpret_cast<int*>(nainv + 128);
    // row maps of all children, back to back, already split into the two address parts of the tile layout: an entry (a, b),
    // a >= b, of the front sits at tiles + rowPart(a) + colPart(b)
    int2* relS = reinterpret_cast<int2*>(fail + 4);
    auto rel_parts = [npb](int r) {
        return make_int2((kMid ? mf_pc_row(r >> 3, npb) : (r >> 3) * ((r >> 3) + 1) / 2) * 128 + (r & 7) * 4, (r >> 3) * 128 + ((r & 4) << 3) + (r & 3));
    };
    // everything that depends on the record alone is requested now: the children's row maps, the first batches of the children's
    // update matrices, the first original entry of every thread (and its value); the latency hides behind the zeroing
    const int nChild = F.nChild;
    {
        int base = 0;
        for (int c = 0; c < nChild; ++c) {
            const int cu = F.cU[c];
            const int* rel = tb.rel + F.cRel[c];
            for (int i = tid; i < cu; i += NT) relS[base + i] = rel_parts(rel[i]);
            base += cu;
        }
    }
    // kMid: inverse row maps of the update rows, child c at invS + c * up: update row a of the front -> row of child c (-1: none)
    int* invS = reinterpret_cast<int*>(relS + ((F.cU[0] + F.cU[1] + F.cU[2] + F.cU[3] + 1) & ~1));
    // Extend-add of the children's update matrices.  Work items = (column group of four, block of 32 rows) of a child's lower
    // triangle (16-byte loads, 64 bytes per lane and item), dealt round-robin to the warps in batches of kBatch.  Every warp
    // walks ITS batches of all children in order with two batches in flight: the loads of batch k+2 are issued before batch k
    // is scattered, across the child boundaries too, so that one global-memory round trip is exposed per front instead of one
    // or two per child.  Children are scattered one after the other (a CTA barrier per child boundary: entries of one child
    // never collide, plain adds, fixed order -> deterministic).
    const double* carena = tb.arena[F.par ^ 1] + (size_t)sys * tb.arenaStride[F.par ^ 1];
    constexpr int kBatch = 1;      // (every instantiation lives on 64 registers)
    struct Batch {
        double2 r01[kBatch], r23[kBatch], i01[kBatch], i23[kBatch];
        int ii[kBatch], jg[kBatch];
        int c;                                    // child, -1: nothing left
    };
    int curC = 0, curQ = warp * kBatch;
    auto load_batch = [&](Batch& bt) {
        while (curC < nChild) {
            const int cu = F.cU[curC];
            if (curQ < (((kMid ? F.cPiv[curC] : cu) + 3) >> 2) * ((cu + 31) >> 5)) break;
            ++curC;
            curQ = warp * kBatch;
        }
        bt.c = curC < nChild ? curC : -1;
        if (bt.c < 0) return;
        const int cu = F.cU[curC], ld = F.cLd[curC], off = F.cFirst[curC];
        const double* U = carena + F.cOff[curC];
        const int ng = ((kMid ? F.cPiv[curC] : cu) + 3) >> 2, nrb = (cu + 31) >> 5;
#pragma unroll
        for (int bq = 0; bq < kBatch; ++bq) {
            const int q = curQ + bq;
            const int jg = nrb == 1 ? q : q / nrb, i = (q - jg * nrb) * 32 + lane;
            bt.jg[bq] = jg;
            bt.ii[bq] = (q < ng * nrb && i < cu && i >= 4 * jg) ? i : -1;
            if (bt.ii[bq] >= 0) {
                const double* pr = U + kg_off(ld, off + i, off + 4 * jg, 0);
                const double* pi = U + kg_off(ld, off + i, off + 4 * jg, 1);
                bt.r01[bq] = *reinterpret_cast<const double2*>(pr); bt.r23[bq] = *reinterpret_cast<const double2*>(pr + 2);
                bt.i01[bq] = *reinterpret_cast<const double2*>(pi); bt.i23[bq] = *reinterpret_cast<const double2*>(pi + 2);
            }
        }
        curQ += NW * kBatch;
    };
    Batch b0, b1;
    load_batch(b0);
    load_batch(b1);
    const cplx* vals = tb.vals + (size_t)sys * tb.valStride;
    OrigEntry oe0{0, 0, -1};
    cplx ov0 = mk(0.0, 0.0);
    if (tid < F.nOrig) {
        oe0 = tb.orig[F.origPtr + tid];
        ov0 = oe0.src < 0 ? mk(1.0, 0.0) : vals[oe0.src];
    }
    for (int i = tid; i < nT * 64; i += NT) reinterpret_cast<double2*>(tiles)[i] = make_double2(0.0, 0.0);
    if (kMid)
        for (int i = tid; i < nChild * F.up; i += NT) invS[i] = -1;
    if (tid == 0) *fail = 0;
    __syncthreads();
    MF_PROF_MARK(0);
    if (kMid) {      // (read by phase D only: many barriers away)
        int base = 0;
        for (int c = 0; c < nChild; ++c) {
            const int cu = F.cU[c];
            const int* rel = tb.rel + F.cRel[c];
            for (int i = F.cPiv[c] + tid; i < cu; i += NT) invS[base + rel[i] - F.sp] = i;
            base += F.up;
        }
    }
    auto addr = [&](int a, int b) {       // a >= b
        return tiles + (size_t)((kMid ? mf_pc_row(a >> 3, npb) : (a >> 3) * ((a >> 3) + 1) / 2) + (b >> 3)) * 128 + tl_off(a & 7, b & 7);
    };
    {
        auto scatter = [&](const Batch& bt) {
            const int2* relC = relS + ((bt.c > 0 ? F.cU[0] : 0) + (bt.c > 1 ? F.cU[1] : 0) + (bt.c > 2 ? F.cU[2] : 0));
            const int jEnd = kMid ? F.cPiv[bt.c] : 0;      // kMid: the columns that land in the pivot columns only
#pragma unroll
            for (int bq = 0; bq < kBatch; ++bq) {
                const int i = bt.ii[bq];
                if (i < 0) continue;
                const int jg = bt.jg[bq];
                const double re[4] = {bt.r01[bq].x, bt.r01[bq].y, bt.r23[bq].x, bt.r23[bq].y};
                const double im[4] = {bt.i01[bq].x, bt.i01[bq].y, bt.i23[bq].x, bt.i23[bq].y};
                double* rowp = tiles + relC[i].x;
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    if (4 * jg + jj > i || (kMid && 4 * jg + jj >= jEnd)) break;
                    double* d = rowp + relC[4 * jg + jj].y;
                    d[0] += re[jj];
                    d[64] += im[jj];
                }
            }
        };
        // one child after the other; every warp takes the same nChild trips through the ONE barrier below, whatever its share of
        // the batches (the batches in flight at a child boundary already belong to the next child)
        for (int c = 0; c < nChild; ++c) {
            while (b0.c == c) {
                scatter(b0);
                b0 = b1;
                load_batch(b1);
            }
            __syncwarp();
            __syncthreads();
        }
        if (nChild == 0) __syncthreads();
    }
    MF_PROF_MARK(2);
    // original matrix entries of the pivot columns
    if (tid < F.nOrig) {
        double* d = addr(oe0.lrow, oe0.lcol);
        d[0] += ov0.x;
        d[64] += ov0.y;
    }
    for (int e = tid + NT; e < F.nOrig; e += NT) {
        const OrigEntry oe = tb.orig[F.origPtr + e];
        const cplx v = oe.src < 0 ? mk(1.0, 0.0) : vals[oe.src];
        double* d = addr(oe.lrow, oe.lcol);
        d[0] += v.x;
        d[64] += v.y;
    }
    __syncthreads();
    MF_PROF_MARK(1);
    double* fac = tb.fac + (size_t)sys * tb.facStride;
    mf_front_factor<NW, kMid, STREAM>(tiles, mbuf, mbuf, nainv, fail, nb, npb, F.s, tb.prof ? tb.prof + 32 + _pc * 4 : nullptr,
                                      fac + F.mOff, F.up);
    if (kMid && nub > 0) {
        // ---- D: U = F22 + M' F21^T, lower tiles, two per trip, written from the registers to the update arena.  F22 is gathered
        // from the children's update matrices through the inverse row maps straight into the accumulators: every element starts
        // at +0.0 and takes the children's entries in child order, the very sums the extend-add into a zeroed F22 formed.
        const long long tD = tb.prof ? clock64() : 0;
        const int g = lane >> 2, t = lane & 3, up = F.up;
        double* U = tb.arena[F.par] + (size_t)sys * tb.arenaStride[F.par] + F.uOff;
        auto gather = [&](TileFrag& c, int I, int J) {      // elements (a, b), (a, b + 1) of the update block
            const int a = 8 * I + g, b = 8 * J + 2 * t;
            frag_zero(c);
#pragma unroll
            for (int ch = 0; ch < kSmallChildren; ++ch) {
                const int* inv = invS + ch * up;
                const int ia = ch < nChild ? inv[a] : -1;
                if (ia < 0) continue;
                const int ib0 = inv[b], ib1 = inv[b + 1];
                const double* Uc = carena + F.cOff[ch];
                const int ld = F.cLd[ch], off = F.cFirst[ch];
                if (ib0 >= 0 && ib0 <= ia) { c.re[0] += Uc[kg_off(ld, off + ia, off + ib0, 0)]; c.im[0] += Uc[kg_off(ld, off + ia, off + ib0, 1)]; }
                if (ib1 >= 0 && ib1 <= ia) { c.re[1] += Uc[kg_off(ld, off + ia, off + ib1, 0)]; c.im[1] += Uc[kg_off(ld, off + ia, off + ib1, 1)]; }
            }
        };
        auto store = [&](const TileFrag& c, int I, int J) {
            double* o = U + kg_off(up, 8 * I + g, 8 * J + 2 * t, 0);
            *reinterpret_cast<double2*>(o) = make_double2(c.re[0], c.re[1]);
            *reinterpret_cast<double2*>(o + 4 * up) = make_double2(c.im[0], c.im[1]);
        };
        if (!STREAM) {
            const int nU = nub * (nub + 1) / 2;
            int I = 0, J = warp;
            while (J > I) { J -= I + 1; ++I; }
            for (int L = warp; L < nU; L += 2 * NW) {
                const int I0 = I, J0 = J;
                J += NW;
                while (J > I) { J -= I + 1; ++I; }
                const bool two = L + NW < nU;
                const int I1 = I, J1 = J;
                J += NW;
                while (J > I) { J -= I + 1; ++I; }
                TileFrag c0, x0, c1, x1;
                gather(c0, I0, J0);
                frag_zero(x0);
                if (two) { gather(c1, I1, J1); frag_zero(x1); }
                for (int kb = 0; kb < npb; ++kb) {
                    TileFrag a, b;
                    frag_load(a, mbuf + (size_t)(I0 * npb + kb) * 128, lane);
                    frag_load(b, mf_tile<true>(tiles, npb, npb + J0, kb), lane);
                    frag_mma(c0, x0, a, b);
                    if (two) {
                        frag_load(a, mbuf + (size_t)(I1 * npb + kb) * 128, lane);
                        frag_load(b, mf_tile<true>(tiles, npb, npb + J1, kb), lane);
                        frag_mma(c1, x1, a, b);
                    }
                }
                frag_add(c0, x0);
                store(c0, I0, J0);
                if (two) { frag_add(c1, x1); store(c1, I1, J1); }
            }
        } else {
            // Streamed M': the A operand is -M from the factor arena, written by this CTA's phase C one barrier ago (plain
            // coherent loads, never the non-coherent path).  A work item is up to kRow tiles (I, J0 .. J0 + kRow - 1) of one tile
            // row, so every A fragment read from L2 serves kRow products; the next fragment is requested before the products of
            // the current one.  Per tile the same operations in the same order as above: U is bit-identical to resident M'.
            constexpr int kRow = 4;
            const double* Mg = fac + F.mOff;
            auto load_a = [&](TileFrag& a, int I, int kb) {
#pragma unroll
                for (int kk = 0; kk < 2; ++kk) {
                    const double* p = Mg + kg_off(up, 8 * I + g, 8 * kb + 4 * kk + t, 0);
                    a.re[kk] = -p[0];
                    a.im[kk] = -p[4 * up];
                }
            };
            int I = 0, q = warp;      // item q of row I: tiles J0 = kRow q ...; row I has I / kRow + 1 items
            while (q > I / kRow) { q -= I / kRow + 1; ++I; }
            while (I < nub) {
                const int J0 = kRow * q, nJ = min(kRow, I + 1 - J0);
                TileFrag c[kRow], x[kRow];
#pragma unroll
                for (int r = 0; r < kRow; ++r)
                    if (r < nJ) { gather(c[r], I, J0 + r); frag_zero(x[r]); }
                TileFrag a;
                load_a(a, I, 0);
                for (int kb = 0; kb < npb; ++kb) {
                    TileFrag an;
                    if (kb + 1 < npb) load_a(an, I, kb + 1);
#pragma unroll
                    for (int r = 0; r < kRow; ++r)
                        if (r < nJ) {
                            TileFrag b;
                            frag_load(b, mf_tile<true>(tiles, npb, npb + J0 + r, kb), lane);
                            frag_mma(c[r], x[r], a, b);
                        }
                    a = an;
                }
#pragma unroll
                for (int r = 0; r < kRow; ++r)
                    if (r < nJ) { frag_add(c[r], x[r]); store(c[r], I, J0 + r); }
                q += NW;
                while (I < nub && q > I / kRow) { q -= I / kRow + 1; ++I; }
            }
        }
        if (tb.prof && tid == 0) atomicAdd(tb.prof + 32 + _pc * 4 + 3, (unsigned long long)(clock64() - tD));
    }
    MF_PROF_MARK(4);
    if (tid == 0 && *fail) tb.status[sys] = kErrSingular;
    // outputs, tile by tile: G = -(pivot x pivot), M = -M' (factor arena; streamed: already there), U = update x update (update
    // arena, lower tiles)
    const int sp = F.sp, up = F.up;
    {
        double* G = fac + F.gOff;
        for (int I = warp; I < npb; I += NW)
            for (int J = 0; J < npb; ++J) {
                if (I >= J) mf_store_tile<false>(mf_tile(tiles, I, J), G, sp, I * 8, J * 8, -1.0, lane);
                else mf_store_tile<true>(mf_tile(tiles, J, I), G, sp, I * 8, J * 8, -1.0, lane);
            }
    }
    if (!STREAM && up > 0) {
        double* M = fac + F.mOff;
        for (int I = warp; I < nub; I += NW)
            for (int J = 0; J < npb; ++J) mf_store_tile<false>(mbuf + (size_t)(I * npb + J) * 128, M, up, I * 8, J * 8, -1.0, lane);
    }
    if (!kMid && up > 0) {
        double* U = tb.arena[F.par] + (size_t)sys * tb.arenaStride[F.par] + F.uOff;
        int I = 0, J = warp;
        while (J > I) { J -= I + 1; ++I; }
        for (int L = warp; L < nub * (nub + 1) / 2; L += NW) {
            mf_store_tile<false>(mf_tile(tiles, npb + I, npb + J), U, up, I * 8, J * 8, 1.0, lane);
            J += NW;
            while (J > I) { J -= I + 1; ++I; }
        }
    }
    MF_PROF_MARK(5);
    if (tb.prof && tid == 0) { atomicAdd(tb.prof + _pc * 8 + 6, 1ull); atomicAdd(tb.prof + _pc * 8 + 7, (unsigned long long)npb); }
}

template <int NW>
__global__ void __launch_bounds__(NW * 32, NW <= 4 ? (NW == 1 ? 16 : 32 / NW) : (NW == 8 ? 4 : 2))
mf_small_kernel(Tables tb, const SmallDesc* __restrict__ descs) {
    mf_small_front<NW, false>(tb, descs);
}
// Fronts whose pivot columns fit in shared memory but not together with M' (more than 144 rows): M' goes through the factor
// arena (L2).  Such a front takes most of an SM's shared memory, so one CTA per SM: 16 warps with up to 128 registers.
__global__ void __launch_bounds__(16 * 32, 1) mf_small_stream_kernel(Tables tb, const SmallDesc* __restrict__ descs) {
    mf_small_front<16, true>(tb, descs);
}

// ------------------------------------------------------------------------------------------------------------------------
// large fronts, assembly.  (front, original entry) pairs of one depth: grid (ceil(n/256), nsys)
__global__ void mf_asm_orig_kernel(Tables tb, const int2* __restrict__ pairs, int n) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x, sys = blockIdx.y;
    if (idx >= n) return;
    const int2 pr = pairs[idx];
    const Front& F = tb.fronts[pr.x];
    const OrigEntry oe = tb.orig[pr.y];
    const cplx v = oe.src < 0 ? mk(1.0, 0.0) : tb.vals[(size_t)sys * tb.valStride + oe.src];
    double* A = tb.arena[F.depth & 1] + (size_t)sys * tb.arenaStride[F.depth & 1] + F.frontOff;
    const int fp = F.sp + F.up;
    A[kg_off(fp, oe.lrow, oe.lcol, 0)] += v.x;
    A[kg_off(fp, oe.lrow, oe.lcol, 1)] += v.y;
}
// Assembly of the large fronts by GATHER: one CTA per 64 x 64 lower tile of a front.  Every thread owns (row a, four columns)
// of the tile, collects the contributions of all children through the inverse row maps (front row -> child row, -1: none) and
// writes its 2 x 32 bytes once, coalesced.  The tile is written completely (zeros included, up to the end of the diagonal 8 x 8
// block of each row), so the front needs no memset and no read-modify-write — the scatter version (zero the arena, then one
// pass per child adding 8-byte entries into the k-grouped parent) moved 3-4x the bytes at a quarter of the sector efficiency.
// The original matrix entries are added afterwards by mf_asm_orig_kernel.  Children are summed in child order: deterministic.
struct AsmTile {
    int front, bi, bj;
    int invPtr;             // offset of the front's inverse maps: child c at invMaps + invPtr + c * fp
};
__global__ void __launch_bounds__(256)
mf_asm_gather_kernel(Tables tb, const AsmTile* __restrict__ tilesList, const int* __restrict__ invMaps) {
    const AsmTile at = tilesList[blockIdx.x];
    const int sys = blockIdx.y;
    const Front P = tb.fronts[at.front];
    const int fp = P.sp + P.up, par = P.depth & 1;
    double* A = tb.arena[par] + (size_t)sys * tb.arenaStride[par] + P.frontOff;
    const double* carena = tb.arena[par ^ 1] + (size_t)sys * tb.arenaStride[par ^ 1];
    for (int item = threadIdx.x; item < 64 * 16; item += 256) {
        const int a = at.bi * 64 + (item & 63), b0 = at.bj * 64 + (item >> 6) * 4;
        if (a >= fp || b0 >= ((a >> 3) + 1) * 8) continue;      // beyond the front / beyond the diagonal 8 x 8 block of this row
        double re[4] = {0.0, 0.0, 0.0, 0.0}, im[4] = {0.0, 0.0, 0.0, 0.0};
        for (int c = 0; c < P.nChild; ++c) {
            const int* inv = invMaps + at.invPtr + (size_t)c * fp;
            const int ia = inv[a];
            if (ia < 0) continue;
            const Front& C = tb.fronts[tb.children[P.childPtr + c]];
            const int ld = C.isBig ? C.sp + C.up : C.up, off = C.isBig ? C.sp : 0;
            const double* U = carena + C.frontOff;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (b0 + k > a) break;
                const int ib = inv[b0 + k];
                if (ib < 0) continue;
                re[k] += U[kg_off(ld, off + ia, off + ib, 0)];
                im[k] += U[kg_off(ld, off + ia, off + ib, 1)];
            }
        }
        double* pr = A + kg_off(fp, a, b0, 0);
        double* pi = A + kg_off(fp, a, b0, 1);
        *reinterpret_cast<double2*>(pr) = make_double2(re[0], re[1]); *reinterpret_cast<double2*>(pr + 2) = make_double2(re[2], re[3]);
        *reinterpret_cast<double2*>(pi) = make_double2(im[0], im[1]); *reinterpret_cast<double2*>(pi + 2) = make_double2(im[2], im[3]);
    }
}

// G of the diagonal block of chunk `c` of every listed large front: grid (nfronts, nsys), kInvWarps warps
constexpr int kInvWarps = 8;
__global__ void __launch_bounds__(kInvWarps * 32)
mf_inv_kernel(Tables tb, const int* __restrict__ list, int c) {
    constexpr int NT = kInvWarps * 32;
    extern __shared__ __align__(16) unsigned char mf_smem[];
    const Front F = tb.fronts[list[blockIdx.x]];
    const Chunk ch = tb.chunks[F.chunkPtr + c];
    const int sys = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sc = ch.p1 - ch.p0, nb = sc >> 3, fp = F.sp + F.up;
    const int nT = nb * (nb + 1) / 2;
    double* tiles = reinterpret_cast<double*>(mf_smem);
    double* scratch = tiles + (size_t)nT * 128;
    double* nainv = scratch + (size_t)2 * nb * 128;
    int* fail = reinterpret_cast<int*>(nainv + 128);
    const double* A = tb.arena[F.depth & 1] + (size_t)sys * tb.arenaStride[F.depth & 1] + F.frontOff;
    if (tid == 0) *fail = 0;
    // lower tiles of A[p0:p1][p0:p1]: a (plane, column group) chunk of a tile is 32 consecutive doubles on both sides
    for (int idx = tid; idx < nT * 64; idx += NT) {
        const int L = idx >> 6, w = idx & 63, chunk = w >> 4, pl = chunk >> 1, cg = chunk & 1, r = (w & 15) >> 1, c2 = (w & 1) * 2;
        int I = 0, J = L;
        while (J > I) { J -= I + 1; ++I; }
        const double* src = A + kg_off(fp, ch.p0 + I * 8 + r, ch.p0 + J * 8 + cg * 4, pl) + c2;
        *reinterpret_cast<double2*>(tiles + (size_t)L * 128 + chunk * 32 + (w & 15) * 2) = *reinterpret_cast<const double2*>(src);
    }
    __syncthreads();
    // pivots of the chunk that are real unknowns (the identity padding sits at the end of the front's pivot range)
    const int sReal = F.s - ch.p0 < sc ? (F.s - ch.p0 < 0 ? 0 : F.s - ch.p0) : sc;
    mf_front_factor<kInvWarps>(tiles, scratch, scratch, nainv, fail, nb, nb, sReal);
    if (tid == 0 && *fail) tb.status[sys] = kErrSingular;
    double* G = tb.fac + (size_t)sys * tb.facStride + ch.gOff;
    for (int q = warp; q < nb * nb; q += kInvWarps) {
        const int I = q / nb, J = q - I * nb;
        if (I >= J) mf_store_tile<false>(mf_tile(tiles, I, J), G, sc, I * 8, J * 8, -1.0, lane);
        else mf_store_tile<true>(mf_tile(tiles, J, I), G, sc, I * 8, J * 8, -1.0, lane);
    }
}

// ------------------------------------------------------------------------------------------------------------------------
// batched complex GEMM  C (64x64 tile) = beta C + alpha A B^T  on the FP64 tensor cores; A (m x K), B (n x K), C (m x n) k-grouped.
// space: 0 / 1 = depth-parity arena, 2 = factor arena
struct GemmJob {
    int64_t aOff, bOff, cOff;
    int aSp, bSp, cSp;
    int ldA, rA, kA, ldB, rB, kB, ldC, rC, cC;
    int m, n, K;
    int lower, beta;
    double alpha;
};
struct GemmTile {
    int job, bi, bj;
};
constexpr int kGemmKC = 16, kGemmStages = 3, kGemmThreads = 256;
constexpr int kGemmStageDoubles = 2 * (kGemmKC / 4) * 2 * 64 * 4;      // A + B operand images of one stage
constexpr size_t kGemmSmemBytes = (size_t)kGemmStages * kGemmStageDoubles * sizeof(double);

__global__ void __launch_bounds__(kGemmThreads)
mf_gemm_kernel(Tables tb, const GemmJob* __restrict__ jobs, const GemmTile* __restrict__ tilesList) {
    extern __shared__ __align__(16) unsigned char mf_smem[];
    double* sm = reinterpret_cast<double*>(mf_smem);
    const GemmTile gt = tilesList[blockIdx.x];
    const GemmJob jb = jobs[gt.job];
    const int sys = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int g = lane >> 2, t = lane & 3;
    const int wr = warp >> 1, wc = warp & 1;          // warp tile: rows [16 wr, +16), cols [32 wc, +32)
    auto base = [&](int sp, int64_t off) -> double* {
        return (sp == 2 ? tb.fac + (size_t)sys * tb.facStride : tb.arena[sp] + (size_t)sys * tb.arenaStride[sp]) + off;
    };
    const double* A = base(jb.aSp, jb.aOff);
    const double* B = base(jb.bSp, jb.bOff);
    double* C = base(jb.cSp, jb.cOff);
    const int r0 = gt.bi * 64, c0 = gt.bj * 64;
    const int nk = (jb.K + kGemmKC - 1) / kGemmKC;
    // stage image: [A|B][group][plane][64][4]
    auto load_stage = [&](int ks, int st) {
        double* dst = sm + (size_t)st * kGemmStageDoubles;
        const int k0 = ks * kGemmKC;
#pragma unroll
        for (int it = 0; it < 2 * (kGemmKC / 4) * 2 * 128 / kGemmThreads; ++it) {
            const int c = tid + it * kGemmThreads;
            const int which = c / ((kGemmKC / 4) * 2 * 128);         // 0: A, 1: B
            const int cc = c - which * ((kGemmKC / 4) * 2 * 128);
            const int grp = cc >> 8, pl = (cc >> 7) & 1, row = (cc & 127) >> 1, half = cc & 1;
            const int k = k0 + 4 * grp;
            const double* src;
            bool ok;
            if (which == 0) {
                ok = (r0 + row < jb.m) && (k < jb.K);
                src = A + kg_off(jb.ldA, jb.rA + r0 + row, jb.kA + k, pl) + half * 2;
            } else {
                ok = (c0 + row < jb.n) && (k < jb.K);
                src = B + kg_off(jb.ldB, jb.rB + c0 + row, jb.kB + k, pl) + half * 2;
            }
            cp_async16(dst + (size_t)c * 2, ok ? src : A, ok ? 16u : 0u);
        }
        cp_async_commit();
    };
    double cre[2][4][2], cim[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) cre[a][b][0] = cre[a][b][1] = cim[a][b][0] = cim[a][b][1] = 0.0;
    // 8x8 blocks of this warp that hold anything the epilogue stores: inside the m x n job and, for the lower-triangle jobs, not
    // strictly above the diagonal.  Fronts are padded to multiples of 8, not 64: on the trailing tiles of a front and on its
    // diagonal tiles up to half of the blocks are skipped, and with them their DMMAs (the warp still helps loading the stages).
    unsigned act = 0;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int rb = r0 + wr * 16 + a * 8, cb = c0 + wc * 32 + b * 8;
            if (rb < jb.m && cb < jb.n && !(jb.lower && jb.cC + cb > jb.rC + rb)) act |= 1u << (a * 4 + b);
        }
    for (int s = 0; s < kGemmStages - 1; ++s) {
        if (s < nk) load_stage(s, s); else cp_async_commit();
    }
    for (int ks = 0; ks < nk; ++ks) {
        cp_async_wait<kGemmStages - 2>();
        __syncthreads();
        if (ks + kGemmStages - 1 < nk) load_stage(ks + kGemmStages - 1, (ks + kGemmStages - 1) % kGemmStages); else cp_async_commit();
        if (!act) continue;
        const double* sA = sm + (size_t)(ks % kGemmStages) * kGemmStageDoubles;
        const double* sB = sA + (kGemmKC / 4) * 2 * 64 * 4;
        const int ngrp = min(kGemmKC / 4, (jb.K - ks * kGemmKC + 3) >> 2);      // K is a multiple of 8, not of the stage depth
#pragma unroll
        for (int grp = 0; grp < kGemmKC / 4; ++grp) {
            if (grp >= ngrp) break;
            double are[2], aim[2], nai[2], bre[4], bim[4];
#pragma unroll
            for (int a = 0; a < 2; ++a) {
                are[a] = sA[((grp * 2 + 0) * 64 + wr * 16 + a * 8 + g) * 4 + t];
                aim[a] = sA[((grp * 2 + 1) * 64 + wr * 16 + a * 8 + g) * 4 + t];
                nai[a] = -aim[a];
            }
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                bre[b] = sB[((grp * 2 + 0) * 64 + wc * 32 + b * 8 + g) * 4 + t];
                bim[b] = sB[((grp * 2 + 1) * 64 + wc * 32 + b * 8 + g) * 4 + t];
            }
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int on = (act >> (a * 4 + b)) & 1;
                    dmma884_p(cre[a][b], are[a], bre[b], on);
                    dmma884_p(cim[a][b], are[a], bim[b], on);
                }
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int on = (act >> (a * 4 + b)) & 1;
                    dmma884_p(cre[a][b], nai[a], bim[b], on);
                    dmma884_p(cim[a][b], aim[a], bre[b], on);
                }
        }
    }
    cp_async_wait<0>();
    // epilogue: C fragments straight to / from global memory (16-byte pairs)
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int rb = r0 + wr * 16 + a * 8, cb = c0 + wc * 32 + b * 8;
            if (!((act >> (a * 4 + b)) & 1)) continue;
            double* pr = C + kg_off(jb.ldC, jb.rC + rb + g, jb.cC + cb + 2 * t, 0);
            double* pi = C + kg_off(jb.ldC, jb.rC + rb + g, jb.cC + cb + 2 * t, 1);
            double2 vr = make_double2(jb.alpha * cre[a][b][0], jb.alpha * cre[a][b][1]);
            double2 vi = make_double2(jb.alpha * cim[a][b][0], jb.alpha * cim[a][b][1]);
            if (jb.beta) {
                const double2 orr = *reinterpret_cast<const double2*>(pr), oi = *reinterpret_cast<const double2*>(pi);
                vr.x += orr.x; vr.y += orr.y; vi.x += oi.x; vi.y += oi.y;
            }
            *reinterpret_cast<double2*>(pr) = vr;
            *reinterpret_cast<double2*>(pi) = vi;
        }
}

// ------------------------------------------------------------------------------------------------------------------------
// values of the MT stencil systems: vals[sys] = [dr + i omega dm | e1 | e2]  (pattern: mf_grid_entries).  grid (ceil(3N/256), nsys)
__global__ void mf_mt_vals_kernel(int N, const MtValSys* __restrict__ sysv, cplx* __restrict__ vals, int64_t valStride) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x, sys = blockIdx.y;
    if (e >= 3 * N) return;
    const MtValSys sv = sysv[sys];
    cplx v;
    if (e < N) v = mk(sv.planes[e], sv.omega * sv.planes[N + e]);
    else v = mk(sv.planes[(size_t)N + e], 0.0);      // e in [N,2N): e1 = planes[2N + q] ; [2N,3N): e2 = planes[3N + q]
    vals[(size_t)sys * valStride + e] = v;
}

// ------------------------------------------------------------------------------------------------------------------------
// solves.  One CTA per (front, right-hand side); vec = blockIdx.y indexes (system, rhs): sys = vec / nrhs.
//   v   : pivot parts of the eliminated rhs (forward), overwritten by the solution (backward), padded permuted numbering;
//         vector `vec` at v + vec*vStride
//   upd : update vectors handed from the children to their parent, vector `vec` at upd + vec*uStride
// The solver's workspace holds maxRhs slots per system (Solver::solve_args): a call with one vector per system strides over
// the other slots, so that a solve on slot 1 leaves the slot-0 vectors of the same systems intact.
struct SolveArgs {
    const cplx* B;      // right-hand sides, original numbering, vector `vec` at B + vec*ldb
    cplx* X;            // solutions, same layout (may alias B)
    int64_t ldb, ldx;
    cplx* v;
    cplx* upd;
    int64_t vStride, uStride;
    int nrhs;
};
// block size: kSolveMfThreads (mf_symbolic.h) at most; launched with 128 threads where no front of the depth exceeds 144 rows

__global__ void __launch_bounds__(kSolveMfThreads)
mf_fwd_kernel(Tables tb, SolveArgs sa, const int* __restrict__ list) {
    extern __shared__ __align__(16) unsigned char mf_smem[];
    cplx* w = reinterpret_cast<cplx*>(mf_smem);
    const Front F = tb.fronts[list[blockIdx.x]];
    const int vec = blockIdx.y, sys = vec / sa.nrhs, tid = threadIdx.x, nthr = blockDim.x;
    const int fp = F.sp + F.up;
    const cplx* b = sa.B + (size_t)vec * sa.ldb;
    cplx* v = sa.v + (size_t)vec * sa.vStride;
    cplx* upd = sa.upd + (size_t)vec * sa.uStride;
    for (int i = tid; i < fp; i += nthr) {
        cplx x = mk(0.0, 0.0);
        if (i < F.s) x = b[tb.pos2orig[F.cbp + i]];
        w[i] = x;
    }
    __syncthreads();
    for (int c = 0; c < F.nChild; ++c) {
        const Front& C = tb.fronts[tb.children[F.childPtr + c]];
        const int* rel = tb.rel + C.rowPtr;
        const cplx* uv = upd + C.updOff;
        const int cu = C.u;
        for (int i = tid; i < cu; i += nthr) w[rel[i]] += uv[i];
        __syncthreads();
    }
    const double* fac = tb.fac + (size_t)sys * tb.facStride;
    for (int c = 0; c < F.nChunk; ++c) {
        const Chunk ch = tb.chunks[F.chunkPtr + c];
        const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
        const double* M = fac + ch.mOff;
        for (int i = tid; i < mr; i += nthr) {
            cplx acc = mk(0.0, 0.0);
            for (int kg = 0; kg < (sc >> 2); ++kg) {
                const double* pr = M + kg_off(mr, i, 4 * kg, 0);
                const double* pi = M + kg_off(mr, i, 4 * kg, 1);
                const double2 r01 = *reinterpret_cast<const double2*>(pr), r23 = *reinterpret_cast<const double2*>(pr + 2);
                const double2 i01 = *reinterpret_cast<const double2*>(pi), i23 = *reinterpret_cast<const double2*>(pi + 2);
                const cplx* wk = w + ch.p0 + 4 * kg;
                cfma(acc, mk(r01.x, i01.x), wk[0]);
                cfma(acc, mk(r01.y, i01.y), wk[1]);
                cfma(acc, mk(r23.x, i23.x), wk[2]);
                cfma(acc, mk(r23.y, i23.y), wk[3]);
            }
            w[ch.p1 + i] -= acc;
        }
        __syncthreads();
    }
    for (int i = tid; i < F.sp; i += nthr) v[F.cbp + i] = w[i];
    for (int i = tid; i < F.up; i += nthr) upd[F.updOff + i] = w[F.sp + i];
}

// Backward substitution of one front for NV vectors of the same system: every G / M element is loaded once and applied to all
// of them, each vector with exactly the arithmetic of the single-vector sweep.  xf[t]: [fp] then the stage tmp[t]: [largest chunk].
template <int NV>
__device__ __forceinline__ void mf_bwd_front(const Tables& tb, const Front& F, int sys, cplx* const (&v)[NV], cplx* const (&x)[NV],
                                             cplx* smem) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
    const int fp = F.sp + F.up;
    cplx* xf[NV];
    cplx* tmp[NV];
#pragma unroll
    for (int t = 0; t < NV; ++t) { xf[t] = smem + t * fp; tmp[t] = smem + NV * fp + t * F.sp; }
    const int* rows = tb.rows + F.rowPtr;
    for (int i = tid; i < fp; i += nthr) {
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            cplx val = mk(0.0, 0.0);
            if (i < F.sp) val = v[t][F.cbp + i];
            else if (i - F.sp < F.u) val = v[t][rows[i - F.sp]];
            xf[t][i] = val;
        }
    }
    __syncthreads();
    const double* fac = tb.fac + (size_t)sys * tb.facStride;
    const int NWS = nthr / 32;
    for (int c = F.nChunk - 1; c >= 0; --c) {
        const Chunk ch = tb.chunks[F.chunkPtr + c];
        const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
        const double* G = fac + ch.gOff;
        const double* M = fac + ch.mOff;
        // x1[k] = sum_j G[j][k] w1[j] - sum_i M[i][k] x2[i] : one warp per group of four k
        for (int kg = warp; kg < (sc >> 2); kg += NWS) {
            cplx a0[NV], a1[NV], a2[NV], a3[NV];
#pragma unroll
            for (int t = 0; t < NV; ++t) a0[t] = a1[t] = a2[t] = a3[t] = mk(0.0, 0.0);
            for (int j = lane; j < sc; j += 32) {
                const double* pr = G + kg_off(sc, j, 4 * kg, 0);
                const double* pi = G + kg_off(sc, j, 4 * kg, 1);
                const double2 r01 = *reinterpret_cast<const double2*>(pr), r23 = *reinterpret_cast<const double2*>(pr + 2);
                const double2 i01 = *reinterpret_cast<const double2*>(pi), i23 = *reinterpret_cast<const double2*>(pi + 2);
#pragma unroll
                for (int t = 0; t < NV; ++t) {
                    const cplx wj = xf[t][ch.p0 + j];
                    cfma(a0[t], mk(r01.x, i01.x), wj); cfma(a1[t], mk(r01.y, i01.y), wj);
                    cfma(a2[t], mk(r23.x, i23.x), wj); cfma(a3[t], mk(r23.y, i23.y), wj);
                }
            }
            for (int i = lane; i < mr; i += 32) {
                const double* pr = M + kg_off(mr, i, 4 * kg, 0);
                const double* pi = M + kg_off(mr, i, 4 * kg, 1);
                const double2 r01 = *reinterpret_cast<const double2*>(pr), r23 = *reinterpret_cast<const double2*>(pr + 2);
                const double2 i01 = *reinterpret_cast<const double2*>(pi), i23 = *reinterpret_cast<const double2*>(pi + 2);
#pragma unroll
                for (int t = 0; t < NV; ++t) {
                    const cplx xi = -xf[t][ch.p1 + i];
                    cfma(a0[t], mk(r01.x, i01.x), xi); cfma(a1[t], mk(r01.y, i01.y), xi);
                    cfma(a2[t], mk(r23.x, i23.x), xi); cfma(a3[t], mk(r23.y, i23.y), xi);
                }
            }
#pragma unroll
            for (int t = 0; t < NV; ++t) {
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    a0[t].x += __shfl_xor_sync(0xffffffffu, a0[t].x, off); a0[t].y += __shfl_xor_sync(0xffffffffu, a0[t].y, off);
                    a1[t].x += __shfl_xor_sync(0xffffffffu, a1[t].x, off); a1[t].y += __shfl_xor_sync(0xffffffffu, a1[t].y, off);
                    a2[t].x += __shfl_xor_sync(0xffffffffu, a2[t].x, off); a2[t].y += __shfl_xor_sync(0xffffffffu, a2[t].y, off);
                    a3[t].x += __shfl_xor_sync(0xffffffffu, a3[t].x, off); a3[t].y += __shfl_xor_sync(0xffffffffu, a3[t].y, off);
                }
                if (lane == 0) { tmp[t][4 * kg] = a0[t]; tmp[t][4 * kg + 1] = a1[t]; tmp[t][4 * kg + 2] = a2[t]; tmp[t][4 * kg + 3] = a3[t]; }
            }
        }
        __syncthreads();
        for (int k = tid; k < sc; k += nthr) {
#pragma unroll
            for (int t = 0; t < NV; ++t) xf[t][ch.p0 + k] = tmp[t][k];
        }
        __syncthreads();
    }
    for (int i = tid; i < F.sp; i += nthr) {
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            v[t][F.cbp + i] = xf[t][i];
            if (i < F.s) x[t][tb.pos2orig[F.cbp + i]] = xf[t][i];
        }
    }
}

__global__ void __launch_bounds__(kSolveMfThreads)
mf_bwd_kernel(Tables tb, SolveArgs sa, const int* __restrict__ list) {
    extern __shared__ __align__(16) unsigned char mf_smem[];
    const Front F = tb.fronts[list[blockIdx.x]];
    const int vec = blockIdx.y, sys = vec / sa.nrhs;
    cplx* const v[1] = {sa.v + (size_t)vec * sa.vStride};
    cplx* const x[1] = {sa.X + (size_t)vec * sa.ldx};
    mf_bwd_front<1>(tb, F, sys, v, x, reinterpret_cast<cplx*>(mf_smem));
}

// Paired backward substitution: one CTA per (front, system) solves vector a and vector b of the system (nrhs = 1 each) with one
// pass over the front's factor.  list[0, nBoth): both vectors; list[nBoth, n): vector b only (fronts whose pivot part of a
// already holds the solution — back-substituting it again would start from the solution instead of the eliminated rhs).
__global__ void __launch_bounds__(kSolveMfThreads)
mf_bwd_pair_kernel(Tables tb, SolveArgs sa, SolveArgs sb, const int* __restrict__ list, int nBoth) {
    extern __shared__ __align__(16) unsigned char mf_smem[];
    const Front F = tb.fronts[list[blockIdx.x]];
    const int sys = blockIdx.y;
    cplx* const vb = sb.v + (size_t)sys * sb.vStride;
    cplx* const xb = sb.X + (size_t)sys * sb.ldx;
    if ((int)blockIdx.x < nBoth) {
        cplx* const v[2] = {sa.v + (size_t)sys * sa.vStride, vb};
        cplx* const x[2] = {sa.X + (size_t)sys * sa.ldx, xb};
        mf_bwd_front<2>(tb, F, sys, v, x, reinterpret_cast<cplx*>(mf_smem));
    } else {
        cplx* const v[1] = {vb};
        cplx* const x[1] = {xb};
        mf_bwd_front<1>(tb, F, sys, v, x, reinterpret_cast<cplx*>(mf_smem));
    }
}

// Small fronts (single chunk, fp <= kSolveSmallMax): one WARP per (front, right-hand side), eight fronts per CTA, warp-level
// synchronisation only.  descs[blockIdx.x * 8 + warp] = the front's record: every later load depends on it alone or on one
// further index load, and the loads of the factor are issued before the gathers they will be combined with have arrived —
// a leaf front streams 1..3 KB of factor, so what a sweep costs is the chain of dependent round trips, not the bytes.
constexpr int kSolveSmallMax = 64;
constexpr int kSolveWarpsPerCta = 8;
__global__ void __launch_bounds__(kSolveWarpsPerCta * 32)
mf_fwd_warp_kernel(Tables tb, SolveArgs sa, const SolveDesc* __restrict__ descs, int n) {
    __shared__ cplx wsh[kSolveWarpsPerCta][kSolveSmallMax];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int fi = blockIdx.x * kSolveWarpsPerCta + warp;
    if (fi >= n) return;
    const SolveDesc D = descs[fi];
    const int vec = blockIdx.y, sys = vec / sa.nrhs;
    const int sp = D.sp, up = D.up, fp = sp + up, fs = D.s, fu = D.u, cbp = D.cbp;
    cplx* w = wsh[warp];
    const cplx* b = sa.B + (size_t)vec * sa.ldb;
    cplx* v = sa.v + (size_t)vec * sa.vStride;
    cplx* upd = sa.upd + (size_t)vec * sa.uStride;
    // (a) requests that need the record only: own right-hand-side rows (through pos2orig), the children's row maps and update vectors
    int orow[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) orow[h] = (lane + 32 * h < fs) ? tb.pos2orig[cbp + lane + 32 * h] : -1;
    int crel[kDescChildren];
    cplx cval[kDescChildren];
#pragma unroll
    for (int c = 0; c < kDescChildren; ++c) {
        crel[c] = -1;
        if (c < D.nChild && lane < D.cU[c]) { crel[c] = tb.rel[D.cRel[c] + lane]; cval[c] = upd[D.cUpd[c] + lane]; }
    }
    for (int i = lane; i < fp; i += 32) w[i] = mk(0.0, 0.0);
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) if (orow[h] >= 0) w[lane + 32 * h] = b[orow[h]];
    __syncwarp();
#pragma unroll
    for (int c = 0; c < kDescChildren; ++c) {
        if (c >= D.nChild) break;
        if (crel[c] >= 0) w[crel[c]] += cval[c];
        for (int i = lane + 32; i < D.cU[c]; i += 32) w[tb.rel[D.cRel[c] + i]] += upd[D.cUpd[c] + i];      // (children wider than a warp)
        __syncwarp();
    }
    if (up > 0) {
        const double* M = tb.fac + (size_t)sys * tb.facStride + D.mOff;
        const int ngr = (fs + 3) >> 2;      // column groups holding a real pivot (the rest is padding); real update rows only
        for (int i = lane; i < fu; i += 32) {
            cplx acc = mk(0.0, 0.0);
            for (int kg = 0; kg < ngr; ++kg) {
                const double* pr = M + kg_off(up, i, 4 * kg, 0);
                const double* pi = M + kg_off(up, i, 4 * kg, 1);
                const double2 r01 = *reinterpret_cast<const double2*>(pr), r23 = *reinterpret_cast<const double2*>(pr + 2);
                const double2 i01 = *reinterpret_cast<const double2*>(pi), i23 = *reinterpret_cast<const double2*>(pi + 2);
                const cplx* wk = w + 4 * kg;
                cfma(acc, mk(r01.x, i01.x), wk[0]);
                cfma(acc, mk(r01.y, i01.y), wk[1]);
                cfma(acc, mk(r23.x, i23.x), wk[2]);
                cfma(acc, mk(r23.y, i23.y), wk[3]);
            }
            upd[D.updOff + i] = w[sp + i] - acc;
        }
    }
    for (int i = lane; i < sp; i += 32) v[cbp + i] = w[i];
}

// Backward substitution of one front by one warp for NV vectors of the same system (each G / M element loaded once, applied
// to every vector with the arithmetic of the single-vector sweep); xf[t]: the warp's [kSolveSmallMax] stage of vector t.
template <int NV>
__device__ __forceinline__ void mf_bwd_warp_front(const Tables& tb, const SolveDesc& D, int sys, cplx* const (&v)[NV], cplx* const (&x)[NV],
                                                  cplx* const (&xf)[NV]) {
    const int lane = threadIdx.x & 31;
    const int sp = D.sp, up = D.up, fs = D.s, fu = D.u, cbp = D.cbp;
    const int* rows = tb.rows + D.rowPtr;
    const double* G = tb.fac + (size_t)sys * tb.facStride + D.gOff;
    const double* M = tb.fac + (size_t)sys * tb.facStride + D.mOff;
    // needs the record only: the update-row indices, the own pivot part, where the solution goes
    int urow[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = lane + 32 * h;
        urow[h] = i < fu ? (i < kDescRows ? D.rows[i] : rows[i]) : -1;
    }
#pragma unroll
    for (int t = 0; t < NV; ++t) {
        if (lane < sp) xf[t][lane] = v[t][cbp + lane];
        if (lane + 32 < sp) xf[t][lane + 32] = v[t][cbp + lane + 32];
    }
    // x1[k] = sum_j G[j][k] w1[j] - sum_i M[i][k] x2[i] : one lane per k; when the front has fewer than 32 pivots the rows are
    // split over 32 / width sub-groups of lanes and combined with shuffles.  Only the real pivots / update rows are visited: the
    // identity padding is never read back by anybody.
    const int width = fs <= 8 ? 8 : (fs <= 16 ? 16 : 32), nparts = 32 / width, part = lane / width, kl = lane - part * width;
    const int orig0 = (kl < fs && part == 0) ? tb.pos2orig[cbp + kl] : -1;      // (fronts of at most 32 pivots: the common case)
#pragma unroll
    for (int t = 0; t < NV; ++t)
#pragma unroll
        for (int h = 0; h < 2; ++h) if (urow[h] >= 0) xf[t][sp + lane + 32 * h] = v[t][urow[h]];
    __syncwarp();
    for (int k0 = 0; k0 < fs; k0 += width) {
        const int k = k0 + kl;
        cplx acc[NV];
#pragma unroll
        for (int t = 0; t < NV; ++t) acc[t] = mk(0.0, 0.0);
        if (k < fs) {
            const double* gr = G + kg_off(sp, 0, k, 0);
            const double* gi = G + kg_off(sp, 0, k, 1);
            for (int j = part; j < fs; j += nparts) {
                const cplx g = mk(gr[4 * j], gi[4 * j]);
#pragma unroll
                for (int t = 0; t < NV; ++t) cfma(acc[t], g, xf[t][j]);
            }
            const double* mr = M + kg_off(up, 0, k, 0);
            const double* mi = M + kg_off(up, 0, k, 1);
            for (int i = part; i < fu; i += nparts) {
                const cplx m = mk(-mr[4 * i], -mi[4 * i]);
#pragma unroll
                for (int t = 0; t < NV; ++t) cfma(acc[t], m, xf[t][sp + i]);
            }
        }
        for (int off = width; off < 32; off <<= 1) {
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                acc[t].x += __shfl_xor_sync(0xffffffffu, acc[t].x, off);
                acc[t].y += __shfl_xor_sync(0xffffffffu, acc[t].y, off);
            }
        }
        if (k < fs && part == 0) {
            const int o = k0 == 0 ? orig0 : tb.pos2orig[cbp + k];
#pragma unroll
            for (int t = 0; t < NV; ++t) {
                v[t][cbp + k] = acc[t];
                x[t][o] = acc[t];
            }
        }
    }
}

// Backward substitution, one warp per front.  (Fetching the front's contiguous [G | M] block whole into a shared-memory stage
// with cp.async was measured: no faster than the direct loads below at any stage size, and slower once the stage costs occupancy.)
__global__ void __launch_bounds__(kSolveWarpsPerCta * 32)
mf_bwd_warp_kernel(Tables tb, SolveArgs sa, const SolveDesc* __restrict__ descs, int n) {
    __shared__ cplx xsh[kSolveWarpsPerCta][kSolveSmallMax];
    const int warp = threadIdx.x >> 5;
    const int fi = blockIdx.x * kSolveWarpsPerCta + warp;
    if (fi >= n) return;
    const SolveDesc& D = descs[fi];                // (fields are read as needed; the row indices ride in the same record)
    const int vec = blockIdx.y, sys = vec / sa.nrhs;
    cplx* const v[1] = {sa.v + (size_t)vec * sa.vStride};
    cplx* const x[1] = {sa.X + (size_t)vec * sa.ldx};
    cplx* const xf[1] = {xsh[warp]};
    mf_bwd_warp_front<1>(tb, D, sys, v, x, xf);
}

// Paired backward substitution, one warp per (front, system) for vectors a and b: descs[0, nBoth) both, descs[nBoth, n) b only
// (see mf_bwd_pair_kernel).
__global__ void __launch_bounds__(kSolveWarpsPerCta * 32, 4)
mf_bwd_pair_warp_kernel(Tables tb, SolveArgs sa, SolveArgs sb, const SolveDesc* __restrict__ descs, int n, int nBoth) {
    __shared__ cplx xsh[2][kSolveWarpsPerCta][kSolveSmallMax];
    const int warp = threadIdx.x >> 5;
    const int fi = blockIdx.x * kSolveWarpsPerCta + warp;
    if (fi >= n) return;
    const SolveDesc& D = descs[fi];
    const int sys = blockIdx.y;
    cplx* const vb = sb.v + (size_t)sys * sb.vStride;
    cplx* const xb = sb.X + (size_t)sys * sb.ldx;
    if (fi < nBoth) {
        cplx* const v[2] = {sa.v + (size_t)sys * sa.vStride, vb};
        cplx* const x[2] = {sa.X + (size_t)sys * sa.ldx, xb};
        cplx* const xf[2] = {xsh[0][warp], xsh[1][warp]};
        mf_bwd_warp_front<2>(tb, D, sys, v, x, xf);
    } else {
        cplx* const v[1] = {vb};
        cplx* const x[1] = {xb};
        cplx* const xf[1] = {xsh[1][warp]};
        mf_bwd_warp_front<1>(tb, D, sys, v, x, xf);
    }
}

}  // namespace mf
}  // namespace hmcmt
