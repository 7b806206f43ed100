// Selected inversion on the multifrontal factor (Takahashi / Erisman-Tinney): diag(A^{-1}) from the resident G / M of every chunk.
//
// Each chunk's elimination is A = L diag(F11, S) L^T with L = [I 0; M I] and G = F11^{-1}, so that on a front, with c the chunk's
// pivots and R = rows [p1, fp) of the front, the inverse Z satisfies
//     Z(R, c) = -Z(R, R) M_c,        Z(c, R) = Z(R, c)^T,        Z(c, c) = G_c - Z(c, R) M_c
// (complex symmetric, no conjugation).  The chunks of a front run last to first.  Z(U, U) of a front's update rows is gathered
// from its parent's Z through the front's `rel` map (the extend-add run backwards), so the sweep runs depth by depth from the
// roots down.  Every front's Z is a full fp x fp square (both triangles, k-grouped, plane 0 / 1 = real / imaginary) in a
// depth-parity arena: both products are then plain A B with B = M_c read in its stored layout.
//   mf_selinv_gather_kernel : Z(U, U) of every front of a depth, one CTA per 64 x 64 tile (padded update rows -> 0);
//   mf_selinv_gemm_kernel   : C (64 x 64 tile) = S + alpha A B on the FP64 tensor cores (DMMA.8x8x4), cp.async-staged like
//                             mf_gemm_kernel; optionally C^T written alongside and the diagonal of the real pivots to `out`.
// Every output element is one thread's sum over k in increasing order: repeated calls are bit-identical, independent of how
// the fronts are grouped into launches.  Padded pivots are identity rows without coupling and padded update rows are zero in
// Z(U, U) and in M, so neither reaches a real entry.
#pragma once
#include "mf_kernels.cuh"

namespace hmcmt {
namespace mf {

struct SelTables {
    const Front* fronts;
    const int* rel;
    const int* pos2orig;
    const int64_t* zOff;         // [K] offset (doubles) of front k's Z square in the arena of its depth parity
    const double* fac;           // [nsys][facStride]
    double* zarena[2];           // [nsys][zStride[p]]
    int64_t facStride, zStride[2];
    cplx* out;                   // diagonal of system s at out + s * ldo (original numbering)
    int64_t ldo;
};

// front k's Z square (arena of parity par; selected without indexing the parameter array, which would copy it to the stack)
__device__ __forceinline__ double* zfront(const SelTables& tb, int par, int sys, int k) {
    return (par ? tb.zarena[1] + (size_t)sys * tb.zStride[1] : tb.zarena[0] + (size_t)sys * tb.zStride[0]) + tb.zOff[k];
}

// Z(U, U) of front `front` from its parent's Z: tile (bi, bj) of the up x up block
struct SelGatherTile {
    int front, bi, bj;
};
__global__ void __launch_bounds__(256) mf_selinv_gather_kernel(SelTables tb, const SelGatherTile* __restrict__ list) {
    const SelGatherTile gt = list[blockIdx.x];
    const int sys = blockIdx.y;
    const Front F = tb.fronts[gt.front];
    const Front& P = tb.fronts[F.parent];
    const int fp = F.sp + F.up, pfp = P.sp + P.up, par = F.depth & 1;
    double* Z = zfront(tb, par, sys, gt.front);
    const double* Zp = zfront(tb, par ^ 1, sys, F.parent);
    const int* rel = tb.rel + F.rowPtr;
    for (int item = threadIdx.x; item < 64 * 16; item += 256) {
        const int i = gt.bi * 64 + (item & 63), j0 = gt.bj * 64 + (item >> 6) * 4;
        if (i >= F.up || j0 >= F.up) continue;
        double re[4], im[4];
        const int ri = i < F.u ? rel[i] : -1;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = j0 + k;
            re[k] = im[k] = 0.0;
            if (ri >= 0 && j < F.u) {
                const int rj = rel[j];
                re[k] = Zp[kg_off(pfp, ri, rj, 0)];
                im[k] = Zp[kg_off(pfp, ri, rj, 1)];
            }
        }
        double* pr = Z + kg_off(fp, F.sp + i, F.sp + j0, 0);
        double* pi = Z + kg_off(fp, F.sp + i, F.sp + j0, 1);
        *reinterpret_cast<double2*>(pr) = make_double2(re[0], re[1]); *reinterpret_cast<double2*>(pr + 2) = make_double2(re[2], re[3]);
        *reinterpret_cast<double2*>(pi) = make_double2(im[0], im[1]); *reinterpret_cast<double2*>(pi + 2) = make_double2(im[2], im[3]);
    }
}

// C(i, j) = S(i, j) + alpha sum_k A(i, k) B(k, j), i < m, j < n, k < K (multiples of 8; K may be 0).  All three k-grouped:
//   A(i, k) = Z[rA + i][kA + k] (the front's Z square, ld fp), B(k, j) = M[k][j] (factor arena, ld ldB), C(i, j) = Z[rC + i][cC + j];
//   S(i, j) = G[i][j] (factor arena, ld ldS) when hasS.  transC: C^T is written too, at Z[cC + j][rC + i].
//   diag: C is the front's Z(c, c) of the pivots [rC, rC + m); its diagonal entries of real pivots (< s) go to out[pos2orig[cbp + .]].
struct SelJob {
    int front;
    int64_t bOff, sOff;
    int rA, kA, ldB, ldS, rC, cC;
    int m, n, K;
    int hasS, transC, diag;
    double alpha;
};
struct SelTile {
    int job, bi, bj;
};

// (two CTAs per SM: at most 128 registers, 2 x 96 KB of stages)
__global__ void __launch_bounds__(kGemmThreads, 2)
mf_selinv_gemm_kernel(SelTables tb, const SelJob* __restrict__ jobs, const SelTile* __restrict__ tilesList) {
    extern __shared__ __align__(16) unsigned char mf_smem[];
    double* sm = reinterpret_cast<double*>(mf_smem);
    const SelTile gt = tilesList[blockIdx.x];
    const SelJob jb = jobs[gt.job];
    const Front F = tb.fronts[jb.front];
    const int fp = F.sp + F.up, par = F.depth & 1;
    const int sys = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int g = lane >> 2, t = lane & 3;
    const int wr = warp >> 1, wc = warp & 1;          // warp tile: rows [16 wr, +16), cols [32 wc, +32)
    double* Z = zfront(tb, par, sys, jb.front);
    const double* fac = tb.fac + (size_t)sys * tb.facStride;
    const double* B = fac + jb.bOff;
    const int r0 = gt.bi * 64, c0 = gt.bj * 64;
    const int nk = (jb.K + kGemmKC - 1) / kGemmKC;
    constexpr int kHalf = (kGemmKC / 4) * 2 * 64 * 4;      // doubles of the A (or B) image of one stage
    // stage image: A [k group][plane][64 rows][4]  |  B [column group of 4][plane][kGemmKC k][4]
    auto load_stage = [&](int ks, int st) {
        double* dst = sm + (size_t)st * kGemmStageDoubles;
        const int k0 = ks * kGemmKC;
#pragma unroll
        for (int it = 0; it < 2 * (kGemmKC / 4) * 2 * 128 / kGemmThreads; ++it) {
            const int c = tid + it * kGemmThreads;
            const int which = c / ((kGemmKC / 4) * 2 * 128);
            const int cc = c - which * ((kGemmKC / 4) * 2 * 128);
            const double* src;
            bool ok;
            if (which == 0) {
                const int grp = cc >> 8, pl = (cc >> 7) & 1, row = (cc & 127) >> 1, half = cc & 1, k = k0 + 4 * grp;
                ok = (r0 + row < jb.m) && (k < jb.K);
                src = Z + kg_off(fp, jb.rA + r0 + row, jb.kA + k, pl) + half * 2;
            } else {
                const int half = cc & 1, k = (cc >> 1) & (kGemmKC - 1), pl = (cc >> 5) & 1, ng = cc >> 6;
                ok = (k0 + k < jb.K) && (c0 + 4 * ng < jb.n);
                src = B + kg_off(jb.ldB, k0 + k, c0 + 4 * ng, pl) + half * 2;
            }
            cp_async16(dst + (size_t)c * 2, ok ? src : B, ok ? 16u : 0u);
        }
        cp_async_commit();
    };
    double cre[2][4][2], cim[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) cre[a][b][0] = cre[a][b][1] = cim[a][b][0] = cim[a][b][1] = 0.0;
    unsigned act = 0;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int rb = r0 + wr * 16 + a * 8, cb = c0 + wc * 32 + b * 8;
            if (rb < jb.m && cb < jb.n) act |= 1u << (a * 4 + b);
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
        const double* sB = sA + kHalf;
        const int ngrp = min(kGemmKC / 4, (jb.K - ks * kGemmKC + 3) >> 2);
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
            for (int b = 0; b < 4; ++b) {      // operand B[k = 4 grp + t][n = 8 b + g]
                const int n = wc * 32 + b * 8 + g;
                bre[b] = sB[(((n >> 2) * 2 + 0) * kGemmKC + 4 * grp + t) * 4 + (n & 3)];
                bim[b] = sB[(((n >> 2) * 2 + 1) * kGemmKC + 4 * grp + t) * 4 + (n & 3)];
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
    // epilogue: lane holds C(rb + g, cb + 2t), C(rb + g, cb + 2t + 1)
    const double* Sg = fac + jb.sOff;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            if (!((act >> (a * 4 + b)) & 1)) continue;
            const int i = r0 + wr * 16 + a * 8 + g, j = c0 + wc * 32 + b * 8 + 2 * t;
            double2 vr = make_double2(jb.alpha * cre[a][b][0], jb.alpha * cre[a][b][1]);
            double2 vi = make_double2(jb.alpha * cim[a][b][0], jb.alpha * cim[a][b][1]);
            if (jb.hasS) {
                const double2 sr = *reinterpret_cast<const double2*>(Sg + kg_off(jb.ldS, i, j, 0));
                const double2 si = *reinterpret_cast<const double2*>(Sg + kg_off(jb.ldS, i, j, 1));
                vr.x = sr.x + vr.x; vr.y = sr.y + vr.y; vi.x = si.x + vi.x; vi.y = si.y + vi.y;
            }
            *reinterpret_cast<double2*>(Z + kg_off(fp, jb.rC + i, jb.cC + j, 0)) = vr;
            *reinterpret_cast<double2*>(Z + kg_off(fp, jb.rC + i, jb.cC + j, 1)) = vi;
            if (jb.transC) {
                Z[kg_off(fp, jb.cC + j, jb.rC + i, 0)] = vr.x; Z[kg_off(fp, jb.cC + j + 1, jb.rC + i, 0)] = vr.y;
                Z[kg_off(fp, jb.cC + j, jb.rC + i, 1)] = vi.x; Z[kg_off(fp, jb.cC + j + 1, jb.rC + i, 1)] = vi.y;
            }
            if (jb.diag && (i == j || i == j + 1)) {
                const int p = jb.rC + i;
                if (p < F.s) tb.out[(size_t)sys * tb.ldo + tb.pos2orig[F.cbp + p]] = i == j ? mk(vr.x, vi.x) : mk(vr.y, vi.y);
            }
        }
}

}  // namespace mf
}  // namespace hmcmt
