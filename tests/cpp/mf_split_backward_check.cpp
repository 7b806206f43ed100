// CPU check of the split backward substitution of the gradient evaluation (Solver::backward_slot / backward_pair,
// hmcmt_b200.cu gradient_range) on the tables of mf_symbolic.h, in plain std::complex on the host:
//   - the receiver path (the active set of the receiver rows' pattern, the marking loop of Solver::add_rhs_pattern) holds every
//     unknown of the two receiver rows and is closed under parents;
//   - x on the receiver rows after the receiver-path sweep alone equals the complete solution there;
//   - receiver path on slot 0, then one sweep over both slots that skips slot 0 on the receiver path, gives exactly (bit for
//     bit: the same operations in the same order) the two complete backward substitutions;
//   - the same sweep without the skip (slot 0 back-substituted a second time from its solution) does not.
// Test infrastructure only.
//   usage: mf_split_backward_check <nl> <nf> <leaf> <fSmall> <cross> <push> <f0>
//          grid nl x nf (the plan's numbering: q = l*nf + f, f along the fast axis); receiver rows f = f0, f0 + 1
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <random>

#include "../../hmcmt2d_b200/csrc/mf_symbolic.h"

using namespace hmcmt::mf;
typedef std::complex<double> cd;

static void invert(std::vector<cd>& A, int n) {      // Gauss-Jordan without pivoting
    std::vector<cd> B((size_t)n * n, cd(0));
    for (int i = 0; i < n; ++i) B[(size_t)i * n + i] = 1.0;
    for (int k = 0; k < n; ++k) {
        cd p = 1.0 / A[(size_t)k * n + k];
        for (int j = 0; j < n; ++j) { A[(size_t)k * n + j] *= p; B[(size_t)k * n + j] *= p; }
        for (int i = 0; i < n; ++i) if (i != k) {
            cd f = A[(size_t)i * n + k];
            if (f == cd(0)) continue;
            for (int j = 0; j < n; ++j) { A[(size_t)i * n + j] -= f * A[(size_t)k * n + j]; B[(size_t)i * n + j] -= f * B[(size_t)k * n + j]; }
        }
    }
    A = B;
}

int main(int argc, char** argv) {
    if (argc < 8) return 2;
    const int nl = atoi(argv[1]), nf = atoi(argv[2]), leaf = atoi(argv[3]), fSmall = atoi(argv[4]), cross = atoi(argv[5]),
              push = atoi(argv[6]), f0 = atoi(argv[7]);
    if (f0 < 0 || f0 + 1 >= nf) return 2;
    const int N = nl * nf;
    std::vector<Entry> ent;
    std::vector<std::vector<int>> sn;
    mf_grid_entries(nl, nf, ent);
    mf_order_grid(nl, nf, leaf, sn, cross, push);
    std::mt19937_64 rng(11);
    std::uniform_real_distribution<double> un(0.1, 1.0);
    int nsrc = 0;
    for (auto& e : ent) nsrc = std::max(nsrc, e.src + 1);
    std::vector<cd> vals(nsrc);
    std::vector<double> rowsum(N, 0.0);
    for (auto& e : ent) if (e.row != e.col) { double v = -un(rng); vals[e.src] = v; rowsum[e.row] += -v; rowsum[e.col] += -v; }
    for (auto& e : ent) if (e.row == e.col) vals[e.src] = cd(rowsum[e.row] + 0.01, 0.3 * un(rng));
    Symbolic S;
    if (!mf_symbolic(N, sn, ent, fSmall, S)) { printf("symbolic failed\n"); return 1; }

    // numeric factorisation (the arithmetic of mf_tables_check.cpp)
    std::vector<std::vector<cd>> U(S.K), G(S.chunks.size()), M(S.chunks.size());
    auto run_front = [&](int k) {
        const Front& F = S.fronts[k];
        const int fp = F.fp();
        std::vector<cd> A((size_t)fp * fp, cd(0));
        for (int e = 0; e < F.nOrig; ++e) {
            const OrigEntry& oe = S.orig[F.origPtr + e];
            A[(size_t)oe.lrow * fp + oe.lcol] += oe.src < 0 ? cd(1.0) : vals[oe.src];
        }
        for (int c = 0; c < F.nChild; ++c) {
            const int ck = S.children[F.childPtr + c];
            const Front& C = S.fronts[ck];
            const int* rel = S.rel.data() + C.rowPtr;
            for (int i = 0; i < C.u; ++i) for (int j = 0; j <= i; ++j) A[(size_t)rel[i] * fp + rel[j]] += U[ck][(size_t)i * C.up + j];
            std::vector<cd>().swap(U[ck]);
        }
        for (int i = 0; i < fp; ++i) for (int j = 0; j < i; ++j) A[(size_t)j * fp + i] = A[(size_t)i * fp + j];
        for (int c = 0; c < F.nChunk; ++c) {
            const Chunk& ch = S.chunks[F.chunkPtr + c];
            const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
            std::vector<cd> g((size_t)sc * sc);
            for (int i = 0; i < sc; ++i) for (int j = 0; j < sc; ++j) g[(size_t)i * sc + j] = A[(size_t)(ch.p0 + i) * fp + ch.p0 + j];
            invert(g, sc);
            std::vector<cd> m((size_t)mr * sc, cd(0));
            for (int i = 0; i < mr; ++i) for (int kk = 0; kk < sc; ++kk) {
                cd a = A[(size_t)(ch.p1 + i) * fp + ch.p0 + kk];
                if (a == cd(0)) continue;
                for (int j = 0; j < sc; ++j) m[(size_t)i * sc + j] += a * g[(size_t)kk * sc + j];
            }
            for (int i = 0; i < mr; ++i) for (int j = 0; j < mr; ++j) {
                cd acc = 0;
                for (int kk = 0; kk < sc; ++kk) acc += m[(size_t)i * sc + kk] * A[(size_t)(ch.p1 + j) * fp + ch.p0 + kk];
                A[(size_t)(ch.p1 + i) * fp + ch.p1 + j] -= acc;
            }
            G[F.chunkPtr + c] = std::move(g);
            M[F.chunkPtr + c] = std::move(m);
        }
        U[k].assign((size_t)F.up * F.up, cd(0));
        for (int i = 0; i < F.up; ++i) for (int j = 0; j < F.up; ++j) U[k][(size_t)i * F.up + j] = A[(size_t)(F.sp + i) * fp + F.sp + j];
    };
    for (int d = S.maxDepth; d >= 0; --d) {
        for (int k : S.byDepthBig[d]) run_front(k);
        for (int k : S.byDepthSmall[d]) run_front(k);
    }

    // receiver rows and their active set (Solver::add_rhs_pattern)
    std::vector<unsigned char> rx(N, 0);
    for (int l = 0; l < nl; ++l) rx[l * nf + f0] = rx[l * nf + f0 + 1] = 1;
    std::vector<char> active(S.K, 0);
    for (int k = 0; k < S.K; ++k) {
        const Front& F = S.fronts[k];
        for (int i = 0; i < F.s && !active[k]; ++i) {
            const int o = S.pos2orig[F.cbp + i];
            if (o >= 0 && rx[o]) active[k] = 1;
        }
        if (active[k] && F.parent >= 0) active[F.parent] = 1;
    }
    int nActive = 0, nLeaf = 0, nLeafActive = 0;
    double bytesAll = 0, bytesActive = 0;
    std::vector<char> covered(N, 0);
    for (int k = 0; k < S.K; ++k) {
        const Front& F = S.fronts[k];
        if (active[k] && F.parent >= 0 && !active[F.parent]) { printf("receiver path not closed under parents\n"); return 1; }
        for (int i = 0; i < F.s; ++i) {
            const int o = S.pos2orig[F.cbp + i];
            if (o >= 0 && active[k]) covered[o] = 1;
        }
        double b = 0;
        for (int c = 0; c < F.nChunk; ++c) {
            const Chunk& ch = S.chunks[F.chunkPtr + c];
            const double sc = ch.p1 - ch.p0, mr = F.fp() - ch.p1;
            b += 16.0 * (sc * sc + mr * sc);
        }
        bytesAll += b;
        nActive += active[k];
        nLeaf += F.nChild == 0;
        if (active[k]) { bytesActive += b; nLeafActive += F.nChild == 0; }
    }
    for (int q = 0; q < N; ++q)
        if (rx[q] && !covered[q]) { printf("receiver unknown %d outside the receiver path\n", q); return 1; }
    printf("fronts %d, receiver path %d (%d of %d leaves), G/M bytes %.2f of %.2f MB = %.1f %%\n", S.K, nActive, nLeafActive, nLeaf,
           bytesActive / 1e6, bytesAll / 1e6, 100.0 * bytesActive / bytesAll);

    // solves: forward elimination (only the fronts of `act` if given: the others hand zero update vectors), backward of one front
    auto forward = [&](const std::vector<cd>& b, const std::vector<char>* act, std::vector<cd>& v, std::vector<cd>& upd) {
        v.assign(S.Np, cd(0));
        upd.assign(S.updEntries, cd(0));
        for (int d = S.maxDepth; d >= 0; --d)
            for (int pass = 0; pass < 2; ++pass)
                for (int k : (pass ? S.byDepthSmall[d] : S.byDepthBig[d])) {
                    if (act && !(*act)[k]) continue;
                    const Front& F = S.fronts[k];
                    const int fp = F.fp();
                    std::vector<cd> w(fp, cd(0));
                    for (int i = 0; i < F.s; ++i) w[i] = b[S.pos2orig[F.cbp + i]];
                    for (int c = 0; c < F.nChild; ++c) {
                        const Front& C = S.fronts[S.children[F.childPtr + c]];
                        for (int i = 0; i < C.u; ++i) w[S.rel[C.rowPtr + i]] += upd[C.updOff + i];
                    }
                    for (int c = 0; c < F.nChunk; ++c) {
                        const Chunk& ch = S.chunks[F.chunkPtr + c];
                        const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
                        for (int i = 0; i < mr; ++i) {
                            cd acc = 0;
                            for (int kk = 0; kk < sc; ++kk) acc += M[F.chunkPtr + c][(size_t)i * sc + kk] * w[ch.p0 + kk];
                            w[ch.p1 + i] -= acc;
                        }
                    }
                    for (int i = 0; i < F.sp; ++i) v[F.cbp + i] = w[i];
                    for (int i = 0; i < F.up; ++i) upd[F.updOff + i] = w[F.sp + i];
                }
    };
    auto backward_front = [&](int k, std::vector<cd>& v, std::vector<cd>& x) {
        const Front& F = S.fronts[k];
        const int fp = F.fp();
        std::vector<cd> xf(fp, cd(0));
        for (int i = 0; i < F.sp; ++i) xf[i] = v[F.cbp + i];
        for (int i = 0; i < F.u; ++i) xf[F.sp + i] = v[S.rows[F.rowPtr + i]];
        for (int c = F.nChunk - 1; c >= 0; --c) {
            const Chunk& ch = S.chunks[F.chunkPtr + c];
            const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
            std::vector<cd> t(sc, cd(0));
            for (int kk = 0; kk < sc; ++kk) {
                cd acc = 0;
                for (int j = 0; j < sc; ++j) acc += G[F.chunkPtr + c][(size_t)j * sc + kk] * xf[ch.p0 + j];
                for (int i = 0; i < mr; ++i) acc -= M[F.chunkPtr + c][(size_t)i * sc + kk] * xf[ch.p1 + i];
                t[kk] = acc;
            }
            for (int kk = 0; kk < sc; ++kk) xf[ch.p0 + kk] = t[kk];
        }
        for (int i = 0; i < F.sp; ++i) { v[F.cbp + i] = xf[i]; if (i < F.s) x[S.pos2orig[F.cbp + i]] = xf[i]; }
    };
    // root first, depth by depth: `which(k)` = 0 skip, 1 vector a only, 2 vector b only, 3 both
    auto sweep = [&](auto which, std::vector<cd>& va, std::vector<cd>& xa, std::vector<cd>& vb, std::vector<cd>& xb) {
        for (int d = 0; d <= S.maxDepth; ++d)
            for (int pass = 0; pass < 2; ++pass)
                for (int k : (pass ? S.byDepthSmall[d] : S.byDepthBig[d])) {
                    const int w = which(k);
                    if (w & 1) backward_front(k, va, xa);
                    if (w & 2) backward_front(k, vb, xb);
                }
    };

    // x: dense right-hand side; lam: non-zero on the receiver rows only (pruned forward elimination, as the adjoint)
    std::vector<cd> bx(N), bl(N, cd(0));
    for (auto& z : bx) z = cd(un(rng) - 0.5, un(rng) - 0.5);
    for (int q = 0; q < N; ++q) if (rx[q]) bl[q] = cd(un(rng) - 0.5, un(rng) - 0.5);
    std::vector<cd> va, ua, vb, ub, xa(N, cd(0)), xb(N, cd(0)), refA(N, cd(0)), refB(N, cd(0));
    // reference: the complete solves, one after the other
    forward(bx, nullptr, va, ua);
    sweep([](int) { return 1; }, va, refA, vb, refB);
    forward(bl, &active, vb, ub);
    sweep([](int) { return 2; }, va, refA, vb, refB);
    // split order: receiver path of x, receiver rows, forward of lam, paired sweep that skips x on the receiver path
    const cd poison(1e300, -1e300);
    for (auto& z : xa) z = poison;
    for (auto& z : xb) z = poison;
    forward(bx, nullptr, va, ua);
    sweep([&](int k) { return active[k] ? 1 : 0; }, va, xa, vb, xb);
    for (int q = 0; q < N; ++q)
        if (rx[q] && xa[q] != refA[q]) { printf("receiver-row x after the receiver-path sweep differs at %d\n", q); return 1; }
    std::vector<cd> vaSplit = va;
    forward(bl, &active, vb, ub);
    sweep([&](int k) { return active[k] ? 2 : 3; }, va, xa, vb, xb);
    for (int q = 0; q < N; ++q)
        if (xa[q] != refA[q] || xb[q] != refB[q]) { printf("split order differs from the complete solves at %d\n", q); return 1; }
    // the in-place trap: back-substituting x again on the receiver path starts from the solution, not the eliminated rhs
    std::vector<cd> xt(N, cd(0)), xt2(N, cd(0));
    forward(bl, &active, vb, ub);
    sweep([](int) { return 3; }, vaSplit, xt, vb, xt2);
    double err = 0;
    for (int q = 0; q < N; ++q) err = std::max(err, std::abs(xt[q] - refA[q]));
    if (!(err > 0)) { printf("recomputing x on the receiver path went unnoticed\n"); return 1; }
    printf("split order bit-identical to the complete solves; recomputing x on the receiver path: max error %.3e\n", err);
    return 0;
}
