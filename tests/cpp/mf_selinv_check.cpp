// CPU check of the selected inversion (hmcmt2d_b200/csrc/mf_selinv.cuh, Solver::inverse_diag): from the very Symbolic tables,
// factorise as tests/cpp/mf_tables_check.cpp does (G = F11^-1, M = F21 G, U = F22 - M F21^T, chunked pivots), then run the
// top-down recursion of the device code in std::complex<long double> — roots first, Z(U, U) gathered from the parent's Z through
// `rel`, chunks last to first, Z(R, c) = -Z(R, R) M_c, Z(c, R) = Z(R, c)^T, Z(c, c) = G_c - Z(c, R) M_c — and compare EVERY entry of
// every front's Z (real rows) with a dense inverse of A computed independently (Gauss-Jordan with partial pivoting, double).
// Entries of padded rows / columns must come out exactly zero (padded pivots: exactly the identity), so that they never reach a
// real entry.  Test infrastructure only.
//   usage: mf_selinv_check grid <nl> <nf> <leaf> <fSmall> [cross] [push]
//          mf_selinv_check active <nl> <nf> <leaf> <fSmall> <seed>      (five-point graph of a random active-cell set, mf_order_graph)
//          mf_selinv_check graph3d <nx> <ny> <nz> <leaf> <fSmall>
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>

#include "../../hmcmt2d_b200/csrc/mf_symbolic.h"

using namespace hmcmt::mf;
typedef std::complex<long double> cl;
typedef std::complex<double> cd;

static void invert(std::vector<cl>& A, int n) {      // Gauss-Jordan without pivoting (the factor's own arithmetic)
    std::vector<cl> B((size_t)n * n, cl(0));
    for (int i = 0; i < n; ++i) B[(size_t)i * n + i] = 1.0L;
    for (int k = 0; k < n; ++k) {
        cl p = 1.0L / A[(size_t)k * n + k];
        for (int j = 0; j < n; ++j) { A[(size_t)k * n + j] *= p; B[(size_t)k * n + j] *= p; }
        for (int i = 0; i < n; ++i) if (i != k) {
            cl f = A[(size_t)i * n + k];
            if (f == cl(0)) continue;
            for (int j = 0; j < n; ++j) { A[(size_t)i * n + j] -= f * A[(size_t)k * n + j]; B[(size_t)i * n + j] -= f * B[(size_t)k * n + j]; }
        }
    }
    A = B;
}

static void graph_order(int N, const std::vector<Entry>& ent, int leaf, std::vector<std::vector<int>>& sn) {
    std::vector<int> ptr(N + 1, 0), adj;
    for (auto& e : ent) if (e.row != e.col) { ++ptr[e.row + 1]; ++ptr[e.col + 1]; }
    for (int i = 0; i < N; ++i) ptr[i + 1] += ptr[i];
    adj.resize(ptr[N]);
    std::vector<int> at(ptr.begin(), ptr.end() - 1);
    for (auto& e : ent) if (e.row != e.col) { adj[at[e.row]++] = e.col; adj[at[e.col]++] = e.row; }
    mf_order_graph(N, ptr, adj, leaf, sn);
}

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    std::vector<Entry> ent;
    std::vector<std::vector<int>> sn;
    int N = 0, fSmall = 144;
    if (!strcmp(argv[1], "grid")) {
        const int nl = atoi(argv[2]), nf = atoi(argv[3]), leaf = atoi(argv[4]);
        fSmall = atoi(argv[5]);
        N = nl * nf;
        mf_grid_entries(nl, nf, ent);
        mf_order_grid(nl, nf, leaf, sn, argc > 6 ? atoi(argv[6]) : 0, argc > 7 ? atoi(argv[7]) : 0);
    } else if (!strcmp(argv[1], "active")) {
        // the model cells of a five-point mesh below a ragged top (air and topography removed), numbered column by column:
        // the pattern of Wm, ordered through mf_order_graph as the plan orders it
        const int nl = atoi(argv[2]), nf = atoi(argv[3]), leaf = atoi(argv[4]);
        fSmall = atoi(argv[5]);
        std::mt19937_64 r(atoi(argv[6]));
        std::vector<int> id((size_t)nl * nf, -1);
        for (int l = 0; l < nl; ++l) {
            const int top = (int)(r() % 4);
            for (int f = top; f < nf; ++f) id[(size_t)l * nf + f] = N++;
        }
        int src = 0;
        for (int l = 0; l < nl; ++l)
            for (int f = 0; f < nf; ++f) {
                const int q = id[(size_t)l * nf + f];
                if (q < 0) continue;
                ent.push_back(Entry{q, q, src++});
                if (f > 0 && id[(size_t)l * nf + f - 1] >= 0) ent.push_back(Entry{q, id[(size_t)l * nf + f - 1], src++});
                if (l > 0 && id[(size_t)(l - 1) * nf + f] >= 0) ent.push_back(Entry{q, id[(size_t)(l - 1) * nf + f], src++});
            }
        graph_order(N, ent, leaf, sn);
    } else {
        const int nx = atoi(argv[2]), ny = atoi(argv[3]), nz = atoi(argv[4]), leaf = atoi(argv[5]);
        fSmall = atoi(argv[6]);
        N = nx * ny * nz;
        auto id = [&](int i, int j, int k) { return (k * ny + j) * nx + i; };
        int src = 0;
        for (int k = 0; k < nz; ++k) for (int j = 0; j < ny; ++j) for (int i = 0; i < nx; ++i) {
            const int q = id(i, j, k);
            ent.push_back(Entry{q, q, src++});
            if (i > 0) ent.push_back(Entry{q, id(i - 1, j, k), src++});
            if (j > 0) ent.push_back(Entry{q, id(i, j - 1, k), src++});
            if (k > 0) ent.push_back(Entry{q, id(i, j, k - 1), src++});
        }
        graph_order(N, ent, leaf, sn);
    }
    if (N > 3000) { printf("n %d: too large for the dense reference\n", N); return 2; }
    // values: complex symmetric, diagonally dominant (pivot-free elimination well defined)
    std::mt19937_64 rng(7);
    std::uniform_real_distribution<double> un(0.1, 1.0);
    int nsrc = 0;
    for (auto& e : ent) nsrc = std::max(nsrc, e.src + 1);
    std::vector<cd> vals(nsrc);
    std::vector<double> rowsum(N, 0.0);
    for (auto& e : ent) if (e.row != e.col) { double v = -un(rng); vals[e.src] = cd(v, 0.2 * v); rowsum[e.row] += -v; rowsum[e.col] += -v; }
    for (auto& e : ent) if (e.row == e.col) vals[e.src] = cd(rowsum[e.row] + 0.05, 0.3 * un(rng));
    Symbolic S;
    if (!mf_symbolic(N, sn, ent, fSmall, S)) { printf("symbolic failed\n"); return 1; }
    int nbig = 0, maxChunks = 0;
    for (auto& F : S.fronts) { nbig += F.isBig; maxChunks = std::max(maxChunks, F.nChunk); }
    printf("N %d K %d depth %d maxFp %d big %d maxChunks %d factor flops %.3e selinv flops %.3e\n", S.N, S.K, S.maxDepth, S.maxFp, nbig,
           maxChunks, S.flops, S.selinvFlops);
    // ---- numeric factorisation (mf_tables_check.cpp), long double ----
    std::vector<std::vector<cl>> U(S.K), G(S.chunks.size()), M(S.chunks.size());
    auto run_front = [&](int k) {
        const Front& F = S.fronts[k];
        const int fp = F.fp();
        std::vector<cl> A((size_t)fp * fp, cl(0));
        for (int e = 0; e < F.nOrig; ++e) {
            const OrigEntry& oe = S.orig[F.origPtr + e];
            const cd v = oe.src < 0 ? cd(1.0) : vals[oe.src];
            A[(size_t)oe.lrow * fp + oe.lcol] += cl(v.real(), v.imag());
        }
        for (int c = 0; c < F.nChild; ++c) {
            const int ck = S.children[F.childPtr + c];
            const Front& C = S.fronts[ck];
            const int* rel = S.rel.data() + C.rowPtr;
            for (int i = 0; i < C.u; ++i) for (int j = 0; j <= i; ++j) A[(size_t)rel[i] * fp + rel[j]] += U[ck][(size_t)i * C.up + j];
            std::vector<cl>().swap(U[ck]);
        }
        for (int i = 0; i < fp; ++i) for (int j = 0; j < i; ++j) A[(size_t)j * fp + i] = A[(size_t)i * fp + j];
        for (int c = 0; c < F.nChunk; ++c) {
            const Chunk& ch = S.chunks[F.chunkPtr + c];
            const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
            std::vector<cl> g((size_t)sc * sc);
            for (int i = 0; i < sc; ++i) for (int j = 0; j < sc; ++j) g[(size_t)i * sc + j] = A[(size_t)(ch.p0 + i) * fp + ch.p0 + j];
            invert(g, sc);
            std::vector<cl> m((size_t)mr * sc, cl(0));
            for (int i = 0; i < mr; ++i) for (int kk = 0; kk < sc; ++kk) {
                const cl a = A[(size_t)(ch.p1 + i) * fp + ch.p0 + kk];
                if (a == cl(0)) continue;
                for (int j = 0; j < sc; ++j) m[(size_t)i * sc + j] += a * g[(size_t)kk * sc + j];
            }
            for (int i = 0; i < mr; ++i) for (int j = 0; j < mr; ++j) {
                cl acc = 0;
                for (int kk = 0; kk < sc; ++kk) acc += m[(size_t)i * sc + kk] * A[(size_t)(ch.p1 + j) * fp + ch.p0 + kk];
                A[(size_t)(ch.p1 + i) * fp + ch.p1 + j] -= acc;
            }
            G[F.chunkPtr + c] = std::move(g);
            M[F.chunkPtr + c] = std::move(m);
        }
        U[k].assign((size_t)F.up * F.up, cl(0));
        for (int i = 0; i < F.up; ++i) for (int j = 0; j < F.up; ++j) U[k][(size_t)i * F.up + j] = A[(size_t)(F.sp + i) * fp + F.sp + j];
    };
    for (int d = S.maxDepth; d >= 0; --d) {
        for (int k : S.byDepthBig[d]) run_front(k);
        for (int k : S.byDepthSmall[d]) run_front(k);
    }
    // ---- selected inversion, top-down, the device's schedule ----
    std::vector<std::vector<cl>> Z(S.K);
    std::vector<cl> diag(N, cl(0));
    std::vector<int> seen(N, 0);
    for (int d = 0; d <= S.maxDepth; ++d) {
        std::vector<int> fr(S.byDepthBig[d]);
        fr.insert(fr.end(), S.byDepthSmall[d].begin(), S.byDepthSmall[d].end());
        for (int k : fr) {
            const Front& F = S.fronts[k];
            const int fp = F.fp();
            std::vector<cl>& z = Z[k];
            z.assign((size_t)fp * fp, cl(0));
            if (F.u) {      // Z(U, U): gather from the parent (padded update rows stay 0)
                const Front& P = S.fronts[F.parent];
                const int pfp = P.fp();
                const int* rel = S.rel.data() + F.rowPtr;
                for (int i = 0; i < F.u; ++i) for (int j = 0; j < F.u; ++j)
                    z[(size_t)(F.sp + i) * fp + F.sp + j] = Z[F.parent][(size_t)rel[i] * pfp + rel[j]];
            }
            for (int c = F.nChunk - 1; c >= 0; --c) {
                const Chunk& ch = S.chunks[F.chunkPtr + c];
                const int sc = ch.p1 - ch.p0, mr = fp - ch.p1;
                const std::vector<cl>& m = M[F.chunkPtr + c];
                const std::vector<cl>& g = G[F.chunkPtr + c];
                for (int i = 0; i < mr; ++i) for (int kk = 0; kk < sc; ++kk) {
                    cl acc = 0;
                    for (int j = 0; j < mr; ++j) acc += z[(size_t)(ch.p1 + i) * fp + ch.p1 + j] * m[(size_t)j * sc + kk];
                    z[(size_t)(ch.p1 + i) * fp + ch.p0 + kk] = -acc;
                    z[(size_t)(ch.p0 + kk) * fp + ch.p1 + i] = -acc;
                }
                for (int a = 0; a < sc; ++a) for (int b = 0; b < sc; ++b) {
                    cl acc = 0;
                    for (int j = 0; j < mr; ++j) acc += z[(size_t)(ch.p0 + a) * fp + ch.p1 + j] * m[(size_t)j * sc + b];
                    z[(size_t)(ch.p0 + a) * fp + ch.p0 + b] = g[(size_t)a * sc + b] - acc;
                }
            }
            for (int i = 0; i < F.s; ++i) { const int o = S.pos2orig[F.cbp + i]; diag[o] = z[(size_t)i * fp + i]; ++seen[o]; }
        }
    }
    for (int o = 0; o < N; ++o) if (seen[o] != 1) { printf("unknown %d written %d times\n", o, seen[o]); return 1; }
    // ---- dense reference: Gauss-Jordan with partial pivoting in double, independent of the tables ----
    std::vector<cd> A((size_t)N * N, cd(0)), Ai((size_t)N * N, cd(0));
    for (auto& e : ent) { A[(size_t)e.row * N + e.col] += vals[e.src]; if (e.row != e.col) A[(size_t)e.col * N + e.row] += vals[e.src]; }
    for (int i = 0; i < N; ++i) Ai[(size_t)i * N + i] = 1.0;
    for (int k = 0; k < N; ++k) {
        int p = k;
        for (int i = k + 1; i < N; ++i) if (std::abs(A[(size_t)i * N + k]) > std::abs(A[(size_t)p * N + k])) p = i;
        if (p != k) for (int j = 0; j < N; ++j) { std::swap(A[(size_t)p * N + j], A[(size_t)k * N + j]); std::swap(Ai[(size_t)p * N + j], Ai[(size_t)k * N + j]); }
        const cd piv = 1.0 / A[(size_t)k * N + k];
        for (int j = 0; j < N; ++j) { A[(size_t)k * N + j] *= piv; Ai[(size_t)k * N + j] *= piv; }
        for (int i = 0; i < N; ++i) if (i != k) {
            const cd f = A[(size_t)i * N + k];
            if (f == cd(0)) continue;
            cd* ai = &A[(size_t)i * N]; const cd* ak = &A[(size_t)k * N];
            cd* bi = &Ai[(size_t)i * N]; const cd* bk = &Ai[(size_t)k * N];
            for (int j = k; j < N; ++j) ai[j] -= f * ak[j];
            for (int j = 0; j < N; ++j) bi[j] -= f * bk[j];
        }
    }
    double zmax = 0.0;
    for (auto& v : Ai) zmax = std::max(zmax, std::abs(v));
    // ---- every entry of every front's Z ----
    double err = 0.0, derr = 0.0;
    long long checked = 0;
    for (int k = 0; k < S.K; ++k) {
        const Front& F = S.fronts[k];
        const int fp = F.fp();
        auto orig = [&](int a) {      // original index of local row a, -1: padding
            if (a < F.sp) return a < F.s ? S.pos2orig[F.cbp + a] : -1;
            return a - F.sp < F.u ? S.pos2orig[S.rows[F.rowPtr + a - F.sp]] : -1;
        };
        for (int a = 0; a < fp; ++a) for (int b = 0; b < fp; ++b) {
            const cl v = Z[k][(size_t)a * fp + b];
            const int oa = orig(a), ob = orig(b);
            if (oa < 0 || ob < 0) {
                const cl want = (a == b && a >= F.s && a < F.sp) ? cl(1) : cl(0);
                if (v != want) { printf("front %d: padded entry (%d, %d) = (%Lg, %Lg)\n", k, a, b, v.real(), v.imag()); return 1; }
                continue;
            }
            const cd r = Ai[(size_t)oa * N + ob];
            err = std::max(err, (double)std::abs(v - cl(r.real(), r.imag())) / zmax);
            ++checked;
        }
    }
    for (int o = 0; o < N; ++o) {
        const cd r = Ai[(size_t)o * N + o];
        derr = std::max(derr, (double)std::abs(diag[o] - cl(r.real(), r.imag())) / zmax);
    }
    printf("entries of Z checked %lld  max |Z - inv(A)| / max|inv(A)| %.3e  diagonal %.3e\n", checked, err, derr);
    if (err > 1e-11 || derr > 1e-11) { printf("FAIL\n"); return 1; }
    printf("selected inversion matches the dense inverse\n");
    return 0;
}
