// CPU check of the assembly of the mid-size fronts (mf_small_kernel<8> / <16>, mf_kernels.cuh) on the tables of mf_symbolic.h.
// Those kernels keep only the pivot columns of a front in shared memory: the extend-add scatters the columns of every child
// that land in the pivot columns, and the Schur product gathers F22 from the children through inverse row maps.  For every
// front of the single-CTA path with children, checks that
//   - the rows of a child that land in the pivot columns (rel < sp) are a prefix of its rows, of the length the host puts in
//     the front's record (SmallDesc::cPiv, computed here the same way);
//   - the scatter work items restricted to that prefix (column groups of four, the straddling group masked) visit every child
//     entry in the pivot columns exactly once and nothing else;
//   - the inverse row maps (front update row -> child row) reach every child entry of the update x update block exactly once;
//   - F22 formed by the gather (each element from +0.0, children in child order) equals F22 formed by the scatter into a zeroed
//     block, bit for bit, on child values that include signed zeros;
//   - mf_mid_front_smem_bytes never exceeds mf_front_smem_bytes, and the classification does not depend on it.
// Test infrastructure only.
//   usage: mf_mid_gather_check grid <nl> <nf> <leaf> <fSmall> [cross] [push]  |  mf_mid_gather_check graph3d <nx> <ny> <nz> <leaf> <fSmall>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>

#include "../../hmcmt2d_b200/csrc/mf_symbolic.h"

using namespace hmcmt::mf;

int main(int argc, char** argv) {
    if (argc < 6) return 2;
    std::vector<Entry> ent;
    std::vector<std::vector<int>> sn;
    int N = 0, fSmall = 144;
    if (!strcmp(argv[1], "grid")) {
        const int nl = atoi(argv[2]), nf = atoi(argv[3]), leaf = atoi(argv[4]);
        fSmall = atoi(argv[5]);
        N = nl * nf;
        mf_grid_entries(nl, nf, ent);
        mf_order_grid(nl, nf, leaf, sn, argc > 6 ? atoi(argv[6]) : 0, argc > 7 ? atoi(argv[7]) : 0);
    } else {
        if (argc < 7) return 2;
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
        std::vector<int> ptr(N + 1, 0), adj;
        for (const Entry& e : ent) if (e.row != e.col) { ++ptr[e.row + 1]; ++ptr[e.col + 1]; }
        for (int i = 0; i < N; ++i) ptr[i + 1] += ptr[i];
        adj.resize(ptr[N]);
        std::vector<int> fill(ptr.begin(), ptr.end() - 1);
        for (const Entry& e : ent) if (e.row != e.col) { adj[fill[e.row]++] = e.col; adj[fill[e.col]++] = e.row; }
        mf_order_graph(N, ptr, adj, leaf, sn);
    }
    Symbolic S;
    if (!mf_symbolic(N, sn, ent, fSmall, S)) { printf("symbolic failed\n"); return 1; }

    std::mt19937_64 rng(5);
    std::uniform_real_distribution<double> un(-1.0, 1.0);
    auto value = [&]() {      // a quarter signed zeros: +0.0 + (-0.0) and friends must come out as the scatter forms them
        const int r = (int)(rng() % 8);
        return r == 0 ? 0.0 : (r == 1 ? -0.0 : un(rng));
    };
    int checked = 0, maxChild = 0, bad = 0;
    long long f22Entries = 0, pivEntries = 0;
    for (int k = 0; k < S.K; ++k) {
        const Front& F = S.fronts[k];
        if (F.isBig || F.nChild == 0) continue;
        const int sp = F.sp, up = F.up, fp = F.fp(), nb = fp / 8, npb = sp / 8;
        if (mf_mid_front_smem_bytes(nb, npb, mf_rel_total(S, k), F.nChild) > mf_front_smem_bytes(nb, npb, mf_rel_total(S, k))) {
            printf("front %d: mid layout larger than the full one\n", k);
            ++bad;
        }
        ++checked;
        maxChild = std::max(maxChild, F.nChild);
        // F22 of the front, lower triangle (a >= b), update-local indices; scatter order and gather order
        std::vector<double> scat((size_t)up * up, 0.0), gath((size_t)up * up, 0.0);
        std::vector<std::vector<int>> inv(F.nChild, std::vector<int>(up, -1));
        std::vector<std::vector<double>> Uc(F.nChild);
        for (int c = 0; c < F.nChild; ++c) {
            const Front& C = S.fronts[S.children[F.childPtr + c]];
            const int* rel = S.rel.data() + C.rowPtr;
            const int cu = C.u;
            int piv = 0;      // SmallDesc::cPiv as the host computes it
            while (piv < cu && rel[piv] < sp) ++piv;
            for (int i = 0; i < cu; ++i)
                if ((rel[i] < sp) != (i < piv)) { printf("front %d child %d: pivot-column rows are not a prefix\n", k, c); ++bad; break; }
            // scatter work items of the pivot columns: (column group jg < ceil(piv / 4), row i >= 4 jg), column masked below piv
            std::vector<int> hit((size_t)cu * cu, 0);
            for (int jg = 0; jg < (piv + 3) / 4; ++jg)
                for (int i = 4 * jg; i < cu; ++i)
                    for (int jj = 0; jj < 4; ++jj) {
                        const int j = 4 * jg + jj;
                        if (j > i || j >= piv) break;
                        ++hit[(size_t)i * cu + j];
                    }
            for (int i = 0; i < cu; ++i)
                for (int j = 0; j <= i; ++j) {
                    const int want = rel[j] < sp ? 1 : 0;
                    if (hit[(size_t)i * cu + j] != want) { printf("front %d child %d: entry (%d,%d) scattered %d times\n", k, c, i, j, hit[(size_t)i * cu + j]); ++bad; }
                    pivEntries += want;
                }
            // the child's update matrix (lower triangle used), and the scatter of its update x update part into F22
            Uc[c].resize((size_t)cu * cu);
            for (double& v : Uc[c]) v = value();
            for (int i = piv; i < cu; ++i)
                for (int j = piv; j <= i; ++j) scat[(size_t)(rel[i] - sp) * up + rel[j] - sp] += Uc[c][(size_t)i * cu + j];
            for (int i = piv; i < cu; ++i) inv[c][rel[i] - sp] = i;
        }
        // gather: every lower element of F22 (the upper half of a diagonal tile stays +0.0), children in order
        std::vector<std::vector<int>> reached(F.nChild);
        for (int c = 0; c < F.nChild; ++c) reached[c].assign((size_t)S.fronts[S.children[F.childPtr + c]].u * S.fronts[S.children[F.childPtr + c]].u, 0);
        for (int a = 0; a < up; ++a)
            for (int b = 0; b <= a; ++b) {
                double v = 0.0;
                for (int c = 0; c < F.nChild; ++c) {
                    const int ia = inv[c][a], ib = inv[c][b];
                    if (ia < 0 || ib < 0 || ib > ia) continue;
                    const int cu = S.fronts[S.children[F.childPtr + c]].u;
                    v += Uc[c][(size_t)ia * cu + ib];
                    ++reached[c][(size_t)ia * cu + ib];
                }
                gath[(size_t)a * up + b] = v;
            }
        for (int c = 0; c < F.nChild; ++c) {
            const Front& C = S.fronts[S.children[F.childPtr + c]];
            const int* rel = S.rel.data() + C.rowPtr;
            for (int i = 0; i < C.u; ++i)
                for (int j = 0; j <= i; ++j) {
                    const int want = rel[j] >= sp ? 1 : 0;
                    if (reached[c][(size_t)i * C.u + j] != want) { printf("front %d child %d: entry (%d,%d) gathered %d times\n", k, c, i, j, reached[c][(size_t)i * C.u + j]); ++bad; }
                    f22Entries += want;
                }
        }
        if (memcmp(scat.data(), gath.data(), scat.size() * sizeof(double)) != 0) { printf("front %d: gathered F22 differs from the scattered one\n", k); ++bad; }
        if (bad > 20) break;
    }
    if (bad) { printf("%d failures\n", bad); return 1; }
    printf("%d fronts (up to %d children): %lld pivot-column and %lld update entries of the children, gather bit-identical to the scatter\n",
           checked, maxChild, pivEntries, f22Entries);
    return 0;
}
