// Host side of the multifrontal solver: owns the symbolic tables on the device, the per-batch arenas and the launch
// schedule (depth by depth, deepest first).  Used by the Level-2 plan (hmcmt_b200.cu) for wide meshes and by the Level-1
// shim (mumps_shim.cu) for arbitrary symmetric matrices.
#pragma once
#include <cstdint>
#include <vector>

#include "common.cuh"
#include "mf_symbolic.h"

namespace hmcmt {
namespace mf {

// one MT stencil system: planes = [dr | dm | e1 | e2] (4 N doubles, internal ordering of mt_kernels.cuh), A = dr + i omega dm on
// the diagonal, e1 / e2 the in-line / cross-line couplings
struct MtValSys {
    const double* planes;
    double omega;
};

// Everything the single-CTA front kernel needs to know about a front, in one record (one global-memory round trip instead of
// the chain list -> front -> child ids -> child fronts): offsets in doubles into the per-system factor / depth-parity arenas.
constexpr int kDescChildren = kSmallChildren;      // fronts with more children take the global-memory path (mf_symbolic)
struct SmallDesc {
    int sp, up, s, nChild;
    int nOrig, origPtr, par, front;       // par: depth parity (arena that takes its update matrix); front: id in Symbolic::fronts
    int64_t gOff, mOff, uOff;
    int64_t cOff[kDescChildren];          // child update matrices (arena of the other parity)
    int cLd[kDescChildren], cFirst[kDescChildren], cU[kDescChildren], cRel[kDescChildren];   // ld, first row / column, real rows, rel offset
    unsigned char cPiv[kDescChildren];    // the child's rows that land in the pivot columns (a prefix: the rows are sorted)
};

// The same for the warp-per-front solve kernels (fronts of at most 64 rows, a single pivot chunk): offsets / counts of the front
// and of its children's update vectors in one 96-byte record.
constexpr int kDescRows = 40;                      // update-row indices carried inside the record (fronts of up to 48 rows)
struct SolveDesc {
    int sp, up, s, u;
    int cbp, rowPtr, updOff, nChild;
    int64_t gOff, mOff;                        // factor arena (doubles)
    int cRel[kDescChildren], cUpd[kDescChildren], cU[kDescChildren];      // children: row map offset, update vector offset, real rows
    int rows[kDescRows];                       // the first min(u, kDescRows) update rows (positions in the permuted numbering)
};

struct DepthSchedule {
    int nSmall = 0, smallWarps = 4;
    bool smallStream = false;                // M' streamed through the factor arena (mf_small_stream_kernel, 16 warps)
    size_t smallSmem = 0;
    const SmallDesc* smallDescs = nullptr;
    int nBig = 0;
    const int* bigList = nullptr;
    int nOrigPairs = 0;
    const int2* origPairs = nullptr;
    const void* asmTiles = nullptr;          // AsmTile[nAsmTiles]: 64 x 64 lower tiles of the large fronts (gather assembly)
    int nAsmTiles = 0;
    struct ChunkStep {
        const int* invList = nullptr;
        int nInv = 0;
        size_t invSmem = 0;
        const void* jobs = nullptr;          // GemmJob[2*nInv]: panel jobs then trailing-update jobs
        const void* panelTiles = nullptr;
        int nPanelTiles = 0;
        const void* schurTiles = nullptr;
        int nSchurTiles = 0;
    };
    std::vector<ChunkStep> chunkSteps;
    size_t bigBytes = 0;                     // leading part of the depth arena holding the large fronts
    const SolveDesc* solveWarpList = nullptr;      // solves: fronts handled one per warp (records) / one per CTA (front ids)
    const int* solveCtaList = nullptr;
    int nSolveWarp = 0, nSolveCta = 0;
    int solveCtaThreads = 256;               // threads per CTA of the CTA-per-front solve kernels at this depth
};

struct Tables;
struct SolveArgs;

class Solver {
  public:
    // S is consumed.  nsys systems are factorised together; up to maxRhs right-hand sides per system in one solve call;
    // valCount complex values per system (the sources referenced by the pattern entries).
    static Solver* create(Symbolic&& S, int nsys, int maxRhs, int64_t valCount, int* rc);
    ~Solver();
    cplx* vals() { return d_vals; }
    int64_t val_stride() const { return valCount; }
    const Symbolic& symbolic() const { return S; }
    // fills vals() of every system from its stencil planes (pattern of mf_grid_entries: [diag N | e1 N | e2 N])
    // Every call below covers the systems [sys0, sys0 + n) (n < 0: all from sys0); disjoint ranges may be in flight on different
    // streams at the same time (the per-system arenas, factors and workspaces do not overlap).
    int set_mt_values(cudaStream_t st, int N, const MtValSys* dSys, int sys0 = 0, int n = -1);
    // numeric factorisation from vals(); status: device array [nsys] (set to -10 on a singular pivot block)
    int factor(cudaStream_t st, int* dStatus, int64_t* nLaunches = nullptr, int sys0 = 0, int n = -1);
    // nrhs right-hand sides per system: vector (sys, r) at B + (sys*nrhs + r)*ldb, original numbering; X may alias B
    // (B and X are the bases of the whole batch; the range is applied inside).  Uses the workspace slots 0 .. nrhs-1.
    // pattern: 0 = dense right-hand sides, > 0 = an id returned by add_rhs_pattern (the rows outside it MUST be zero)
    int solve(cudaStream_t st, int nrhs, const cplx* B, int64_t ldb, cplx* X, int64_t ldx, int64_t* nLaunches = nullptr, int sys0 = 0,
              int n = -1, int pattern = 0);
    // The two phases of solve() for one vector per system in workspace slot `slot` (< maxRhs), so that two solves with the same
    // factors can be interleaved (B, X: vector sys at B + sys*ldb; sys0 / n / pattern as in solve()):
    //   forward_slot   : forward elimination (leaves the other slots alone);
    //   backward_slot  : backward substitution of the fronts of pattern's active set only — the fronts whose subtree holds a
    //                    row of the pattern: the unknowns of those rows and all their ancestors — writing X on their unknowns;
    //   backward_pair  : backward substitution of slot 0 into Xa and slot 1 into Xb in one pass over the factor, complete except
    //                    that on the fronts of `done`'s active set only slot 1 is solved: backward_slot(0, done) has already
    //                    overwritten their slot-0 pivot parts with the solution, which the sweep reads as its ancestors' values.
    int forward_slot(cudaStream_t st, int slot, const cplx* B, int64_t ldb, int64_t* nLaunches, int sys0, int n, int pattern);
    int backward_slot(cudaStream_t st, int slot, cplx* X, int64_t ldx, int64_t* nLaunches, int sys0, int n, int pattern);
    int backward_pair(cudaStream_t st, cplx* Xa, cplx* Xb, int64_t ldx, int64_t* nLaunches, int sys0, int n, int done);
    // Right-hand sides with a known sparsity pattern (nz[i] != 0: row i, original numbering, may be non-zero).  The forward
    // elimination then visits only the fronts whose subtree holds such a row — every other front would hand a zero update
    // vector to its parent — which prunes most of the tree when the sources sit on a few grid lines (MT right-hand sides:
    // the nodes next to the Dirichlet boundary, the two receiver rows of the adjoint sources).  The backward substitution of
    // solve() is always complete.  Returns the pattern id (> 0), or a negative error code.
    int add_rhs_pattern(const std::vector<unsigned char>& nz);
    // fronts visited by the forward elimination of a pattern (0: all), for diagnostics
    int fwd_fronts(int pattern) const;
    size_t device_bytes() const { return bytes; }
    double factor_flops() const { return S.flops; }
    int64_t factor_doubles() const { return S.factorDoubles; }

  private:
    Solver() = default;
    int build(int nsys, int maxRhs, int64_t valCount);
    template <typename Tp>
    int upload(const std::vector<Tp>& h, Tp** d);
    int upload_solve_descs(const std::vector<int>& fronts, const SolveDesc** d);
    Tables tables(int sys0) const;
    SolveArgs solve_args(const cplx* B, int64_t ldb, cplx* X, int64_t ldx, int sys0, int nrhs, int slot) const;
    int set_solve_attributes();
    int clear_ws(cudaStream_t st, const SolveArgs& sa, int nvec);
    int fwd_sweep(cudaStream_t st, const Tables& tb, const SolveArgs& sa, int nvec, int pattern, int64_t& nl);
    Symbolic S;
    int nsys = 0, maxRhs = 1;
    int64_t valCount = 0;
    size_t bytes = 0;
    std::vector<void*> owned;
    std::vector<DepthSchedule> sched;
    struct PatternLists {                        // launch lists of one right-hand-side pattern, per depth
        std::vector<const SolveDesc*> warpList;  // its active set: forward elimination, backward_slot
        std::vector<const int*> ctaList;
        std::vector<int> nWarp, nCta;
        int nFronts = 0;
        std::vector<const SolveDesc*> pairWarpList;   // backward_pair(done = this pattern): every front of the depth, those
        std::vector<const int*> pairCtaList;          // outside the active set first (both slots), then the active set (slot 1)
        std::vector<int> nPairWarpBoth, nPairCtaBoth;
    };
    std::vector<PatternLists> patterns;
    // device tables
    Front* d_fronts = nullptr;
    int *d_rows = nullptr, *d_rel = nullptr, *d_children = nullptr, *d_pos2orig = nullptr;
    OrigEntry* d_orig = nullptr;
    Chunk* d_chunks = nullptr;
    double* d_fac = nullptr;
    double* d_arena[2] = {nullptr, nullptr};
    cplx *d_vals = nullptr, *d_v = nullptr, *d_upd = nullptr;
    int* d_invMaps = nullptr;                  // inverse row maps (front row -> child row) of the large fronts
    size_t solveSmem = 0;
    size_t pairSmem = 0;                       // mf_bwd_pair_kernel: two vectors of the largest front and their chunk stages
    unsigned long long* d_prof = nullptr;      // HMCMT_MF_PROF=1: phase cycle counters of mf_small_kernel
};

}  // namespace mf
}  // namespace hmcmt
