// ps_part.hpp -- z-slab decomposition of one Stokes step over several GPUs (SURVEY.md section 8e).
//
// One process per GPU.  The grid is cut along z at multiples of lcm(16, tileSize): the reference numbers DOFs
// in UT_VoxelArray order (16^3 tiles, tile index z-slowest; exec/HDK_PolyStokesSolver_Classifier.cpp:1738-1770),
// so every rank owns ONE contiguous index range per sample slot, and reduced tiles (aligned to multiples of
// tileSize, S_Cls:736-738) never straddle a cut.  Classification and the (cheap, stencil) matrix fill are
// computed redundantly by every rank in the global numbering -- no setup communication, bit-identical to the
// single-GPU result -- while the per-region Gram builds, the operator rows and all CG vector work are
// restricted to the owned ranges.  Per CG iteration: one halo exchange of p, one of w, two scalar all-reduces.
#pragma once
#include "ps_grid.hpp"

namespace ps {

// up to 7 disjoint ascending ranges of a global index space, passed by value to kernels: local item l in
// [0, total) <-> global index.  Neighbouring threads map to neighbouring indices except at the <= 6 seams.
template <int N>
struct RangeSetN {
    int n = 0;
    int64_t lo[N] = {};
    int64_t pre[N + 1] = {};     // pre[k] = items before range k; pre[n] = total
    void add(int64_t a, int64_t b) {             // adjacent ranges are merged, empty ones dropped: one GPU => one range
        if (b <= a) return;
        if (n > 0 && lo[n - 1] + count(n - 1) == a) { pre[n] += b - a; return; }
        lo[n] = a; pre[n + 1] = pre[n] + (b - a); ++n;
    }
    PS_HD int64_t total() const { return pre[n]; }
    PS_HD int64_t count(int k) const { return pre[k + 1] - pre[k]; }
    PS_HD int64_t at(int64_t l) const {
        int64_t base = lo[0];
#pragma unroll
        for (int i = 1; i < N; ++i) if (i < n && l >= pre[i]) base = lo[i] - pre[i];
        return base + l;
    }
    PS_HD bool has(int64_t gidx) const {
        bool in = false;
#pragma unroll
        for (int i = 0; i < N; ++i) if (i < n && gidx >= lo[i] && gidx < lo[i] + (pre[i + 1] - pre[i])) in = true;
        return in;
    }
};
// Grid-stride walk over the concatenation of the ranges: thread t visits local items t, t+stride, ... so the work
// is balanced over the whole set (no per-range tail), and the common step is one add + one compare.
template <int N>
struct RangeWalk {
    int k; int64_t j, end;
    PS_HD RangeWalk(const RangeSetN<N>& s, int64_t l) {
        k = 0;
        while (k < s.n && l >= s.pre[k + 1]) ++k;
        if (k < s.n) { j = s.lo[k] + (l - s.pre[k]); end = s.lo[k] + s.count(k); } else { j = 0; end = 0; }
    }
    PS_HD bool valid(const RangeSetN<N>& s) const { return k < s.n; }
    PS_HD void step(const RangeSetN<N>& s, int64_t stride) {
        j += stride;
        while (j >= end) {
            const int64_t over = j - end;
            if (++k >= s.n) return;
            j = s.lo[k] + over; end = s.lo[k] + s.count(k);
        }
    }
};
typedef RangeSetN<7> RangeSet;    // the system vector: p | xx | yy | zz | yz | xz | xy
typedef RangeSetN<4> RowSet;      // operator rows: K_ext (x, y, z faces + coupled reduced rows) and the K_ext^T blocks
inline RowSet one_range(int64_t a, int64_t b) { RowSet r; r.add(a, b); return r; }

// host description of who owns what (identical on every rank: derived from the replicated classification)
struct Partition {
    int rank = 0, nranks = 1;
    std::vector<int> zCut;                              // [nranks+1]; rank k owns cells z in [zCut[k], zCut[k+1])
    std::vector<int64_t> slotCut[N_SLOTS];              // [nranks+1] active-index cut of every sample slot
    std::vector<int32_t> regionCut;                     // [nranks+1] region-id cut
    std::vector<int64_t> redRowCut;                     // [nranks+1] coupled-reduced-row cut (relative to nActiveVs)
    bool multi() const { return nranks > 1; }
    // Slab-local setup: every rank uploads, classifies, numbers and assembles only its slab plus `halo` cell layers; global DOF /
    // region / row numbers follow from an all-gather of the per-slab counts (the reference numbering is a scan in tile order, tiles
    // z-slowest, and a slab is a whole number of tile layers), the halo layers of the label / index fields come from the neighbour.
    // Needs regions that cannot interact across a cut: reduced regions off, or tiles with padding >= 2 (the boundary fix-up
    // S_Cls:1073-1172 never fires then).  Otherwise the setup is replicated on every rank as in round 1.
    bool local = false;
    int halo = 0;
    // Reduced regions that may cross a cut (doTile off, or tiles without padding): the setup is replicated, a region belongs to the
    // rank of its first cell (regions are numbered in voxel order, so regionCut stays monotone), and a region with reduced faces in
    // more than one slab is SHARED: its coupled rows follow the slab of the face (the convention of the active rows, slotCut), and
    // every operator apply sums its moments over the ranks (Solver::sharedApply).
    bool spanning = false;
};

}  // namespace ps
