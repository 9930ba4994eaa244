// ps_scan.cu -- DOF numbering primitives.
//
// tile_order_scan reproduces serialAssignFieldIndices (exec/HDK_PolyStokesSolver_Classifier.cpp:1738-1770):
// a running counter over the voxels for which a predicate holds, visited in UT_VoxelArray order
// (16^3 tiles, x->y->z, x fastest inside).  The reference does this serially; here one CTA owns one
// 16^3 tile: (1) per-tile counts, (2) one-CTA exclusive scan of the tile counts, (3) per-tile local
// scan + write.  A thread owns one z-column of its tile, so every slice is read and written as 16 rows of 16 contiguous voxels.
#include "ps_solver.hpp"
#ifndef PS_EMULATE
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#endif

namespace ps {

#ifndef PS_EMULATE

struct TileGeom { int rx, ry, rz, tx, ty, tz; };

// Thread t of a tile's CTA owns the voxel column (x0 + (t & 15), y0 + (t >> 4), z0 + 0..15): in every z-slice the 256 threads
// read 16 x 16 contiguous bytes and their thread order IS the voxel order of the slice (voxels beyond a ragged tile's
// width / height count as unset).  Returns the 16 slice flags of the column as a bit mask; base = voxel of slice 0.
__device__ __forceinline__ unsigned column_mask(const uint8_t* __restrict__ flag, const TileGeom& t, int tile, int tid, int64_t& base, int64_t& zStride, int& depth) {
    const int ti = tile % t.tx, tj = (tile / t.tx) % t.ty, tk = tile / (t.tx * t.ty);
    const int x = (ti << 4) + (tid & 15), y = (tj << 4) + (tid >> 4), z0 = tk << 4;
    zStride = (int64_t)t.rx * t.ry;
    depth = min(16, t.rz - z0);
    base = (int64_t)x + (int64_t)t.rx * ((int64_t)y + (int64_t)t.ry * z0);
    if (x >= t.rx || y >= t.ry) { depth = 0; return 0u; }
    unsigned m = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) if (k < depth && flag[base + k * zStride]) m |= 1u << k;
    return m;
}

// block-wide exclusive scan of one int per thread (256 threads), returns total in `total`
__device__ __forceinline__ int block_exclusive_scan_256(int v, int& total) {
    __shared__ int warpSums[8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
    if (lane == 31) warpSums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int s = lane < 8 ? warpSums[lane] : 0;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += n; }
        if (lane < 8) warpSums[lane] = s;
    }
    __syncthreads();
    total = warpSums[7];
    const int warpBase = wid == 0 ? 0 : warpSums[wid - 1];
    __syncthreads();
    return warpBase + inc - v;
}

__global__ void __launch_bounds__(256) tile_count_kernel(const uint8_t* __restrict__ flag, TileGeom t, int32_t* tileCounts, int tile0) {
    int64_t base, zStride; int depth;
    const int c = __popc(column_mask(flag, t, tile0 + blockIdx.x, threadIdx.x, base, zStride, depth));
    int total;
    block_exclusive_scan_256(c, total);
    if (threadIdx.x == 0) tileCounts[blockIdx.x] = total;
}

// single CTA: exclusive scan of nTiles counts in place; tileCounts[nTiles] = grand total
__global__ void __launch_bounds__(256) tile_offsets_kernel(int32_t* tileCounts, int nTiles) {
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < nTiles; base += 256) {
        const int i = base + threadIdx.x;
        const int v = i < nTiles ? tileCounts[i] : 0;
        int total;
        const int ex = block_exclusive_scan_256(v, total);
        const int c = carry;
        if (i < nTiles) tileCounts[i] = c + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) tileCounts[nTiles] = carry;
}

__global__ void __launch_bounds__(256) tile_write_kernel(const uint8_t* __restrict__ flag, TileGeom t, const int32_t* tileOffsets, int32_t* __restrict__ out, int tile0) {
    __shared__ int part[16 * 8 + 1];      // set voxels per (slice, warp), then their exclusive prefix in slice-major order
    int64_t base, zStride; int depth;
    const unsigned m = column_mask(flag, t, tile0 + blockIdx.x, threadIdx.x, base, zStride, depth);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const unsigned b = __ballot_sync(0xffffffffu, (m >> k) & 1u);
        if (lane == 0) part[k * 8 + wid] = __popc(b);
    }
    __syncthreads();
    if (wid == 0) {        // 128 entries: lane owns 4 consecutive ones
        int v[4], s = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[i] = part[4 * lane + i]; s += v[i]; }
        int inc = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
        int run = inc - s;
#pragma unroll
        for (int i = 0; i < 4; ++i) { part[4 * lane + i] = run; run += v[i]; }
    }
    __syncthreads();
    const int tileBase = tileOffsets[blockIdx.x];
    const unsigned below = (1u << lane) - 1u;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const unsigned b = __ballot_sync(0xffffffffu, (m >> k) & 1u);
        if (k < depth) out[base + k * zStride] = ((m >> k) & 1u) ? tileBase + part[k * 8 + wid] + __popc(b & below) : -1;
    }
}

int64_t tile_order_scan(cudaStream_t st, const Geom& g, int slot, const uint8_t* flag, int32_t* out, DBuf<int32_t>& tileCounts,
                        const std::vector<int>* zCut, std::vector<int64_t>* cuts, const int* tileZ) {
    TileGeom t;
    t.rx = g.r[slot][0]; t.ry = g.r[slot][1]; t.rz = g.r[slot][2];
    t.tx = (t.rx + 15) >> 4; t.ty = (t.ry + 15) >> 4; t.tz = (t.rz + 15) >> 4;
    const int tzA = tileZ ? std::max(0, std::min(tileZ[0], t.tz)) : 0, tzB = tileZ ? std::max(tzA, std::min(tileZ[1], t.tz)) : t.tz;
    const int tile0 = t.tx * t.ty * tzA, nTiles = t.tx * t.ty * (tzB - tzA);
    tileCounts.alloc((size_t)nTiles + 1);
    if (nTiles <= 0) return 0;
    tile_count_kernel<<<nTiles, 256, 0, st>>>(flag, t, tileCounts.p, tile0);
    PS_COUNT_LAUNCH(1);
    tile_offsets_kernel<<<1, 256, 0, st>>>(tileCounts.p, nTiles);
    PS_COUNT_LAUNCH(1);
    tile_write_kernel<<<nTiles, 256, 0, st>>>(flag, t, tileCounts.p, out, tile0);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
    if (zCut && cuts) {
        // tiles are visited z-slowest, so the rank of the first voxel of a z cut is the offset of the cut's first tile
        std::vector<int32_t> off = tileCounts.to_host(st, (size_t)nTiles + 1);
        const int nc = (int)zCut->size();
        cuts->assign((size_t)nc, 0);
        for (int k = 0; k < nc; ++k) {
            const int z = (*zCut)[k];
            const int64_t tile = (int64_t)std::max(0, (z >> 4) - tzA) * t.tx * t.ty;
            (*cuts)[k] = (k == nc - 1 || tile >= nTiles) ? off[nTiles] : off[tile];
        }
        (*cuts)[0] = 0;
        return off[nTiles];
    }
    int32_t total = 0;
    copy_d2h(&total, tileCounts.p + nTiles, sizeof(int32_t), st);
    return total;
}

// Per-CTA histogram in shared memory: the lanes of a warp that hit the same bin add once (rows of one region share their z), and every CTA
// adds its bins to the global counters once.
__global__ void __launch_bounds__(256) unit_counts_kernel(Geom g, int unit, int nUnits, const uint32_t* __restrict__ rowXYZ, int64_t rLo, int64_t nRows,
                                                          const int32_t* __restrict__ cellList, const int32_t* __restrict__ cellStart, int32_t regLo,
                                                          int64_t n, int* counts) {
    __shared__ int h[2 * MAX_UNITS];
    for (int i = threadIdx.x; i < 2 * nUnits; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < n; base += (int64_t)gridDim.x * blockDim.x) {      // uniform per warp
        const int64_t i = base + threadIdx.x;
        int bin = -1;
        if (i < nRows) bin = 2 * min((int)((rowXYZ[rLo + i] >> 20) & 1023u) / unit, nUnits - 1);
        else if (i < n) {
            const int32_t r = regLo + (int32_t)(i - nRows);
            if (cellStart[r + 1] > cellStart[r]) bin = 2 * min(delin(g, SL_CENTER, cellList[cellStart[r]]).z / unit, nUnits - 1) + 1;
        }
        const unsigned same = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && lane == __ffs(same) - 1) atomicAdd(&h[bin], __popc(same));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * nUnits; i += blockDim.x) if (h[i]) atomicAdd(&counts[i], h[i]);
}

void k_unit_counts(cudaStream_t st, const Geom& g, int unit, int nUnits, const uint32_t* rowXYZ, int64_t rLo, int64_t rHi,
                   const int32_t* cellList, const int32_t* cellStart, int32_t regLo, int32_t regHi, int* counts) {
    if (nUnits > MAX_UNITS) throw Error("k_unit_counts: more z-units than MAX_UNITS");
    const int64_t n = (rHi - rLo) + (regHi - regLo);
    if (n <= 0) return;
    const int64_t blocks = std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 4);
    unit_counts_kernel<<<(unsigned)blocks, 256, 0, st>>>(g, unit, nUnits, rowXYZ, rLo, rHi - rLo, cellList, cellStart, regLo, n, counts);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}

// ascending list of the indices i < n with flag[i] != 0, written to out[outOffset...]; returns the count
int64_t select_flagged(cudaStream_t st, int64_t n, const uint8_t* flag, DBuf<int32_t>& out, int64_t outOffset) {
    if (n <= 0) return 0;
    DBuf<uint8_t>& tmp = scratch().selTmp;
    DBuf<int32_t>& cnt = scratch().selCnt; DBuf<int32_t>& staging = scratch().selStaging;
    cnt.alloc(1); staging.alloc((size_t)n);
    cub::CountingInputIterator<int32_t> idx(0);
    size_t tmpBytes = 0;
    PS_CUDA(cub::DeviceSelect::Flagged(nullptr, tmpBytes, idx, flag, staging.p, cnt.p, (int)n, st));
    tmp.alloc(tmpBytes);
    PS_CUDA(cub::DeviceSelect::Flagged(tmp.p, tmpBytes, idx, flag, staging.p, cnt.p, (int)n, st));
    PS_COUNT_LAUNCH(1);
    int32_t c = 0;
    copy_d2h(&c, cnt.p, sizeof c, st);
    if (c > 0) {
        if (out.n < (size_t)(outOffset + c)) {      // grow, keeping what is already there
            DBuf<int32_t> bigger; bigger.alloc((size_t)(outOffset + c));
            if (outOffset > 0) copy_d2d(bigger.p, out.p, (size_t)outOffset * sizeof(int32_t), st);
            stream_sync(st);
            std::swap(out.p, bigger.p); std::swap(out.n, bigger.n);
        }
        copy_d2d(out.p + outOffset, staging.p, (size_t)c * sizeof(int32_t), st);
    }
    return c;
}

void sort_pairs_by_key(cudaStream_t st, int64_t n, int keyBits, DBuf<int32_t>& keys, DBuf<int32_t>& vals, DBuf<int32_t>& keysTmp, DBuf<int32_t>& valsTmp) {
    if (n <= 0) return;
    keysTmp.alloc((size_t)n); valsTmp.alloc((size_t)n);
    size_t tmpBytes = 0;
    PS_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmpBytes, keys.p, keysTmp.p, vals.p, valsTmp.p, (int)n, 0, keyBits, st));
    DBuf<uint8_t>& tmp = scratch().sortTmp;
    tmp.alloc(tmpBytes);
    PS_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmpBytes, keys.p, keysTmp.p, vals.p, valsTmp.p, (int)n, 0, keyBits, st));
    copy_d2d(keys.p, keysTmp.p, (size_t)n * sizeof(int32_t), st);
    copy_d2d(vals.p, valsTmp.p, (size_t)n * sizeof(int32_t), st);
}

int64_t exclusive_scan_i64(cudaStream_t st, int64_t n, const int64_t* in, int64_t* out) {
    if (n <= 0) return 0;
    size_t tmpBytes = 0;
    PS_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, in, out, (int)n, st));
    DBuf<uint8_t>& tmp = scratch().scanTmp;
    tmp.alloc(tmpBytes);
    PS_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, in, out, (int)n, st));
    int64_t last[2] = {0, 0};
    copy_d2h(&last[0], out + (n - 1), sizeof(int64_t), st);
    copy_d2h(&last[1], in + (n - 1), sizeof(int64_t), st);
    return last[0] + last[1];
}

#else  // ---- PS_EMULATE: serial twins (test-only build) ----

int64_t exclusive_scan_i64(cudaStream_t, int64_t n, const int64_t* in, int64_t* out) {
    int64_t s = 0;
    for (int64_t i = 0; i < n; ++i) { const int64_t v = in[i]; out[i] = s; s += v; }
    return s;
}

int64_t tile_order_scan(cudaStream_t, const Geom& g, int slot, const uint8_t* flag, int32_t* out, DBuf<int32_t>&,
                        const std::vector<int>* zCut, std::vector<int64_t>* cuts, const int* tileZ) {
    const int rx = g.r[slot][0], ry = g.r[slot][1], rz = g.r[slot][2];
    int32_t n = 0;
    const int zA = tileZ ? std::max(0, tileZ[0] * 16) : 0, zB = tileZ ? std::min(rz, tileZ[1] * 16) : rz;
    if (zCut && cuts) { cuts->assign(zCut->size(), -1); for (size_t k = 0; k < zCut->size(); ++k) if ((*zCut)[k] < zA) (*cuts)[k] = 0; }
    for (int tk = zA; tk < zB; tk += 16) for (int tj = 0; tj < ry; tj += 16) for (int ti = 0; ti < rx; ti += 16) {
        if (zCut && cuts && tj == 0 && ti == 0) for (size_t k = 0; k < zCut->size(); ++k) if ((*zCut)[k] == tk) (*cuts)[k] = n;
        for (int k = tk; k < std::min(tk + 16, rz); ++k) for (int j = tj; j < std::min(tj + 16, ry); ++j) for (int i = ti; i < std::min(ti + 16, rx); ++i) {
            const int64_t q = (int64_t)i + (int64_t)rx * ((int64_t)j + (int64_t)ry * k);
            out[q] = flag[q] ? n++ : -1;
        }
    }
    if (zCut && cuts) { for (size_t k = 0; k < cuts->size(); ++k) if ((*cuts)[k] < 0 || k + 1 == cuts->size()) (*cuts)[k] = n; (*cuts)[0] = 0; }
    return n;
}

void k_unit_counts(cudaStream_t, const Geom& g, int unit, int nUnits, const uint32_t* rowXYZ, int64_t rLo, int64_t rHi,
                   const int32_t* cellList, const int32_t* cellStart, int32_t regLo, int32_t regHi, int* counts) {
    if (nUnits > MAX_UNITS) throw Error("k_unit_counts: more z-units than MAX_UNITS");
    for (int64_t i = rLo; i < rHi; ++i) ++counts[2 * std::min((int)((rowXYZ[i] >> 20) & 1023u) / unit, nUnits - 1)];
    for (int32_t r = regLo; r < regHi; ++r)
        if (cellStart[r + 1] > cellStart[r]) ++counts[2 * std::min(delin(g, SL_CENTER, cellList[cellStart[r]]).z / unit, nUnits - 1) + 1];
}

int64_t select_flagged(cudaStream_t, int64_t n, const uint8_t* flag, DBuf<int32_t>& out, int64_t outOffset) {
    std::vector<int32_t> keep;
    if (outOffset > 0) keep.assign(out.p, out.p + outOffset);
    for (int64_t i = 0; i < n; ++i) if (flag[i]) keep.push_back((int32_t)i);
    const int64_t c = (int64_t)keep.size() - outOffset;
    if (out.n < keep.size()) { DBuf<int32_t> bigger; bigger.alloc(keep.size()); std::swap(out.p, bigger.p); std::swap(out.n, bigger.n); }
    std::copy(keep.begin(), keep.end(), out.p);
    return c;
}

void sort_pairs_by_key(cudaStream_t, int64_t n, int, DBuf<int32_t>& keys, DBuf<int32_t>& vals, DBuf<int32_t>&, DBuf<int32_t>&) {
    std::vector<int64_t> ord((size_t)n);
    for (int64_t i = 0; i < n; ++i) ord[i] = i;
    std::stable_sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) { return keys.p[a] < keys.p[b]; });
    std::vector<int32_t> k2((size_t)n), v2((size_t)n);
    for (int64_t i = 0; i < n; ++i) { k2[i] = keys.p[ord[i]]; v2[i] = vals.p[ord[i]]; }
    std::copy(k2.begin(), k2.end(), keys.p); std::copy(v2.begin(), v2.end(), vals.p);
}

#endif

}  // namespace ps
