// ps_classify.cu -- Classifier kernels (SURVEY.md section 8a rows C1-C12, K1-K8, K16) and the
// integration-weight kernel (8f rank 1).  Every kernel is a memory-bound voxel sweep: one thread
// per voxel, x-fastest so a warp reads 32 consecutive voxels.
//
// Reference behaviour being reproduced bit-exactly: exec/HDK_PolyStokesSolver_Classifier.cpp and
// exec/HDK_PolyStokesSolver.cpp:238-326 (weights); the HDK pieces are the shim of BASELINE.md 3.
#include "ps_solver.hpp"

namespace ps {

// every sweep visits the rank's window of the grid only (Geom::wzLo / wzHi; the whole grid on one GPU): voxel indices stay global
template <class F>
static inline void for_window(cudaStream_t st, const Geom& g, int slot, F f, int margin = 0) {
    int64_t lo, hi;
    z_range(g, slot, g.wzLo - margin, g.wzHi + margin, lo, hi);
    ps_for_range(st, lo, hi, f);
}

// ---------------------------------------------------------------------------------------------
// Integration weights.  HDK computeSDFWeightsSampled(sdf, 2, false, 0) (call sites
// exec/HDK_PolyStokesSolver.cpp:304, 322-323) -- shim: 2x2x2 sub-samples at +-dx/4, trilinear SDF
// evaluated in double (all products exact), liquid counts sdf < 0, fluid counts collision >= 0.
// One thread per sample computes BOTH weights of its slot (the 8 sub-sample stencils are shared).
// ---------------------------------------------------------------------------------------------
void k_build_weights(cudaStream_t st, const Geom& g, const Fields& F, uint8_t* signX, uint8_t* signBox) {
    // Pre-pass: signBox[c] = OR over the (clamped) 3x3x3 cell block around c of {1: surface < 0, 2: surface >= 0,
    // 4: collision < 0, 8: collision >= 0}, separably (x taps from the SDFs, then the 3x3 y/z taps of the x result).
    // Every slot's sub-sample stencil at index c lies inside that block (base cells c-1..c per axis, +1 for the upper
    // trilinear corner; an index one past the centre range clamps into the block of the last cell), so where the block
    // has one sign the eighth-counts are 0 or 8 without touching the SDFs again; the exact per-slot test below only
    // runs near the interfaces.  A NaN sets both bits of its field: a sub-sample whose interpolation meets a NaN is
    // NaN, and counts as neither liquid nor fluid, which only the exact test gets right.
    {
        const float* surf = F.surface; const float* coll = F.collision;
        for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
            const I3 c = delin(g, SL_CENTER, q);
            int code = 0;
            for (int d = -1; d <= 1; ++d) {
                const int64_t l = lin(g, SL_CENTER, clamped(g, SL_CENTER, I3{c.x + d, c.y, c.z}));
                const float sv = surf[l], cv = coll[l];
                code |= (sv < 0.f ? 1 : 0) | (sv >= 0.f ? 2 : 0) | (cv < 0.f ? 4 : 0) | (cv >= 0.f ? 8 : 0)
                      | (sv != sv ? 3 : 0) | (cv != cv ? 12 : 0);
            }
            signX[q] = (uint8_t)code;
        }, 1);
        for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
            const I3 c = delin(g, SL_CENTER, q);
            int code = 0;
            for (int dz = -1; dz <= 1; ++dz) for (int dy = -1; dy <= 1; ++dy)
                code |= signX[lin(g, SL_CENTER, clamped(g, SL_CENTER, I3{c.x, c.y + dy, c.z + dz}))];
            signBox[q] = (uint8_t)code;
        });
    }
    for (int slot = 0; slot < N_SLOTS; ++slot) {
        int off2[3] = {1, 1, 1};   // 2 * SamplingOffset (exec/HDK_PolyStokesSolver.h:193-222)
        if (slot >= SL_FACE && slot < SL_EDGE) off2[slot - SL_FACE] = 0;
        else if (slot >= SL_EDGE) { for (int a = 0; a < 3; ++a) if (a != slot - SL_EDGE) off2[a] = 0; }
        const int o0 = off2[0], o1 = off2[1], o2 = off2[2];
        const float* surf = F.surface; const float* coll = F.collision;
        uint8_t* lw = F.liqW[slot]; uint8_t* fw = F.fluW[slot];
        for_window(st, g, slot, PS_LAMBDA(int64_t q) {
            const I3 c = delin(g, slot, q);
            {
                const int box = signBox[lin(g, SL_CENTER, clamped(g, SL_CENTER, c))];
                if ((box & 3) != 3 && (box & 12) != 12) {      // one sign each, no NaN
                    lw[q] = (uint8_t)((box & 3) != 2 ? 8 : 0); fw[q] = (uint8_t)((box & 12) != 4 ? 8 : 0);
                    return;
                }
            }
            const int idx[3] = {c.x, c.y, c.z};
            const int o[3] = {o0, o1, o2};
            // per axis: two sub-sample positions -> base cell and fraction (1/4 or 3/4)
            int base[3][2]; double fr[3][2];
            for (int a = 0; a < 3; ++a)
                for (int s = 0; s < 2; ++s) {
                    const int qq = 4 * idx[a] + 2 * o[a] - 2 + (s ? 1 : -1);
                    const int fl = (qq >= 0) ? (qq >> 2) : -((-qq + 3) >> 2);
                    base[a][s] = fl; fr[a][s] = (double)(qq - 4 * fl) * 0.25;
                }
            // Every sub-sample is a convex combination (all 8 trilinear weights are positive: fractions are 1/4 or 3/4)
            // of the SDF values in the <= 3x3x3 cell block below, so away from the interfaces the count is decided
            // by the signs alone -- exactly, rounding included -- and the fp64 interpolation is skipped.  fminf / fmaxf
            // skip a NaN, so a NaN in the block forces the exact test.
            float minS = 3.4e38f, maxS = -3.4e38f, minC = 3.4e38f, maxC = -3.4e38f;
            bool nanS = false, nanC = false;
            {
                int lo[3], hi[3];
                for (int a = 0; a < 3; ++a) { lo[a] = min(base[a][0], base[a][1]); hi[a] = max(base[a][0], base[a][1]) + 1; }
                for (int z = lo[2]; z <= hi[2]; ++z) for (int y = lo[1]; y <= hi[1]; ++y) for (int x = lo[0]; x <= hi[0]; ++x) {
                    const int64_t l = lin(g, SL_CENTER, clamped(g, SL_CENTER, I3{x, y, z}));
                    const float sv = surf[l], cv = coll[l];
                    minS = fminf(minS, sv); maxS = fmaxf(maxS, sv); minC = fminf(minC, cv); maxC = fmaxf(maxC, cv);
                    nanS |= sv != sv; nanC |= cv != cv;
                }
            }
            const bool needL = nanS || !(minS >= 0.f || maxS < 0.f), needF = nanC || !(minC >= 0.f || maxC < 0.f);
            int nl = (maxS < 0.f) ? 8 : 0, nf = (minC >= 0.f) ? 8 : 0;
            if (needL || needF) {
                int cl = 0, cf = 0;
                for (int sz = 0; sz < 2; ++sz) for (int sy = 0; sy < 2; ++sy) for (int sx = 0; sx < 2; ++sx) {
                    double accL = 0.0, accF = 0.0;
                    for (int dz = 0; dz < 2; ++dz) for (int dy = 0; dy < 2; ++dy) for (int dxx = 0; dxx < 2; ++dxx) {
                        const double w = mul_rn(mul_rn(dxx ? fr[0][sx] : 1.0 - fr[0][sx], dy ? fr[1][sy] : 1.0 - fr[1][sy]), dz ? fr[2][sz] : 1.0 - fr[2][sz]);
                        const I3 cc = clamped(g, SL_CENTER, I3{base[0][sx] + dxx, base[1][sy] + dy, base[2][sz] + dz});
                        const int64_t l = lin(g, SL_CENTER, cc);
                        accL = add_rn(accL, mul_rn(w, (double)surf[l]));
                        accF = add_rn(accF, mul_rn(w, (double)coll[l]));
                    }
                    cl += (accL < 0.0); cf += (accF >= 0.0);
                }
                if (needL) nl = cl;
                if (needF) nf = cf;
            }
            lw[q] = (uint8_t)nl; fw[q] = (uint8_t)nf;
        });
    }
}

// C1 classifyCells (S_Cls:56-128), fused with the GENERICFLUID -> ACTIVEFLUID overwrite of
// constructOnlyActiveRegions (S_Cls:192-199) when reduced regions are off.
void k_classify_cells(cudaStream_t st, const Geom& g, const Fields& F, bool genericToActive) {
    int8_t* L = F.label[SL_CENTER];
    const uint8_t* clw = F.liqW[SL_CENTER]; const uint8_t* cfw = F.fluW[SL_CENTER];
    const uint8_t* fx = F.liqW[SL_FACE + 0]; const uint8_t* fy = F.liqW[SL_FACE + 1]; const uint8_t* fz = F.liqW[SL_FACE + 2];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        const I3 c = delin(g, SL_CENTER, q);
        bool inSolve = clw[q] > 0;
        if (!inSolve) {
            inSolve = fx[lin(g, SL_FACE + 0, c)] > 0 || fx[lin(g, SL_FACE + 0, shifted(c, 0, 1))] > 0
                   || fy[lin(g, SL_FACE + 1, c)] > 0 || fy[lin(g, SL_FACE + 1, shifted(c, 1, 1))] > 0
                   || fz[lin(g, SL_FACE + 2, c)] > 0 || fz[lin(g, SL_FACE + 2, shifted(c, 2, 1))] > 0;
        }
        const bool inFluid = cfw[q] != 0;
        int8_t lab = L_UNSOLVED;
        if (inSolve) lab = inFluid ? (genericToActive ? L_ACTIVEFLUID : L_GENERICFLUID) : L_SOLID;
        L[q] = lab;
    });
}

// C2 constructAirBoundaryLayer (S_Cls:291-508).  The reference grows frontier lists; on the GPU the
// flood is a sequence of full-grid dilation sweeps.  stamp[q] = layer+1 marks the sweep in which a
// cell was activated, so a sweep only expands from cells of the previous sweep (no in-place hazard).
void k_air_layer_seed(cudaStream_t st, const Geom& g, const Fields& F, uint8_t* stamp) {
    int8_t* L = F.label[SL_CENTER];
    const uint8_t* fw0 = F.liqW[SL_FACE + 0]; const uint8_t* fw1 = F.liqW[SL_FACE + 1]; const uint8_t* fw2 = F.liqW[SL_FACE + 2];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        stamp[q] = 0;
        if (L[q] != L_GENERICFLUID) return;
        const I3 c = delin(g, SL_CENTER, q);
        bool boundary = false;
        for (int axis = 0; axis < 3; ++axis)
            for (int dir = 0; dir < 2; ++dir) {
                const I3 adj = shifted(c, axis, dir ? 1 : -1);
                if (!in_bounds(g, SL_CENTER, adj)) continue;
                const I3 face = dir ? shifted(c, axis, 1) : c;
                // neighbour labels other than UNSOLVED are never changed by this sweep, so reading L in place is safe
                if (L[lin(g, SL_CENTER, adj)] == L_UNSOLVED) boundary = true;
                const uint8_t* fw = axis == 0 ? fw0 : axis == 1 ? fw1 : fw2;
                if (fw[lin(g, SL_FACE + axis, face)] < 8) boundary = true;
            }
        if (boundary) stamp[q] = 1;
    });
}
// marks stamped cells of `layer` ACTIVE (setActiveLayerCells, S.cpp:2022-2060)
void k_layer_commit(cudaStream_t st, const Geom& g, const Fields& F, const uint8_t* stamp, int layerStamp) {
    int8_t* L = F.label[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) { if (stamp[q] == layerStamp) L[q] = L_ACTIVEFLUID; });
}
// buildNextLiquidBoundaryLayer (S_Cls:432-508): GENERICFLUID neighbours of the previous layer through
// faces with liquid weight > 0
void k_air_layer_grow(cudaStream_t st, const Geom& g, const Fields& F, uint8_t* stamp, int prevStamp) {
    const int8_t* L = F.label[SL_CENTER];
    const uint8_t* fw0 = F.liqW[SL_FACE + 0]; const uint8_t* fw1 = F.liqW[SL_FACE + 1]; const uint8_t* fw2 = F.liqW[SL_FACE + 2];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        if (L[q] != L_GENERICFLUID || stamp[q] != 0) return;
        const I3 c = delin(g, SL_CENTER, q);
        bool hit = false;
        for (int axis = 0; axis < 3; ++axis)
            for (int dir = 0; dir < 2; ++dir) {
                const I3 adj = shifted(c, axis, dir ? 1 : -1);
                if (!in_bounds(g, SL_CENTER, adj)) continue;
                if (stamp[lin(g, SL_CENTER, adj)] != prevStamp) continue;
                const I3 face = dir ? shifted(c, axis, 1) : c;
                const uint8_t* fw = axis == 0 ? fw0 : axis == 1 ? fw1 : fw2;
                if (fw[lin(g, SL_FACE + axis, face)] > 0) hit = true;
            }
        if (hit) stamp[q] = (uint8_t)(prevStamp + 1);
    });
}

// C3 constructSolidBoundaryLayer (S_Cls:510-703): seeds = GENERIC/ACTIVE cells next to a SOLID cell
// or to the domain wall; then S-1 growth sweeps through liquid faces into unvisited GENERIC/ACTIVE cells.
void k_solid_layer_seed(cudaStream_t st, const Geom& g, const Fields& F, uint8_t* stamp) {
    const int8_t* L = F.label[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        stamp[q] = 0;
        const int lab = L[q];
        if (lab != L_GENERICFLUID && lab != L_ACTIVEFLUID) return;
        const I3 c = delin(g, SL_CENTER, q);
        bool boundary = false;
        for (int axis = 0; axis < 3; ++axis)
            for (int dir = 0; dir < 2; ++dir) {
                const I3 adj = shifted(c, axis, dir ? 1 : -1);
                if (!in_bounds(g, SL_CENTER, adj)) { boundary = true; continue; }
                if (L[lin(g, SL_CENTER, adj)] == L_SOLID) boundary = true;
            }
        if (boundary) stamp[q] = 1;
    });
}
void k_solid_layer_grow(cudaStream_t st, const Geom& g, const Fields& F, uint8_t* stamp, int prevStamp) {
    const int8_t* L = F.label[SL_CENTER];
    const uint8_t* fw0 = F.liqW[SL_FACE + 0]; const uint8_t* fw1 = F.liqW[SL_FACE + 1]; const uint8_t* fw2 = F.liqW[SL_FACE + 2];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        const int lab = L[q];
        if ((lab != L_GENERICFLUID && lab != L_ACTIVEFLUID) || stamp[q] != 0) return;   // stamp != 0 <=> VISITED
        const I3 c = delin(g, SL_CENTER, q);
        bool hit = false;
        for (int axis = 0; axis < 3; ++axis)
            for (int dir = 0; dir < 2; ++dir) {
                const I3 adj = shifted(c, axis, dir ? 1 : -1);
                if (!in_bounds(g, SL_CENTER, adj)) continue;
                if (stamp[lin(g, SL_CENTER, adj)] != prevStamp) continue;
                const I3 face = dir ? shifted(c, axis, 1) : c;
                const uint8_t* fw = axis == 0 ? fw0 : axis == 1 ? fw1 : fw2;
                if (fw[lin(g, SL_FACE + axis, face)] > 0) hit = true;
            }
        if (hit) stamp[q] = (uint8_t)(prevStamp + 1);
    });
}

// C4 constructTiles (S_Cls:705-746) fused with the final GENERICFLUID -> REDUCED overwrite (S_Cls:189)
void k_tiles_and_reduce(cudaStream_t st, const Geom& g, const Fields& F, bool doTile, int tileSize, int tilePadding) {
    int8_t* L = F.label[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        if (L[q] != L_GENERICFLUID) return;
        const I3 c = delin(g, SL_CENTER, q);
        bool pad = false;
        if (doTile) pad = (c.x % tileSize) < tilePadding || (c.y % tileSize) < tilePadding || (c.z % tileSize) < tilePadding;
        L[q] = pad ? L_ACTIVEFLUID : L_REDUCED;
    });
}

// C8 classifyFaces -> findFaceLabelFromCenter (S_Cls:784-832)
void k_classify_faces(cudaStream_t st, const Geom& g, const Fields& F) {
    for (int axis = 0; axis < 3; ++axis) {
        int8_t* FL = F.label[SL_FACE + axis];
        const uint8_t* clw = F.liqW[SL_CENTER];
        const uint8_t* ffw = F.fluW[SL_FACE + axis];
        const int e1 = (axis + 1) % 3, e2 = (axis + 2) % 3;
        const uint8_t* ew1 = F.liqW[SL_EDGE + e1]; const uint8_t* ew2 = F.liqW[SL_EDGE + e2];
        for_window(st, g, SL_FACE + axis, PS_LAMBDA(int64_t q) {
            const I3 f = delin(g, SL_FACE + axis, q);
            bool activeVel = false;
            const I3 c0 = shifted(f, axis, -1);
            if (in_bounds(g, SL_CENTER, c0) && clw[lin(g, SL_CENTER, c0)] > 0) activeVel = true;
            if (in_bounds(g, SL_CENTER, f) && clw[lin(g, SL_CENTER, f)] > 0) activeVel = true;
            if (!activeVel) {
                // faceToEdgeMap(face, axis, edgeAxis, dir): +dir on axis 3-axis-edgeAxis (always in bounds)
                const int o1 = 3 - axis - e1, o2 = 3 - axis - e2;
                activeVel = ew1[lin(g, SL_EDGE + e1, f)] > 0 || ew1[lin(g, SL_EDGE + e1, shifted(f, o1, 1))] > 0
                         || ew2[lin(g, SL_EDGE + e2, f)] > 0 || ew2[lin(g, SL_EDGE + e2, shifted(f, o2, 1))] > 0;
            }
            int8_t lab = L_UNSOLVED;
            if (activeVel) lab = (ffw[q] < 4) ? L_SOLID : L_GENERICFLUID;     // faceFluidW < 0.5
            FL[q] = lab;
        });
    }
}

// C9 classifyEdges -> findEdgeLabelFromFaceAlt (S_Cls:1021-1067)
void k_classify_edges(cudaStream_t st, const Geom& g, const Fields& F) {
    for (int e = 0; e < 3; ++e) {
        int8_t* EL = F.label[SL_EDGE + e];
        const uint8_t* elw = F.liqW[SL_EDGE + e]; const uint8_t* efw = F.fluW[SL_EDGE + e];
        const int fa0 = (e == 0) ? 1 : 0, fa1 = (e == 2) ? 1 : 2;   // XY->(X,Y)  XZ->(X,Z)  YZ->(Y,Z)
        const uint8_t* w0 = F.liqW[SL_FACE + fa0]; const uint8_t* w1 = F.liqW[SL_FACE + fa1];
        for_window(st, g, SL_EDGE + e, PS_LAMBDA(int64_t q) {
            const I3 ed = delin(g, SL_EDGE + e, q);
            bool in = elw[q] != 0 && efw[q] != 0;
            if (in) {
                // face(i,j,k) [clamped read, as the reference reads it unguarded] && !oob(back) && face(back)
                const I3 b0 = shifted(ed, 3 - fa0 - e, -1), b1 = shifted(ed, 3 - fa1 - e, -1);
                in = weight8_at(g, w0, SL_FACE + fa0, ed) != 0 && in_bounds(g, SL_FACE + fa0, b0) && w0[lin(g, SL_FACE + fa0, b0)] != 0
                  && weight8_at(g, w1, SL_FACE + fa1, ed) != 0 && in_bounds(g, SL_FACE + fa1, b1) && w1[lin(g, SL_FACE + fa1, b1)] != 0;
            }
            EL[q] = in ? L_GENERICFLUID : L_UNSOLVED;
        });
    }
}

// ---------------------------------------------------------------------------------------------
// C5 connected components (HDK SIM_VolumetricConnectedComponentBuilder, shim): label-equivalence
// propagation on dense cell ids (min-id representative, pointer jumping), then components are ranked
// by the tile-order key of their first cell.
// ---------------------------------------------------------------------------------------------
void k_cc_init(cudaStream_t st, const Geom& g, const Fields& F, int32_t* parent) {
    const int8_t* L = F.label[SL_CENTER];
    // Only the rank's own cells take part: with slab-local setup a region never crosses a z cut (tiles are aligned to the cuts), so
    // the components of the own cells ARE the own regions; REDUCED cells of the halo keep region -1 until the neighbour's ids arrive.
    const int64_t plane = (int64_t)g.r[SL_CENTER][0] * g.r[SL_CENTER][1];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) { const int z = (int)(q / plane); parent[q] = (L[q] == L_REDUCED && (!g.slabLocal || (z >= g.zLo && z < g.zHi))) ? (int32_t)q : -1; });
}
void k_cc_sweep(cudaStream_t st, const Geom& g, const Fields& F, int32_t* parent, int* changed) {
    const uint8_t* fw0 = F.liqW[SL_FACE + 0]; const uint8_t* fw1 = F.liqW[SL_FACE + 1]; const uint8_t* fw2 = F.liqW[SL_FACE + 2];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        int32_t mine = parent[q];
        if (mine < 0) return;
        const I3 c = delin(g, SL_CENTER, q);
        int32_t best = mine;
        for (int axis = 0; axis < 3; ++axis)
            for (int dir = 0; dir < 2; ++dir) {
                const I3 adj = shifted(c, axis, dir ? 1 : -1);
                if (!in_bounds(g, SL_CENTER, adj)) continue;
                const int32_t pa = parent[lin(g, SL_CENTER, adj)];
                if (pa < 0) continue;
                const I3 face = dir ? shifted(c, axis, 1) : c;
                const uint8_t* fw = axis == 0 ? fw0 : axis == 1 ? fw1 : fw2;
                if (!(fw[lin(g, SL_FACE + axis, face)] > 0)) continue;
                if (pa < best) best = pa;
            }
        // pointer jumping: follow representatives (labels only ever decrease, races are benign)
        int32_t root = best;
        for (int hop = 0; hop < 64; ++hop) { const int32_t up = parent[root]; if (up == root || up < 0) break; root = up; }
        if (root < mine) { atomic_min(&parent[q], root); atomic_min(&parent[mine], root); *changed = 1; }
    });
}
// every member posts its tile-order key to its representative
void k_cc_minkey(cudaStream_t st, const Geom& g, const int32_t* parent, int32_t* minKey) {
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        const int32_t root = parent[q];
        if (root < 0) return;
        atomic_min(&minKey[root], (int32_t)tile_key(g, SL_CENTER, delin(g, SL_CENTER, q)));
    });
}
// flag = 1 on the first cell (in tile order) of every component
void k_cc_first_flags(cudaStream_t st, const Geom& g, const int32_t* parent, const int32_t* minKey, uint8_t* flag) {
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        const int32_t root = parent[q];
        flag[q] = (root >= 0 && minKey[root] == (int32_t)tile_key(g, SL_CENTER, delin(g, SL_CENTER, q))) ? 1 : 0;
    });
}
// firstRank[q] (from the tile-order scan of the flags) is valid on first cells; publish it on the root,
// then every member reads its root's id
void k_cc_publish(cudaStream_t st, const Geom& g, const int32_t* parent, const uint8_t* flag, const int32_t* firstRank, int32_t* rootId) {
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) { if (flag[q]) rootId[parent[q]] = firstRank[q]; });
}
void k_cc_assign(cudaStream_t st, const Geom& g, const Fields& F, const int32_t* parent, const int32_t* rootId) {
    int32_t* R = F.ridx[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) { const int32_t root = parent[q]; R[q] = root >= 0 ? rootId[root] : -1; });
}

// ---------------------------------------------------------------------------------------------
// C6 fixReducedRegionBoundaries (S_Cls:1073-1172).  The reference sweep is serial, in place and
// order dependent.  It is reproduced EXACTLY by solving the recurrence
//     F[c] = activeAt(c) and  #distinct regions among { n in N6(c) : reduced0[n], n not yet removed } >= 2
//     "n removed before c"  <=>  some c'' in N6(n) with key(c'') < key(c) has F[c''] = 1
//     activeAt(c) = active0[c] or (reduced0[c] and c removed before c)
// by fixed-point iteration F <- G(F) from F = 0.  F[c] depends only on cells earlier in tile order,
// so the recurrence has a unique solution and any fixed point of G is that solution (induction on the
// visiting order).  Only cells whose initial neighbourhood already holds >= 2 regions can ever fire.
// ---------------------------------------------------------------------------------------------
PS_D bool fix_fires(const Geom& g, const int8_t* L, const int32_t* R, const uint8_t* fired, const I3& c, int64_t q) {
    const int lab = L[q];
    const int64_t myKey = tile_key(g, SL_CENTER, c);
    auto removedBefore = [&](const I3& n) -> bool {   // n was converted by an earlier-firing neighbour
        for (int a = 0; a < 3; ++a)
            for (int d = -1; d <= 1; d += 2) {
                const I3 cc = shifted(n, a, d);
                if (!in_bounds(g, SL_CENTER, cc)) continue;
                const int64_t qq = lin(g, SL_CENTER, cc);
                if (fired[qq] && tile_key(g, SL_CENTER, cc) < myKey) return true;
            }
        return false;
    };
    bool activeAt = (lab == L_ACTIVEFLUID);
    if (!activeAt && lab == L_REDUCED) activeAt = removedBefore(c);
    if (!activeAt) return false;
    bool seen = false, fix = false; int region = 0;
    for (int axis = 0; axis < 3; ++axis)
        for (int dir = 0; dir < 2; ++dir) {
            const I3 n = shifted(c, axis, dir ? 1 : -1);
            if (!in_bounds(g, SL_CENTER, n)) continue;
            const int64_t qn = lin(g, SL_CENTER, n);
            if (L[qn] != L_REDUCED) continue;
            if (removedBefore(n)) continue;
            if (!seen) { seen = true; region = R[qn]; }
            else if (R[qn] != region) fix = true;
        }
    return fix;
}
// candidates: fluid cells whose initial 6-neighbourhood touches >= 2 different regions
void k_fix_candidates(cudaStream_t st, const Geom& g, const Fields& F, uint8_t* cand, uint8_t* firedA, uint8_t* firedB, int* anyCand) {
    const int8_t* L = F.label[SL_CENTER]; const int32_t* R = F.ridx[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        firedA[q] = 0; firedB[q] = 0;
        uint8_t isCand = 0;
        const int lab = L[q];
        if (lab == L_ACTIVEFLUID || lab == L_REDUCED) {
            const I3 c = delin(g, SL_CENTER, q);
            bool seen = false; int region = 0;
            for (int axis = 0; axis < 3; ++axis)
                for (int dir = 0; dir < 2; ++dir) {
                    const I3 n = shifted(c, axis, dir ? 1 : -1);
                    if (!in_bounds(g, SL_CENTER, n)) continue;
                    const int64_t qn = lin(g, SL_CENTER, n);
                    if (L[qn] != L_REDUCED) continue;
                    if (!seen) { seen = true; region = R[qn]; }
                    else if (R[qn] != region) isCand = 1;
                }
        }
        cand[q] = isCand;
        if (isCand) *anyCand = 1;
    });
}
void k_fix_iterate(cudaStream_t st, const Geom& g, const Fields& F, const uint8_t* cand, const uint8_t* firedIn, uint8_t* firedOut, int* changed) {
    const int8_t* L = F.label[SL_CENTER]; const int32_t* R = F.ridx[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        uint8_t f = 0;
        if (cand[q]) f = fix_fires(g, L, R, firedIn, delin(g, SL_CENTER, q), q) ? 1 : 0;
        firedOut[q] = f;
        if (f != firedIn[q]) *changed = 1;
    });
}
// end of sweep: every REDUCED cell adjacent to a fired cell becomes ACTIVEFLUID / UNASSIGNED
void k_fix_apply(cudaStream_t st, const Geom& g, const Fields& F, const uint8_t* fired, int* anyFired) {
    int8_t* L = F.label[SL_CENTER]; int32_t* R = F.ridx[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        if (fired[q]) *anyFired = 1;
        if (L[q] != L_REDUCED) return;
        const I3 c = delin(g, SL_CENTER, q);
        bool hit = false;
        for (int a = 0; a < 3; ++a)
            for (int d = -1; d <= 1; d += 2) {
                const I3 cc = shifted(c, a, d);
                if (in_bounds(g, SL_CENTER, cc) && fired[lin(g, SL_CENTER, cc)]) hit = true;
            }
        // labels of other cells are only read through `fired` (a separate array), so in-place is safe
        if (hit) { L[q] = L_ACTIVEFLUID; R[q] = -1; }
    });
}

// C7 fixSmallReducedRegions (S_Cls:1174-1313, 1418-1467): bounding boxes by atomics
void k_region_bbox(cudaStream_t st, const Geom& g, const Fields& F, int* bbMin, int* bbMax) {
    const int8_t* L = F.label[SL_CENTER]; const int32_t* R = F.ridx[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        if (L[q] != L_REDUCED) return;
        const int r = R[q];
        if (r < 0) return;                    // REDUCED cell of a neighbour's region (halo)
        const I3 c = delin(g, SL_CENTER, q);
        atomic_min(&bbMin[3 * r + 0], c.x); atomic_min(&bbMin[3 * r + 1], c.y); atomic_min(&bbMin[3 * r + 2], c.z);
        atomic_max(&bbMax[3 * r + 0], c.x); atomic_max(&bbMax[3 * r + 1], c.y); atomic_max(&bbMax[3 * r + 2], c.z);
    });
}
void k_region_remap(cudaStream_t st, const Geom& g, const Fields& F, const int32_t* remap) {
    int8_t* L = F.label[SL_CENTER]; int32_t* R = F.ridx[SL_CENTER];
    for_window(st, g, SL_CENTER, PS_LAMBDA(int64_t q) {
        if (L[q] != L_REDUCED || R[q] < 0) return;
        const int nr = remap[R[q]];
        if (nr < 0) { L[q] = L_ACTIVEFLUID; R[q] = -1; } else R[q] = nr;
    });
}

// C10a constructFacesReducedIndices (S_Cls:1473-1528)
void k_faces_reduced(cudaStream_t st, const Geom& g, const Fields& F) {
    const int8_t* CL = F.label[SL_CENTER]; const int32_t* CR = F.ridx[SL_CENTER];
    for (int axis = 0; axis < 3; ++axis) {
        int8_t* FL = F.label[SL_FACE + axis]; int32_t* FR = F.ridx[SL_FACE + axis];
        for_window(st, g, SL_FACE + axis, PS_LAMBDA(int64_t q) {
            const I3 f = delin(g, SL_FACE + axis, q);
            int idx = -1;
            const I3 c0 = shifted(f, axis, -1);
            if (in_bounds(g, SL_CENTER, f) && CL[lin(g, SL_CENTER, f)] == L_REDUCED) idx = CR[lin(g, SL_CENTER, f)];
            else if (in_bounds(g, SL_CENTER, c0) && CL[lin(g, SL_CENTER, c0)] == L_REDUCED) idx = CR[lin(g, SL_CENTER, c0)];
            FR[q] = idx;
            if (idx != -1) FL[q] = L_REDUCED;
        });
    }
}

// C10b constructEdgesReducedIndices (S_Cls:1534-1659), including the index-source quirk of the
// all-four-reduced case (XY, XZ: faceX(i,j,k); YZ: faceY(i,j-1,k))
void k_edges_reduced(cudaStream_t st, const Geom& g, const Fields& F) {
    for (int e = 0; e < 3; ++e) {
        int8_t* EL = F.label[SL_EDGE + e]; int32_t* ER = F.ridx[SL_EDGE + e];
        const int fa0 = (e == 0) ? 1 : 0, fa1 = (e == 2) ? 1 : 2;
        const int8_t* L0 = F.label[SL_FACE + fa0]; const int8_t* L1 = F.label[SL_FACE + fa1];
        const int32_t* R0 = F.ridx[SL_FACE + fa0]; const int32_t* R1 = F.ridx[SL_FACE + fa1];
        const int32_t* RX = F.ridx[SL_FACE + 0]; const int32_t* RY = F.ridx[SL_FACE + 1];
        for_window(st, g, SL_EDGE + e, PS_LAMBDA(int64_t q) {
            const I3 ed = delin(g, SL_EDGE + e, q);
            const I3 f[4] = {ed, shifted(ed, 3 - fa0 - e, -1), ed, shifted(ed, 3 - fa1 - e, -1)};
            bool red[4];
            red[0] = label_at(g, L0, SL_FACE + fa0, f[0]) == L_REDUCED;
            red[1] = label_at(g, L0, SL_FACE + fa0, f[1]) == L_REDUCED;
            red[2] = label_at(g, L1, SL_FACE + fa1, f[2]) == L_REDUCED;
            red[3] = label_at(g, L1, SL_FACE + fa1, f[3]) == L_REDUCED;
            int label = L_UNASSIGNED, idx = -1;
            if (red[0] && red[1] && red[2] && red[3]) {
                idx = (e == 0) ? index_at(g, RY, SL_FACE + 1, shifted(ed, 1, -1)) : index_at(g, RX, SL_FACE + 0, ed);
                label = L_REDUCED;
            } else if (red[0]) { idx = R0[lin(g, SL_FACE + fa0, f[0])]; label = L_BOUNDARY; }
            else if (red[1]) { idx = R0[lin(g, SL_FACE + fa0, f[1])]; label = L_BOUNDARY; }
            else if (red[2]) { idx = R1[lin(g, SL_FACE + fa1, f[2])]; label = L_BOUNDARY; }
            else if (red[3]) { idx = R1[lin(g, SL_FACE + fa1, f[3])]; label = L_BOUNDARY; }
            ER[q] = idx;
            if (idx != -1) EL[q] = (int8_t)label;
        });
    }
}

// GENERICFLUID -> ACTIVEFLUID (S_Cls:260-280) and the isActive flag the tile-order scan consumes
void k_generic_to_active_flags(cudaStream_t st, const Geom& g, int slot, int8_t* L, uint8_t* flag) {
    for_window(st, g, slot, PS_LAMBDA(int64_t q) {
        int lab = L[q];
        if (lab == L_GENERICFLUID) { lab = L_ACTIVEFLUID; L[q] = L_ACTIVEFLUID; }
        flag[q] = is_active(lab) ? 1 : 0;
    });
}

// C12 buildValidFaces (S_Cls:4-54)
void k_valid_faces(cudaStream_t st, const Geom& g, const Fields& F, float* const valid[3]) {
    for (int axis = 0; axis < 3; ++axis) {
        const int8_t* FL = F.label[SL_FACE + axis]; float* v = valid[axis];
        for_window(st, g, SL_FACE + axis, PS_LAMBDA(int64_t q) { const int l = FL[q]; v[q] = (l == L_UNSOLVED || l == L_UNASSIGNED) ? 0.f : 1.f; });
    }
}

}  // namespace ps
