// ps_reduced.cu -- reduced-region dense algebra (SURVEY.md section 8a rows D1-D6, K9-K10).
//
// Per region r the reference accumulates three 26x26 matrices and one 26-vector from rank-1 updates
// over the region's faces (exec/HDK_PolyStokesSolver.cpp:1330-1399 least squares, 1405-1482 mass,
// 1484-1694 viscosity), then solves/inverts them with Eigen (S.cpp:415, S_AB:195-244).  GPU layout:
//   * REDUCED cells are listed sorted by (region, voxel order); the list is cut into fixed-size chunks
//     that never straddle a region, one CTA per chunk;
//   * a CTA stages, per batch of faces, the basis rows c_f, the viscosity rows d_f and the weights in
//     shared memory and forms the partial Grams  sum c c^T (x2)  and  sum c d^T  (Phi^T W Phi);
//   * partials are summed per region in chunk order (deterministic), then one thread per region does
//     the 26x26 complete-pivoting solve and the partial-pivoting inverse.
#include "ps_solver.hpp"

namespace ps {

// D2 computeCenterOfMasses (S.cpp:328-372, 1274-1324): integer coordinate sums are exact, so the
// atomics below give the reference's value bit for bit: COM = sum * (dx / count).
void k_region_com(cudaStream_t st, const Geom& g, const Fields& F, int32_t R, unsigned long long* sums, double* com) {
    const int8_t* L = F.label[SL_CENTER]; const int32_t* Rg = F.ridx[SL_CENTER];
    dev_memset(sums, 0, (size_t)R * 4 * sizeof(unsigned long long), st);
    int64_t lo, hi;
    z_range(g, SL_CENTER, g.zLo, g.zHi, lo, hi);          // the rank's own cells: with slab-local setup a region never crosses a z cut
    if (!g.slabLocal) { lo = 0; hi = g.n[SL_CENTER]; }     // one GPU / replicated setup (regions crossing cuts included): every region
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) {
        if (L[q] != L_REDUCED) return;
        const int r = Rg[q];
        if (r < 0) return;
        const I3 c = delin(g, SL_CENTER, q);
        atomic_add(&sums[4 * r + 0], (unsigned long long)c.x); atomic_add(&sums[4 * r + 1], (unsigned long long)c.y);
        atomic_add(&sums[4 * r + 2], (unsigned long long)c.z); atomic_add(&sums[4 * r + 3], 1ull);
    });
    const double dx = g.dx;
    ps_for(st, R, PS_LAMBDA(int64_t r) {
        if (sums[4 * r + 3] == 0ull) return;              // a region of another rank
        const double s = dx / (double)sums[4 * r + 3];
        for (int a = 0; a < 3; ++a) com[3 * r + a] = mul_rn((double)sums[4 * r + a], s);
    });
}

// scatter (region, voxel) pairs of flagged voxels to their voxel-order rank (input of the stable sort)
void k_collect_region_keys(cudaStream_t st, const Geom& g, const int32_t* rank, const uint8_t* flag, const int32_t* region, int64_t lo, int64_t hi, int32_t tag, int32_t rankOffset, int32_t* keys, int32_t* vals) {
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) {
        if (!flag[q]) return;
        const int64_t pos = (int64_t)rankOffset + rank[q];
        keys[pos] = region[q]; vals[pos] = (int32_t)q | tag;
    });
}

// SIM_RawField::getValue(indexToPos(sample)) shim: trilinear viscosity at a sample, fractions 0 or 1/2,
// lerp x, y, z as a + t*(b-a) in fp32 (BASELINE.md section 3)
PS_D float local_viscosity(const Geom& g, const float* visc, int slot, const I3& idx) {
    int o[3] = {1, 1, 1};
    if (slot >= SL_FACE && slot < SL_EDGE) o[slot - SL_FACE] = 0;
    else if (slot >= SL_EDGE) { for (int a = 0; a < 3; ++a) if (a != slot - SL_EDGE) o[a] = 0; }
    const int b0 = o[0] ? idx.x : idx.x - 1, b1 = o[1] ? idx.y : idx.y - 1, b2 = o[2] ? idx.z : idx.z - 1;
    const float t0 = o[0] ? 0.f : 0.5f, t1 = o[1] ? 0.f : 0.5f, t2 = o[2] ? 0.f : 0.5f;
    float cz[2];
    for (int dz = 0; dz < 2; ++dz) {
        float cy[2];
        for (int dy = 0; dy < 2; ++dy) {
            const float a = float_at(g, visc, SL_CENTER, I3{b0, b1 + dy, b2 + dz});
            const float b = float_at(g, visc, SL_CENTER, I3{b0 + 1, b1 + dy, b2 + dz});
            cy[dy] = fadd_rn(a, fmul_rn(t0, fsub_rn(b, a)));
        }
        cz[dz] = fadd_rn(cy[0], fmul_rn(t1, fsub_rn(cy[1], cy[0])));
    }
    return fadd_rn(cz[0], fmul_rn(t2, fsub_rn(cz[1], cz[0])));
}

// ---------------------------------------------------------------------------------------------------------------
// Region matrices from polynomial moments.
//
// The reference accumulates  M_r = rho sum_f c_f c_f^T,  N_r = sum_surface c_f c_f^T,  rhs_r = sum_surface u_f c_f  and
// (JD^T mu DJ^T)_r = sum_f c_f d_f^T  as 26x26 rank-1 updates per face (S.cpp:1330-1694): ~2000 FMAs per face.  But
//   * c_f = S_a m(o_f): a fixed sparse 26x10 image S_a (per face axis a) of the 10 monomials m = {1,x,y,z,xx,xy,xz,yy,yz,zz}
//     of the face offset o_f (buildConversionCoefficients, S.cpp:2107-2149), so  sum_f w_f c_f c_f^T = S_a Q_a S_a^T  with
//     the 10x10 moment matrix  Q_a = sum_f w_f m m^T  (55 numbers per axis and weight);
//   * the viscosity block is  sum over stress samples s of  kappa_s e_s e_s^T  where e_s = sum over the faces around s of
//     +-c_f is the discrete strain rate of the basis at s (S.cpp:1537-1683 visits every (face, partner face) pair of a
//     REDUCED cell / strictly REDUCED edge exactly once).  Central differences of quadratics are exact, so e_s is LINEAR
//     in the sample position: e_s = dx A (1,x,y,z)^T with a constant 26x4 matrix A per sample type, and the block is
//       sum_a A_a T^c A_a^T + 1/2 sum_e H_e T^e H_e^T,   T = sum_s mu_s (1,x,y,z)(1,x,y,z)^T   (10 numbers per type).
// So a region needs 400 moments (2 x 3 x 55 + 3 x 10 + 10 + 3 x 10) accumulated over its cells in a FIXED order (chunks of
// the (region, voxel order) sorted cell list, then chunk order): bit-reproducible, ~25x fewer flops and no 26x26
// shared-memory traffic.  The tables S_a, A_a, H_e are generated from conversion_coefficients itself at integer points
// (exact arithmetic), not typed in.
// ---------------------------------------------------------------------------------------------------------------
constexpr int MOM_QM = 0, MOM_QN = 165, MOM_RHS = 330, MOM_TC = 360, MOM_TE = 370, MOM_COUNT = 400;
constexpr int TAB_S = 0, TAB_A = 3 * RDOF * 10, TAB_H = TAB_A + 3 * RDOF * 4, TAB_COUNT = TAB_H + 3 * RDOF * 4;
constexpr int GRAM_CELLS = 256;          // cells per chunk (build_chunks in ps_solver.cu)
constexpr int STAGE_DOUBLES = 3 + 18 + 1 + 12;   // per cell: index (3), wM/wN/wN*u of 6 faces, mu, mu of the <= 12 owned REDUCED edges

PS_HD double monomial(int k, double x, double y, double z) {
    switch (k) { case 0: return 1.; case 1: return x; case 2: return y; case 3: return z; case 4: return x * x; case 5: return x * y;
                 case 6: return x * z; case 7: return y * y; case 8: return y * z; default: return z * z; }
}
// (k, l), k <= l, of the q-th entry of a symmetric n x n matrix stored row-wise upper triangle
PS_HD void sym_pair(int n, int q, int& k, int& l) { k = 0; while (q >= n - k) { q -= n - k; ++k; } l = k + q; }
PS_HD int sym_index(int n, int k, int l) { if (k > l) { const int t = k; k = l; l = t; } return k * n - k * (k - 1) / 2 + (l - k); }

// host: S_a (26x10), A_a (26x4), H_e (26x4) from conversion_coefficients at small integer points (all values exact)
static void build_region_tables(double* T) {
    auto cc = [](double x, double y, double z, int axis, double* v) { conversion_coefficients(x, y, z, axis, v); };
    for (int i = 0; i < TAB_COUNT; ++i) T[i] = 0.;
    // S_a: column k = response to the k-th monomial; probe with points whose monomial vectors form an invertible system
    // -- simpler: every entry of c is +-{1, 2, 1/2} times ONE monomial, so two probes identify (monomial, coefficient)
    const double P[2][3] = {{2., 3., 5.}, {7., 11., 13.}};
    for (int a = 0; a < 3; ++a) {
        double v0[RDOF], v1[RDOF];
        cc(P[0][0], P[0][1], P[0][2], a, v0); cc(P[1][0], P[1][1], P[1][2], a, v1);
        for (int n = 0; n < RDOF; ++n) {
            if (v0[n] == 0. && v1[n] == 0.) continue;
            bool found = false;
            for (int k = 0; k < 10 && !found; ++k) {
                const double m0 = monomial(k, P[0][0], P[0][1], P[0][2]), m1 = monomial(k, P[1][0], P[1][1], P[1][2]);
                const double c = v0[n] / m0;
                if (c * m1 == v1[n]) { T[TAB_S + (a * RDOF + n) * 10 + k] = c; found = true; }
            }
            if (!found) throw Error("region tables: basis row is not a single monomial");
        }
    }
    // A_a: (c_a(p + e_a) - c_a(p - e_a)) / 2 = d/da c_a, linear in p; H_e likewise for the two axes != e
    auto strain = [&](int type, bool edge, double x, double y, double z, double* out) {
        for (int n = 0; n < RDOF; ++n) out[n] = 0.;
        double hi[RDOF], lo[RDOF];
        if (!edge) {
            const int a = type; double p[3] = {x, y, z}, q[3] = {x, y, z};
            p[a] += 1.; q[a] -= 1.;
            cc(p[0], p[1], p[2], a, hi); cc(q[0], q[1], q[2], a, lo);
            for (int n = 0; n < RDOF; ++n) out[n] = (hi[n] - lo[n]) / 2.;
        } else {
            const int e = type;
            for (int a = 0; a < 3; ++a) {
                if (a == e) continue;
                const int b = 3 - a - e;
                double p[3] = {x, y, z}, q[3] = {x, y, z};
                p[b] += 1.; q[b] -= 1.;
                cc(p[0], p[1], p[2], a, hi); cc(q[0], q[1], q[2], a, lo);
                for (int n = 0; n < RDOF; ++n) out[n] += (hi[n] - lo[n]) / 2.;
            }
        }
    };
    for (int pass = 0; pass < 2; ++pass)
        for (int t = 0; t < 3; ++t) {
            double f0[RDOF], f1[RDOF];
            strain(t, pass == 1, 0., 0., 0., f0);
            double* dst = T + (pass ? TAB_H : TAB_A) + t * RDOF * 4;
            for (int n = 0; n < RDOF; ++n) dst[n * 4 + 0] = f0[n];
            for (int d = 0; d < 3; ++d) {
                strain(t, pass == 1, d == 0 ? 1. : 0., d == 1 ? 1. : 0., d == 2 ? 1. : 0., f1);
                for (int n = 0; n < RDOF; ++n) dst[n * 4 + 1 + d] = f1[n] - f0[n];
            }
        }
}

// phase 1: everything the moments need from one REDUCED cell, staged as stage[field * GRAM_CELLS + slot]:
// fields 0-2 the cell-centre offset from the region's COM, 3-8 wM, 9-14 wN, 15-20 wN*u of the 6 faces, 21 mu, 22-33 mu of
// the owned REDUCED edges
PS_D void stage_cell(const Geom& g, const Fields& F, const double* com, int64_t cellQ, int slot, double* stage) {
    const I3 c = delin(g, SL_CENTER, cellQ);
    stage[0 * GRAM_CELLS + slot] = sub_rn(mul_rn((double)c.x, g.dx), com[0]);
    stage[1 * GRAM_CELLS + slot] = sub_rn(mul_rn((double)c.y, g.dx), com[1]);
    stage[2 * GRAM_CELLS + slot] = sub_rn(mul_rn((double)c.z, g.dx), com[2]);
    const int8_t* CL = F.label[SL_CENTER];
    for (int axis = 0; axis < 3; ++axis)
        for (int dir = 0; dir < 2; ++dir) {
            const I3 face = dir ? shifted(c, axis, 1) : c;
            const bool nbrActive = is_active(label_at(g, CL, SL_CENTER, shifted(c, axis, dir ? 1 : -1)));
            const double wM = (dir == 0 || nbrActive) ? g.density : 0.;            // S.cpp:1442-1472
            const double wN = nbrActive ? 1. : 0.;                                  // S.cpp:1369-1390
            const double u = (double)F.vel[axis][lin(g, SL_FACE + axis, face)];
            const int f = axis * 2 + dir;
            stage[(3 + f) * GRAM_CELLS + slot] = wM; stage[(9 + f) * GRAM_CELLS + slot] = wN; stage[(15 + f) * GRAM_CELLS + slot] = wN * u;
        }
    stage[21 * GRAM_CELLS + slot] = (double)F.viscosity[cellQ];
    // strictly REDUCED edges (S.cpp:1605-1683), each owned by the first REDUCED cell among its 4 cells in the order
    // (0,0), (-a), (-b), (-a,-b) with a < b the axes across the edge
    for (int e = 0; e < 3; ++e) {
        const int a = e == 0 ? 1 : 0, b = e == 2 ? 1 : 2;
        for (int db = 0; db < 2; ++db) for (int da = 0; da < 2; ++da) {
            const I3 ed = shifted(shifted(c, a, da), b, db);
            double mu = 0.;
            if (F.label[SL_EDGE + e][lin(g, SL_EDGE + e, ed)] == L_REDUCED) {
                // cells around the edge, in priority order; this cell is ed - (da, db)
                bool owner = true;
                const I3 cand[4] = {ed, shifted(ed, a, -1), shifted(ed, b, -1), shifted(shifted(ed, a, -1), b, -1)};
                const int mine = da + 2 * db;                 // index of this cell in cand[]
                for (int k = 0; k < mine; ++k) if (label_at(g, CL, SL_CENTER, cand[k]) == L_REDUCED) owner = false;
                if (owner) mu = (double)local_viscosity(g, F.viscosity, SL_EDGE + e, ed);
            }
            stage[(22 + e * 4 + db * 2 + da) * GRAM_CELLS + slot] = mu;
        }
    }
}

#ifndef PS_EMULATE
// ---- the same moments on the FP64 tensor cores (DMMA.8x8x4) ------------------------------------------------------------------
// Per face axis a the moments are one dense contraction over the 2 x 256 face samples of the chunk,
//     Phi_a^T [ W_M Phi_a | W_N Phi_a | W_N u ]        Phi_a : 512 x 10 (monomials of the face offsets),   10 x 21 outputs,
// i.e. Q^M_a, Q^N_a (both triangles) and the least-squares right-hand side in one product: 2 x 3 tiles of mma.m8n8k4.f64, 128
// k-steps, split over the 8 warps of the CTA (64 samples each), 6 independent accumulators per warp.  The stress moments are
// Gram products of (1, x, y, z) at the cell centres (T^c) and at the four owned edges around a cell (T^e): two sample positions
// share one 8 x 8 tile (rows / columns 0-3 and 4-7; the off-diagonal blocks are not read).  Partial tiles are summed over the
// warps in warp order, so the result is reproducible run to run; against the serial sum it differs by the association order only.
constexpr int PHI_DOUBLES = 2 * GRAM_CELLS * 10;                 // Phi_a, reused for the cross-warp sums (8 warps x 12 x 32)
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
__global__ void __launch_bounds__(GRAM_CELLS, 2) gram_moments_dmma_kernel(Geom g, Fields F, const double* __restrict__ com, const int32_t* __restrict__ cellList,
                                                                        const int32_t* __restrict__ chunk, double* __restrict__ partial, int chunk0) {
    extern __shared__ double stage[];              // [STAGE_DOUBLES][GRAM_CELLS] | Phi / warp partials [PHI_DOUBLES]
    double* phi = stage + STAGE_DOUBLES * GRAM_CELLS;
    const int ch = chunk0 + blockIdx.x;
    const int region = chunk[3 * ch + 0], begin = chunk[3 * ch + 1], end = chunk[3 * ch + 2];
    const int nCells = end - begin;
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31, r = lane >> 2, q = lane & 3;
    if (tid < nCells) stage_cell(g, F, com + 3 * region, cellList[begin + tid], tid, stage);
    else for (int f = 0; f < STAGE_DOUBLES; ++f) stage[f * GRAM_CELLS + tid] = 0.;          // empty slots: zero weights, zero offsets
    double* out = partial + (size_t)ch * MOM_COUNT;
    const double h = 0.5 * g.dx;
    __syncthreads();
    // ---- faces ----
    for (int a = 0; a < 3; ++a) {
        {   // Phi_a: sample s = dir * 256 + cell
            double o[3] = {stage[tid], stage[GRAM_CELLS + tid], stage[2 * GRAM_CELLS + tid]};
            const double ca = o[a];
#pragma unroll
            for (int dir = 0; dir < 2; ++dir) {
                o[a] = dir ? ca + h : ca - h;
                double* m = phi + (size_t)(dir * GRAM_CELLS + tid) * 10;
                m[0] = 1.; m[1] = o[0]; m[2] = o[1]; m[3] = o[2]; m[4] = o[0] * o[0]; m[5] = o[0] * o[1]; m[6] = o[0] * o[2]; m[7] = o[1] * o[1]; m[8] = o[1] * o[2]; m[9] = o[2] * o[2];
            }
        }
        __syncthreads();
        double acc[2][3][2];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int t = 0; t < 3; ++t) { acc[i][t][0] = 0.; acc[i][t][1] = 0.; }
        // column r of the three B tiles: [wM m_r] [wM m_8, wM m_9, wN m_0 .. wN m_5] [wN m_6 .. wN m_9, wN u, 0, 0, 0]
        const int k1 = r < 2 ? r + 8 : r - 2, k2 = r < 4 ? r + 6 : 0;
#pragma unroll 4
        for (int ks = 0; ks < 16; ++ks) {
            const int sIdx = wid * 64 + ks * 4 + q;
            const int dir = sIdx >> 8, cell = sIdx & (GRAM_CELLS - 1);
            const double* m = phi + (size_t)sIdx * 10;
            const double mr = m[r], m1 = m[k1], m2 = m[k2];
            const double wM = stage[(3 + 2 * a + dir) * GRAM_CELLS + cell], wN = stage[(9 + 2 * a + dir) * GRAM_CELLS + cell], wU = stage[(15 + 2 * a + dir) * GRAM_CELLS + cell];
            const double a0 = mr, a1 = r < 2 ? m1 : 0.;
            const double b0 = wM * mr, b1 = (r < 2 ? wM : wN) * m1, b2 = r < 4 ? wN * m2 : (r == 4 ? wU : 0.);
            dmma884(acc[0][0][0], acc[0][0][1], a0, b0); dmma884(acc[0][1][0], acc[0][1][1], a0, b1); dmma884(acc[0][2][0], acc[0][2][1], a0, b2);
            dmma884(acc[1][0][0], acc[1][0][1], a1, b0); dmma884(acc[1][1][0], acc[1][1][1], a1, b1); dmma884(acc[1][2][0], acc[1][2][1], a1, b2);
        }
        __syncthreads();                 // every warp is done reading Phi_a: it becomes the table of warp partials [wid][row 16][col 24]
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int t = 0; t < 3; ++t)
#pragma unroll
                for (int e = 0; e < 2; ++e) phi[(size_t)wid * 384 + (r + 8 * i) * 24 + 8 * t + 2 * q + e] = acc[i][t][e];
        __syncthreads();
        if (tid < 120) {                 // 55 + 55 + 10 outputs of this axis, summed over the warps in warp order
            int row, col;
            if (tid < 110) { int k, l; sym_pair(10, tid % 55, k, l); row = k; col = l + (tid < 55 ? 0 : 10); }
            else { row = tid - 110; col = 20; }
            double sum = 0.;
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) sum += phi[(size_t)w8 * 384 + row * 24 + col];
            if (tid < 55) out[MOM_QM + a * 55 + tid] = sum;
            else if (tid < 110) out[MOM_QN + a * 55 + (tid - 55)] = sum;
            else out[MOM_RHS + a * 10 + (tid - 110)] = sum;
        }
        __syncthreads();
    }
    // ---- stresses: T^c (cell centres) and T^e (edge axis e, four owned edges around the cell) ----
    {
        double tc[2] = {0., 0.}, te[3][2] = {{0., 0.}, {0., 0.}, {0., 0.}};
        const int comp = r & 3, hiHalf = r >> 2;          // rows / columns 0-3: first sample position, 4-7: second
#pragma unroll 2
        for (int ks = 0; ks < 8; ++ks) {
            const int cell = wid * 32 + ks * 4 + q;
            const double x = stage[cell], y = stage[GRAM_CELLS + cell], z = stage[2 * GRAM_CELLS + cell];
            {
                const double v = comp == 0 ? 1. : (comp == 1 ? x : (comp == 2 ? y : z));
                const double av = hiHalf ? 0. : v;
                dmma884(tc[0], tc[1], av, stage[21 * GRAM_CELLS + cell] * av);
            }
#pragma unroll
            for (int e = 0; e < 3; ++e) {
                const int ea = e == 0 ? 1 : 0, eb = e == 2 ? 1 : 2;
#pragma unroll
                for (int db = 0; db < 2; ++db) {
                    // first position (da = 0) in rows 0-3, second (da = 1) in rows 4-7
                    double o[3] = {x, y, z};
                    o[ea] = hiHalf ? o[ea] + h : o[ea] - h;
                    o[eb] = db ? o[eb] + h : o[eb] - h;
                    const double v = comp == 0 ? 1. : (comp == 1 ? o[0] : (comp == 2 ? o[1] : o[2]));
                    const double mu = stage[(22 + e * 4 + db * 2 + hiHalf) * GRAM_CELLS + cell];
                    dmma884(te[e][0], te[e][1], v, mu * v);
                }
            }
        }
        // warp partials: [wid][4 tiles][row 8][col 8]
#pragma unroll
        for (int e2 = 0; e2 < 2; ++e2) {
            phi[(size_t)wid * 256 + 0 * 64 + r * 8 + 2 * q + e2] = tc[e2];
#pragma unroll
            for (int e = 0; e < 3; ++e) phi[(size_t)wid * 256 + (1 + e) * 64 + r * 8 + 2 * q + e2] = te[e][e2];
        }
        __syncthreads();
        if (tid < 40) {
            const int tile = tid / 10; int k, l; sym_pair(4, tid % 10, k, l);
            double sum = 0.;
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) {
                const double* t8 = phi + (size_t)w8 * 256 + tile * 64;
                sum += tile == 0 ? t8[k * 8 + l] : t8[k * 8 + l] + t8[(k + 4) * 8 + l + 4];
            }
            if (tile == 0) out[MOM_TC + tid] = sum; else out[MOM_TE + (tile - 1) * 10 + tid % 10] = sum;
        }
    }
}
void region_gram_partials(cudaStream_t st, const Geom& g, const Fields& F, const RegionData& RG, double* partial) {
    if (RG.cellChunkHi <= RG.cellChunkLo) return;
    const size_t smem = (size_t)(STAGE_DOUBLES * GRAM_CELLS + PHI_DOUBLES) * sizeof(double);
    // a per-DEVICE attribute: set on every call (a process-wide "done" flag left the second GPU of a multi-device handle without it)
    PS_CUDA(cudaFuncSetAttribute(gram_moments_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gram_moments_dmma_kernel<<<RG.cellChunkHi - RG.cellChunkLo, GRAM_CELLS, smem, st>>>(g, F, RG.com.p, RG.cellList.p, RG.cellChunk.p, partial, RG.cellChunkLo);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
#else
// the emulation twin: the moments one at a time (phase 2 below), each a serial sum in cell order
// v^e for e in 0..4 without divergent control flow
PS_HD double pow_small(double v, int e) {
    const double v2 = v * v;
    double r = (e & 1) ? v : 1.;
    if (e & 2) r *= v2;
    if (e & 4) r *= v2 * v2;
    return r;
}
// exponents (ex, ey, ez) of monomial k of {1,x,y,z,xx,xy,xz,yy,yz,zz}, packed 4 bits each
PS_HD int monomial_exps(int k) {
    const int t[10] = {0x000, 0x001, 0x010, 0x100, 0x002, 0x011, 0x101, 0x020, 0x110, 0x200};
    return t[k];
}
// phase 2: moment `item` (0..234 work items, see the layout constants) over the staged cells, in cell order.
// A face of axis a sits at the cell-centre offset -+ dx/2 on axis a; an edge of axis e at -+ dx/2 on the two other axes.
PS_D void accumulate_item(const Geom& g, const double* stage, int nCells, int item, double* out) {
    const double h = 0.5 * g.dx;
    if (item < 195) {
        const bool rhs = item >= 165;
        const int a = rhs ? (item - 165) / 10 : item / 55;
        int ex;
        if (rhs) ex = monomial_exps((item - 165) % 10);
        else { int k, l; sym_pair(10, item % 55, k, l); ex = monomial_exps(k) + monomial_exps(l); }
        const int e[3] = {ex & 15, (ex >> 4) & 15, (ex >> 8) & 15};
        const int b = (a + 1) % 3, c = (a + 2) % 3;
        const double* pa = stage + a * GRAM_CELLS; const double* pb = stage + b * GRAM_CELLS; const double* pc = stage + c * GRAM_CELLS;
        const double* w0 = stage + ((rhs ? 15 : 3) + 2 * a) * GRAM_CELLS;    // wM (or wN*u) of the two faces of axis a
        const double* w1 = stage + (9 + 2 * a) * GRAM_CELLS;                  // wN
        double acc0 = 0., acc1 = 0.;
        for (int s = 0; s < nCells; ++s) {
            const double base = pow_small(pb[s], e[b]) * pow_small(pc[s], e[c]);
            for (int dir = 0; dir < 2; ++dir) {
                const double wa = w0[dir * GRAM_CELLS + s], wb = rhs ? 0. : w1[dir * GRAM_CELLS + s];
                if (wa == 0. && wb == 0.) continue;
                const double pr = base * pow_small(dir ? pa[s] + h : pa[s] - h, e[a]);
                acc0 += wa * pr; acc1 += wb * pr;
            }
        }
        if (rhs) out[MOM_RHS + (item - 165)] = acc0;
        else { out[MOM_QM + item] = acc0; out[MOM_QN + item] = acc1; }
    } else if (item < 205) {                             // T^c: cell-centred stresses, sum mu (1,x,y,z)(1,x,y,z)^T
        int k, l; sym_pair(4, item - 195, k, l);
        const int ex = monomial_exps(k) + monomial_exps(l);
        const double* mu = stage + 21 * GRAM_CELLS;
        double acc = 0.;
        for (int s = 0; s < nCells; ++s)
            acc += mu[s] * (pow_small(stage[s], ex & 15) * pow_small(stage[GRAM_CELLS + s], (ex >> 4) & 15) * pow_small(stage[2 * GRAM_CELLS + s], (ex >> 8) & 15));
        out[MOM_TC + (item - 195)] = acc;
    } else {                                             // T^e: edge-centred stresses of edge axis e
        const int e = (item - 205) / 10; int k, l; sym_pair(4, (item - 205) % 10, k, l);
        const int ex = monomial_exps(k) + monomial_exps(l);
        const int ee[3] = {ex & 15, (ex >> 4) & 15, (ex >> 8) & 15};
        const int a = e == 0 ? 1 : 0, b = e == 2 ? 1 : 2;
        const double* pe = stage + e * GRAM_CELLS; const double* pa = stage + a * GRAM_CELLS; const double* pb = stage + b * GRAM_CELLS;
        double acc = 0.;
        for (int s = 0; s < nCells; ++s) {
            const double along = pow_small(pe[s], ee[e]);
            for (int db = 0; db < 2; ++db) for (int da = 0; da < 2; ++da) {
                const double mu = stage[(22 + e * 4 + db * 2 + da) * GRAM_CELLS + s];
                if (mu == 0.) continue;
                acc += mu * (along * pow_small(da ? pa[s] + h : pa[s] - h, ee[a]) * pow_small(db ? pb[s] + h : pb[s] - h, ee[b]));
            }
        }
        out[MOM_TE + (item - 205)] = acc;
    }
}
constexpr int MOM_ITEMS = 235;
void region_gram_partials(cudaStream_t, const Geom& g, const Fields& F, const RegionData& RG, double* partial) {
    std::vector<double> stage((size_t)STAGE_DOUBLES * GRAM_CELLS);
    for (int ch = RG.cellChunkLo; ch < RG.cellChunkHi; ++ch) {
        const int region = RG.cellChunk.p[3 * ch], begin = RG.cellChunk.p[3 * ch + 1], end = RG.cellChunk.p[3 * ch + 2];
        for (int i = begin; i < end; ++i) stage_cell(g, F, RG.com.p + 3 * region, RG.cellList.p[i], i - begin, stage.data());
        for (int item = 0; item < MOM_ITEMS; ++item) accumulate_item(g, stage.data(), end - begin, item, partial + (size_t)ch * MOM_COUNT);
    }
}
#endif

// dense 26x26 factorisations.  Same elimination order, pivot choice and per-element operations as the serial
// algorithms (so the results are bit-identical to them), with the independent element updates spread over `nl` lanes.
// PS_LANE_SYNC is a warp barrier in the CUDA build and nothing in the serial emulation (nl = 1).
#ifndef PS_EMULATE
#define PS_LANE_SYNC() __syncwarp()
#else
#define PS_LANE_SYNC()
#endif
// S_AB:209 .inverse() -> PartialPivLU (extern/eigen/Eigen/src/LU/InverseImpl.h:25-31).  lu, inv, perm live in shared / private memory.
PS_D void inverse_partial_piv(double* lu, double* inv, int* perm, int lane, int nl) {
    const int n = RDOF;
    for (int i = lane; i < n; i += nl) perm[i] = i;
    PS_LANE_SYNC();
    for (int k = 0; k < n; ++k) {
        int piv = k; double best = fabs(lu[k * n + k]);
        for (int i = k + 1; i < n; ++i) { const double a = fabs(lu[i * n + k]); if (a > best) { best = a; piv = i; } }     // every lane, same answer
        PS_LANE_SYNC();
        if (piv != k) {
            for (int j = lane; j < n; j += nl) { const double t = lu[k * n + j]; lu[k * n + j] = lu[piv * n + j]; lu[piv * n + j] = t; }
            if (lane == 0) { const int t = perm[k]; perm[k] = perm[piv]; perm[piv] = t; }
        }
        PS_LANE_SYNC();
        const double dg = lu[k * n + k];
        PS_LANE_SYNC();
        if (dg != 0.) for (int i = k + 1 + lane; i < n; i += nl) lu[i * n + k] /= dg;
        PS_LANE_SYNC();
        const int m = n - k - 1;
        for (int e = lane; e < m * m; e += nl) { const int i = k + 1 + e / m, j = k + 1 + e % m; lu[i * n + j] -= lu[i * n + k] * lu[k * n + j]; }
        PS_LANE_SYNC();
    }
    for (int c = lane; c < n; c += nl) {          // one right-hand side (unit vector) per lane
        double col[RDOF];
        for (int i = 0; i < n; ++i) col[i] = (perm[i] == c) ? 1. : 0.;
        for (int i = 0; i < n; ++i) { double s = col[i]; for (int j = 0; j < i; ++j) s -= lu[i * n + j] * col[j]; col[i] = s; }
        for (int i = n - 1; i >= 0; --i) { double s = col[i]; for (int j = i + 1; j < n; ++j) s -= lu[i * n + j] * col[j]; col[i] = s / lu[i * n + i]; }
        for (int i = 0; i < n; ++i) inv[i * n + c] = col[i];
    }
    PS_LANE_SYNC();
}
// S.cpp:415 fullPivLu().solve(): complete pivoting, rank threshold maxPivot * eps * n, free variables 0
PS_D void solve_full_piv(double* lu, const double* rhs, double* x, int* rowT, int* colT, int lane, int nl) {
    const int n = RDOF;
    int nonzero = n; double maxPivot = 0.;
    for (int k = 0; k < n; ++k) {
        // first maximum of |lu| over the trailing block in row-major order (the serial scan keeps the first on ties)
        double best = 0.; int bestIdx = k * n + k;
        const int m = n - k;
        for (int e = lane; e < m * m; e += nl) { const int idx = (k + e / m) * n + (k + e % m); const double a = fabs(lu[idx]); if (a > best || (a == best && a > 0. && idx < bestIdx)) { best = a; bestIdx = idx; } }
#ifndef PS_EMULATE
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o); const int oi = __shfl_xor_sync(0xffffffffu, bestIdx, o);
            if (ob > best || (ob == best && ob > 0. && oi < bestIdx)) { best = ob; bestIdx = oi; }
        }
#endif
        const int pr = bestIdx / n, pc = bestIdx % n;
        if (best == 0.) { nonzero = k; for (int i = k + lane; i < n; i += nl) { rowT[i] = i; colT[i] = i; } break; }
        if (best > maxPivot) maxPivot = best;
        if (lane == 0) { rowT[k] = pr; colT[k] = pc; }
        PS_LANE_SYNC();
        if (pr != k) for (int j = lane; j < n; j += nl) { const double t = lu[k * n + j]; lu[k * n + j] = lu[pr * n + j]; lu[pr * n + j] = t; }
        PS_LANE_SYNC();
        if (pc != k) for (int i = lane; i < n; i += nl) { const double t = lu[i * n + k]; lu[i * n + k] = lu[i * n + pc]; lu[i * n + pc] = t; }
        PS_LANE_SYNC();
        const double dg = lu[k * n + k];
        PS_LANE_SYNC();
        for (int i = k + 1 + lane; i < n; i += nl) lu[i * n + k] /= dg;
        PS_LANE_SYNC();
        const int mm = n - k - 1;
        for (int e = lane; e < mm * mm; e += nl) { const int i = k + 1 + e / mm, j = k + 1 + e % mm; lu[i * n + j] -= lu[i * n + k] * lu[k * n + j]; }
        PS_LANE_SYNC();
    }
    PS_LANE_SYNC();
    if (lane == 0) {
        const double thr = maxPivot * (2.220446049250313e-16 * n);
        int rank = 0;
        for (int i = 0; i < nonzero; ++i) if (fabs(lu[i * n + i]) > thr) ++rank;
        double c[RDOF];
        for (int i = 0; i < n; ++i) c[i] = rhs[i];
        for (int k = 0; k < n; ++k) if (rowT[k] != k) { const double t = c[k]; c[k] = c[rowT[k]]; c[rowT[k]] = t; }
        for (int i = 0; i < n; ++i) { double s = c[i]; for (int j = 0; j < i; ++j) s -= lu[i * n + j] * c[j]; c[i] = s; }
        for (int i = rank - 1; i >= 0; --i) { double s = c[i]; for (int j = i + 1; j < rank; ++j) s -= lu[i * n + j] * c[j]; c[i] = s / lu[i * n + i]; }
        for (int i = rank; i < n; ++i) c[i] = 0.;
        for (int k = n - 1; k >= 0; --k) if (colT[k] != k) { const double t = c[k]; c[k] = c[colT[k]]; c[colT[k]] = t; }
        for (int i = 0; i < n; ++i) x[i] = c[i];
    }
    PS_LANE_SYNC();
}

// per region: v* = fullPivLu(N).solve(rhs) (S.cpp:412-416); B = M/dt + 2 V, B^-1 = B.inverse() (S_AB:195-244); rhs_r = M v* (S_AB:356-367)
PS_D void region_factor(double invDt, const double* Mr, const double* Vi, const double* Nm, const double* lsq, double* fit, double* Binv, double* rhsR,
                        double* a, double* b, int* piv, int lane, int nl) {
    const int NN = RDOF * RDOF;
    for (int e = lane; e < NN; e += nl) { a[e] = Nm[e]; b[e] = invDt * Mr[e] + 2. * Vi[e]; }
    PS_LANE_SYNC();
    solve_full_piv(a, lsq, fit, piv, piv + RDOF, lane, nl);
    inverse_partial_piv(b, Binv, piv + 2 * RDOF, lane, nl);
    for (int i = lane; i < RDOF; i += nl) { double s = 0.; for (int j = 0; j < RDOF; ++j) s += Mr[i * RDOF + j] * fit[j]; rhsR[i] = s; }
}
#ifndef PS_EMULATE
__global__ void __launch_bounds__(32) region_factor_kernel(double invDt, int region0, const double* __restrict__ Mr, const double* __restrict__ Vi, const double* __restrict__ Nm,
                                                          const double* __restrict__ lsq, double* fit, double* Binv, double* rhsR) {
    __shared__ double a[RDOF * RDOF], b[RDOF * RDOF], inv[RDOF * RDOF], x[RDOF], out[RDOF];
    __shared__ int piv[3 * RDOF];
    const int r = region0 + blockIdx.x, NN = RDOF * RDOF;
    region_factor(invDt, Mr + (size_t)r * NN, Vi + (size_t)r * NN, Nm + (size_t)r * NN, lsq + (size_t)r * RDOF, x, inv, out, a, b, piv, threadIdx.x, 32);
    __syncwarp();
    for (int e = threadIdx.x; e < NN; e += 32) Binv[(size_t)r * NN + e] = inv[e];
    if (threadIdx.x < RDOF) { fit[(size_t)r * RDOF + threadIdx.x] = x[threadIdx.x]; rhsR[(size_t)r * RDOF + threadIdx.x] = out[threadIdx.x]; }
}
#endif

// sums the chunk moments of every owned region in chunk order, expands them to M_r, N_r, (JD^T mu DJ^T)_r and the
// least-squares right-hand side, then factorises
void region_gram_finish(cudaStream_t st, const Geom& g, RegionData& RG, int nChunks) {
    // only the regions this rank builds [bldLo, regHi) (all of them on one GPU)
    const int R0 = RG.bldLo, R = RG.regHi - RG.bldLo;
    if (R <= 0) return;
    if (RG.tables.n < (size_t)TAB_COUNT) { std::vector<double> T(TAB_COUNT); build_region_tables(T.data()); RG.tables.from_host(st, T.data(), T.size()); }
    RG.moments.alloc((size_t)RG.count * MOM_COUNT);
    const double* partial = RG.partial.p; const int32_t* chunkStart = RG.cellChunkStart.p;
    double* mom = RG.moments.p; const double* T = RG.tables.p;
    double* Mr = RG.Mr.p; double* Vi = RG.Visc.p; double* Nm = RG.N.p; double* Binv = RG.Binv.p;
    double* lsq = RG.lsqRhs.p; double* fit = RG.bestFit.p; double* rhsR = RG.rhsR.p;
    const int NN = RDOF * RDOF;
    ps_for(st, (int64_t)R * MOM_COUNT, PS_LAMBDA(int64_t ql) {
        const int r = R0 + (int)(ql / MOM_COUNT), e = (int)(ql % MOM_COUNT);
        double s = 0.;
        for (int ch = chunkStart[r]; ch < chunkStart[r + 1]; ++ch) s += partial[(size_t)ch * MOM_COUNT + e];
        mom[(size_t)r * MOM_COUNT + e] = s;
    });
    ps_for(st, (int64_t)R * NN, PS_LAMBDA(int64_t ql) {
        const int r = R0 + (int)(ql / NN), e = (int)(ql % NN), i = e / RDOF, j = e % RDOF;
        const double* m = mom + (size_t)r * MOM_COUNT;
        double M = 0., N = 0., V = 0.;
        for (int a = 0; a < 3; ++a) {
            const double* Si = T + TAB_S + (a * RDOF + i) * 10; const double* Sj = T + TAB_S + (a * RDOF + j) * 10;
            for (int k = 0; k < 10; ++k) {
                if (Si[k] == 0.) continue;
                for (int l = 0; l < 10; ++l) {
                    if (Sj[l] == 0.) continue;
                    const int q = a * 55 + sym_index(10, k, l);
                    M += Si[k] * Sj[l] * m[MOM_QM + q]; N += Si[k] * Sj[l] * m[MOM_QN + q];
                }
            }
            const double* Ai = T + TAB_A + (a * RDOF + i) * 4; const double* Aj = T + TAB_A + (a * RDOF + j) * 4;
            const double* Hi = T + TAB_H + (a * RDOF + i) * 4; const double* Hj = T + TAB_H + (a * RDOF + j) * 4;
            for (int k = 0; k < 4; ++k) for (int l = 0; l < 4; ++l) {
                const int q = sym_index(4, k, l);
                V += Ai[k] * Aj[l] * m[MOM_TC + q] + 0.5 * (Hi[k] * Hj[l]) * m[MOM_TE + a * 10 + q];
            }
        }
        const size_t o = (size_t)r * NN + e;
        Mr[o] = M; Nm[o] = N; Vi[o] = V;
    });
    ps_for(st, (int64_t)R * RDOF, PS_LAMBDA(int64_t ql) {
        const int r = R0 + (int)(ql / RDOF), i = (int)(ql % RDOF);
        const double* m = mom + (size_t)r * MOM_COUNT;
        double s = 0.;
        for (int a = 0; a < 3; ++a) { const double* Si = T + TAB_S + (a * RDOF + i) * 10; for (int k = 0; k < 10; ++k) s += Si[k] * m[MOM_RHS + a * 10 + k]; }
        lsq[(size_t)r * RDOF + i] = s;
    });
#ifndef PS_EMULATE
    region_factor_kernel<<<R, 32, 0, st>>>(g.invDt, R0, Mr, Vi, Nm, lsq, fit, Binv, rhsR);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
#else
    for (int r = R0; r < R0 + R; ++r) {
        double a[RDOF * RDOF], b[RDOF * RDOF]; int piv[3 * RDOF];
        region_factor(g.invDt, Mr + (size_t)r * NN, Vi + (size_t)r * NN, Nm + (size_t)r * NN, lsq + (size_t)r * RDOF, fit + (size_t)r * RDOF, Binv + (size_t)r * NN,
                      rhsR + (size_t)r * RDOF, a, b, piv, 0, 1);
    }
#endif
    (void)nChunks;
}

// a REDUCED face is a row of K_ext iff it has at least one entry of G / D^T (S_CMB:393-639):
// an adjacent cell with a pressure index and positive coefficient, or an adjacent isActive edge
// (only faces of the regions [regLo, regHi) this rank owns; lo / hi = the voxel range to visit)
void k_flag_coupled_faces(cudaStream_t st, const Geom& g, const Fields& F, int axis, uint8_t* flag, int32_t regLo, int32_t regHi, int64_t lo, int64_t hi) {
    const int8_t* FL = F.label[SL_FACE + axis]; const uint8_t* ffw = F.fluW[SL_FACE + axis]; const int32_t* FR = F.ridx[SL_FACE + axis];
    const int32_t* CA = F.aidx[SL_CENTER]; const uint8_t* clw = F.liqW[SL_CENTER];
    const int e1 = axis == 0 ? 1 : 0, e2 = axis == 2 ? 1 : 2;
    const int8_t* EL1 = F.label[SL_EDGE + e1]; const int8_t* EL2 = F.label[SL_EDGE + e2];
    const uint8_t* ew1 = F.liqW[SL_EDGE + e1]; const uint8_t* ew2 = F.liqW[SL_EDGE + e2];
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) {
        uint8_t f = 0;
        if (FL[q] == L_REDUCED && ffw[q] > 0 && FR[q] >= regLo && FR[q] < regHi) {
            const I3 fc = delin(g, SL_FACE + axis, q);
            for (int dir = 0; dir < 2; ++dir) {
                const I3 cell = dir ? fc : shifted(fc, axis, -1);
                if (!in_bounds(g, SL_CENTER, cell)) continue;
                const int64_t qc = lin(g, SL_CENTER, cell);
                if (CA[qc] >= 0 && clw[qc] > 0) f = 1;
            }
            for (int dir = 0; dir < 2; ++dir) {
                const I3 ed1 = dir ? shifted(fc, 3 - axis - e1, 1) : fc;
                const int64_t q1 = lin(g, SL_EDGE + e1, ed1);
                if (is_active(EL1[q1]) && ew1[q1] > 0) f = 1;
                const I3 ed2 = dir ? shifted(fc, 3 - axis - e2, 1) : fc;
                const int64_t q2 = lin(g, SL_EDGE + e2, ed2);
                if (is_active(EL2[q2]) && ew2[q2] > 0) f = 1;
            }
        }
        flag[q] = f;
    });
}

}  // namespace ps
