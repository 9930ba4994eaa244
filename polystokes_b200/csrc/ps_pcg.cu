// ps_pcg.cu -- the per-iteration hot path: factored operator apply + CG vector kernels
// (SURVEY.md section 8a rows O1, O2, W1, W2; K13-K15).
//
// Reference: y = A x as a product of stored factors (lib/include/ApplyPressureStressMatrix.h:102-179)
//     y = -dt K^T Mc^-1 K x  -  J^T B^-1 J x  -  1/2 [0; mu^-1 x_tau],   K = [G D^T], J = [JG JD^T]
// and the CG loop lib/include/pcg.h:268-340.  Here J is never stored: J = C K_red (see ps_assemble.cu), so
//   pass 1 : w = K_ext x, one thread per face row (8-wide slot-major ELL, coalesced 8B/4B streams, x gathered
//            through L1/L2); active rows are scaled by dt Mc^-1, coupled reduced rows keep the raw product
//   reduced: ONE CTA per region: 10 monomial moments of its rows per face axis -> t_r -> s_r = B_r^-1 t_r -> sigma_r ->
//            the same threads overwrite their rows with w_f = sigma . monomials(f)
//            (regions too large for one CTA -- doTile off -- use the chunked kernels moments -> solve -> expand instead)
//   pass 2 : y = -K_ext^T w - 1/2 mu^-1 x_tau         (one thread per DOF row, ELL widths 6/2/4), fused with
//            the dot products p.Ap, r.Ap, Ap.Ap (warp shuffle -> CTA partial -> last CTA finishes in fixed order)
// All CG scalars live in device memory; the host only polls a convergence flag every few iterations.
#include "ps_solver.hpp"
#include "ps_peer.hpp"

namespace ps {

// ---- row functors (reference semantics of one row; the emulation twins call them directly) ----
// face row r of K_ext: sum over the slots p-, p+, c-, c+, e0..e3 in this order (CompactOp, ps_solver.hpp)
PS_D double k_row(const OpArgs& A, int64_t r, const double* __restrict__ x) {
    const uint64_t word = A.kcode[r];
    const int32_t c0w = A.kcol[r];
    const int64_t cOff = A.nP + (int64_t)((uint32_t)c0w >> 30) * A.nC;
    int64_t col[8];
    col[0] = c0w & OP_COL_MASK; col[1] = A.kcol[A.nRowsExt + r]; col[2] = cOff + col[0]; col[3] = cOff + col[1];
    for (int k = 0; k < 4; ++k) col[4 + k] = A.kcol[(int64_t)(2 + k) * A.nRowsExt + r];
    double s = 0.;
    for (int k = 0; k < 8; ++k) { const int code = op_code(word, k); if (code) s += ((double)code * A.valScale) * x[col[k]]; }
    return s;
}
// cell ci: pressure row and the three centre-stress rows (same face columns, opposite sign); out[0] = (K^T w)_p, out[1+a] = (K^T w)_aa
PS_D void kt_cell_rows(const OpArgs& A, int64_t ci, const double* __restrict__ w, double* out) {
    const uint64_t word = A.ccode[ci];
    double v[6], wv[6];
    for (int k = 0; k < 6; ++k) { const int code = op_code(word, k); v[k] = (double)code * A.valScale; wv[k] = code ? w[A.ccol[(int64_t)k * A.nC + ci]] : 0.; }
    double s = 0.;
    for (int k = 0; k < 6; ++k) s += v[k] * wv[k];
    out[0] = s;
    for (int a = 0; a < 3; ++a) { double t = 0.; t += (-v[2 * a]) * wv[2 * a]; t += (-v[2 * a + 1]) * wv[2 * a + 1]; out[1 + a] = t; }
}
PS_D double kt_edge_row(const OpArgs& A, int64_t e, const double* __restrict__ w) {
    const uint64_t word = A.ecode[e];
    double s = 0.;
    for (int k = 0; k < 4; ++k) { const int code = op_code(word, k); if (code) s += ((double)code * A.valScale) * w[A.ecol[(int64_t)k * A.nE + e]]; }
    return s;
}

// t (26) from the per-axis moments M[3][10]
PS_D void moments_to_t(const double* M, double* t) {
    for (int n = 0; n < RDOF; ++n) t[n] = 0.;
    const double* A = M; const double* B = M + 10; const double* Cz = M + 20;
    t[0] = A[0]; t[3] = A[1]; t[4] = A[2]; t[5] = A[3]; for (int k = 0; k < 6; ++k) t[6 + k] = A[4 + k];
    t[1] = B[0]; t[12] = B[1]; t[13] = B[2]; t[14] = B[3]; for (int k = 0; k < 6; ++k) t[15 + k] = B[4 + k];
    t[2] += Cz[0]; t[3] += -Cz[3]; t[6] += -2. * Cz[6]; t[7] += -Cz[8]; t[8] += -0.5 * Cz[9];
    t[13] += -Cz[3]; t[16] += -Cz[6]; t[18] += -2. * Cz[8]; t[19] += -0.5 * Cz[9];
    t[21] += Cz[1]; t[22] += Cz[2]; t[23] += Cz[4]; t[24] += Cz[5]; t[25] += Cz[7];
}
// sigma[3][10] from s (26): w_f = sum_m sigma[axis][m] * mono_m
PS_D void s_to_sigma(const double* s, double* sg) {
    sg[0] = s[0]; sg[1] = s[3]; sg[2] = s[4]; sg[3] = s[5]; for (int k = 0; k < 6; ++k) sg[4 + k] = s[6 + k];
    sg[10] = s[1]; sg[11] = s[12]; sg[12] = s[13]; sg[13] = s[14]; for (int k = 0; k < 6; ++k) sg[14 + k] = s[15 + k];
    double* z = sg + 20;
    z[0] = s[2]; z[1] = s[21]; z[2] = s[22]; z[3] = -s[3] - s[13]; z[4] = s[23]; z[5] = s[24];
    z[6] = -2. * s[6] - s[16]; z[7] = s[25]; z[8] = -s[7] - 2. * s[18]; z[9] = -0.5 * s[8] - 0.5 * s[19];
}

// fixed-order finish of a dot product: called by the last CTA (or the emulation) over the CTA partials
PS_D double sum_partials(const double* p, int n) { double s = 0.; for (int i = 0; i < n; ++i) s += p[i]; return s; }

// CG scalar bookkeeping.  Every dot product is first summed per rank (fixed order) into S->red[], then --
// with more than one rank -- all-reduced in place by the host-enqueued collective (or inside the kernels over peer
// memory); the consumers below read the global value.  alpha = rsold / p.Ap (pcg.h:313).
//
// pcg.h:313-336 sweeps the vectors five times per iteration (x += a p, r -= a Ap, r.r, x.x, p = r + b p) with two
// reductions (p.Ap before, r.r between).  Here ONE kernel does all three updates:
//   update : x += alpha p, r -= alpha Ap, p = r + beta p, fused r.r, x.p, p.p      reads x, r, p, Ap   writes x, r, p   (56 B / row)
// beta = r_new.r_new / r.r is needed before r_new exists; it follows from the dots pass 2 takes while Ap is in registers:
//   |r - alpha Ap|^2 = r.r - 2 alpha r.Ap + alpha^2 Ap.Ap
// an identity of the computed vectors (no conjugacy assumed), exact up to a few ulp of r.r.  r.r itself is re-summed directly
// by the update every iteration (it is the next alpha's numerator and the base of the next recurrence step), so nothing drifts.
// The stop test needs x.x of the new x as well; it follows from the dots of the PREVIOUS update by
//   |x + alpha p|^2 = x.x + 2 alpha x.p + alpha^2 p.p
// (x_0 = 0; in CG every term is >= 0 -- |x_k| grows monotonically -- so the recurrence does not cancel).
// One reduction is consumed right after it is produced (pass 2 -> update); the update's own sums are consumed one
// whole operator apply later.
// stop test of pcg.h:316-325: min(rr, rr/xx) < tol^2
PS_D double cg_rre2(double rr, double xx) { double rre = rr; if (rr / xx < rre) rre = rr / xx; return rre; }
PS_D double cg_next_xx(double xx, double alpha, double xp, double pp) { return xx + (2. * alpha) * xp + (alpha * alpha) * pp; }
PS_D double cg_next_rr(double rr, double alpha, double rAp, double ApAp) { return (rr - (2. * alpha) * rAp) + (alpha * alpha) * ApAp; }
// the element updates of r and p, written once: the halo push recomputes the new p on the boundary entries and must round like the update
PS_D double cg_r_new(double r, double alpha, double Ap) { return fma(-alpha, Ap, r); }
PS_D double cg_p_new(double rNew, double beta, double p) { return fma(beta, p, rNew); }
// once per iteration, after every reader of the scalars is done (last CTA of the update): pcg.h:326-336
PS_D void cg_advance(PcgScalars* S, double rsold, double rr, double xx, double alpha, double pAp) {
    const double rre = cg_rre2(rr, xx);
    S->rsnew = rr; S->xmag = xx; S->xx = xx; S->rre = rre; S->pAp = pAp; S->alpha = alpha;
    if (rre < S->tol2) { S->done = 1; return; }
    S->beta = rr / rsold;
    S->rsold = rr;
    S->iter += 1;
    if (S->iter >= S->maxIter) S->done = 2;
}

#ifndef PS_EMULATE
constexpr int HOT_THREADS = 256;
constexpr int HOT_MAX_BLOCKS = 1 << 14;      // bound of the partial-sum tables; the grids themselves are SM count x resident CTAs (hot_blocks)
static_assert(HOT_THREADS == SCHED_BLOCK, "one schedule block per CTA iteration");

// Programmatic dependent launch (PDL): the kernels of the CG loop form one dependency chain on one stream, ~10 launches
// per iteration of 20-120 us each.  Every kernel of the chain is launched with programmatic stream serialization and
// starts with pdl_sync(): "launch_dependents" lets the NEXT kernel's CTAs take SM slots as soon as this kernel's CTAs
// drain (their launch latency and prologue hide under this kernel's tail), "wait" blocks until the PREVIOUS kernel has
// completed and flushed -- so nothing that reads or writes global memory may precede it (kernel parameters are fine).
__device__ __forceinline__ void pdl_sync() { asm volatile("griddepcontrol.launch_dependents;\n\tgriddepcontrol.wait;" ::: "memory"); }
template <class... KA, class... AA>
static inline void launch_chain(void (*kernel)(KA...), unsigned grid, unsigned block, cudaStream_t st, AA&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    PS_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<AA>(args)...));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
// CTA reduce; result valid in thread 0
__device__ __forceinline__ double block_sum(double v) {
    __shared__ double ws[HOT_THREADS / 32];
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.;
    if (threadIdx.x < 32) { s = threadIdx.x < HOT_THREADS / 32 ? ws[threadIdx.x] : 0.; s = warp_sum(s); }
    __syncthreads();
    return s;
}
// fixed-order sum of the CTA partials by the last CTA (thread i takes partials i, i+256, ...)
__device__ __forceinline__ double block_sum_partials(const double* p, int n) {
    double s = 0.;
    for (int i = threadIdx.x; i < n; i += HOT_THREADS) s += __ldcg(p + i);
    return block_sum(s);
}
// returns true (in every thread) for the last CTA to arrive: all partials are visible to it
__device__ __forceinline__ bool last_block(unsigned int* ticket) {
    __shared__ bool last;
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned t = atomicInc(ticket, gridDim.x - 1);
        last = (t == gridDim.x - 1);
        if (last) __threadfence();
    }
    __syncthreads();
    return last;
}

// pass 1: one thread per face row.  Per row: 8 B of codes + 6 x 4 B columns (+ 1 B mass code) in coalesced slot-major
// streams, <= 8 gathers of x (L1 / L2), 8 B of w out.  No barrier, no atomics: the 8 warps of a CTA walk their rows independently,
// two rows in flight per thread -- the sweep is bound by the two dependent round trips of a row (columns, then gathers), so
// anything that stalls a warp between rows (tickets, fences; an acquire also invalidates the L1 the gathers live in) costs more
// than it saves: the fused region term measured 2 - 4x slower than sweep + region kernel (profiles/r02_probe_s3_256_v1..v4.log).
// (6 resident CTAs per SM at 40 registers; forcing 7 or 8 spills and costs 18 %, profiles/r01_sweep_occupancy.log)
// one 256-row block of the sweep: entry e of a block schedule (SchedRanges, ps_solver.hpp)
__device__ __forceinline__ void pass1_block(const OpArgs& A, const double* __restrict__ x, double* __restrict__ w, double activeScale, const double* lut, int32_t e) {
    const int k = (int)((uint32_t)e >> 28);
    const int64_t r = A.s1.lo[k] + (int64_t)(e & 0x0fffffff) * SCHED_BLOCK + threadIdx.x;
    if (r >= A.s1.hi[k]) return;
    const double sc = A.valScale;
    const uint64_t word = __ldcs(A.kcode + r);
    int32_t c[6];
#pragma unroll
    for (int k2 = 0; k2 < 6; ++k2) c[k2] = __ldcs(A.kcol + (int64_t)k2 * A.nRowsExt + r);
    const int64_t cOff = A.nP + (int64_t)((uint32_t)c[0] >> 30) * A.nC;
    const int64_t c0 = c[0] & OP_COL_MASK, c1 = c[1];
    const int64_t col[8] = {c0, c1, cOff + c0, cOff + c1, c[2], c[3], c[4], c[5]};
    double xv[8];
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) xv[k2] = ((word >> (8 * k2)) & 0xffull) ? x[col[k2]] : 0.;
    double s = 0.;
#pragma unroll
    for (int k2 = 0; k2 < 8; ++k2) s += ((double)op_code(word, k2) * sc) * xv[k2];
    w[r] = r < A.nActiveVs ? activeScale * lut[__ldcs(A.kmc + r)] * s : s;     // coupled reduced rows keep the raw (K_red x)_f
}
__global__ void __launch_bounds__(HOT_THREADS, 6) pass1_kernel(const __grid_constant__ OpArgs A, const double* __restrict__ x, double* __restrict__ w, double activeScale, const PcgScalars* S,
                                                             const int32_t* __restrict__ sched, int nSched, const __grid_constant__ VecLink V) {    pdl_sync();

    __shared__ double lut[65];
    if (S && S->done) return;
    if (threadIdx.x < 65) lut[threadIdx.x] = A.mcInvLut[threadIdx.x];
    __syncthreads();
    if (!vec_wait(V)) { if (threadIdx.x == 0) const_cast<PcgScalars*>(S)->peerError = 1; return; }      // the neighbours' entries of x (direct halo stores)
    // owned rows in the merged block order of the ranges (SchedRanges, ps_solver.hpp)
#pragma unroll 2
    for (int g = blockIdx.x; g < nSched; g += gridDim.x) pass1_block(A, x, w, activeScale, lut, __ldg(sched + g));
}
// last CTA of a producer: v0..v2 are valid in thread 0; every rank's block receives this rank's partial sums
__device__ __forceinline__ void publish_partials(const PeerCtx& P, int slot, double v0, double v1, double v2) {
    __shared__ double pv[PEER_VALS];
    if (threadIdx.x == 0) { pv[0] = v0; pv[1] = v1; pv[2] = v2; }
    __syncthreads();
    const double vals[PEER_VALS] = {pv[0], pv[1], pv[2]};
    peer_reduce_push(P, slot, vals, PEER_VALS);
}
// y = -K_ext^T w - muScale * mu^-1 x_tau + add.  mode bit 0: accumulate dot(x, y) (p.Ap) -> S->red[0] / the peers; bit 1: also
// dot(r2, y) and dot(y, y) (r.Ap, Ap.Ap) -> red[1], red[2] while y is in registers (the update kernel's beta, see above).
// Cell sweep: one thread computes the pressure row and the xx / yy / zz stress rows of its cell from ONE set of 6
// columns, codes and w gathers (32 B of matrix per cell); edge sweep: 4 columns + 4 codes (20 B per edge).
// 6 resident CTAs per SM.  Measured on S3 256^3 (profiles/r01_sweep_occupancy.log): 4 -> 0.148 ms, 5 -> 0.137 ms, 6 -> 0.132 ms,
// 7 / 8 spill and fall back to 0.137 ms
__global__ void __launch_bounds__(HOT_THREADS, 6) pass2_kernel(const __grid_constant__ OpArgs A, const double* __restrict__ w, const double* __restrict__ x, double* __restrict__ y,
                                                            double muScale, const double* __restrict__ add, double* dotPartial, PcgScalars* S, int mode, const __grid_constant__ PeerCtx P,
                                                            const double* __restrict__ r2, const __grid_constant__ VecLink V) {    pdl_sync();

    if (S && S->done) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) vec_raise(V);                     // this rank's rows of w are in the neighbours' vectors (the push launch before this one)
    if (!vec_wait(V)) { if (threadIdx.x == 0) S->peerError = 1; return; }      // the neighbours' rows of w (direct halo stores)
    const bool dot = mode & 1, dot3 = mode & 2;
    const double sc = A.valScale;
    const int64_t nC = A.nC, nP = A.nP, oE = A.nP + 3 * A.nC;
    double acc = 0., accR = 0., accY = 0.;
    // owned rows in the merged block order: range 0 = cells, 1..3 = yz / xz / xy edges (SchedRanges, ps_solver.hpp)
#pragma unroll 1
    for (int g = blockIdx.x; g < A.nSched2; g += gridDim.x) {
        const int32_t se = __ldg(A.sched2 + g);
        const int k = (int)((uint32_t)se >> 28);
        const int64_t row = A.s2.lo[k] + (int64_t)(se & 0x0fffffff) * SCHED_BLOCK + threadIdx.x;
        if (row >= A.s2.hi[k]) continue;
        if (k == 0) {
            const int64_t ci = row;
            const uint64_t word = __ldcs(A.ccode + ci);
            double v[6], wv[6];
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                const int32_t c = __ldcs(A.ccol + (int64_t)q * nC + ci);
                v[q] = (double)op_code(word, q) * sc;
                wv[q] = ((word >> (8 * q)) & 0xffull) ? w[c] : 0.;
            }
            double s = 0.;
#pragma unroll
            for (int q = 0; q < 6; ++q) s += v[q] * wv[q];
            double yp = -s;
            if (add) yp += add[ci];
            y[ci] = yp;
            if (dot) acc += x[ci] * yp;
            if (dot3) { accR += r2[ci] * yp; accY += yp * yp; }
            const double ui = muScale != 0. ? muScale * A.uInv[ci] : 0.;      // mu^-1 is the same for xx, yy, zz of a cell
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                double t = 0.;
                t += (-v[2 * a]) * wv[2 * a]; t += (-v[2 * a + 1]) * wv[2 * a + 1];
                const int64_t jj = nP + a * nC + ci;
                const double xj = x ? x[jj] : 0.;
                double yt = -t;
                if (muScale != 0.) yt -= ui * xj;
                if (add) yt += add[jj];
                y[jj] = yt;
                acc += xj * yt;
                if (dot3) { accR += r2[jj] * yt; accY += yt * yt; }
            }
        } else {
            const int64_t e = row;
            const uint32_t word = __ldcs(A.ecode + e);
            double s = 0.;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int32_t c = __ldcs(A.ecol + (int64_t)q * A.nE + e);
                const double wv = ((word >> (8 * q)) & 0xffu) ? w[c] : 0.;
                s += ((double)op_code(word, q) * sc) * wv;
            }
            const int64_t jj = oE + e;
            const double xj = x ? x[jj] : 0.;
            double yt = -s;
            if (muScale != 0.) yt -= muScale * A.uInv[3 * nC + e] * xj;
            if (add) yt += add[jj];
            y[jj] = yt;
            acc += xj * yt;
            if (dot3) { accR += r2[jj] * yt; accY += yt * yt; }
        }
    }
    if (dot) {
        const double bs = block_sum(acc);
        if (threadIdx.x == 0) dotPartial[blockIdx.x] = bs;
        if (dot3) {
            const double bR = block_sum(accR), bY = block_sum(accY);
            if (threadIdx.x == 0) { dotPartial[gridDim.x + blockIdx.x] = bR; dotPartial[2 * gridDim.x + blockIdx.x] = bY; }
        }
        if (last_block(&S->ticket[0])) {
            const double t = block_sum_partials(dotPartial, gridDim.x);
            double tR = 0., tY = 0.;
            if (dot3) { tR = block_sum_partials(dotPartial + gridDim.x, gridDim.x); tY = block_sum_partials(dotPartial + 2 * gridDim.x, gridDim.x); }
            if (threadIdx.x == 0) { S->red[0] = t; S->red[1] = tR; S->red[2] = tY; }
            if (P.nranks > 1) publish_partials(P, 0, t, tR, tY);     // fused all-reduce, producer side (ps_peer.hpp)
        }
    }
}
// The three vector updates of one CG iteration in one sweep (see the comment above cg_rre2): alpha from the global p.Ap of
// pass 2 and the global r.r of the previous update, beta from |r - alpha Ap|^2 = r.r - 2 alpha r.Ap + alpha^2 Ap.Ap.
// x += alpha p always (pcg.h:314 runs before the stop test); r and p are only advanced if the stop test did not fire.
// The last CTA then advances the CG state (every CTA has read the scalars by then).
// (3 resident CTAs per SM at 80 registers: without the bound ptxas takes 64 and spills)
__global__ void __launch_bounds__(HOT_THREADS, 3) cg_update_kernel(RangeSet own, double* __restrict__ x, double* __restrict__ r, double* __restrict__ p, const double* __restrict__ Ap,
                                                               double* dotPartial, PcgScalars* S, const __grid_constant__ PeerCtx P, const __grid_constant__ VecLink V) {    pdl_sync();

    if (S->done) return;
    double a[3] = {S->red[0], S->red[1], S->red[2]}, b[3] = {S->red[3], S->red[4], S->red[5]};
    if (P.nranks > 1) {        // fused all-reduces, consumer side: this iteration's pass 2, and the previous update (or init)
        if (!peer_reduce_wait(P, 0, P.seqIn, a, 3)) { if (threadIdx.x == 0) S->peerError = 1; return; }
        if (!peer_reduce_wait(P, 1, P.seqIn2, b, 3)) { if (threadIdx.x == 0) S->peerError = 1; return; }
    }
    const double rsold = b[0], alpha = rsold / a[0];
    const double rrNew = cg_next_rr(rsold, alpha, a[1], a[2]);
    const double xxNew = cg_next_xx(S->xx, alpha, b[1], b[2]);
    const bool converged = cg_rre2(rrNew, xxNew) < S->tol2;
    const double beta = rrNew / rsold;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    double rr = 0., xp = 0., pp = 0.;
    if (!converged && own.n == 1 && !(own.lo[0] & 1)) {
        // one owned range (a single GPU): two consecutive elements per thread and step as 16-byte accesses -- half the memory
        // instructions of the scalar walk below
        const int64_t base = own.lo[0], total = own.total(), pairs = total >> 1;
#pragma unroll 2
        for (int64_t q = tid; q < pairs; q += stride) {
            const int64_t i = base + 2 * q;
            const double2 pv = *reinterpret_cast<const double2*>(p + i), xv = *reinterpret_cast<const double2*>(x + i);
            const double2 rv = *reinterpret_cast<const double2*>(r + i), av = __ldcs(reinterpret_cast<const double2*>(Ap + i));
            double2 xo, ro, po;
            xo.x = xv.x + alpha * pv.x; ro.x = cg_r_new(rv.x, alpha, av.x); po.x = cg_p_new(ro.x, beta, pv.x);
            xo.y = xv.y + alpha * pv.y; ro.y = cg_r_new(rv.y, alpha, av.y); po.y = cg_p_new(ro.y, beta, pv.y);
            *reinterpret_cast<double2*>(x + i) = xo; *reinterpret_cast<double2*>(r + i) = ro; *reinterpret_cast<double2*>(p + i) = po;
            rr += ro.x * ro.x; xp += xo.x * po.x; pp += po.x * po.x;
            rr += ro.y * ro.y; xp += xo.y * po.y; pp += po.y * po.y;
        }
        if ((total & 1) && tid == 0) {
            const int64_t i = base + total - 1;
            const double pi = p[i];
            const double xi = x[i] + alpha * pi, ri = cg_r_new(r[i], alpha, Ap[i]);
            const double pn = cg_p_new(ri, beta, pi);
            x[i] = xi; r[i] = ri; p[i] = pn;
            rr += ri * ri; xp += xi * pn; pp += pn * pn;
        }
    } else if (!converged) {
#pragma unroll 4
        for (RangeWalk<7> it(own, tid); it.valid(own); it.step(own, stride)) {
            const int64_t i = it.j;
            const double pi = p[i];
            const double xi = x[i] + alpha * pi, ri = cg_r_new(r[i], alpha, Ap[i]);
            const double pn = cg_p_new(ri, beta, pi);
            x[i] = xi; r[i] = ri; p[i] = pn;
            rr += ri * ri; xp += xi * pn; pp += pn * pn;
        }
    } else {
#pragma unroll 4
        for (RangeWalk<7> it(own, tid); it.valid(own); it.step(own, stride)) { const int64_t i = it.j; x[i] += alpha * p[i]; }
    }
    const double brr = block_sum(rr), bxp = block_sum(xp), bpp = block_sum(pp);
    if (threadIdx.x == 0) { dotPartial[blockIdx.x] = brr; dotPartial[gridDim.x + blockIdx.x] = bxp; dotPartial[2 * gridDim.x + blockIdx.x] = bpp; }
    if (last_block(&S->ticket[3])) {
        if (!converged && threadIdx.x == 0) vec_raise(V);      // the boundary entries of the new p reached the neighbours with the push launch before this one
        const double trr = block_sum_partials(dotPartial, gridDim.x), txp = block_sum_partials(dotPartial + gridDim.x, gridDim.x), tpp = block_sum_partials(dotPartial + 2 * gridDim.x, gridDim.x);
        if (threadIdx.x == 0) { cg_advance(S, rsold, rrNew, xxNew, alpha, a[0]); S->red[3] = trr; S->red[4] = txp; S->red[5] = tpp; }
        if (P.nranks > 1) publish_partials(P, 1, trr, txp, tpp);
    }
}
__global__ void __launch_bounds__(HOT_THREADS) cg_init_kernel(RangeSet own, const double* __restrict__ b, double* x, double* r, double* p, double* dotPartial, PcgScalars* S, double tol, int maxIter,
                                                             const __grid_constant__ PeerCtx P) {    pdl_sync();

    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    double rr = 0.;
    for (RangeWalk<7> it(own, tid); it.valid(own); it.step(own, stride)) {
        const int64_t i = it.j;
        const double bi = b[i];
        x[i] = 0.; r[i] = bi; p[i] = bi; rr += bi * bi;
    }
    const double brr = block_sum(rr);
    if (threadIdx.x == 0) dotPartial[blockIdx.x] = brr;
    if (last_block(&S->ticket[2])) {
        const double rs = block_sum_partials(dotPartial, gridDim.x);
        if (threadIdx.x == 0) {
            S->rsold = 0.; S->pAp = 0.; S->alpha = 0.; S->beta = 0.; S->rsnew = 0.; S->xmag = 0.; S->rre = 0.;
            S->red[0] = 0.; S->red[1] = 0.; S->red[2] = 0.; S->red[3] = rs; S->red[4] = 0.; S->red[5] = rs; S->red[6] = rs; S->xx = 0.;      // r = p = b: r.r = p.p = b.b; x = 0: x.p = 0
            S->iter = 0; S->done = 0; S->maxIter = maxIter; S->tol2 = tol * tol;
            S->ticket[0] = 0; S->ticket[3] = 0; S->ticket[4] = 0; S->ticket[5] = 0;      // nothing else is in flight: heal tickets after an aborted solve
        }
        if (P.nranks > 1) publish_partials(P, 1, rs, 0., rs);
    }
}
// after the all-reduce of b.b: rsold, and the b == 0 early out
__global__ void cg_begin_kernel(PcgScalars* S, const __grid_constant__ PeerCtx P) {    pdl_sync();

    double bb[3] = {S->red[3], S->red[4], S->red[5]};
    if (P.nranks > 1 && !peer_reduce_wait(P, 1, P.seqIn, bb, 3)) { if (threadIdx.x == 0) { S->peerError = 1; S->done = 1; } return; }
    if (threadIdx.x == 0) { S->red[6] = bb[0]; S->rsold = bb[0]; S->done = (bb[0] == 0.) ? 1 : 0; }
}
// Halo push over peer memory with the entries stored at their FINAL place: the neighbours map this rank's vector arena (PeerLink::vecBase), entry j
// of my vector goes to entry j of theirs (vectors are global-length everywhere).  Nothing is unpacked on the other side: the kernel
// that consumes the vector there waits for the flag at its head (VecLink).  This launch never waits, so it cannot stall behind a
// slower neighbour; its tail (two system fences + the flag's NVLink trip) hides under the consumer's launch.
__global__ void __launch_bounds__(256) halo_push_direct_kernel(int64_t n0, int64_t n1, const int32_t* __restrict__ idx, const double* __restrict__ v,
                                                              double* __restrict__ dst0, double* __restrict__ dst1, const PcgScalars* S) {    pdl_sync();

    if (S && S->done) return;
    const int64_t n = n0 + n1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t j = idx[i];
        const double val = v[j];
        if (i < n0) dst0[j] = val; else dst1[j] = val;
    }
}
// The push of the NEW p, launched before the x/r/p update: p_new = (r - alpha Ap) + beta p on the boundary entries, from the old
// vectors and the same scalars the update is about to form (same reductions, same expressions -- bit-identical values).
__global__ void __launch_bounds__(256) halo_push_p_kernel(int64_t n0, int64_t n1, const int32_t* __restrict__ idx, const double* __restrict__ r, const double* __restrict__ p,
                                                         const double* __restrict__ Ap, double* __restrict__ dst0, double* __restrict__ dst1, PcgScalars* S, const __grid_constant__ PeerCtx P) {
    pdl_sync();
    if (S->done) return;
    double a[3] = {S->red[0], S->red[1], S->red[2]}, b[3] = {S->red[3], S->red[4], S->red[5]};
    if (P.nranks > 1) {
        if (!peer_reduce_wait(P, 0, P.seqIn, a, 3)) { if (threadIdx.x == 0) S->peerError = 1; return; }
        if (!peer_reduce_wait(P, 1, P.seqIn2, b, 3)) { if (threadIdx.x == 0) S->peerError = 1; return; }
    }
    const double rsold = b[0], alpha = rsold / a[0];
    const double rrNew = cg_next_rr(rsold, alpha, a[1], a[2]);
    const double xxNew = cg_next_xx(S->xx, alpha, b[1], b[2]);
    if (cg_rre2(rrNew, xxNew) < S->tol2) return;          // the update will stop here: nobody reads another p
    const double beta = rrNew / rsold;
    const int64_t n = n0 + n1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t j = idx[i];
        const double val = cg_p_new(cg_r_new(r[j], alpha, Ap[j]), beta, p[j]);
        if (i < n0) dst0[j] = val; else dst1[j] = val;
    }
}
// Both sides in ONE launch (<= one CTA per SM, so every CTA is resident): each CTA first pushes its share of my boundary
// entries, the last CTA to finish raises the neighbours' flags, then every CTA waits for MY flags and scatters its share of
// what the neighbours stored here.  No CTA waits before it has pushed, so two ranks can never wait on each other.
__global__ void __launch_bounds__(256) halo_exchange_kernel(int64_t ns0, int64_t ns1, const int32_t* __restrict__ sendIdx, double* __restrict__ dst0, double* __restrict__ dst1,
                                                           unsigned long long* dflag0, unsigned long long* dflag1,
                                                           int64_t nr0, int64_t nr1, const int32_t* __restrict__ recvIdx, const double* src0, const double* src1,
                                                           const unsigned long long* sflag0, const unsigned long long* sflag1,
                                                           unsigned long long seq, double* v, PcgScalars* S, int respectDone, unsigned int* ticket) {
    pdl_sync();
    if (respectDone && S->done) return;
    const int64_t ns = ns0 + ns1, nr = nr0 + nr1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += (int64_t)gridDim.x * blockDim.x) {
        const double val = v[sendIdx[i]];
        if (i < ns0) dst0[i] = val; else dst1[i - ns0] = val;
    }
    // One system fence per CTA, not per thread (membar.sys by every warp costs ~20 us here): the CTA barrier orders
    // all threads' stores before thread 0's fence, the fence makes them visible system-wide before the ticket,
    // and the last CTA's release store publishes the flag after every CTA's fence (cumulative).
    __shared__ int ok;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        const unsigned t = atomicInc(ticket, gridDim.x - 1);
        if (t == gridDim.x - 1) {
            __threadfence_system();
            if (dflag0) peer_st_flag(dflag0, seq);
            if (dflag1) peer_st_flag(dflag1, seq);
        }
        bool good = true;
        if (sflag0) good = peer_wait_flag(sflag0, seq) && good;
        if (sflag1) good = peer_wait_flag(sflag1, seq) && good;
        ok = good ? 1 : 0;
    }
    __syncthreads();
    if (!ok) { if (threadIdx.x == 0) S->peerError = 1; return; }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nr; i += (int64_t)gridDim.x * blockDim.x)
        v[recvIdx[i]] = __ldcg(i < nr0 ? src0 + i : src1 + (i - nr0));
}
__global__ void __launch_bounds__(256) halo_pack_kernel(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ v, double* __restrict__ buf, const PcgScalars* S) {    pdl_sync();

    if (S && S->done) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) buf[i] = v[idx[i]];
}
__global__ void __launch_bounds__(256) halo_unpack_kernel(int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ buf, double* __restrict__ v, const PcgScalars* S) {    pdl_sync();

    if (S && S->done) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v[idx[i]] = buf[i];
}
// persistent grid-stride sizing: exactly one wave = SM count x resident CTAs of this kernel (no partial second wave)
template <class K>
static inline int hot_blocks(K kernel, int64_t n) {
    static thread_local std::vector<std::pair<const void*, int>> cache;
    int resident = 0;
    for (auto& e : cache) if (e.first == (const void*)kernel) resident = e.second;
    if (!resident) {
        int per = 1;
        const int sms = sm_count();
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kernel, HOT_THREADS, 0);
        resident = std::min(sms * std::max(per, 1), HOT_MAX_BLOCKS);
        cache.push_back({(const void*)kernel, resident});
    }
    int64_t b = (n + HOT_THREADS - 1) / HOT_THREADS;
    if (b > resident) b = resident;
    if (b < 1) b = 1;
    return (int)b;
}

void k_pass1(cudaStream_t st, const OpArgs& A, const double* x, double* w, double activeScale, const PcgScalars* S, const VecLink& V) {
    const int n = A.nSched1;
    if (n <= 0 && !V.waitSeq) return;
    launch_chain(pass1_kernel, hot_blocks(pass1_kernel, (int64_t)std::max(n, 1) * HOT_THREADS), HOT_THREADS, st, A, x, w, activeScale, S, A.sched1, n, V);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_pass2(cudaStream_t st, const OpArgs& A, const double* w, const double* x, double* y, double muScale, const double* add, double* dotPartial, const PeerCtx& P, PcgScalars* scal, int mode, const double* r2, const VecLink& V) {
    const int64_t rows = A.rowsP.total() + A.rowsE.total();
    if (rows <= 0 && !(mode & 1)) return;
    launch_chain(pass2_kernel, hot_blocks(pass2_kernel, rows), HOT_THREADS, st, A, w, x, y, muScale, add, dotPartial, scal, mode, P, r2, V);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_cg_update(cudaStream_t st, const RangeSet& own, double* x, double* r, double* p, const double* Ap, double* dotPartial, PcgScalars* scal, const PeerCtx& P, const VecLink& V) {
    launch_chain(cg_update_kernel, hot_blocks(cg_update_kernel, own.total()), HOT_THREADS, st, own, x, r, p, Ap, dotPartial, scal, P, V);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_cg_init(cudaStream_t st, const RangeSet& own, const double* b, double* x, double* r, double* p, double* dotPartial, PcgScalars* scal, double tol, int maxIter, const PeerCtx& P) {
    launch_chain(cg_init_kernel, hot_blocks(cg_init_kernel, own.total()), HOT_THREADS, st, own, b, x, r, p, dotPartial, scal, tol, maxIter, P);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_cg_begin(cudaStream_t st, PcgScalars* scal, const PeerCtx& P) {
    launch_chain(cg_begin_kernel, 1, 32, st, scal, P);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_halo_pack(cudaStream_t st, int64_t n, const int32_t* idx, const double* v, double* buf, const PcgScalars* S) {
    if (n <= 0) return;
    launch_chain(halo_pack_kernel, (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 4), 256, st, n, idx, v, buf, S);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_halo_push_direct(cudaStream_t st, int64_t n0, int64_t n1, const int32_t* idx, const double* v, double* dst0, double* dst1, const PcgScalars* S) {
    const int64_t n = n0 + n1;
    if (n <= 0) return;
    launch_chain(halo_push_direct_kernel, (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)sm_count())), 256, st, n0, n1, idx, v, dst0, dst1, S);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_halo_push_p(cudaStream_t st, int64_t n0, int64_t n1, const int32_t* idx, const double* r, const double* p, const double* Ap, double* dst0, double* dst1, PcgScalars* S, const PeerCtx& P) {
    const int64_t n = n0 + n1;
    if (n <= 0) return;
    launch_chain(halo_push_p_kernel, (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)sm_count())), 256, st, n0, n1, idx, r, p, Ap, dst0, dst1, S, P);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_halo_exchange_peer(cudaStream_t st, int64_t ns0, int64_t ns1, const int32_t* sendIdx, double* dst0, double* dst1, unsigned long long* dflag0, unsigned long long* dflag1,
                          int64_t nr0, int64_t nr1, const int32_t* recvIdx, const double* src0, const double* src1, const unsigned long long* sflag0, const unsigned long long* sflag1,
                          unsigned long long seq, double* v, PcgScalars* S, bool respectDone, unsigned int* ticket) {
    const int64_t n = std::max(ns0 + ns1, nr0 + nr1);
    launch_chain(halo_exchange_kernel, (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)sm_count())), 256, st, ns0, ns1, sendIdx, dst0, dst1, dflag0, dflag1,
                 nr0, nr1, recvIdx, src0, src1, sflag0, sflag1, seq, v, S, respectDone ? 1 : 0, ticket);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void k_halo_unpack(cudaStream_t st, int64_t n, const int32_t* idx, const double* buf, double* v, const PcgScalars* S) {
    if (n <= 0) return;
    launch_chain(halo_unpack_kernel, (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)sm_count() * 4), 256, st, n, idx, buf, v, S);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
#else  // ---- serial twins ----
void k_pass1(cudaStream_t, const OpArgs& A, const double* x, double* w, double activeScale, const PcgScalars* S, const VecLink&) {
    if (S && S->done) return;
    for (int64_t l = 0; l < A.rowsK.total(); ++l) { const int64_t r = A.rowsK.at(l); const double s = k_row(A, r, x); w[r] = r < A.nActiveVs ? activeScale * A.mcInvLut[A.kmc[r]] * s : s; }
}
void k_pass2(cudaStream_t, const OpArgs& A, const double* w, const double* x, double* y, double muScale, const double* add, double*, const PeerCtx&, PcgScalars* S, int mode, const double* r2, const VecLink&) {
    if (S && S->done) return;
    double acc = 0., accR = 0., accY = 0.;
    auto finish = [&](int64_t j, double ktw) {
        double v = -ktw;
        const double xj = (mode & 1) || j >= A.nP ? (x ? x[j] : 0.) : 0.;
        if (j >= A.nP && muScale != 0.) v -= muScale * A.uInv[j - A.nP] * xj;
        if (add) v += add[j];
        y[j] = v; acc += xj * v;
        if (mode & 2) { accR += r2[j] * v; accY += v * v; }
    };
    for (int64_t l = 0; l < A.rowsP.total(); ++l) {
        const int64_t ci = A.rowsP.at(l);
        double out[4];
        kt_cell_rows(A, ci, w, out);
        finish(ci, out[0]);
        for (int a = 0; a < 3; ++a) finish(A.nP + a * A.nC + ci, out[1 + a]);
    }
    for (int64_t l = 0; l < A.rowsE.total(); ++l) { const int64_t e = A.rowsE.at(l); finish(A.nP + 3 * A.nC + e, kt_edge_row(A, e, w)); }
    if (mode & 1) { S->red[0] = acc; S->red[1] = accR; S->red[2] = accY; }
}
void k_cg_update(cudaStream_t, const RangeSet& own, double* x, double* r, double* p, const double* Ap, double*, PcgScalars* S, const PeerCtx&, const VecLink&) {
    if (S->done) return;
    const double rsold = S->red[3], alpha = rsold / S->red[0];
    const double rrNew = cg_next_rr(rsold, alpha, S->red[1], S->red[2]);
    const double xxNew = cg_next_xx(S->xx, alpha, S->red[4], S->red[5]);
    const bool converged = cg_rre2(rrNew, xxNew) < S->tol2;
    const double beta = rrNew / rsold;
    double rr = 0., xp = 0., pp = 0.;
    for (int64_t l = 0; l < own.total(); ++l) {
        const int64_t i = own.at(l);
        x[i] += alpha * p[i];
        if (!converged) { r[i] = cg_r_new(r[i], alpha, Ap[i]); p[i] = cg_p_new(r[i], beta, p[i]); rr += r[i] * r[i]; xp += x[i] * p[i]; pp += p[i] * p[i]; }
    }
    cg_advance(S, rsold, rrNew, xxNew, alpha, S->red[0]);
    S->red[3] = rr; S->red[4] = xp; S->red[5] = pp;
}
void k_cg_init(cudaStream_t, const RangeSet& own, const double* b, double* x, double* r, double* p, double*, PcgScalars* S, double tol, int maxIter, const PeerCtx&) {
    double rr = 0.;
    for (int64_t l = 0; l < own.total(); ++l) { const int64_t i = own.at(l); x[i] = 0.; r[i] = b[i]; p[i] = b[i]; rr += b[i] * b[i]; }
    S->rsold = S->pAp = S->alpha = S->beta = S->rsnew = S->xmag = S->rre = S->xx = 0.; S->red[0] = S->red[1] = S->red[2] = 0.; S->red[3] = rr; S->red[4] = 0.; S->red[5] = rr; S->red[6] = rr;
    S->iter = 0; S->done = 0; S->maxIter = maxIter; S->tol2 = tol * tol;
}
void k_cg_begin(cudaStream_t, PcgScalars* S, const PeerCtx&) { S->red[6] = S->red[3]; S->rsold = S->red[3]; S->done = (S->red[3] == 0.) ? 1 : 0; }
void k_halo_pack(cudaStream_t, int64_t n, const int32_t* idx, const double* v, double* buf, const PcgScalars* S) { if (S && S->done) return; for (int64_t i = 0; i < n; ++i) buf[i] = v[idx[i]]; }
void k_halo_unpack(cudaStream_t, int64_t n, const int32_t* idx, const double* buf, double* v, const PcgScalars* S) { if (S && S->done) return; for (int64_t i = 0; i < n; ++i) v[idx[i]] = buf[i]; }
#endif

// ---- BiCGSTAB fallback (bicgstab_external_matrix_A, lib/include/pcg.h:134-200) ---------------------------------
// One generic sweep: f(i, a, b) updates element i and may add to two running sums; the sums end up rank-local in
// S->bred[0..1] (CTA partials summed by the last CTA in fixed order).  The fallback runs only after CG has used
// up maxSolverIterations, so these kernels favour clarity; each is still one coalesced pass over the vectors.
// scalar bookkeeping of one iteration, in the reference's statement order
PS_D void bicg_stage(PcgScalars* S, int stage) {
    if (S->done) return;
    if (stage == 0) {            // pcg.h:171-173
        S->rhoOld = S->rhoCurr; S->rhoCurr = S->bred[0];
        S->beta = (S->rhoCurr / S->rhoOld) * (S->alpha / S->omega);
    } else if (stage == 1) {     // pcg.h:176
        S->alpha = S->rhoCurr / S->bred[0];
    } else if (stage == 2) {     // pcg.h:181
        S->omega = S->bred[0] / S->bred[1];
    } else {                     // pcg.h:185-193: the reference compares rre with tol (not tol^2) here
        const double xmag = sqrt(S->bred[0]), rsnew = S->bred[1];
        double rre = rsnew;
        if (sqrt(rsnew) / xmag < rre) rre = sqrt(rsnew) / xmag;
        S->xmag = xmag; S->rsnew = rsnew; S->rre = rre;
        if (rre < S->tol) { S->done = 1; return; }
        S->iter += 1;
        if (S->iter >= S->maxIter) S->done = 2;
    }
}
#ifndef PS_EMULATE
template <class F>
__global__ void __launch_bounds__(HOT_THREADS) vec_sweep_kernel(RangeSet own, double* dotPartial, PcgScalars* S, int nred, int slot, bool respectDone, F f) {
    if (respectDone && S->done) return;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    double a = 0., b = 0.;
    for (RangeWalk<7> it(own, tid); it.valid(own); it.step(own, stride)) f(it.j, a, b);
    if (nred > 0) {
        const double ba = block_sum(a), bb = block_sum(b);
        if (threadIdx.x == 0) { dotPartial[blockIdx.x] = ba; dotPartial[gridDim.x + blockIdx.x] = bb; }
        if (last_block(&S->ticket[6])) {
            const double ta = block_sum_partials(dotPartial, gridDim.x), tb = block_sum_partials(dotPartial + gridDim.x, gridDim.x);
            if (threadIdx.x == 0) { S->bred[slot] = ta; if (nred > 1) S->bred[slot + 1] = tb; }
        }
    }
}
template <class F>
static void vec_sweep(cudaStream_t st, const RangeSet& own, double* dotPartial, PcgScalars* S, int nred, int slot, bool respectDone, F f) {
    vec_sweep_kernel<<<hot_blocks(vec_sweep_kernel<F>, own.total()), HOT_THREADS, 0, st>>>(own, dotPartial, S, nred, slot, respectDone, f);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
#else
template <class F>
static void vec_sweep(cudaStream_t, const RangeSet& own, double*, PcgScalars* S, int nred, int slot, bool respectDone, F f) {
    if (respectDone && S->done) return;
    double a = 0., b = 0.;
    for (int64_t l = 0; l < own.total(); ++l) f(own.at(l), a, b);
    if (nred > 0) { S->bred[slot] = a; if (nred > 1) S->bred[slot + 1] = b; }
}
#endif
// pcg.h:149-168: x = 0 => r = b - A 0 = b, rhat = r, p = v = 0, rho = alpha = omega = 1
void k_bicg_init(cudaStream_t st, const RangeSet& own, const double* b, double* x, double* r, double* rhat, double* p, double* v, PcgScalars* S, double tol, int maxIter) {
    vec_sweep(st, own, nullptr, S, 0, 0, false, PS_LAMBDA(int64_t i, double&, double&) { const double bi = b[i]; x[i] = 0.; r[i] = bi; rhat[i] = bi; p[i] = 0.; v[i] = 0.; });
    ps_for(st, 1, PS_LAMBDA(int64_t) {
        S->rhoCurr = 1.; S->rhoOld = 1.; S->alpha = 1.; S->beta = 0.; S->omega = 1.; S->xmag = 0.; S->rsnew = 0.; S->rre = 0.;
        S->bred[0] = 0.; S->bred[1] = 0.; S->tol = tol; S->tol2 = tol * tol; S->iter = 0; S->maxIter = maxIter; S->done = maxIter > 0 ? 0 : 2;
        S->ticket[6] = 0;
    });
}
void k_bicg_dot(cudaStream_t st, const RangeSet& own, const double* a0, const double* b0, const double* a1, const double* b1, double* dotPartial, PcgScalars* S) {
    if (a1) vec_sweep(st, own, dotPartial, S, 2, 0, true, PS_LAMBDA(int64_t i, double& a, double& b) { a += a0[i] * b0[i]; b += a1[i] * b1[i]; });
    else vec_sweep(st, own, dotPartial, S, 1, 0, true, PS_LAMBDA(int64_t i, double& a, double&) { a += a0[i] * b0[i]; });
}
void k_bicg_stage(cudaStream_t st, PcgScalars* S, int stage) { ps_for(st, 1, PS_LAMBDA(int64_t) { bicg_stage(S, stage); }); }
// pcg.h:174  p = r + beta (p - omega v)
void k_bicg_update_p(cudaStream_t st, const RangeSet& own, double* p, const double* r, const double* v, const PcgScalars* S) {
    vec_sweep(st, own, nullptr, const_cast<PcgScalars*>(S), 0, 0, true, PS_LAMBDA(int64_t i, double&, double&) { p[i] = r[i] + S->beta * (p[i] - S->omega * v[i]); });
}
// pcg.h:177-179  h = x + alpha p (kept in x),  s = r - alpha v
void k_bicg_update_hs(cudaStream_t st, const RangeSet& own, double* x, double* s, const double* r, const double* p, const double* v, const PcgScalars* S) {
    vec_sweep(st, own, nullptr, const_cast<PcgScalars*>(S), 0, 0, true, PS_LAMBDA(int64_t i, double&, double&) { const double al = S->alpha; x[i] = x[i] + al * p[i]; s[i] = r[i] - al * v[i]; });
}
// pcg.h:182-185  x = h + omega s, fused x.x
void k_bicg_update_x(cudaStream_t st, const RangeSet& own, double* x, const double* s, double* dotPartial, PcgScalars* S) {
    vec_sweep(st, own, dotPartial, S, 1, 0, true, PS_LAMBDA(int64_t i, double& a, double&) { const double xi = x[i] + S->omega * s[i]; x[i] = xi; a += xi * xi; });
}
// pcg.h:186-187  err = b - A x, rsnew = err.err  (into bred[1]; bred[0] keeps x.x)
void k_bicg_err(cudaStream_t st, const RangeSet& own, const double* b, const double* Ax, double* dotPartial, PcgScalars* S) {
    vec_sweep(st, own, dotPartial, S, 1, 1, true, PS_LAMBDA(int64_t i, double& a, double&) { const double e = b[i] - Ax[i]; a += e * e; });
}
// pcg.h:195  r = s - omega t
void k_bicg_update_r(cudaStream_t st, const RangeSet& own, double* r, const double* s, const double* t, const PcgScalars* S) {
    vec_sweep(st, own, nullptr, const_cast<PcgScalars*>(S), 0, 0, true, PS_LAMBDA(int64_t i, double&, double&) { r[i] = s[i] - S->omega * t[i]; });
}

// halo discovery: flag[c] = 1 for every column c of a non-empty slot of the given rows that `colsOwned` contains
void k_mark_K_columns(cudaStream_t st, const OpArgs& A, const RowSet& rows, const RangeSet& colsOwned, uint8_t* flag) {
    const RowSet R = rows; const RangeSet Cs = colsOwned;
    const uint64_t* kcode = A.kcode; const int32_t* kcol = A.kcol; const int64_t nRows = A.nRowsExt, nP = A.nP, nC = A.nC;
    ps_for(st, R.total(), PS_LAMBDA(int64_t l) {
        const int64_t r = R.at(l);
        const uint64_t word = kcode[r];
        const int32_t c0w = kcol[r];
        const int64_t cOff = nP + (int64_t)((uint32_t)c0w >> 30) * nC;
        int64_t col[8];
        col[0] = c0w & OP_COL_MASK; col[1] = kcol[nRows + r]; col[2] = cOff + col[0]; col[3] = cOff + col[1];
        for (int k = 0; k < 4; ++k) col[4 + k] = kcol[(int64_t)(2 + k) * nRows + r];
        for (int k = 0; k < 8; ++k) if (op_code(word, k) && Cs.has(col[k])) flag[col[k]] = 1;
    });
}
void k_mark_Kt_columns(cudaStream_t st, const OpArgs& A, const RowSet& cellRows, const RowSet& edgeRows, const RowSet& colsOwned, uint8_t* flag) {
    const RowSet Rc = cellRows, Re = edgeRows, Cs = colsOwned;
    const uint64_t* ccode = A.ccode; const int32_t* ccol = A.ccol; const uint32_t* ecode = A.ecode; const int32_t* ecol = A.ecol;
    const int64_t nC = A.nC, nE = A.nE;
    ps_for(st, Rc.total(), PS_LAMBDA(int64_t l) {
        const int64_t ci = Rc.at(l);
        const uint64_t word = ccode[ci];
        for (int k = 0; k < 6; ++k) { const int32_t c = ccol[(int64_t)k * nC + ci]; if (op_code(word, k) && Cs.has(c)) flag[c] = 1; }
    });
    ps_for(st, Re.total(), PS_LAMBDA(int64_t l) {
        const int64_t e = Re.at(l);
        const uint64_t word = ecode[e];
        for (int k = 0; k < 4; ++k) { const int32_t c = ecol[(int64_t)k * nE + e]; if (op_code(word, k) && Cs.has(c)) flag[c] = 1; }
    });
}

// ---- reduced regions -------------------------------------------------------------------------------
// t_r = J_r x = sum_f c_f (K_red x)_f ;  s_r = B_r^-1 (extraScale*extra_r + tScale*t_r) ;  w_f = scale * c_f . s_r
// Every entry of c_f is +-{1, 1/2, 2} times one of the 10 monomials {1,x,y,z,xx,xy,xz,yy,yz,zz} of the face
// offset (S.cpp:2107-2149), so a chunk of same-axis rows only accumulates 10 moments per row; the 26-vector
// t_r is a fixed sparse image of the 3x10 moments, and w_f is a 10-term polynomial with coefficients
// sigma[axis] = (that image)^T s_r.
#ifndef PS_EMULATE
constexpr int RED_THREADS = 256;
constexpr int MOM_THREADS = 64;
// the small solve of one region, shared by reduced_finish_kernel and the fused tail of reduced_moments_kernel (lane = thread
// index, at least 32 threads, all of them call): ordered sum of the chunk partials -> t -> s = B^-1 t -> sigma
__device__ __forceinline__ void region_solve(int r, int lane, const int32_t* __restrict__ chunkStart, const int32_t* __restrict__ chunk, const double* partial,
                                             const double* __restrict__ Binv, const double* __restrict__ extra, double extraScale, double tScale,
                                             double* tOut, double* sOut, double* __restrict__ sigma, double* M, double* t, double* sv) {
    if (lane < 30) {
        const int axis = lane / 10, k = lane % 10;
        double s = 0.;
        if (tScale != 0.)
            for (int ch = chunkStart[r]; ch < chunkStart[r + 1]; ++ch) if (chunk[4 * ch + 3] == axis) s += __ldcg(partial + (size_t)ch * 10 + k);
        M[lane] = s;
    }
    __syncthreads();
    if (lane == 0) moments_to_t(M, t);
    __syncthreads();
    if (lane < RDOF) {
        double v = tScale * t[lane];
        if (extra) v += extraScale * extra[(size_t)r * RDOF + lane];
        t[lane] = v; if (tOut) tOut[(size_t)r * RDOF + lane] = v;
    }
    __syncthreads();
    if (lane < RDOF) {
        const double* B = Binv + (size_t)r * RDOF * RDOF + lane * RDOF;
        double s = 0.;
#pragma unroll
        for (int j = 0; j < RDOF; ++j) s += B[j] * t[j];
        sv[lane] = s; if (sOut) sOut[(size_t)r * RDOF + lane] = s;
    }
    __syncthreads();
    if (lane == 0) { double sg[30]; s_to_sigma(sv, sg); for (int k = 0; k < 30; ++k) sigma[(size_t)r * 30 + k] = sg[k]; }
}
// one small CTA per (region, axis) chunk of coupled reduced rows: 10 monomial moments of w_f = (K_red x)_f (written by pass 1).
// With `regionTicket` the LAST chunk of a region to finish also runs the region's small solve (t -> s = B^-1 t -> sigma):
// the sums are taken in chunk order whoever comes last, so the result does not depend on the schedule.
__global__ void __launch_bounds__(MOM_THREADS) reduced_moments_kernel(double dx, const uint32_t* __restrict__ rowXYZ, const int32_t* __restrict__ chunk, const int32_t* __restrict__ chunkStart,
                                                                     const double* __restrict__ com, const double* __restrict__ wRows, double* partial, const double* __restrict__ Binv,
                                                                     double* __restrict__ sigma, unsigned int* regionTicket, const PcgScalars* S, int chunk0) {    pdl_sync();

    if (S && S->done) return;
    __shared__ double red[MOM_THREADS / 32][10];
    __shared__ double M[30], t[RDOF], sv[RDOF];
    __shared__ bool last;
    const int ch = chunk0 + blockIdx.x;
    const int region = chunk[4 * ch], begin = chunk[4 * ch + 1], end = chunk[4 * ch + 2];
    const double cm[3] = {com[3 * region], com[3 * region + 1], com[3 * region + 2]};
    double acc[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) acc[k] = 0.;
#pragma unroll 4
    for (int row = begin + threadIdx.x; row < end; row += MOM_THREADS) {
        const double gk = __ldcs(wRows + row);
        double m[10];
        row_monomials(dx, __ldcs(rowXYZ + row), cm, m);
#pragma unroll
        for (int k = 0; k < 10; ++k) acc[k] += m[k] * gk;
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        const double v = warp_sum(acc[k]);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 10) {
        double s = 0.;
#pragma unroll
        for (int wI = 0; wI < MOM_THREADS / 32; ++wI) s += red[wI][threadIdx.x];
        partial[(size_t)ch * 10 + threadIdx.x] = s;
    }
    if (!regionTicket) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned nch = (unsigned)(chunkStart[region + 1] - chunkStart[region]);
        const unsigned tk = atomicInc(regionTicket + region, nch - 1);
        last = (tk == nch - 1);
        if (last) __threadfence();
    }
    __syncthreads();
    if (last) region_solve(region, threadIdx.x, chunkStart, chunk, partial, Binv, nullptr, 0., 1., nullptr, nullptr, sigma, M, t, sv);
}
// one warp per region: ordered sum of the chunk partials -> t -> s = B^-1 t -> sigma
__global__ void __launch_bounds__(32) reduced_finish_kernel(const int32_t* __restrict__ chunkStart, const int32_t* __restrict__ chunk, const double* __restrict__ partial,
                                                           const double* __restrict__ Binv, const double* __restrict__ extra, double extraScale, double tScale,
                                                           double* __restrict__ tOut, double* __restrict__ sOut, double* __restrict__ sigma, const PcgScalars* S, int region0) {    pdl_sync();

    if (S && S->done) return;
    __shared__ double M[30], t[RDOF], sv[RDOF];
    region_solve(region0 + blockIdx.x, threadIdx.x, chunkStart, chunk, partial, Binv, extra, extraScale, tScale, tOut, sOut, sigma, M, t, sv);
}
// w_f = scale * sigma[region][axis] . monomials(f): one thread per coupled reduced row (sigma / com of a region are shared by
// neighbouring rows and come through L1)
__global__ void __launch_bounds__(RED_THREADS) reduced_expand_kernel(double dx, const uint32_t* __restrict__ rowXYZ, const int32_t* __restrict__ rowRegion, const double* __restrict__ com,
                                                                    const double* __restrict__ sigma, double* __restrict__ wRows, double scale, const PcgScalars* S, int rowLo, int rowHi) {    pdl_sync();

    if (S && S->done) return;
    for (int row = rowLo + blockIdx.x * RED_THREADS + threadIdx.x; row < rowHi; row += gridDim.x * RED_THREADS) {
        const uint32_t xyz = __ldcs(rowXYZ + row);
        const int region = __ldcs(rowRegion + row), axis = (int)(xyz >> 30);
        const double cm[3] = {__ldg(com + 3 * region), __ldg(com + 3 * region + 1), __ldg(com + 3 * region + 2)};
        const double* sg = sigma + (size_t)region * 30 + axis * 10;
        double m[10];
        row_monomials(dx, xyz, cm, m);
        double v = 0.;
#pragma unroll
        for (int k = 0; k < 10; ++k) v += __ldg(sg + k) * m[k];
        wRows[row] = scale * v;
    }
}
// The whole reduced term of one apply for tiled regions, ONE CTA per region: w_f <- scale * c_f . B_r^-1 (sum_f c_f w_f).
// Three groups of REG_GROUP threads take the region's x / y / z rows (rowAxisStart), so every load of the region is in flight
// at once; the 3 x 10 moments are reduced in a fixed order (warp shuffles, then the group's warps in order), B^-1 (staged in
// shared memory while the rows stream in) is applied by 26 threads, and the same threads that read a row overwrite it with the
// expanded value.  No inter-CTA hand-off: this replaces moments + last-chunk solve + expand (3 dependent stages, 2 launches)
// by one launch whose critical path is one row round trip + one 26x26 product.  Regions too large for one CTA (doTile off)
// keep the chunked kernels above.
// GROUP threads per axis, ROWS rows per thread kept in registers between the two phases (0: re-read rowXYZ through L1/L2)
template <int GROUP, int ROWS, int MINB>
__global__ void __launch_bounds__(3 * GROUP, MINB) reduced_region_kernel(double dx, const uint32_t* __restrict__ rowXYZ, const int32_t* __restrict__ rowAxisStart, const double* __restrict__ com,
                                                                       const double* __restrict__ Binv, double* __restrict__ wRows, double scale, const PcgScalars* S, int region0) {
    constexpr int NW = GROUP / 32, KEEP = ROWS > 0 ? ROWS : 1;
    __shared__ double Bs[RDOF * RDOF];
    __shared__ double red[3][NW][10];
    __shared__ double M[30], t[RDOF], sv[RDOF], sg[30];
    const int r = region0 + blockIdx.x;
    // B^-1, the row table and the centres of mass are setup data: they may be fetched before the previous kernel has finished
    for (int i = threadIdx.x; i < RDOF * RDOF; i += 3 * GROUP) Bs[i] = __ldg(Binv + (size_t)r * RDOF * RDOF + i);
    const int axis = threadIdx.x / GROUP, lane = threadIdx.x % GROUP;
    const int begin = __ldg(rowAxisStart + 3 * r + axis), end = __ldg(rowAxisStart + 3 * r + axis + 1);
    const double cm[3] = {__ldg(com + 3 * r), __ldg(com + 3 * r + 1), __ldg(com + 3 * r + 2)};
    pdl_sync();
    if (S && S->done) return;
    double acc[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) acc[k] = 0.;
    uint32_t xyz[KEEP];
    if (ROWS > 0) {
        double gk[KEEP];
#pragma unroll
        for (int i = 0; i < KEEP; ++i) {
            const int row = begin + lane + i * GROUP;
            xyz[i] = row < end ? __ldcs(rowXYZ + row) : 0u;
            gk[i] = row < end ? __ldcs(wRows + row) : 0.;
        }
#pragma unroll
        for (int i = 0; i < KEEP; ++i) {
            double m[10];
            row_monomials(dx, xyz[i], cm, m);
#pragma unroll
            for (int k = 0; k < 10; ++k) acc[k] += m[k] * gk[i];
        }
    }
#pragma unroll 4
    for (int row = begin + lane + ROWS * GROUP; row < end; row += GROUP) {
        double m[10];
        row_monomials(dx, __ldg(rowXYZ + row), cm, m);
        const double g1 = __ldcs(wRows + row);
#pragma unroll
        for (int k = 0; k < 10; ++k) acc[k] += m[k] * g1;
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        const double v = warp_sum(acc[k]);
        if ((lane & 31) == 0) red[axis][lane >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 30) {
        const int a = threadIdx.x / 10, k = threadIdx.x % 10;
        double s = 0.;
#pragma unroll
        for (int wI = 0; wI < NW; ++wI) s += red[a][wI][k];
        M[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) moments_to_t(M, t);
    __syncthreads();
    if (threadIdx.x < RDOF) {
        const double* B = Bs + threadIdx.x * RDOF;
        double s = 0.;
#pragma unroll
        for (int j = 0; j < RDOF; ++j) s += B[j] * t[j];
        sv[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_to_sigma(sv, sg);
    __syncthreads();
    double sgl[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) sgl[k] = sg[axis * 10 + k];
    if (ROWS > 0) {
#pragma unroll
        for (int i = 0; i < KEEP; ++i) {
            const int row = begin + lane + i * GROUP;
            if (row < end) {
                double m[10];
                row_monomials(dx, xyz[i], cm, m);
                double v = 0.;
#pragma unroll
                for (int k = 0; k < 10; ++k) v += sgl[k] * m[k];
                wRows[row] = scale * v;
            }
        }
    }
#pragma unroll 4
    for (int row = begin + lane + ROWS * GROUP; row < end; row += GROUP) {
        double m[10];
        row_monomials(dx, __ldg(rowXYZ + row), cm, m);
        double v = 0.;
#pragma unroll
        for (int k = 0; k < 10; ++k) v += sgl[k] * m[k];
        wRows[row] = scale * v;
    }
}
// regions with more coupled rows than this take the chunked kernels (reduced_moments_kernel + reduced_expand_kernel)
static int region_fuse_limit() {
    static const int fuseLimit = getenv("PS_REGION_FUSE_MAX") ? atoi(getenv("PS_REGION_FUSE_MAX")) : 16384;
    return fuseLimit;
}
template <int GROUP, int ROWS, int MINB>
static void launch_region(cudaStream_t st, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    launch_chain(reduced_region_kernel<GROUP, ROWS, MINB>, (unsigned)(RG.regHi - RG.regLo), 3 * GROUP, st, g.dx, RG.rowXYZ.p, RG.rowAxisStart.p, RG.com.p, RG.Binv.p, wRows, scale, S, RG.regLo);
}
// which kernels carry the reduced term of a forward apply (reduced_apply): -1 no owned region, 0 reduced_region_kernel with 64 lanes per
// axis, 1 with 128 lanes, 2 the chunked kernels.  64 lanes per axis and 6 CTAs per SM for many regions (throughput); few regions per GPU
// (slab decomposition) are latency bound -- 128 lanes per axis with the rows kept in registers put every load of a region in flight at once
int region_path(const RegionData& RG) {
    if (RG.regHi <= RG.regLo) return -1;
    if (RG.maxRegionRows > region_fuse_limit()) return 2;
    return RG.regHi - RG.regLo <= 900 ? 1 : 0;
}
// w_f <- scale * c_f . B^-1 J w on the coupled reduced rows (the reduced term of one operator apply)
void reduced_apply(cudaStream_t st, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    if (RG.regHi <= RG.regLo) return;
    const int path = region_path(RG);
    if (path == 2) { reduced_moments(st, g, RG, wRows, S, true); reduced_expand(st, g, RG, wRows, scale, S); return; }
    if (path == 1) launch_region<128, 8, 2>(st, g, RG, wRows, scale, S);
    else launch_region<64, 0, 6>(st, g, RG, wRows, scale, S);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void reduced_moments(cudaStream_t st, const Geom& g, const RegionData& RG, const double* wRows, const PcgScalars* S, bool solve) {
    if (RG.rowChunkHi <= RG.rowChunkLo) return;
    launch_chain(reduced_moments_kernel, (unsigned)(RG.rowChunkHi - RG.rowChunkLo), MOM_THREADS, st, g.dx, RG.rowXYZ.p, RG.rowChunk.p, RG.rowChunkStart.p, RG.com.p, wRows, RG.partial.p, RG.Binv.p, RG.sigma.p,
                                                                                 solve ? RG.regionTicket.p : nullptr, S, RG.rowChunkLo);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void reduced_finish(cudaStream_t st, const Geom&, const RegionData& RG, const double* extra, double extraScale, double tScale, const PcgScalars* S) {
    if (RG.regHi <= RG.regLo) return;
    launch_chain(reduced_finish_kernel, (unsigned)(RG.regHi - RG.regLo), 32, st, RG.rowChunkStart.p, RG.rowChunk.p, RG.partial.p, RG.Binv.p, extra, extraScale, tScale, RG.t.p, RG.s.p, RG.sigma.p, S, RG.regLo);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void reduced_expand(cudaStream_t st, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    if (RG.ownRowHi <= RG.ownRowLo) return;
    const int n = RG.ownRowHi - RG.ownRowLo;
    launch_chain(reduced_expand_kernel, (unsigned)std::min((n + RED_THREADS - 1) / RED_THREADS, sm_count() * 8), RED_THREADS, st, g.dx, RG.rowXYZ.p, RG.rowRegion.p, RG.com.p, RG.sigma.p, wRows, scale, S, RG.ownRowLo, RG.ownRowHi);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void shared_moments(cudaStream_t st, const Geom& g, const RegionData& RG, const double* wRows, const PcgScalars* S) {
    if (RG.nShChunks <= 0) return;
    launch_chain(reduced_moments_kernel, (unsigned)RG.nShChunks, MOM_THREADS, st, g.dx, RG.rowXYZ.p, RG.shChunk.p, RG.shChunkStart.p, RG.com.p, wRows, RG.shPartial.p, RG.Binv.p, RG.sigma.p,
                 (unsigned int*)nullptr, S, 0);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
void shared_expand(cudaStream_t st, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    if (RG.shRowHi <= RG.shRowLo) return;
    const int n = RG.shRowHi - RG.shRowLo;
    launch_chain(reduced_expand_kernel, (unsigned)std::min((n + RED_THREADS - 1) / RED_THREADS, sm_count() * 8), RED_THREADS, st, g.dx, RG.rowXYZ.p, RG.rowRegion.p, RG.com.p, RG.sigma.p, wRows, scale, S, RG.shRowLo, RG.shRowHi);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
#else
void shared_moments(cudaStream_t, const Geom& g, const RegionData& RG, const double* wRows, const PcgScalars* S) {
    if (S && S->done) return;
    for (int ch = 0; ch < RG.nShChunks; ++ch) {
        const int region = RG.shChunk.p[4 * ch], begin = RG.shChunk.p[4 * ch + 1], end = RG.shChunk.p[4 * ch + 2];
        double acc[10] = {0};
        for (int row = begin; row < end; ++row) {
            double m[10]; row_monomials(g.dx, RG.rowXYZ.p[row], RG.com.p + 3 * region, m);
            for (int k = 0; k < 10; ++k) acc[k] += m[k] * wRows[row];
        }
        for (int k = 0; k < 10; ++k) RG.shPartial.p[(size_t)ch * 10 + k] = acc[k];
    }
}
void shared_expand(cudaStream_t, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    if (S && S->done) return;
    for (int row = RG.shRowLo; row < RG.shRowHi; ++row) {
        const int region = RG.rowRegion.p[row], axis = (int)(RG.rowXYZ.p[row] >> 30);
        double m[10]; row_monomials(g.dx, RG.rowXYZ.p[row], RG.com.p + 3 * region, m);
        double v = 0.;
        for (int k = 0; k < 10; ++k) v += RG.sigma.p[(size_t)region * 30 + axis * 10 + k] * m[k];
        wRows[row] = scale * v;
    }
}
void reduced_finish(cudaStream_t, const Geom&, const RegionData& RG, const double* extra, double extraScale, double tScale, const PcgScalars* S);
void reduced_moments(cudaStream_t st, const Geom& g, const RegionData& RG, const double* wRows, const PcgScalars* S, bool solve) {
    if (S && S->done) return;
    for (int ch = RG.rowChunkLo; ch < RG.rowChunkHi; ++ch) {
        const int region = RG.rowChunk.p[4 * ch], begin = RG.rowChunk.p[4 * ch + 1], end = RG.rowChunk.p[4 * ch + 2];
        double acc[10] = {0};
        for (int row = begin; row < end; ++row) {
            const double gk = wRows[row];
            double m[10]; row_monomials(g.dx, RG.rowXYZ.p[row], RG.com.p + 3 * region, m);
            for (int k = 0; k < 10; ++k) acc[k] += m[k] * gk;
        }
        for (int k = 0; k < 10; ++k) RG.partial.p[(size_t)ch * 10 + k] = acc[k];
    }
    if (solve) reduced_finish(st, g, RG, nullptr, 0.0, 1.0, S);
}
void reduced_finish(cudaStream_t, const Geom&, const RegionData& RG, const double* extra, double extraScale, double tScale, const PcgScalars* S) {
    if (S && S->done) return;
    for (int r = RG.regLo; r < RG.regHi; ++r) {
        double M[30] = {0}, t[RDOF], sv[RDOF], sg[30];
        if (tScale != 0.)
            for (int ch = RG.rowChunkStart.p[r]; ch < RG.rowChunkStart.p[r + 1]; ++ch)
                for (int k = 0; k < 10; ++k) M[RG.rowChunk.p[4 * ch + 3] * 10 + k] += RG.partial.p[(size_t)ch * 10 + k];
        moments_to_t(M, t);
        for (int n = 0; n < RDOF; ++n) { t[n] = tScale * t[n] + (extra ? extraScale * extra[(size_t)r * RDOF + n] : 0.); RG.t.p[(size_t)r * RDOF + n] = t[n]; }
        for (int i = 0; i < RDOF; ++i) { double s = 0.; for (int j = 0; j < RDOF; ++j) s += RG.Binv.p[(size_t)r * RDOF * RDOF + i * RDOF + j] * t[j]; sv[i] = s; RG.s.p[(size_t)r * RDOF + i] = s; }
        s_to_sigma(sv, sg);
        for (int k = 0; k < 30; ++k) RG.sigma.p[(size_t)r * 30 + k] = sg[k];
    }
}
void reduced_apply(cudaStream_t st, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    reduced_moments(st, g, RG, wRows, S, true); reduced_expand(st, g, RG, wRows, scale, S);
}
int region_path(const RegionData& RG) { return RG.regHi > RG.regLo ? 2 : -1; }      // the twin has the chunked form only
void reduced_expand(cudaStream_t, const Geom& g, const RegionData& RG, double* wRows, double scale, const PcgScalars* S) {
    if (S && S->done) return;
    for (int ch = RG.rowChunkLo; ch < RG.rowChunkHi; ++ch) {
        const int region = RG.rowChunk.p[4 * ch], begin = RG.rowChunk.p[4 * ch + 1], end = RG.rowChunk.p[4 * ch + 2], axis = RG.rowChunk.p[4 * ch + 3];
        for (int row = begin; row < end; ++row) {
            double m[10]; row_monomials(g.dx, RG.rowXYZ.p[row], RG.com.p + 3 * region, m);
            double v = 0.;
            for (int k = 0; k < 10; ++k) v += RG.sigma.p[(size_t)region * 30 + axis * 10 + k] * m[k];
            wRows[row] = scale * v;
        }
    }
}
#endif
// [nShared][3][10]: this rank's chunk partials of every shared slot, summed in chunk order (0 where it holds no rows); the caller sums
// the table over the ranks.  Runs after `done` too: the all-reduce that follows is summed every time.
void shared_pack(cudaStream_t st, const RegionData& RG) {
    const int32_t* cs = RG.shChunkStart.p; const int32_t* chunk = RG.shChunk.p; const double* partial = RG.shPartial.p; double* mom = RG.shMoments.p;
    ps_for(st, (int64_t)RG.nShared * 30, PS_LAMBDA(int64_t i) {
        const int j = (int)(i / 30), axis = (int)(i % 30) / 10, k = (int)(i % 10);
        double s = 0.;
        for (int ch = cs[j]; ch < cs[j + 1]; ++ch) if (chunk[4 * ch + 3] == axis) s += partial[(size_t)ch * 10 + k];
        mom[i] = s;
    });
}
// the small solve of one shared region from its summed moments M: t, s = B^-1 (extraScale extra + tScale t), sigma (both transports)
PS_D void shared_solve_slot(const double* M, int r, const double* Binv, const double* extra, double extraScale, double tScale, double* sOut, double* sigma) {
    double t[RDOF], sv[RDOF], sg[30];
    moments_to_t(M, t);
    for (int n = 0; n < RDOF; ++n) { double v = tScale * t[n]; if (extra) v += extraScale * extra[(size_t)r * RDOF + n]; t[n] = v; }
    const double* B = Binv + (size_t)r * RDOF * RDOF;
    for (int a = 0; a < RDOF; ++a) { double s = 0.; for (int b = 0; b < RDOF; ++b) s += B[a * RDOF + b] * t[b]; sv[a] = s; if (sOut) sOut[(size_t)r * RDOF + a] = s; }
    s_to_sigma(sv, sg);
    for (int k = 0; k < 30; ++k) sigma[(size_t)r * 30 + k] = sg[k];
}
// the small solve of the slots this rank takes part in, from shMoments (summed over the ranks by the communicator)
// (every rank that holds rows of the region forms the same s from the same sums)
void shared_finish(cudaStream_t st, const RegionData& RG, const double* extra, double extraScale, double tScale, double* sOut, const PcgScalars* S) {
    const int32_t* mine = RG.shMine.p; const int32_t* reg = RG.shRegion.p; const double* mom = RG.shMoments.p; const double* Binv = RG.Binv.p;
    double* sigma = RG.sigma.p;
    ps_for(st, RG.nShMine, PS_LAMBDA(int64_t i) {
        if (S && S->done) return;
        const int j = mine[i];
        double M[30];
        for (int k = 0; k < 30; ++k) M[k] = tScale != 0. ? mom[(size_t)j * 30 + k] : 0.;
        shared_solve_slot(M, reg[j], Binv, extra, extraScale, tScale, sOut, sigma);
    });
}
#ifndef PS_EMULATE
// Peer transport.  CTA d packs this rank's [nShared][30] moments (chunk partials summed in chunk order, as shared_pack) straight into
// row [parity][rank] of rank d's moment area, fences, and raises flag [parity][rank] there.  Runs after `done` too: the finish kernels
// of every rank wait for every exchange, so the sequence numbers stay in step.
__global__ void __launch_bounds__(256) shared_push_kernel(const int32_t* __restrict__ cs, const int32_t* __restrict__ chunk, const double* __restrict__ partial, int nShared,
                                                          const __grid_constant__ SharedPeer P) {    pdl_sync();
    const int d = blockIdx.x, par = (int)(P.seq & 1ull);
    double* dst = P.val[d] + ((size_t)par * PEER_MAX_RANKS + P.rank) * P.stride;
    for (int i = threadIdx.x; i < nShared * 30; i += blockDim.x) {
        const int j = i / 30, axis = (i % 30) / 10, k = i % 10;
        double s = 0.;
        for (int ch = cs[j]; ch < cs[j + 1]; ++ch) if (chunk[4 * ch + 3] == axis) s += partial[(size_t)ch * 10 + k];
        peer_st_f64(dst + i, s);
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) peer_st_flag(P.flag[d] + par * PEER_MAX_RANKS + P.rank, P.seq);
}
// one warp per slot this rank takes part in: wait for the N ranks' rows of this exchange (time-out -> peerError), sum them in rank
// order (the same sums on every rank), then the slot's small solve
__global__ void __launch_bounds__(32) shared_finish_peer_kernel(const int32_t* __restrict__ mine, const int32_t* __restrict__ reg, const double* __restrict__ Binv,
                                                                const double* __restrict__ extra, double extraScale, double tScale, double* sOut, double* sigma,
                                                                const PcgScalars* S, PcgScalars* err, const __grid_constant__ SharedPeer P) {    pdl_sync();
    __shared__ double M[30];
    const int lane = threadIdx.x, par = (int)(P.seq & 1ull);
    bool good = true;
    if (lane < P.nranks) good = peer_wait_flag(P.flag[P.rank] + par * PEER_MAX_RANKS + lane, P.seq);
    good = __all_sync(0xffffffffu, good);
    if (!good) { if (lane == 0) err->peerError = 1; return; }
    if (S && S->done) return;
    const int j = mine[blockIdx.x];
    if (lane < 30) {
        double s = 0.;
        for (int q = 0; q < P.nranks; ++q) s += peer_ld_f64(P.val[P.rank] + ((size_t)par * PEER_MAX_RANKS + q) * P.stride + (size_t)j * 30 + lane);
        M[lane] = s;
    }
    __syncwarp();
    if (lane == 0) shared_solve_slot(M, reg[j], Binv, extra, extraScale, tScale, sOut, sigma);
}
void shared_exchange_peer(cudaStream_t st, const RegionData& RG, const SharedPeer& P, const double* extra, double extraScale, double tScale, double* sOut,
                          const PcgScalars* S, PcgScalars* err) {
    launch_chain(shared_push_kernel, (unsigned)P.nranks, 256, st, RG.shChunkStart.p, RG.shChunk.p, RG.shPartial.p, (int)RG.nShared, P);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
    if (RG.nShMine <= 0) return;
    launch_chain(shared_finish_peer_kernel, (unsigned)RG.nShMine, 32, st, RG.shMine.p, RG.shRegion.p, RG.Binv.p, extra, extraScale, tScale, sOut, RG.sigma.p, S, err, P);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
#endif

// ---- solverType EIGEN (exec/HDK_PolyStokesSolver.cpp:814-862) ---------------------------------------------------
// The reference hands the explicit A to Eigen::ConjugateGradient<SparseMatrix, Lower|Upper> (default
// DiagonalPreconditioner) and starts from guessVector.  Here the operator stays factored (same A up to rounding) and only
// diag(A) is formed, row by row, from the factors:
//   A_ii = -dt sum_{active f} K_fi^2 / Mc_f  -  v_i^T B_r^-1 v_i  -  1/2 mu^-1_i [stress rows],   v_i = sum_{f in region r} K_fi c_f
// (column i of J_r = C_r K_red; the coupled reduced faces of one DOF belong to one region after C6, several are handled anyway).
struct DiagCtx { const int32_t* rowRegion; const uint32_t* rowXYZ; const double* com; const double* Binv; double dx, dt; };
template <int NS>
PS_D double diag_row(const OpArgs& A, const DiagCtx& D, const int64_t* f, const double* val) {
    double uni = 0., red = 0.;
    bool used[NS];
    for (int k = 0; k < NS; ++k) {
        used[k] = (val[k] == 0.) || f[k] < A.nActiveVs;
        if (val[k] != 0. && f[k] < A.nActiveVs) uni += val[k] * val[k] * A.mcInvLut[A.kmc[f[k]]];
    }
    for (int k = 0; k < NS; ++k) {
        if (used[k]) continue;
        const int region = D.rowRegion[f[k] - A.nActiveVs];
        double V[RDOF], c[RDOF], m[10];
        for (int n = 0; n < RDOF; ++n) V[n] = 0.;
        for (int q = k; q < NS; ++q) {
            if (used[q] || D.rowRegion[f[q] - A.nActiveVs] != region) continue;
            used[q] = true;
            const uint32_t packed = D.rowXYZ[f[q] - A.nActiveVs];
            row_monomials(D.dx, packed, D.com + 3 * region, m);
            conversion_coefficients(m[1], m[2], m[3], (int)(packed >> 30), c);
            for (int n = 0; n < RDOF; ++n) V[n] += val[q] * c[n];
        }
        const double* B = D.Binv + (size_t)region * RDOF * RDOF;
        for (int i = 0; i < RDOF; ++i) { double t = 0.; for (int j = 0; j < RDOF; ++j) t += B[i * RDOF + j] * V[j]; red += V[i] * t; }
    }
    return -D.dt * uni - red;
}
void k_diag_A(cudaStream_t st, const Geom& g, const OpArgs& A, const RegionData& RG, double* diag) {
    const DiagCtx D = {RG.rowRegion.p, RG.rowXYZ.p, RG.com.p, RG.Binv.p, g.dx, g.dt};
    ps_for(st, A.nC, PS_LAMBDA(int64_t ci) {
        const uint64_t word = A.ccode[ci];
        int64_t f[6]; double v[6];
        for (int k = 0; k < 6; ++k) { const int code = op_code(word, k); v[k] = (double)code * A.valScale; f[k] = code ? A.ccol[(int64_t)k * A.nC + ci] : 0; }
        diag[ci] = diag_row<6>(A, D, f, v);
        for (int a = 0; a < 3; ++a) {
            const double va[2] = {-v[2 * a], -v[2 * a + 1]};
            const int64_t j = (int64_t)a * A.nC + ci;
            diag[A.nP + j] = diag_row<2>(A, D, f + 2 * a, va) - 0.5 * A.uInv[j];
        }
    });
    ps_for(st, A.nE, PS_LAMBDA(int64_t e) {
        const uint32_t word = A.ecode[e];
        int64_t f[4]; double v[4];
        for (int k = 0; k < 4; ++k) { const int code = op_code(word, k); v[k] = (double)code * A.valScale; f[k] = code ? A.ecol[(int64_t)k * A.nE + e] : 0; }
        const int64_t j = 3 * A.nC + e;
        diag[A.nP + j] = diag_row<4>(A, D, f, v) - 0.5 * A.uInv[j];
    });
}
// warm start (S.cpp:521-531): sigma of v*_r without the B^-1 solve, so that expand gives w_f = c_f . v*_r
void k_sigma_from_s(cudaStream_t st, int32_t R, const double* s, double* sigma) {
    ps_for(st, R, PS_LAMBDA(int64_t r) { double sg[30]; s_to_sigma(s + r * RDOF, sg); for (int k = 0; k < 30; ++k) sigma[r * 30 + k] = sg[k]; });
}
// guess holds -K_ext^T w; the stress part becomes -2 mu^-1 (-D u - DJ^T v*) (S.cpp:530, uInv_Matrix as written there)
void k_guess_finish(cudaStream_t st, const OpArgs& A, double* guess) {
    ps_for(st, A.nT, PS_LAMBDA(int64_t i) { guess[A.nP + i] = (-2. * A.uInv[i]) * guess[A.nP + i]; });
}
// Eigen's m_invdiag: 1 / A_jj, 1 where the diagonal entry is absent or zero (BasicPreconditioners.h:75-84)
PS_D double eig_invdiag(double d) { return d != 0. ? 1. / d : 1.; }
// scalar bookkeeping in the statement order of ConjugateGradient.h:44-90
PS_D void eig_stage(PcgScalars* S, int stage) {
    if (S->done) return;
    if (stage == 0) {            // :46-61  bred = {b.b, r.r}
        const double rhsNorm2 = S->bred[0], residualNorm2 = S->bred[1];
        S->eigRhsNorm2 = rhsNorm2;
        if (rhsNorm2 == 0.) { S->rre = 0.; S->done = 3; return; }                      // x.setZero(), 0 iterations
        const double t = S->tol * S->tol * rhsNorm2;
        S->eigThreshold = t > 2.2250738585072014e-308 ? t : 2.2250738585072014e-308;
        S->rre = sqrt(residualNorm2 / rhsNorm2);
        if (residualNorm2 < S->eigThreshold) S->done = 1;
        else if (S->maxIter <= 0) S->done = 2;
    } else if (stage == 1) {     // :67  absNew = r.p
        S->eigAbsNew = S->bred[0];
    } else {                     // :78-88  bred = {r.r, r.z}
        const double residualNorm2 = S->bred[0];
        S->rsnew = residualNorm2; S->rre = sqrt(residualNorm2 / S->eigRhsNorm2);
        if (residualNorm2 < S->eigThreshold) { S->done = 1; return; }
        const double absOld = S->eigAbsNew;
        S->eigAbsNew = S->bred[1];
        S->beta = S->eigAbsNew / absOld;
        S->iter += 1;
        if (S->iter >= S->maxIter) S->done = 2;
    }
}
void k_eig_stage(cudaStream_t st, PcgScalars* S, int stage) { ps_for(st, 1, PS_LAMBDA(int64_t) { eig_stage(S, stage); }); }
// :40-48  residual = rhs - mat * x, |rhs|^2, |residual|^2
void k_eig_init(cudaStream_t st, const RangeSet& own, const double* b, const double* Ax, double* r, double* dotPartial, PcgScalars* S, double tol, int maxIter) {
    ps_for(st, 1, PS_LAMBDA(int64_t) {
        S->alpha = 0.; S->beta = 0.; S->rsnew = 0.; S->rre = 0.; S->red[0] = 0.; S->bred[0] = 0.; S->bred[1] = 0.;
        S->tol = tol; S->tol2 = tol * tol; S->iter = 0; S->maxIter = maxIter; S->done = 0;
        S->ticket[0] = 0; S->ticket[6] = 0;
    });
    vec_sweep(st, own, dotPartial, S, 2, 0, false, PS_LAMBDA(int64_t i, double& a, double& c) { const double bi = b[i], ri = bi - Ax[i]; r[i] = ri; a += bi * bi; c += ri * ri; });
}
// :64-67  p = precond.solve(residual), absNew = residual . p
void k_eig_first_p(cudaStream_t st, const RangeSet& own, const double* diag, const double* r, double* p, double* dotPartial, PcgScalars* S) {
    vec_sweep(st, own, dotPartial, S, 1, 0, true, PS_LAMBDA(int64_t i, double& a, double&) { const double ri = r[i], pi = eig_invdiag(diag[i]) * ri; p[i] = pi; a += ri * pi; });
}
// :73-84  alpha = absNew / p.tmp (p.tmp left in red[0] by pass 2), x += alpha p, residual -= alpha tmp, |residual|^2, residual . z
void k_eig_update_xr(cudaStream_t st, const RangeSet& own, const double* diag, double* x, double* r, const double* p, const double* Ap, double* dotPartial, PcgScalars* S) {
    vec_sweep(st, own, dotPartial, S, 2, 0, true, PS_LAMBDA(int64_t i, double& a, double& c) {
        const double alpha = S->eigAbsNew / S->red[0];
        x[i] += alpha * p[i];
        const double ri = r[i] - alpha * Ap[i];
        r[i] = ri; a += ri * ri; c += ri * (eig_invdiag(diag[i]) * ri);
    });
}
// :81, :87  p = z + beta p
void k_eig_update_p(cudaStream_t st, const RangeSet& own, const double* diag, double* p, const double* r, const PcgScalars* S) {
    vec_sweep(st, own, nullptr, const_cast<PcgScalars*>(S), 0, 0, true, PS_LAMBDA(int64_t i, double&, double&) { p[i] = eig_invdiag(diag[i]) * r[i] + S->beta * p[i]; });
}

// W1 recoverVelocityFromPressureStress, active part (S.cpp:507): u = dt Mc^-1 (rhs_u/dt - G p - D^T tau)
// (wAct already holds dt Mc^-1 K x from pass 1)
void k_recover_active(cudaStream_t st, const Geom& g, const RowSet& rows, const double* wAct, const double* mcInv, const double* rhsU, double* velSol) {
    const double dt = g.dt, invDt = g.invDt;
    const RowSet R = rows;
    ps_for(st, R.total(), PS_LAMBDA(int64_t l) { const int64_t i = R.at(l); velSol[i] = dt * (mcInv[i] * (invDt * rhsU[i])) - wAct[i]; });
}

PS_HD bool face_is_mine(const FaceOwner& own, int ri, int z) {
    if (own.shared && own.shared[ri]) return z >= own.zLo && (z < own.zHi || own.zHi >= own.nz);
    return ri >= own.regLo && ri < own.regHi;
}
// W2 applySolutionToVelocity (S.cpp:937-1028) fused with buildValidFaces (S_Cls:4-54).  With several ranks a
// face carrying a DOF is written by the rank that owns the DOF; faces without one are written by everybody.
// Visits the faces [lo, hi); `valid` is written on [validLo, validHi) only (the part of the field this rank delivers).
void k_writeback_velocity(cudaStream_t st, const Geom& g, const Fields& F, const Counts& C, const RegionData& RG, const double* velSol, int axis, float* velOut, bool writeValid, float* validOut, FaceOwner own,
                          int64_t lo, int64_t hi, int64_t validLo, int64_t validHi) {
    const int8_t* FL = F.label[SL_FACE + axis]; const int32_t* FA = F.aidx[SL_FACE + axis]; const int32_t* FR = F.ridx[SL_FACE + axis];
    const float* cvel = F.colvel[axis];
    const double* com = RG.com.p;
    const int64_t faceOff = C.faceOff[axis], nAct = C.nActiveVs;
    const bool haveReduced = RG.count > 0;
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) {
        const int lab = FL[q];
        const bool valid = !(lab == L_UNSOLVED || lab == L_UNASSIGNED);
        if (writeValid && q >= validLo && q < validHi) validOut[q] = valid ? 1.f : 0.f;
        if (!valid || !velOut) return;
        double v = 0.;
        const int ri = haveReduced ? FR[q] : -1;
        const int ai = FA[q];
        if (ri >= 0) {
            const I3 f = delin(g, SL_FACE + axis, q);
            if (!face_is_mine(own, ri, f.z)) return;
            double ox, oy, oz, c[RDOF];
            face_offset(g, f, axis, com + 3 * ri, ox, oy, oz);
            conversion_coefficients(ox, oy, oz, axis, c);
            for (int n = 0; n < RDOF; ++n) v += velSol[nAct + (int64_t)RDOF * ri + n] * c[n];
        } else if (ai >= 0) {
            if (ai < own.aLo || ai >= own.aHi) return;
            v = velSol[faceOff + ai];
        }
        else if (lab == L_SOLID) v = (double)cvel[q];
        velOut[q] = (float)v;
    });
}

// the z-face plane shared by two slabs holds DOFs of both ranks: take the peer's value where the peer owns the DOF
void k_merge_face_plane(cudaStream_t st, const Geom& g, const Fields& F, int axis, int k, const float* peerPlane, float* velOut, FaceOwner own) {
    const int8_t* FL = F.label[SL_FACE + axis]; const int32_t* FA = F.aidx[SL_FACE + axis]; const int32_t* FR = F.ridx[SL_FACE + axis];
    const int64_t plane = (int64_t)g.r[SL_FACE + axis][0] * g.r[SL_FACE + axis][1], base = plane * k;
    ps_for(st, plane, PS_LAMBDA(int64_t i) {
        const int64_t q = base + i;
        const int lab = FL[q];
        if (lab == L_UNSOLVED || lab == L_UNASSIGNED) return;
        const int ri = FR[q], ai = FA[q];
        const bool mine = ri >= 0 ? face_is_mine(own, ri, k) : (ai >= 0 ? (ai >= own.aLo && ai < own.aHi) : true);
        if (!mine) velOut[q] = peerPlane[i];
    });
}

}  // namespace ps
