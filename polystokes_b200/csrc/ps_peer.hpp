// ps_peer.hpp -- the collectives of the distributed CG fused INTO the compute kernels over NVLink peer memory.
//
// NCCL (ps_comm.cu) needs one host-enqueued collective kernel per halo exchange / all-reduce: at 256^3 on 8 GPUs
// a CG iteration is ~0.1 ms of HBM work, so four ~30 us NCCL launches per iteration would dominate.  Here every
// rank owns one small *symmetric block* (cudaMalloc'd, exported with cudaIpcGetMemHandle, mapped by every other rank):
//   * halo exchange = the sender's pack kernel STORES its boundary entries straight into the receiver's block through
//     NVLink (contiguous, coalesced), then raises a sequence flag there; the receiver's unpack kernel spins on its own
//     flag and scatters into its vector.  No staging copy, no collective launch.
//   * all-reduce of the CG dot products = the LAST CTA of the producing kernel (pass 2 / x,r update / init) stores the
//     rank's partial sum into slot [rank] of EVERY rank's block and raises a flag; the FIRST thing the consuming
//     kernel does is wait for all N flags and add the N partials in rank order -- bit-identical on every rank, so
//     all ranks take the same stop decision.  Zero extra kernels per iteration.
// Buffers are double-buffered by the parity of a host-side sequence number; reuse is safe because a rank can only
// start operation s+2 after it consumed operation s+1 of the peer, which the peer issued after finishing s
// (stream order on both sides).  Every spin has a time-out that flags the solve as failed instead of hanging.
// The NCCL path stays as the fallback (no peer access, PS_COMM=nccl) and carries the IPC handles at start-up.
#pragma once
#include "ps_rt.hpp"

namespace ps {

constexpr int PEER_MAX_RANKS = 8;
constexpr int PEER_SLOTS = 2;      // reduction slots: 0 (p.Ap, r.Ap, Ap.Ap) of pass 2, 1 (r.r, x.p, p.p) of the x/r/p update (or b.b, 0, b.b from init)
constexpr int PEER_VALS = 3;       // values per reduction
// Shared-region moments (Solver::sharedApply): behind the halo buffers every block holds flags [parity][source rank] and values
// [parity][source rank][PEER_SH_CAP][30]; a step with more shared regions takes the communicator's all-reduce instead
constexpr int PEER_SH_CAP = 4096;
constexpr size_t PEER_SH_FLAG_BYTES = 256;

struct PeerSync {                  // head of every rank's symmetric block
    unsigned long long haloFlag[2][2][2];                      // [kind x|w][parity][side: from below | from above]
    unsigned long long redFlag[2][PEER_SLOTS][PEER_MAX_RANKS]; // [parity][slot][source rank]
    double redVal[2][PEER_SLOTS][PEER_VALS][PEER_MAX_RANKS];   // [parity][slot][value][source rank]
    unsigned long long vecFlag[2][2];                          // [kind p|w][side: from below | from above] direct halo stores (VecLink)
    unsigned long long pad[12];
};

// Halo exchange without unpacking: p and w are global-length on every rank and live in one arena per rank that the z-neighbours map
// (PeerLink::vecBase).  A small push launch stores the entries a neighbour reads at their FINAL place in the neighbour's copy -- and
// does nothing else: no fence, no ticket, no flag, so it ends as soon as the stores are issued.  The flags are raised by ONE thread of
// the launch that FOLLOWS on this rank, after a system fence (the launch boundary orders the stores before that thread, the fence is
// cumulative): for p the push runs BEFORE the x/r/p update -- it recomputes p_new = (r - alpha Ap) + beta p on the boundary entries
// from the old vectors -- so the NVLink trip of the data hides under the update, whose last CTA raises the flags; for w the push
// follows the reduced term and the head of pass 2 raises the flags before it waits for its own.  The consuming kernel (pass 1 for
// p, pass 2 for w) waits for its two flags at its head (VecLink) -- no receive buffer, no scatter, no launch that sits waiting.
// Reuse is safe without a second buffer: a neighbour pushes p after its x/r/p update, which consumed the reductions of this rank's
// pass 2, i.e. every read of the old values (pass 1) is over; it pushes w after its pass 1, which waited for this rank's p push,
// issued after this rank's update -- behind the last reader of the old w (pass 2).
struct VecLink {
    const unsigned long long* wait[2] = {nullptr, nullptr}; // this rank's flags for what comes from below / above
    unsigned long long waitSeq = 0;                         // 0: nothing to wait for
    unsigned long long* raise[2] = {nullptr, nullptr};      // the neighbours' flags for what the PREVIOUS launch of this rank stored into their vectors
    unsigned long long raiseSeq = 0;                        // 0: nothing to announce
};

struct PeerCtx {                   // passed by value to the CG kernels; nranks <= 1 means "no peers"
    int nranks = 1, rank = 0;
    unsigned long long seqIn = 0, seqOut = 0;   // sequence numbers of the reduction this kernel consumes / produces
    unsigned long long seqIn2 = 0;              // the x/r/p update also consumes slot 1 of the previous update (or of init)
    PeerSync* sync[PEER_MAX_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

// the moment exchange of the shared regions, by value to its two kernels: every rank's flags and values, this exchange's sequence number
struct SharedPeer {
    int nranks = 1, rank = 0;
    unsigned long long seq = 0;
    size_t stride = 0;                            // doubles per [parity][source rank] row (shCap * 30)
    unsigned long long* flag[PEER_MAX_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double* val[PEER_MAX_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

// host-side state of the peer transport of one solver
struct PeerLink {
    bool on = false;
    bool needResync = false;                      // a wait timed out / a solve was cancelled: flags and sequence numbers are re-agreed at the next setup
    int rank = 0, nranks = 1;
    void* block[PEER_MAX_RANKS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // block[rank] = mine, others IPC-mapped
    bool sameProcess[PEER_MAX_RANKS] = {false, false, false, false, false, false, false, false};          // peers of this process: plain peer access to their pointer
    size_t cap = 0;                               // doubles per halo receive buffer
    unsigned long long seqHalo[2] = {0, 0}, seqRed[PEER_SLOTS] = {0, 0}, seqVec[2] = {0, 0};
    // direct halo stores: the neighbours' vector arena ([below, above]; p at offset 0, w at vecOffW doubles), this rank's published arena
    void* vecBase[2] = {nullptr, nullptr};
    bool vecIpc[2] = {false, false};
    void* vecPublished = nullptr;
    size_t vecOffW = 0;                          // offset of w in EVERY rank's arena this step (doubles; from the global system size)
    bool vecReady = false;
    size_t shCap = 0;                            // shared-region slots of the moment area
    unsigned long long seqSh = 0;
    PeerSync* sync(int r) const { return (PeerSync*)block[r]; }
    double* recv(int r, int kind, int par, int side) const { return (double*)((char*)block[r] + sizeof(PeerSync)) + ((size_t)((kind * 2 + par) * 2 + side)) * cap; }
    size_t shOff() const { return sizeof(PeerSync) + 8 * cap * sizeof(double); }
    unsigned long long* shFlag(int r) const { return (unsigned long long*)((char*)block[r] + shOff()); }          // [2][PEER_MAX_RANKS]
    double* shVal(int r) const { return (double*)((char*)block[r] + shOff() + PEER_SH_FLAG_BYTES); }             // [2][PEER_MAX_RANKS][shCap * 30]
    size_t bytes() const { return shOff() + PEER_SH_FLAG_BYTES + (size_t)2 * PEER_MAX_RANKS * shCap * 30 * sizeof(double); }
    PeerCtx ctx() const { PeerCtx c; if (on) { c.nranks = nranks; c.rank = rank; for (int r = 0; r < nranks; ++r) c.sync[r] = sync(r); } return c; }
};

#if !defined(PS_EMULATE) && defined(__CUDACC__)
constexpr long long PEER_TIMEOUT_CYCLES = 20000000000ll;     // ~10 s at 2 GHz

__device__ __forceinline__ unsigned long long peer_ld_flag(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void peer_st_flag(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double peer_ld_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void peer_st_f64(double* p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" :: "l"(p), "d"(v) : "memory");
}
// spin until *flag >= seq; false on time-out
__device__ __forceinline__ bool peer_wait_flag(const unsigned long long* flag, unsigned long long seq) {
    const long long t0 = clock64();
    while (peer_ld_flag(flag) < seq) {
        if (clock64() - t0 > PEER_TIMEOUT_CYCLES) return false;
        __nanosleep(20);
    }
    return true;
}
// ---- VecLink ----
// head of a consuming kernel, every thread of the CTA: false on time-out.  The acquire also drops this SM's L1 copies of the
// entries the neighbours have rewritten since the last sweep.
__device__ __forceinline__ bool vec_wait(const VecLink& V) {
    if (!V.waitSeq) return true;
    __shared__ int okv;
    if (threadIdx.x == 0) {
        bool good = true;
        if (V.wait[0]) good = peer_wait_flag(V.wait[0], V.waitSeq) && good;
        if (V.wait[1]) good = peer_wait_flag(V.wait[1], V.waitSeq) && good;
        okv = good ? 1 : 0;
    }
    __syncthreads();
    const bool good = okv != 0;
    __syncthreads();
    return good;
}
// one thread, after the launch that stored into the neighbours' vectors has completed: make those stores visible system-wide, then announce
__device__ __forceinline__ void vec_raise(const VecLink& V) {
    if (!V.raiseSeq) return;
    __threadfence_system();
    if (V.raise[0]) peer_st_flag(V.raise[0], V.raiseSeq);
    if (V.raise[1]) peer_st_flag(V.raise[1], V.raiseSeq);
}
// called by every thread of ONE CTA (the last CTA of the producer): thread r stores this rank's partials into rank r's block
__device__ __forceinline__ void peer_reduce_push(const PeerCtx& P, int slot, const double* vals, int nvals) {
    if ((int)threadIdx.x < P.nranks) {
        PeerSync* d = P.sync[threadIdx.x];
        const int par = (int)(P.seqOut & 1ull);
        for (int v = 0; v < nvals; ++v) peer_st_f64(&d->redVal[par][slot][v][P.rank], vals[v]);
        __threadfence_system();
        peer_st_flag(&d->redFlag[par][slot][P.rank], P.seqOut);
    }
}
// called by every thread of a CTA: waits for the N partials of reduction (slot, seq) and returns their rank-ordered
// sums in out[0..nvals); returns false (in every thread) on time-out
__device__ __forceinline__ bool peer_reduce_wait(const PeerCtx& P, int slot, unsigned long long seq, double* out, int nvals) {
    __shared__ double sh[PEER_VALS];
    __shared__ int ok;
    if (threadIdx.x < 32) {
        const PeerSync* m = P.sync[P.rank];
        const int par = (int)(seq & 1ull);
        bool good = true;
        if ((int)threadIdx.x < P.nranks) good = peer_wait_flag(&m->redFlag[par][slot][threadIdx.x], seq);
        good = __all_sync(0xffffffffu, good);
        if (threadIdx.x == 0) {
            ok = good ? 1 : 0;
            for (int v = 0; v < nvals; ++v) { double s = 0.; for (int r = 0; r < P.nranks; ++r) s += peer_ld_f64(&m->redVal[par][slot][v][r]); sh[v] = s; }
        }
    }
    __syncthreads();
    for (int v = 0; v < nvals; ++v) out[v] = sh[v];
    const bool good = ok != 0;
    __syncthreads();
    return good;
}
#endif

}  // namespace ps
