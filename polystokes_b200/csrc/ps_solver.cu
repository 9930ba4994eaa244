// ps_solver.cu -- host orchestration of one Stokes step: the same stage sequence as
// HDK_PolyStokes::solveGasSubclass (exec/HDK_PolyStokes.C:344-584), every stage a few kernels on one stream.
#include "ps_solver.hpp"
#include <climits>
#include <chrono>
#include <memory>
#include <unistd.h>

namespace ps {

thread_local std::string g_lastError;
thread_local int64_t g_launches = 0;
thread_local Scratch* g_scratch = nullptr;
thread_local std::vector<void*>* g_deferredFree = nullptr;
thread_local const char* volatile* g_where = nullptr;

// ---- small helper kernels (free functions: extended lambdas may not live in private members) ----
static void k_flag_label(cudaStream_t st, int64_t lo, int64_t hi, const int8_t* L, int value, uint8_t* flag) {
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) { flag[q] = (L[q] == value) ? 1 : 0; });
}
static void k_krow_active(cudaStream_t st, int64_t lo, int64_t hi, const int32_t* aidx, int32_t offset, int32_t* krow) {
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) { const int a = aidx[q]; krow[q] = a >= 0 ? a + offset : -1; });
}
static void k_krow_reduced(cudaStream_t st, int64_t nRows, const int32_t* rowFace, int32_t base, int32_t* kr0, int32_t* kr1, int32_t* kr2) {
    ps_for(st, nRows, PS_LAMBDA(int64_t i) {
        const int32_t packed = rowFace[i];
        const int axis = (packed >> 29) & 3;
        int32_t* kr = axis == 0 ? kr0 : axis == 1 ? kr1 : kr2;
        kr[packed & 0x1fffffff] = base + (int32_t)i;
    });
}
// per (region, face axis) row counts + the bit-field form of the row list used by the hot kernels
static void k_rows_finalize(cudaStream_t st, const Geom& g, int64_t n, const int32_t* region, const int32_t* rowFace, int* counts, uint32_t* rowXYZ) {
    ps_for(st, n, PS_LAMBDA(int64_t i) {
        const int32_t packed = rowFace[i];
        const int axis = (packed >> 29) & 3;
        const I3 f = delin(g, SL_FACE + axis, (int64_t)(packed & 0x1fffffff));
        rowXYZ[i] = (uint32_t)f.x | ((uint32_t)f.y << 10) | ((uint32_t)f.z << 20) | ((uint32_t)axis << 30);
        atomic_add(&counts[3 * region[i] + axis], 1);
    });
}
static void k_scale_rows(cudaStream_t st, int64_t n, const double* a, const double* b, double* out) {
    ps_for(st, n, PS_LAMBDA(int64_t i) { out[i] = a[i] * b[i]; });
}
// slab of a face plane / cell layer z: rank k holds [zCut[k], zCut[k+1]), the last one also z = nz (the convention of slotCut)
PS_HD int slab_of(const int32_t* zCut, int nranks, int z) { int k = 0; while (k + 1 < nranks && z >= zCut[k + 1]) ++k; return k; }
static void k_gather_first(cudaStream_t st, int32_t R, const int32_t* list, const int32_t* start, int32_t* first) {
    ps_for(st, R, PS_LAMBDA(int64_t r) { first[r] = list[start[r]]; });
}
// touch[region * nranks + k] = 1 if the region has a reduced face in slab k
static void k_region_face_slabs(cudaStream_t st, const Geom& g, int slot, const int32_t* FR, const int32_t* zCut, int nranks, uint8_t* touch) {
    ps_for(st, g.n[slot], PS_LAMBDA(int64_t q) {
        const int ri = FR[q];
        if (ri >= 0) touch[(int64_t)ri * nranks + slab_of(zCut, nranks, delin(g, slot, q).z)] = 1;
    });
}
// sort key of a coupled reduced row: (slab of the face, shared, region) -- a rank's own rows first, those of shared regions last
static void k_span_row_keys(cudaStream_t st, const Geom& g, int64_t n, const int32_t* rowFace, const uint8_t* shared, const int32_t* zCut, int nranks, int32_t R, int32_t* keys) {
    ps_for(st, n, PS_LAMBDA(int64_t i) {
        const int32_t packed = rowFace[i], r = keys[i];
        const int axis = (packed >> 29) & 3;
        const int k = slab_of(zCut, nranks, delin(g, SL_FACE + axis, (int64_t)(packed & 0x1fffffff)).z);
        keys[i] = (2 * k + shared[r]) * R + r;
    });
}
static void k_key_region(cudaStream_t st, int64_t n, const int32_t* keys, int32_t R, int32_t* region) {
    ps_for(st, n, PS_LAMBDA(int64_t i) { region[i] = keys[i] % R; });
}
static void k_copy_reduced_solution(cudaStream_t st, int64_t n, const double* s, double* velSolReduced) {
    ps_for(st, n, PS_LAMBDA(int64_t i) { velSolReduced[i] = s[i]; });
}

// ---- stage timers ----
struct StageTimer {
#ifndef PS_EMULATE
    cudaEvent_t a, b; cudaStream_t st; double* acc;
    StageTimer(cudaStream_t s, double* dst) : st(s), acc(dst) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, st); }
    ~StageTimer() { cudaEventRecord(b, st); cudaEventSynchronize(b); float ms = 0; cudaEventElapsedTime(&ms, a, b); *acc += ms; cudaEventDestroy(a); cudaEventDestroy(b); }
#else
    std::chrono::steady_clock::time_point t0; double* acc;
    StageTimer(cudaStream_t, double* dst) : t0(std::chrono::steady_clock::now()), acc(dst) {}
    ~StageTimer() { *acc += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
#endif
};

Solver::Solver(const ps_params& p) : P(p) {
    if (p.nx <= 0 || p.ny <= 0 || p.nz <= 0 || !(p.dx > 0) || !(p.dt > 0)) throw Error("ps_create: invalid grid / dx / dt");
    if ((int64_t)(p.nx + 1) * (p.ny + 1) * (p.nz + 1) >= (1ll << 29)) throw Error("ps_create: grid too large for 29-bit packed face indices");
    if (p.nx + 1 > 1023 || p.ny + 1 > 1023 || p.nz + 1 > 1023) throw Error("ps_create: grid axis longer than 1022 cells (10-bit packed row coordinates)");
    g = make_geom(p.nx, p.ny, p.nz, p.dx, p.dt, p.constantDensity);
#ifndef PS_EMULATE
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw Error("ps_create: no CUDA device (this library has no CPU path)");
    PS_CUDA(cudaSetDevice(p.device));
    smCount = sm_count();
    PS_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    PS_CUDA(cudaStreamCreateWithFlags(&stIn, cudaStreamNonBlocking));
    PS_CUDA(cudaStreamCreateWithFlags(&stOut, cudaStreamNonBlocking));
#endif
    flags.alloc(64);
    scal.alloc(1);
    scal.zero(st, 1);
    memset(&F, 0, sizeof F);
    part.zCut = {0, p.nz};
}

static int gcd_i(int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; }

// z cuts at multiples of lcm(16, tileSize): the caller's (ps_set_partition, ps_rebalance) or as even as the unit allows (ps_part.hpp)
void Solver::initComm(Comm* c) {
    std::unique_ptr<Comm> guard(c);
    if (c->nranks < 1 || c->rank < 0 || c->rank >= c->nranks) throw Error("ps_comm_init: bad rank / nranks");
    computePartition(c->rank, c->nranks);
    delete comm;
    comm = guard.release();
    haveSetup = false;
}
int Solver::cutUnit() const { return (P.doReducedRegions && P.doTile && P.tileSize >= 1) ? 16 / gcd_i(16, P.tileSize) * P.tileSize : 16; }
std::vector<int> Solver::unitBounds() const {
    const int unit = cutUnit(), nUnits = (g.nz + unit - 1) / unit;
    std::vector<int> b((size_t)nUnits + 1, g.nz);
    for (int u = 0; u < nUnits; ++u) b[u] = u * unit;
    return b;
}
// the slab decomposition as a function of the grid, the tiling / layer parameters and the caller's cuts (ps_comm_init, ps_set_params,
// ps_set_partition, ps_rebalance)
void Solver::computePartition(int rank, int nranks) {
    const int unit = cutUnit();
    // untiled regions, or tiles without padding, may reach across a cut: shared regions (ps_part.hpp), replicated setup
    part.spanning = nranks > 1 && P.doReducedRegions && (!P.doTile || P.tilePadding < 1 || P.tileSize < 1);
    const int nUnits = (g.nz + unit - 1) / unit;
    if (nranks > nUnits) throw Error("ps_comm_init: more ranks than z-slabs of lcm(16, tileSize) cells");
    part.rank = rank; part.nranks = nranks;
    // the caller's cuts while they are multiples of the unit (ps_set_params may change it), the even cuts otherwise
    if (!userCut.empty() && !valid_cuts(userCut, nranks, g.nz, unit)) userCut.clear();
    if (!userCut.empty()) part.zCut = userCut;
    else {
        part.zCut.assign((size_t)nranks + 1, 0);
        for (int k = 0; k <= nranks; ++k) part.zCut[k] = std::min(g.nz, (int)(((int64_t)k * nUnits + nranks / 2) / nranks) * unit);
        part.zCut[0] = 0; part.zCut[nranks] = g.nz;
    }
    for (int k = 0; k < nranks; ++k) if (part.zCut[k + 1] <= part.zCut[k]) throw Error("ps_comm_init: empty z-slab");
    g.zLo = part.zCut[rank]; g.zHi = part.zCut[rank + 1];
    // slab-local setup where regions cannot interact across a cut (ps_part.hpp), unless a step with these tiling / layer
    // parameters has fallen back to the replicated setup (NeedReplicatedSetup)
    part.local = nranks > 1 && !replicatedSetup && (!P.doReducedRegions || (P.doTile && P.tilePadding >= 2));
    part.halo = std::min(16, std::max(4, P.activeLiquidBoundaryLayerSize + P.activeSolidBoundaryLayerSize + 3));
    if (part.local && P.activeLiquidBoundaryLayerSize + P.activeSolidBoundaryLayerSize + 3 > 16) part.local = false;      // the floods reach further than one tile layer
    g.wzLo = part.local ? std::max(0, g.zLo - part.halo) : 0;
    g.wzHi = part.local ? std::min(g.nz, g.zHi + part.halo) : g.nz;
    g.slabLocal = part.local ? 1 : 0;
}
// ps_set_params: everything but the grid and the device may change between steps (dt and density change every substep in a DOP
// network); the buffers, streams and the communicator stay
void Solver::setParams(const ps_params& p) {
    if (p.nx != P.nx || p.ny != P.ny || p.nz != P.nz || p.dx != P.dx) throw Error("ps_set_params: the grid (nx, ny, nz, dx) is fixed at ps_create");
    if (!(p.dt > 0)) throw Error("ps_set_params: invalid dt");
    if (p.doReducedRegions != P.doReducedRegions || p.doTile != P.doTile || p.tileSize != P.tileSize || p.tilePadding != P.tilePadding ||
        p.activeLiquidBoundaryLayerSize != P.activeLiquidBoundaryLayerSize || p.activeSolidBoundaryLayerSize != P.activeSolidBoundaryLayerSize)
        replicatedSetup = false;        // other regions: slab-local setup gets another chance
    const int dev = P.device;
    P = p; P.device = dev;
    const Geom old = g;
    g = make_geom(P.nx, P.ny, P.nz, P.dx, P.dt, P.constantDensity);
    g.zLo = old.zLo; g.zHi = old.zHi; g.wzLo = old.wzLo; g.wzHi = old.wzHi; g.slabLocal = old.slabLocal;
    if (comm) computePartition(part.rank, part.nranks);
    haveSetup = false;
}

// ---- NVLink peer-memory transport (ps_peer.hpp) ----
void Solver::closePeer() {
#ifndef PS_EMULATE
    if (st) cudaStreamSynchronize(st);
    closeVectorMaps();
    for (int r = 0; r < PEER_MAX_RANKS; ++r) {
        if (!peer.block[r]) continue;
        if (r == peer.rank) cudaFree(peer.block[r]); else if (!peer.sameProcess[r]) cudaIpcCloseMemHandle(peer.block[r]);
        peer.block[r] = nullptr;
    }
#endif
    peer = PeerLink();
}

// Collective.  Every rank allocates its symmetric block (flags + reduction slots + 8 halo receive buffers), the IPC
// handles travel by one NCCL all-gather, every rank maps every other block.  Any failure on any rank (no peer
// access, IPC refused) switches ALL ranks back to the NCCL path -- agreed on with one all-reduce.
void Solver::setupPeer() {
#ifndef PS_EMULATE
    PS_WHERE("setupPeer");
    closePeer();
    if (!comm || !part.multi() || part.nranks > PEER_MAX_RANKS) return;
    const char* env = getenv("PS_COMM");
    if (env && std::string(env) == "nccl") return;
    peer.rank = part.rank; peer.nranks = part.nranks;
    peer.cap = (size_t)12 * (g.nx + 1) * (g.ny + 1);
    peer.shCap = PEER_SH_CAP;
    double okLocal = 1.;
    void* mine = nullptr;
    if (cudaMalloc(&mine, peer.bytes()) != cudaSuccess) { cudaGetLastError(); okLocal = 0.; mine = nullptr; }
    // what every rank publishes: an IPC handle for ranks in other processes, the raw pointer + device for ranks of THIS process
    // (ps_create_multi: one host thread per GPU; cudaIpcOpenMemHandle refuses handles of the calling process)
    struct Card { cudaIpcMemHandle_t ipc; unsigned long long pid, ptr; int dev, pad; };
    Card card; memset(&card, 0, sizeof card);
    card.pid = (unsigned long long)getpid(); card.ptr = (unsigned long long)(uintptr_t)mine; card.dev = P.device;
    if (mine) {
        PS_CUDA(cudaMemsetAsync(mine, 0, peer.bytes(), st));
        if (cudaIpcGetMemHandle(&card.ipc, mine) != cudaSuccess) { cudaGetLastError(); okLocal = 0.; }
    }
    DBuf<uint8_t> dSend, dAll;
    DBuf<double> dOk;
    dSend.alloc(sizeof card); dAll.alloc(sizeof card * (size_t)part.nranks); dOk.alloc(1);
    copy_h2d(dSend.p, &card, sizeof card, st);
    comm->allgather(dSend.p, dAll.p, sizeof card, st);
    std::vector<uint8_t> all = dAll.to_host(st, sizeof card * (size_t)part.nranks);
    peer.block[part.rank] = mine;
    if (okLocal > 0.) {
        for (int r = 0; r < part.nranks && okLocal > 0.; ++r) {
            if (r == part.rank) continue;
            Card c; memcpy(&c, all.data() + sizeof c * (size_t)r, sizeof c);
            void* ptr = nullptr;
            if (c.pid == card.pid) {
                int can = 0;
                if (c.ptr == 0 || cudaDeviceCanAccessPeer(&can, P.device, c.dev) != cudaSuccess || !can) { cudaGetLastError(); okLocal = 0.; break; }
                const cudaError_t e = cudaDeviceEnablePeerAccess(c.dev, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); okLocal = 0.; break; }
                cudaGetLastError();
                ptr = (void*)(uintptr_t)c.ptr;
                peer.sameProcess[r] = true;
            } else if (cudaIpcOpenMemHandle(&ptr, c.ipc, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); okLocal = 0.; break; }
            peer.block[r] = ptr;
        }
    }
    copy_h2d(dOk.p, &okLocal, sizeof(double), st);
    comm->allreduce_sum(dOk.p, 1, st);            // also the barrier: every block is zeroed before anybody writes into it
    double okAll = 0.;
    copy_d2h(&okAll, dOk.p, sizeof(double), st);
    if (okAll < part.nranks - 0.5) { const int rk = part.rank, n = part.nranks; closePeer(); peer.rank = rk; peer.nranks = n; return; }
    peer.on = true;
#endif
}

// sum over the ranks of one host value (collective; a host sync -- setup / poll paths only)
double Solver::hostAllreduceSum(double v) {
    if (!part.multi() || !comm) return v;
    PS_WHERE("hostAllreduceSum");
    hostRed.alloc(1);
    copy_h2d(hostRed.p, &v, sizeof(double), st);
    comm->allreduce_sum(hostRed.p, 1, st);
    copy_d2h(&v, hostRed.p, sizeof(double), st);
    return v;
}
std::vector<double> Solver::hostAllgather(const std::vector<double>& mine) {
    const size_t k = mine.size(), n = k * (size_t)part.nranks;
    std::vector<double> all(n, 0.);
    std::copy(mine.begin(), mine.end(), all.begin() + k * (size_t)part.rank);
    if (!part.multi() || !comm) return all;
    PS_WHERE("hostAllgather");
    hostRed.alloc(n);
    copy_h2d(hostRed.p, all.data(), n * sizeof(double), st);
    comm->allreduce_sum(hostRed.p, (int)n, st);
    copy_d2h(all.data(), hostRed.p, n * sizeof(double), st);
    return all;
}
// prefix sums over the ranks of item `item` of an all-gathered table with `stride` entries per rank
std::vector<int64_t> Solver::cutsFromCounts(const std::vector<double>& all, int stride, int item) const {
    std::vector<int64_t> cut((size_t)part.nranks + 1, 0);
    for (int k = 0; k < part.nranks; ++k) cut[k + 1] = cut[k] + (int64_t)std::llround(all[(size_t)k * stride + item]);
    return cut;
}
// tile layers [tz[0], tz[1]) of the own slab (cuts are multiples of 16); the last slab takes the slot's extra top layer, and
// `extraTop` further tile layers can be added above (faces on the upper cut plane that belong to an own region)
void Solver::ownTileZ(int slot, int tz[2], int extraTop) const {
    const int rz = g.r[slot][2];
    tz[0] = g.zLo >> 4;
    tz[1] = g.zHi >= g.nz ? (rz + 15) >> 4 : std::min((rz + 15) >> 4, (g.zHi >> 4) + extraTop);
}
// Halo layers of grid fields: my lower / upper `halo` layers go to the neighbours, theirs arrive in my halo.  Dense x-fastest
// arrays addressed by global voxel index: a z-range is one contiguous byte range, the same on both sides.
void Solver::exchangeLayers(const std::vector<LayerField>& fields) {
    if (!part.local || !comm) return;
    PS_WHERE("exchangeLayers");
    const int H = part.halo;
    std::vector<int> peers; std::vector<const void*> sb; std::vector<size_t> sby; std::vector<void*> rb; std::vector<size_t> rby;
    for (const LayerField& f : fields) {
        for (int side = 0; side < 2; ++side) {
            const int pr = side == 0 ? part.rank - 1 : part.rank + 1;
            if (pr < 0 || pr >= part.nranks) continue;
            int64_t slo, shi, rlo, rhi;
            if (side == 0) { z_range(g, f.slot, g.zLo, std::min(g.zLo + H, g.zHi), slo, shi); z_range(g, f.slot, std::max(g.zLo - H, part.zCut[pr]), g.zLo, rlo, rhi); }
            else { z_range(g, f.slot, std::max(g.zHi - H, g.zLo), g.zHi, slo, shi); z_range(g, f.slot, g.zHi, std::min(g.zHi + H, part.zCut[pr + 1]), rlo, rhi); }
            // z_range gives the slot's extra top layer to a range that ends at nz: only the last slab may send / receive it
            peers.push_back(pr);
            sb.push_back((const char*)f.base + slo * f.elem); sby.push_back((size_t)(shi - slo) * f.elem);
            rb.push_back((char*)f.base + rlo * f.elem); rby.push_back((size_t)(rhi - rlo) * f.elem);
        }
    }
    if (!peers.empty()) comm->sendrecv((int)peers.size(), peers.data(), sb.data(), sby.data(), rb.data(), rby.data(), st);
}
static void k_merge_max_i32(cudaStream_t st, int64_t n, int32_t* dst, const int32_t* src) {
    ps_for(st, n, PS_LAMBDA(int64_t i) { const int32_t a = dst[i], b = src[i]; dst[i] = a > b ? a : b; });
}
// A z-face plane on a cut carries rows of both ranks: active faces are numbered by the upper slab, coupled reduced faces belong
// to a region of the lower one.  Both sides exchange their copy of the plane and keep the larger entry (-1 = none).
void Solver::mergeSharedPlanes(int32_t* f) {
    if (!part.local || !comm) return;
    PS_WHERE("mergeSharedPlanes");
    const int slot = SL_FACE + 2;
    const int64_t plane = (int64_t)g.r[slot][0] * g.r[slot][1];
    xchgTmp.alloc((size_t)plane * 2 * sizeof(int32_t));
    int32_t* tmp = (int32_t*)xchgTmp.p;
    const int peers[2] = {part.rank > 0 ? part.rank - 1 : -1, part.rank + 1 < part.nranks ? part.rank + 1 : -1};
    const int kz[2] = {g.zLo, g.zHi};
    const void* sb[2] = {f + plane * kz[0], f + plane * kz[1]};
    void* rb[2] = {tmp, tmp + plane};
    const size_t bytes[2] = {peers[0] >= 0 ? (size_t)plane * sizeof(int32_t) : 0, peers[1] >= 0 ? (size_t)plane * sizeof(int32_t) : 0};
    comm->sendrecv(2, peers, sb, bytes, rb, bytes, st);
    for (int i = 0; i < 2; ++i) if (peers[i] >= 0) k_merge_max_i32(st, plane, f + plane * kz[i], tmp + plane * i);
}

// a peer-memory wait that timed out leaves the ranks out of step (sequence numbers, flags): report it once, clear the device flag and
// ask for a collective resynchronisation at the next setup
void Solver::checkPeer(const char* where) {
#ifndef PS_EMULATE
    if (!peer.on) return;
    PS_WHERE("checkPeer (stream sync)");
    int err = 0;
    copy_d2h(&err, &scal.p->peerError, sizeof(int), st);
    if (!err) return;
    dev_memset(&scal.p->peerError, 0, sizeof(int), st);
    peer.needResync = true;
    result = R_FAILED;
    throw Error(std::string("a peer-memory wait timed out in ") + where + " (another rank died or fell out of step)");
#else
    (void)where;
#endif
}
// collective, at the start of every setup: if any rank saw a time-out (or was cancelled mid-solve), every rank zeroes its own
// block and restarts the sequence numbers, so one failed step does not poison the handle
void Solver::peerResync() {
#ifndef PS_EMULATE
    if (!peer.on || !comm || !part.multi()) return;
    const double any = hostAllreduceSum(peer.needResync ? 1. : 0.);
    peer.needResync = false;
    if (any < 0.5) return;
    stream_sync(st);
    PS_CUDA(cudaMemsetAsync(peer.block[peer.rank], 0, sizeof(PeerSync), st));
    PS_CUDA(cudaMemsetAsync(peer.shFlag(peer.rank), 0, PEER_SH_FLAG_BYTES, st));
    dev_memset(&scal.p->peerError, 0, sizeof(int), st);
    peer.seqSh = 0;
    for (auto& q : peer.seqHalo) q = 0;
    for (auto& q : peer.seqRed) q = 0;
    for (auto& q : peer.seqVec) q = 0;
    stream_sync(st);
    hostAllreduceSum(0.);          // barrier: every block is clean before anybody stores into it again
#endif
}

PeerCtx Solver::reduceCtx(int slotIn, int slotOut, int slotIn2) {
    PeerCtx c = peer.ctx();
    if (peer.on) {
        if (slotIn >= 0) c.seqIn = peer.seqRed[slotIn];           // produced by the previous kernel of the chain
        if (slotIn2 >= 0) c.seqIn2 = peer.seqRed[slotIn2];        // read before slotOut advances: the x/r/p update consumes and produces slot 1
        if (slotOut >= 0) c.seqOut = ++peer.seqRed[slotOut];
    }
    return c;
}

Solver::~Solver() {
    closePeer();
    if (arenaGraveyard) { dev_free(arenaGraveyard); arenaGraveyard = nullptr; }
    delete comm;
#ifndef PS_EMULATE
    if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    if (stIn) { cudaStreamSynchronize(stIn); cudaStreamDestroy(stIn); }
    if (stOut) { cudaStreamSynchronize(stOut); cudaStreamDestroy(stOut); }
#endif
}

void Solver::setInputs(const ps_fields_in& in) {
    PS_WHERE("setInputs");
    StageTimer T(st, &stageMs[PS_STAGE_UPLOAD]);
    if (!in.surface || !in.collision || !in.viscosity) throw Error("ps_step: surface / collision / viscosity field missing");
    for (int a = 0; a < 3; ++a) if (!in.velocity[a] || !in.collisionvel[a]) throw Error("ps_step: velocity / collisionvel field missing");
    const bool dev = in.memory == PS_MEM_DEVICE;
    const size_t nc = (size_t)g.n[SL_CENTER];
    dSurface.alloc(nc); dCollision.alloc(nc); dViscosity.alloc(nc);
    // Only the layers of the rank's window (+ the margin the stencils reach) cross PCIe: 1 / nranks of the grid with slab-local
    // setup, everything on one GPU.  The caller's arrays are full-grid either way (global voxel index = offset).
    auto upload = [&](float* d, const float* src, int slot, int margin, cudaStream_t s2) {
        int64_t lo, hi;
        z_range(g, slot, g.wzLo - margin, g.wzHi + margin, lo, hi);
        copy_any2d(d + lo, src + lo, (size_t)(hi - lo) * sizeof(float), dev, s2);
    };
    upload(dSurface.p, in.surface, SL_CENTER, 2, st);
    upload(dCollision.p, in.collision, SL_CENTER, 2, st);
    // host inputs: only the two SDFs are needed at once (weights); the other seven fields are first read by the region
    // matrices, so they cross PCIe on the copy stream while weights / classification / numbering run (waitLateInputs)
    cudaStream_t sLate = st;
#ifndef PS_EMULATE
    if (!dev) {
        sLate = stIn;
        cudaEvent_t e; PS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        PS_CUDA(cudaEventRecord(e, st)); PS_CUDA(cudaStreamWaitEvent(stIn, e, 0)); PS_CUDA(cudaEventDestroy(e));   // earlier readers of the old fields
        lateInputsPending = true;
    }
#endif
    upload(dViscosity.p, in.viscosity, SL_CENTER, 2, sLate);
    for (int a = 0; a < 3; ++a) {
        const size_t nf = (size_t)g.n[SL_FACE + a];
        dVel[a].alloc(nf); dColVel[a].alloc(nf);
        upload(dVel[a].p, in.velocity[a], SL_FACE + a, 1, sLate);
        upload(dColVel[a].p, in.collisionvel[a], SL_FACE + a, 1, sLate);
        F.vel[a] = dVel[a].p; F.colvel[a] = dColVel[a].p;
    }
    validSent = false;
    F.surface = dSurface.p; F.collision = dCollision.p; F.viscosity = dViscosity.p;
    // labels / indices start UNASSIGNED (S.cpp:94-152); byte 0xFF = -1 for int8 and int32 alike (window + the margin stencils reach)
    for (int s = 0; s < N_SLOTS; ++s) {
        const size_t n = (size_t)g.n[s];
        dLiqW[s].alloc(n); dFluW[s].alloc(n); dLabel[s].alloc(n); dAidx[s].alloc(n); dRidx[s].alloc(n);
        int64_t lo, hi;
        z_range(g, s, g.wzLo - 2, g.wzHi + 2, lo, hi);
        dev_memset(dLabel[s].p + lo, 0xFF, (size_t)(hi - lo), st);
        dev_memset(dAidx[s].p + lo, 0xFF, (size_t)(hi - lo) * sizeof(int32_t), st);
        dev_memset(dRidx[s].p + lo, 0xFF, (size_t)(hi - lo) * sizeof(int32_t), st);
        F.liqW[s] = dLiqW[s].p; F.fluW[s] = dFluW[s].p; F.label[s] = dLabel[s].p; F.aidx[s] = dAidx[s].p; F.ridx[s] = dRidx[s].p;
    }
    for (int a = 0; a < 3; ++a) {
        dKrow[a].alloc((size_t)g.n[SL_FACE + a]); F.krow[a] = dKrow[a].p;
        int64_t lo, hi;
        z_range(g, SL_FACE + a, g.wzLo - 2, g.wzHi + 2, lo, hi);
        dev_memset(dKrow[a].p + lo, 0xFF, (size_t)(hi - lo) * sizeof(int32_t), st);
    }
    size_t nmax = 0;
    for (int s = 0; s < N_SLOTS; ++s) nmax = std::max(nmax, (size_t)g.n[s]);
    for (auto& b : scratch8) b.alloc(nmax);
    for (auto& b : scratch32) b.alloc(nmax);
    haveSetup = false;
}

// the compute stream joins the copy stream: from here on viscosity / velocity / collision velocity are read
void Solver::waitLateInputs() {
#ifndef PS_EMULATE
    if (!lateInputsPending) return;
    StageTimer T(st, &stageMs[PS_STAGE_UPLOAD]);
    cudaEvent_t e; PS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    PS_CUDA(cudaEventRecord(e, stIn)); PS_CUDA(cudaStreamWaitEvent(st, e, 0)); PS_CUDA(cudaEventDestroy(e));
    lateInputsPending = false;
#endif
}

// `valid` depends on the face labels only (S_Cls:4-54), which are final after setup: a host caller's three valid fields
// are produced now and cross PCIe on the output stream while the CG loop runs
void Solver::sendValidEarly(const ps_fields_out& out) {
    PS_WHERE("sendValidEarly");
#ifndef PS_EMULATE
    if (out.memory == PS_MEM_DEVICE || !(out.valid[0] && out.valid[1] && out.valid[2])) return;
    float* v[3];
    for (int a = 0; a < 3; ++a) { outStage[3 + a].alloc((size_t)g.n[SL_FACE + a]); v[a] = outStage[3 + a].p; }
    k_valid_faces(st, g, F, v);
    cudaEvent_t e; PS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    PS_CUDA(cudaEventRecord(e, st)); PS_CUDA(cudaStreamWaitEvent(stOut, e, 0)); PS_CUDA(cudaEventDestroy(e));
    for (int a = 0; a < 3; ++a) {
        int64_t lo, hi;
        outRange(SL_FACE + a, lo, hi);
        copy_d2any(out.valid[a] + lo, v[a] + lo, (size_t)(hi - lo) * sizeof(float), false, stOut);
    }
    validSent = true;
#endif
}

void Solver::buildIntegrationWeightsAlt() {
    StageTimer T(st, &stageMs[PS_STAGE_WEIGHTS]);
    k_build_weights(st, g, F, scratch8[0].p, scratch8[1].p);
}

void Solver::classifyCells() {
    k_classify_cells(st, g, F, /*genericToActive=*/!P.doReducedRegions);
}

// constructReducedRegions (S_Cls:179-190)
void Solver::constructReducedRegions() {
    uint8_t* stamp = scratch8[0].p;
    const int L = P.activeLiquidBoundaryLayerSize, S = P.activeSolidBoundaryLayerSize;
    if (L > 255 || S > 255) throw Error("boundary layer size > 255 not supported");
    if (L - 1 >= 1) {   // for (layer = 0; layer < L-1; ++layer) { commit; if (layer < L-2) grow; }
        k_air_layer_seed(st, g, F, stamp);
        k_layer_commit(st, g, F, stamp, 1);
        for (int layer = 1; layer <= L - 2; ++layer) { k_air_layer_grow(st, g, F, stamp, layer); k_layer_commit(st, g, F, stamp, layer + 1); }
    }
    if (S >= 1) {
        k_solid_layer_seed(st, g, F, stamp);
        k_layer_commit(st, g, F, stamp, 1);
        for (int layer = 1; layer <= S - 1; ++layer) { k_solid_layer_grow(st, g, F, stamp, layer); k_layer_commit(st, g, F, stamp, layer + 1); }
    }
    k_tiles_and_reduce(st, g, F, P.doTile != 0, P.tileSize, P.tilePadding);
}

void Solver::classifyFaces() { k_classify_faces(st, g, F); }
void Solver::classifyEdges() { k_classify_edges(st, g, F); }

static int read_flag(cudaStream_t st, const int* dflag) { int v = 0; copy_d2h(&v, dflag, sizeof(int), st); return v; }

// constructCenterReducedIndices (S_Cls:217-239): connected components, stencil-overlap fix, small regions
static void k_add_offset_i32(cudaStream_t st, int64_t lo, int64_t hi, int32_t* f, int32_t off) {
    if (off == 0) return;
    ps_for_range(st, lo, hi, PS_LAMBDA(int64_t q) { const int32_t v = f[q]; if (v >= 0) f[q] = v + off; });
}

void Solver::constructCenterReducedIndices() {
    const int64_t nc = g.n[SL_CENTER];
    int32_t* parent = scratch32[0].p; int32_t* minKey = scratch32[1].p; int32_t* firstRank = scratch32[2].p; int32_t* rootId = scratch32[3].p;
    int* dflag = flags.p;
    int64_t wlo, whi;
    z_range(g, SL_CENTER, g.wzLo, g.wzHi, wlo, whi);
    int tz[2];
    ownTileZ(SL_CENTER, tz);
    k_cc_init(st, g, F, parent);
    for (int sweep = 0; sweep < 100000; ++sweep) {
        dev_memset(dflag, 0, sizeof(int), st);
        k_cc_sweep(st, g, F, parent, dflag);
        if (!read_flag(st, dflag)) break;
    }
    dev_memset(minKey + wlo, 0x7f, (size_t)(whi - wlo) * sizeof(int32_t), st);
    k_cc_minkey(st, g, parent, minKey);
    uint8_t* first = scratch8[0].p;
    k_cc_first_flags(st, g, parent, minKey, first);
    // slab-local: only the own cells are members (k_cc_init), so the first cells all lie in the own tile layers
    int64_t R = tile_order_scan(st, g, SL_CENTER, first, firstRank, tileCounts, nullptr, nullptr, part.local ? tz : nullptr);
    k_cc_publish(st, g, parent, first, firstRank, rootId);
    k_cc_assign(st, g, F, parent, rootId);

    // fixReducedRegionBoundaries (S_Cls:1073-1172), see ps_classify.cu for the recurrence
    fixLoops = 0;
    if (R > 0 || part.local) {
        uint8_t* cand = scratch8[0].p; uint8_t* fa = scratch8[1].p; uint8_t* fb = scratch8[2].p;
        for (;;) {
            fixLoops++;
            dev_memset(dflag, 0, 2 * sizeof(int), st);
            k_fix_candidates(st, g, F, cand, fa, fb, dflag);
            const int any = read_flag(st, dflag);
            if (part.local) {
                // padding >= 2 keeps two regions at least two cells apart: the sweep has nothing to do; anything else would need the
                // serial order across the cuts
                if (hostAllreduceSum(any ? 1. : 0.) > 0.5) throw NeedReplicatedSetup();      // every rank leaves here together (setInputsAndSetup)
                break;
            }
            if (!any) break;            // sweep finds nothing to fix -> done
            uint8_t* in = fa; uint8_t* out = fb;
            for (int it = 0; it < 1000000; ++it) {
                dev_memset(dflag, 0, sizeof(int), st);
                k_fix_iterate(st, g, F, cand, in, out, dflag);
                std::swap(in, out);
                if (!read_flag(st, dflag)) break;
            }
            dev_memset(dflag + 1, 0, sizeof(int), st);
            k_fix_apply(st, g, F, in, dflag + 1);
            if (!read_flag(st, dflag + 1)) break;
        }
    }

    // fixSmallReducedRegions (S_Cls:1174-1262)
    if (R > 0) {
        DBuf<int>& bb = scratch().bb;
        bb.alloc((size_t)6 * R);
        dev_memset(bb.p, 0x7f, (size_t)3 * R * sizeof(int), st);
        dev_memset(bb.p + 3 * R, 0x80, (size_t)3 * R * sizeof(int), st);
        k_region_bbox(st, g, F, bb.p, bb.p + 3 * R);
        std::vector<int> h = bb.to_host(st, (size_t)6 * R);
        std::vector<int32_t> remap((size_t)R, -1);
        int32_t next = 0;
        for (int64_t r = 0; r < R; ++r) {
            bool remove = false;
            for (int a = 0; a < 3; ++a) {
                const int mn = h[3 * r + a], mx = h[3 * R + 3 * r + a];
                if (mx < 0) { remove = true; continue; }          // region emptied by the boundary fix
                if (mx == mn) remove = true;
                if (mn > mx - 3) remove = true;
            }
            if (!remove) remap[r] = next++;
        }
        if (next < R) {
            DBuf<int32_t>& dremap = scratch().dremap;
            dremap.from_host(st, remap.data(), (size_t)R);
            k_region_remap(st, g, F, dremap.p);
            R = next;
        }
    }
    if (part.local) {
        // global region ids: regions are numbered by their first cell in tile order (tiles z-slowest), a slab is a whole number of
        // tile layers and holds its regions entirely => ids of slab k follow those of the slabs below it
        const std::vector<double> all = hostAllgather({(double)R});
        const std::vector<int64_t> cut = cutsFromCounts(all, 1, 0);
        part.regionCut.assign(cut.begin(), cut.end());
        int64_t lo, hi;
        z_range(g, SL_CENTER, g.zLo, g.zHi, lo, hi);
        k_add_offset_i32(st, lo, hi, F.ridx[SL_CENTER], (int32_t)cut[part.rank]);
        R = cut[part.nranks];
        // labels / region ids of the halo cells from their owners (small-region removal is the owner's decision)
        exchangeLayers({{F.label[SL_CENTER], SL_CENTER, 1}, {F.ridx[SL_CENTER], SL_CENTER, 4}});
    }
    (void)nc;
    RG.count = (int32_t)R;
}

void Solver::constructFacesReducedIndices() { k_faces_reduced(st, g, F); }
void Solver::constructEdgesReducedIndices() { k_edges_reduced(st, g, F); }

// construct{Center,Faces,Edges}ActiveIndices (S_Cls:257-284)
void Solver::constructActiveIndices() {
    uint8_t* flag = scratch8[0].p;
    int64_t cnt[N_SLOTS];
    // every scan also tells where each z-unit starts in the numbering: the active counts of the own units (unitLoad); the slab cuts
    // are unit boundaries
    const std::vector<int> ub = unitBounds();
    const int unit = cutUnit(), nUnits = (int)ub.size() - 1, uLo = g.zLo / unit, uHi = (g.zHi + unit - 1) / unit;
    std::vector<int64_t> uc;
    auto ownUnits = [&](int s) {
        unitActive[s].assign((size_t)nUnits, 0);
        for (int u = uLo; u < uHi; ++u) unitActive[s][u] = uc[u + 1] - uc[u];
    };
    if (part.local) {
        // every slab numbers its own voxels from 0 (the scan visits its tile layers only); the global index adds the counts of the
        // slabs below -- exactly the reference's running counter, because tile order is z-slowest
        std::vector<double> mine(N_SLOTS);
        for (int s = 0; s < N_SLOTS; ++s) {
            int tz[2];
            ownTileZ(s, tz);
            k_generic_to_active_flags(st, g, s, F.label[s], flag);
            mine[s] = (double)tile_order_scan(st, g, s, flag, F.aidx[s], tileCounts, &ub, &uc, tz);
            ownUnits(s);
        }
        const std::vector<double> all = hostAllgather(mine);
        for (int s = 0; s < N_SLOTS; ++s) {
            part.slotCut[s] = cutsFromCounts(all, N_SLOTS, s);
            cnt[s] = part.slotCut[s][part.nranks];
            int64_t lo, hi;
            z_range(g, s, g.zLo, g.zHi, lo, hi);
            k_add_offset_i32(st, lo, hi, F.aidx[s], (int32_t)part.slotCut[s][part.rank]);
        }
    } else
    for (int s = 0; s < N_SLOTS; ++s) {
        k_generic_to_active_flags(st, g, s, F.label[s], flag);
        cnt[s] = tile_order_scan(st, g, s, flag, F.aidx[s], tileCounts, &ub, &uc);
        ownUnits(s);
        part.slotCut[s].assign((size_t)part.nranks + 1, cnt[s]);
        for (int k = 0; k < part.nranks; ++k) part.slotCut[s][k] = uc[part.zCut[k] / unit];
    }
    C = Counts();
    C.nCenter = cnt[SL_CENTER];
    for (int a = 0; a < 3; ++a) { C.nFace[a] = cnt[SL_FACE + a]; C.nEdge[a] = cnt[SL_EDGE + a]; }
    // constructMatrixBlocks dimension block (S_CMB:12-21)
    C.nActiveVs = C.nFace[0] + C.nFace[1] + C.nFace[2];
    C.nReducedVs = (int64_t)RG.count * RDOF;
    C.nPressures = C.nCenter;
    C.nStresses = 3 * C.nCenter + C.nEdge[0] + C.nEdge[1] + C.nEdge[2];
    C.nTotalDOFs = C.nActiveVs + C.nReducedVs + C.nPressures + C.nStresses;
    C.nSystemSize = C.nPressures + C.nStresses;
    C.faceOff[0] = 0; C.faceOff[1] = C.nFace[0]; C.faceOff[2] = C.nFace[0] + C.nFace[1];
    C.stressOff[0] = 0; C.stressOff[1] = C.nCenter; C.stressOff[2] = 2 * C.nCenter;
    C.stressOff[3] = 3 * C.nCenter; C.stressOff[4] = 3 * C.nCenter + C.nEdge[0]; C.stressOff[5] = 3 * C.nCenter + C.nEdge[0] + C.nEdge[1];
    if (C.nSystemSize >= INT32_MAX || C.nActiveVs + 26 >= INT32_MAX) throw Error("system too large for int32 column indices");
}

static OpArgs make_op(const Solver& S);
static int key_bits(int64_t n) { int b = 1; while ((1ll << b) < n + 1 && b < 31) ++b; return b; }

// builds (region, begin, end) chunk tables of at most `chunk` items for lists sorted by region
static void build_chunks(const std::vector<int>& perRegion, int chunk, std::vector<int32_t>& start, std::vector<int32_t>& table, std::vector<int32_t>& chunkStart) {
    const size_t R = perRegion.size();
    start.assign(R + 1, 0); chunkStart.assign(R + 1, 0); table.clear();
    for (size_t r = 0; r < R; ++r) start[r + 1] = start[r] + perRegion[r];
    for (size_t r = 0; r < R; ++r) {
        chunkStart[r] = (int32_t)(table.size() / 3);
        for (int32_t b = start[r]; b < start[r + 1]; b += chunk) { table.push_back((int32_t)r); table.push_back(b); table.push_back(std::min(b + chunk, start[r + 1])); }
    }
    chunkStart[R] = (int32_t)(table.size() / 3);
}

// computeCenterOfMasses + computeLeastSquaresFits + computeReducedMassMatrices +
// computeReducedViscosityMatricesInteriorOnly (S.cpp:328-490) + the AssembleBlocks dense part (S_AB)
void Solver::computeReducedRegionMatrices() {
    const int R = RG.count;
    if (!part.local) part.regionCut.assign((size_t)part.nranks + 1, 0);      // slab-local: known since the regions were numbered
    RG.regLo = RG.regHi = 0; RG.cellChunkLo = RG.cellChunkHi = 0; RG.maxRegionCells = RG.minRegionCells = 0;
    if (R <= 0) return;
    const int64_t nc = g.n[SL_CENTER];
    DBuf<unsigned long long>& sums = scratch().sums;
    sums.alloc((size_t)4 * R);
    RG.com.alloc((size_t)3 * R);
    k_region_com(st, g, F, R, sums.p, RG.com.p);
    // REDUCED cells sorted by (region, voxel order)
    uint8_t* flag = scratch8[0].p; int32_t* rank = scratch32[0].p;
    int64_t clo = 0, chi = nc;
    int tz[2];
    ownTileZ(SL_CENTER, tz);
    if (part.local) z_range(g, SL_CENTER, g.zLo, g.zHi, clo, chi);      // the cells of the own regions
    k_flag_label(st, clo, chi, F.label[SL_CENTER], L_REDUCED, flag);
    const int64_t nRed = tile_order_scan(st, g, SL_CENTER, flag, rank, tileCounts, nullptr, nullptr, part.local ? tz : nullptr);
    DBuf<int32_t>& keys = scratch().keys; DBuf<int32_t>& kt = scratch().kt; DBuf<int32_t>& vt = scratch().vt;
    keys.alloc((size_t)nRed); RG.cellList.alloc((size_t)nRed);
    k_collect_region_keys(st, g, rank, flag, F.ridx[SL_CENTER], clo, chi, 0, 0, keys.p, RG.cellList.p);
    sort_pairs_by_key(st, nRed, key_bits(R), keys, RG.cellList, kt, vt);
    std::vector<unsigned long long> hs = sums.to_host(st, (size_t)4 * R);
    std::vector<int> perRegion((size_t)R);
    for (int r = 0; r < R; ++r) perRegion[r] = (int)hs[4 * r + 3];
    std::vector<int32_t> start, table, chunkStart;
    build_chunks(perRegion, 256, start, table, chunkStart);
    RG.cellStart.from_host(st, start.data(), start.size());
    // region -> rank: regions are numbered by their first cell in voxel order (z-slowest tiles) and never span a
    // z cut, so every rank owns one contiguous id range (slab-local setup: already known from the all-gathered counts;
    // regions that may span a cut: classifySharedRegions)
    if (part.spanning) classifySharedRegions();
    else if (!part.local) {
        int owner = 0;
        for (int r = 0; r < R; ++r) {
            const int zmean = (int)(hs[4 * r + 2] / std::max<unsigned long long>(hs[4 * r + 3], 1ull));
            int k = 0;
            while (k + 1 < part.nranks && zmean >= part.zCut[k + 1]) ++k;
            if (k < owner) throw Error("region numbering is not monotone in z: cannot slab-decompose these reduced regions");
            while (owner < k) part.regionCut[++owner] = r;
        }
        while (owner < part.nranks) part.regionCut[++owner] = R;
    }
    RG.regLo = part.regionCut[part.rank]; RG.regHi = part.regionCut[part.rank + 1];
    if (!part.spanning) RG.bldLo = RG.regLo;
    if (RG.regHi > RG.regLo) {
        const auto mm = std::minmax_element(perRegion.begin() + RG.regLo, perRegion.begin() + RG.regHi);
        RG.minRegionCells = *mm.first; RG.maxRegionCells = *mm.second;
    }
    RG.nCellChunks = (int32_t)(table.size() / 3);
    RG.cellChunkLo = chunkStart[RG.bldLo]; RG.cellChunkHi = chunkStart[RG.regHi];
    RG.cellChunk.from_host(st, table.data(), table.size());
    RG.cellChunkStart.from_host(st, chunkStart.data(), chunkStart.size());
    const size_t NN = (size_t)RDOF * RDOF;
    RG.partial.alloc((size_t)RG.nCellChunks * 400);
    RG.Mr.alloc(R * NN); RG.Visc.alloc(R * NN); RG.N.alloc(R * NN); RG.Binv.alloc(R * NN);
    RG.lsqRhs.alloc((size_t)R * RDOF); RG.bestFit.alloc((size_t)R * RDOF); RG.rhsR.alloc((size_t)R * RDOF);
    RG.t.alloc((size_t)R * RDOF); RG.s.alloc((size_t)R * RDOF);
    region_gram_partials(st, g, F, RG, RG.partial.p);
    region_gram_finish(st, g, RG, RG.nCellChunks);
}

// Partition::spanning.  Owner of a region = slab of its first cell in voxel order (RG.cellList is sorted by (region, voxel order)); a
// region with reduced faces in more than one slab, or in one slab that is not its owner's, is shared.  Everything follows from the
// replicated classification: every rank derives the same owners and the same shared list.  This rank builds the region matrices
// of the contiguous id range from the lowest shared region it takes part in (rows or reduced faces in its slab) to its last own
// region: the regions of the lower ranks numbered in between are built too.  When region 0 crosses every cut (one untiled body)
// that is every region up to this rank's last one -- on the top rank the whole Gram build.
void Solver::classifySharedRegions() {
    const int R = RG.count, N = part.nranks, me = part.rank;
    zCutDev.from_host(st, part.zCut.data(), part.zCut.size());
    DBuf<int32_t>& first = scratch().rc;
    first.alloc((size_t)R);
    k_gather_first(st, R, RG.cellList.p, RG.cellStart.p, first.p);
    DBuf<uint8_t>& touch = scratch().haloFlag;
    touch.alloc((size_t)R * N); touch.zero(st, (size_t)R * N);
    for (int a = 0; a < 3; ++a) k_region_face_slabs(st, g, SL_FACE + a, F.ridx[SL_FACE + a], zCutDev.p, N, touch.p);
    const std::vector<int32_t> fh = first.to_host(st, (size_t)R);
    const std::vector<uint8_t> th = touch.to_host(st, (size_t)R * N);
    std::vector<int32_t> shList, mine;
    std::vector<uint8_t> flag((size_t)R, 0);
    int owner = 0, lo = INT_MAX;
    for (int r = 0; r < R; ++r) {
        const int k = slab_of(part.zCut.data(), N, delin(g, SL_CENTER, fh[r]).z);
        if (k < owner) throw Error("region numbering is not monotone in z: cannot slab-decompose these reduced regions");
        while (owner < k) part.regionCut[++owner] = r;
        int slabs = 0;
        for (int j = 0; j < N; ++j) slabs += th[(size_t)r * N + j];
        if (slabs > 1 || (slabs == 1 && !th[(size_t)r * N + k])) {
            flag[r] = 1;
            if (th[(size_t)r * N + me] || k == me) { mine.push_back((int32_t)shList.size()); lo = std::min(lo, r); }
            shList.push_back(r);
        }
    }
    while (owner < N) part.regionCut[++owner] = R;
    RG.bldLo = std::min(lo, part.regionCut[me]);
    RG.nShared = (int32_t)shList.size(); RG.nShMine = (int32_t)mine.size();
    RG.shRegion.from_host(st, shList.data(), shList.size() + 0);
    RG.shMine.from_host(st, mine.data(), mine.size());
    RG.shFlag.from_host(st, flag.data(), flag.size());
    RG.shMoments.alloc((size_t)RG.nShared * 30 + 1);
    stream_sync(st);      // the host vectors die here
}

// constructMatrixBlocks (S_CMB:9-868): row numbering of K_ext, then the ELL fills
void Solver::constructMatrixBlocks() {
    const int R = RG.count;
    // slab-local: the DOF indices of the halo voxels come from their owners (every kernel below reads its neighbours' indices)
    if (part.local) {
        std::vector<LayerField> f;
        for (int s = 0; s < N_SLOTS; ++s) f.push_back({F.aidx[s], s, 4});
        exchangeLayers(f);
    }
    for (int a = 0; a < 3; ++a) {
        int64_t lo, hi;
        z_range(g, SL_FACE + a, g.wzLo, g.wzHi, lo, hi);
        k_krow_active(st, lo, hi, F.aidx[SL_FACE + a], (int32_t)C.faceOff[a], F.krow[a]);
    }
    RG.nRows = 0; RG.nRowChunks = 0; RG.rowChunkLo = RG.rowChunkHi = 0; RG.ownRowLo = RG.ownRowHi = 0; RG.maxRegionRows = RG.maxRegionAxisRows = 0;
    part.redRowCut.assign((size_t)part.nranks + 1, 0);
    if (R > 0) {
        // the coupled reduced faces of the regions this rank builds rows for: all regions (one GPU, replicated setup) or its own;
        // a region's faces reach one plane above the slab (the z-faces on the upper cut)
        const int32_t fLo = part.local ? RG.regLo : 0, fHi = part.local ? RG.regHi : R;
        int64_t cnt[3], off[3];
        for (int a = 0; a < 3; ++a) {
            int64_t lo = 0, hi = g.n[SL_FACE + a];
            int tz[2];
            ownTileZ(SL_FACE + a, tz, 1);
            if (part.local) z_range(g, SL_FACE + a, g.zLo, std::min(g.nz, g.zHi + 1), lo, hi);
            if (part.local) { int64_t tlo, thi; z_range(g, SL_FACE + a, tz[0] * 16, std::min(g.nz, tz[1] * 16), tlo, thi); dev_memset(scratch8[a].p + tlo, 0, (size_t)(thi - tlo), st); }
            k_flag_coupled_faces(st, g, F, a, scratch8[a].p, fLo, fHi, lo, hi);
            cnt[a] = tile_order_scan(st, g, SL_FACE + a, scratch8[a].p, scratch32[a].p, tileCounts, nullptr, nullptr, part.local ? tz : nullptr);
        }
        off[0] = 0; off[1] = cnt[0]; off[2] = cnt[0] + cnt[1];
        const int64_t nLocal = cnt[0] + cnt[1] + cnt[2];
        // global row numbers: the rows are sorted by (region, axis, voxel order) and the regions of a slab are contiguous
        int64_t rowOff = 0, nRows = nLocal;
        if (part.local) {
            const std::vector<double> all = hostAllgather({(double)nLocal});
            part.redRowCut = cutsFromCounts(all, 1, 0);
            rowOff = part.redRowCut[part.rank]; nRows = part.redRowCut[part.nranks];
        }
        RG.nRows = nRows;
        RG.rowFace.alloc((size_t)nRows + 1); RG.rowRegion.alloc((size_t)nRows + 1);
        DBuf<int32_t>& lk = scratch().keys; DBuf<int32_t>& lv = scratch().selStaging;      // local (region, face) pairs
        lk.alloc((size_t)nLocal + 1); lv.alloc((size_t)nLocal + 1);
        for (int a = 0; a < 3; ++a) {
            int64_t lo = 0, hi = g.n[SL_FACE + a];
            if (part.local) z_range(g, SL_FACE + a, g.zLo, std::min(g.nz, g.zHi + 1), lo, hi);
            k_collect_region_keys(st, g, scratch32[a].p, scratch8[a].p, F.ridx[SL_FACE + a], lo, hi, (int32_t)(a << 29), (int32_t)off[a], lk.p, lv.p);
        }
        // shared regions (Partition::spanning): the rows go by the slab of the face, the rank's shared rows after its other rows
        const int KM = part.spanning ? 2 * part.nranks : 1;
        if ((int64_t)R * KM >= INT32_MAX) throw Error("too many reduced regions x ranks for 32-bit row keys");
        if (part.spanning) k_span_row_keys(st, g, nLocal, lv.p, RG.shFlag.p, zCutDev.p, part.nranks, R, lk.p);
        DBuf<int32_t>& kt = scratch().kt; DBuf<int32_t>& vt = scratch().vt;
        sort_pairs_by_key(st, nLocal, key_bits((int64_t)R * KM), lk, lv, kt, vt);
        if (part.spanning) k_key_region(st, nLocal, lk.p, R, RG.rowRegion.p);
        else copy_d2d(RG.rowRegion.p + rowOff, lk.p, (size_t)nLocal * sizeof(int32_t), st);
        copy_d2d(RG.rowFace.p + rowOff, lv.p, (size_t)nLocal * sizeof(int32_t), st);
        if (C.nActiveVs + nRows >= INT32_MAX) throw Error("K_ext has too many rows for int32");
        k_krow_reduced(st, nLocal, RG.rowFace.p + rowOff, (int32_t)(C.nActiveVs + rowOff), F.krow[0], F.krow[1], F.krow[2]);
        DBuf<int>& rc = scratch().rc;
        rc.alloc((size_t)3 * R * KM); rc.zero(st, (size_t)3 * R * KM);
        RG.rowXYZ.alloc((size_t)nRows + 1);
        k_rows_finalize(st, g, nLocal, part.spanning ? lk.p : RG.rowRegion.p + rowOff, RG.rowFace.p + rowOff, rc.p, RG.rowXYZ.p + rowOff);
        const std::vector<int> perRAall = rc.to_host(st, (size_t)3 * R * KM);
        // row counts per (region, axis) of the rows laid out below: all of them, or this rank's rows of its unshared regions
        const int* perRA = perRAall.data() + (part.spanning ? (size_t)3 * R * (2 * part.rank) : 0);
        if (part.spanning) {
            for (int k = 0; k < part.nranks; ++k) {
                int64_t n = 0;
                for (size_t i = (size_t)3 * R * (2 * k); i < (size_t)3 * R * (2 * k + 2); ++i) n += perRAall[i];
                part.redRowCut[k + 1] = part.redRowCut[k] + n;
            }
        }
        // chunk table: rows are sorted by (region, axis, voxel order); a chunk holds <= 2048 rows of one (region, axis)
        std::vector<int32_t> start((size_t)R + 1, 0), chunkStart((size_t)R + 1, 0), table, axisStart((size_t)3 * R + 1, 0);
        for (int r = 0; r < R; ++r) RG.maxRegionRows = std::max(RG.maxRegionRows, (int32_t)(perRA[3 * r] + perRA[3 * r + 1] + perRA[3 * r + 2]));
        for (int i = 0; i < 3 * R; ++i) RG.maxRegionAxisRows = std::max(RG.maxRegionAxisRows, (int32_t)perRA[i]);
        if (part.local) RG.maxRegionRows = (int32_t)std::llround(hostAllreduceSum((double)RG.maxRegionRows));      // every rank takes the same kernels (an upper bound is enough)
        int32_t pos = part.spanning ? (int32_t)part.redRowCut[part.rank] : 0;
        for (int r = 0; r < R; ++r) {
            if (part.local && r == RG.regLo) pos = (int32_t)rowOff;      // the regions below belong to other ranks (no rows here)
            start[r] = pos; chunkStart[r] = (int32_t)(table.size() / 4);
            for (int a = 0; a < 3; ++a) {
                axisStart[3 * r + a] = pos;
                const int32_t e = pos + perRA[3 * r + a];
                for (int32_t b = pos; b < e; b += 2048) { table.push_back(r); table.push_back(b); table.push_back(std::min(b + 2048, e)); table.push_back(a); }
                pos = e;
            }
        }
        start[R] = pos; chunkStart[R] = (int32_t)(table.size() / 4);
        RG.nRowChunks = (int32_t)(table.size() / 4);
        RG.rowChunkLo = chunkStart[RG.regLo]; RG.rowChunkHi = chunkStart[RG.regHi];
        RG.ownRowLo = start[RG.regLo]; RG.ownRowHi = start[RG.regHi];
        RG.regionTicket.alloc((size_t)R + 1); RG.regionTicket.zero(st, (size_t)R + 1);
        if (!part.local && !part.spanning) for (int k = 0; k <= part.nranks; ++k) part.redRowCut[k] = start[part.regionCut[k]];
        if (part.spanning) {      // this rank's rows of the shared regions: chunks of <= 2048 rows of one (region, axis), per slot
            const int* shRA = perRAall.data() + (size_t)3 * R * (2 * part.rank + 1);
            const std::vector<int32_t> shList = RG.shRegion.to_host(st, (size_t)RG.nShared);
            std::vector<int32_t> shTable, shStart((size_t)RG.nShared + 1, 0);
            RG.shRowLo = pos;
            for (int j = 0; j < RG.nShared; ++j) {
                const int r = shList[j];
                shStart[j] = (int32_t)(shTable.size() / 4);
                for (int a = 0; a < 3; ++a) {
                    const int32_t e = pos + shRA[3 * r + a];
                    for (int32_t b = pos; b < e; b += 2048) { shTable.push_back(r); shTable.push_back(b); shTable.push_back(std::min(b + 2048, e)); shTable.push_back(a); }
                    pos = e;
                }
            }
            shStart[RG.nShared] = (int32_t)(shTable.size() / 4);
            RG.shRowHi = pos;
            if (pos != part.redRowCut[part.rank + 1]) throw Error("shared-region row layout does not match the row cut");
            RG.nShChunks = (int32_t)(shTable.size() / 4);
            RG.shChunk.from_host(st, shTable.data(), shTable.size() + 0);
            RG.shChunkStart.from_host(st, shStart.data(), shStart.size());
            RG.shPartial.alloc((size_t)RG.nShChunks * 10 + 1);
            stream_sync(st);
        }
        axisStart[(size_t)3 * R] = pos;
        RG.rowAxisStart.from_host(st, axisStart.data(), axisStart.size());
        RG.rowStart.from_host(st, start.data(), start.size());
        RG.rowChunk.from_host(st, table.data(), table.size());
        RG.rowChunkStart.from_host(st, chunkStart.data(), chunkStart.size());
        RG.partial.alloc(std::max((size_t)RG.nRowChunks * 10, RG.partial.n));
        RG.sigma.alloc((size_t)R * 30);
    }
    if (part.local) {
        // row numbers of the halo faces from their owners; the z-face planes on the cuts hold rows of both sides
        exchangeLayers({{F.krow[0], SL_FACE + 0, 4}, {F.krow[1], SL_FACE + 1, 4}});
        std::vector<LayerField> fz = {{F.krow[2], SL_FACE + 2, 4}};
        mergeSharedPlanes(F.krow[2]);
        exchangeLayers(fz);
        mergeSharedPlanes(F.krow[2]);
    }
    C.nRowsExt = C.nActiveVs + RG.nRows;
    const int64_t nE = C.nEdge[0] + C.nEdge[1] + C.nEdge[2];
    Op.alloc(C.nRowsExt, C.nActiveVs, C.nCenter, nE);
    mcInv.alloc((size_t)C.nActiveVs); mc.alloc((size_t)C.nActiveVs); rhsU.alloc((size_t)C.nActiveVs); oldVs.alloc((size_t)C.nActiveVs);
    computeOwnership();
    RowSet allRows; allRows.add(0, C.nRowsExt);
    k_assemble_K(st, g, F, C, Op, mcInv.p, mc.p, rhsU.p, oldVs.p, part.local ? ownK : allRows);
    uInv.alloc((size_t)C.nStresses); uDiag.alloc((size_t)C.nStresses); rhsPT.alloc((size_t)C.nSystemSize);
    k_assemble_Kt(st, g, F, C, Op, uInv.p, uDiag.p, rhsPT.p, part.local);
    const size_t n = (size_t)C.nSystemSize;
    b.alloc(n); x.alloc(n); r.alloc(n); Ap.alloc(n); allocVectors(n, (size_t)C.nRowsExt + 1);
    velSol.alloc((size_t)(C.nActiveVs + C.nReducedVs) + 1);
    dotPartial.alloc(3 * 16384);      // three partial sums per CTA of a hot sweep (grids: SM count x resident CTAs, at most 2^14: ps_pcg.cu)
    computeOwnership();
    buildSchedules();
    buildHalos();
    exchangeVectorPointers();
}

// p and w: with the peer transport both live in ONE arena of their own (an IPC handle covers exactly that allocation), which the
// z-neighbours map so that the kernels can store halo entries straight into their copies (VecLink, ps_peer.hpp)
void Solver::allocVectors(size_t n, size_t nRows) {
#ifndef PS_EMULATE
    if (peer.on) {
        const size_t offW = (n + 31) & ~(size_t)31;
        const size_t need = offW + nRows;
        if (!vecArena.p || vecArena.n < need) {
            if (arenaGraveyard) { dev_free(arenaGraveyard); arenaGraveyard = nullptr; }
            arenaGraveyard = vecArena.release();          // the neighbours still map it: freed after they have let go (exchangeVectorPointers)
            vecArena.alloc(std::max(need + need / 8, (size_t)1 << 19));
        }
        p.adopt(vecArena.p, n); w.adopt(vecArena.p + offW, nRows);
        peer.vecOffW = offW;
        return;
    }
#endif
    p.alloc(n); w.alloc(nRows);
}
void Solver::closeVectorMaps() {
#ifndef PS_EMULATE
    for (int i = 0; i < 2; ++i) {
        if (peer.vecBase[i] && peer.vecIpc[i]) cudaIpcCloseMemHandle(peer.vecBase[i]);
        peer.vecBase[i] = nullptr; peer.vecIpc[i] = false;
    }
    peer.vecReady = false;
#endif
}
// Collective (every setup with the peer transport on): one host all-reduce tells whether any rank's arena moved (first step, or a
// larger system); only then the arenas are published and mapped again.
void Solver::exchangeVectorPointers() {
    fusedHalo = false;
#ifndef PS_EMULATE
    if (!peer.on || !comm || !part.multi()) return;
    PS_WHERE("exchangeVectorPointers");
    const bool moved = (void*)vecArena.p != peer.vecPublished;
    const bool anyMoved = hostAllreduceSum(moved ? 1. : 0.) > 0.5;
    if (anyMoved) {
        stream_sync(st);
        closeVectorMaps();
        struct Card { cudaIpcMemHandle_t ipc; unsigned long long pid, ptr; int dev, ok; };
        Card card; memset(&card, 0, sizeof card);
        card.pid = (unsigned long long)getpid(); card.ptr = (unsigned long long)(uintptr_t)vecArena.p; card.dev = P.device; card.ok = 1;
        if (cudaIpcGetMemHandle(&card.ipc, vecArena.p) != cudaSuccess) { cudaGetLastError(); card.ok = 0; }
        DBuf<uint8_t> dSend, dAll;
        dSend.alloc(sizeof card); dAll.alloc(sizeof card * (size_t)part.nranks);
        copy_h2d(dSend.p, &card, sizeof card, st);
        comm->allgather(dSend.p, dAll.p, sizeof card, st);
        const std::vector<uint8_t> all = dAll.to_host(st, sizeof card * (size_t)part.nranks);
        bool ok = card.ok != 0;
        for (int i = 0; i < 2; ++i) {
            const int pr = i == 0 ? part.rank - 1 : part.rank + 1;
            if (pr < 0 || pr >= part.nranks) continue;
            Card c; memcpy(&c, all.data() + sizeof c * (size_t)pr, sizeof c);
            if (!c.ok || !c.ptr) { ok = false; continue; }
            void* ptr = nullptr;
            if (c.pid == card.pid) { ptr = (void*)(uintptr_t)c.ptr; peer.vecIpc[i] = false; }              // peer access was enabled in setupPeer
            else if (cudaIpcOpenMemHandle(&ptr, c.ipc, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; continue; }
            else peer.vecIpc[i] = true;
            peer.vecBase[i] = ptr;
        }
        peer.vecPublished = vecArena.p;
        peer.vecReady = hostAllreduceSum(ok ? 0. : 1.) < 0.5;        // also the barrier: every neighbour has closed its mapping of the previous arena
        if (arenaGraveyard) { dev_free(arenaGraveyard); arenaGraveyard = nullptr; }
    }
    fusedHalo = peer.vecReady;
#endif
}

// ---- ownership (ps_part.hpp): row / DOF ranges of rank k in the global numbering ----
RowSet Solver::rowsK(int k) const {
    RowSet r;
    for (int a = 0; a < 3; ++a) r.add(C.faceOff[a] + part.slotCut[SL_FACE + a][k], C.faceOff[a] + part.slotCut[SL_FACE + a][k + 1]);
    r.add(C.nActiveVs + part.redRowCut[k], C.nActiveVs + part.redRowCut[k + 1]);
    return r;
}
RowSet Solver::rowsP(int k) const { return one_range(part.slotCut[SL_CENTER][k], part.slotCut[SL_CENTER][k + 1]); }
RowSet Solver::rowsC(int k) const {   // numbering inside the centre-stress block [xx | yy | zz]
    RowSet r;
    for (int a = 0; a < 3; ++a) r.add(a * C.nCenter + part.slotCut[SL_CENTER][k], a * C.nCenter + part.slotCut[SL_CENTER][k + 1]);
    return r;
}
RowSet Solver::rowsE(int k) const {   // numbering inside the edge-stress block [yz | xz | xy]
    RowSet r;
    for (int e = 0; e < 3; ++e) { const int64_t off = C.stressOff[3 + e] - 3 * C.nCenter; r.add(off + part.slotCut[SL_EDGE + e][k], off + part.slotCut[SL_EDGE + e][k + 1]); }
    return r;
}
RangeSet Solver::rowsSys(int k) const {  // x = [p | xx | yy | zz | yz | xz | xy]
    RangeSet r;
    const RowSet p = rowsP(k), c = rowsC(k), e = rowsE(k);
    for (int i = 0; i < p.n; ++i) r.add(p.lo[i], p.lo[i] + p.count(i));
    for (int i = 0; i < c.n; ++i) r.add(C.nPressures + c.lo[i], C.nPressures + c.lo[i] + c.count(i));
    for (int i = 0; i < e.n; ++i) r.add(C.nPressures + 3 * C.nCenter + e.lo[i], C.nPressures + 3 * C.nCenter + e.lo[i] + e.count(i));
    return r;
}
// K-way merge of the ranges' 256-row blocks by fractional position (j + 1/2) / blocks(k); ties go to the lower range
std::vector<int32_t> merge_schedule(const SchedRanges& R) {
    int64_t nb[4] = {0, 0, 0, 0}, next[4] = {0, 0, 0, 0}, total = 0;
    for (int k = 0; k < R.n; ++k) { nb[k] = R.blocks(k); total += nb[k]; }
    std::vector<int32_t> out;
    out.reserve((size_t)total);
    for (int64_t i = 0; i < total; ++i) {
        int best = -1;
        for (int k = 0; k < R.n; ++k) {
            if (next[k] >= nb[k]) continue;
            // (2 next[k] + 1) / nb[k] < (2 next[best] + 1) / nb[best], in integers
            if (best < 0 || (2 * next[k] + 1) * nb[best] < (2 * next[best] + 1) * nb[k]) best = k;
        }
        if (nb[best] >= (1ll << 28)) throw Error("merge_schedule: range too long for 28-bit block indices");
        out.push_back((int32_t)((uint32_t)best << 28 | (uint32_t)next[best]));
        ++next[best];
    }
    return out;
}
void Solver::buildSchedules() {
    const int k = part.rank;
    sr1 = SchedRanges(); sr2 = SchedRanges();
    for (int a = 0; a < 3; ++a) sr1.add(C.faceOff[a] + part.slotCut[SL_FACE + a][k], C.faceOff[a] + part.slotCut[SL_FACE + a][k + 1]);
    sr1.add(C.nActiveVs + part.redRowCut[k], C.nActiveVs + part.redRowCut[k + 1]);
    sr2.add(part.slotCut[SL_CENTER][k], part.slotCut[SL_CENTER][k + 1]);
    for (int e = 0; e < 3; ++e) { const int64_t off = C.stressOff[3 + e] - 3 * C.nCenter; sr2.add(off + part.slotCut[SL_EDGE + e][k], off + part.slotCut[SL_EDGE + e][k + 1]); }
    const std::vector<int32_t> a = merge_schedule(sr1), b = merge_schedule(sr2);
    nSched1 = (int)a.size(); nSched2 = (int)b.size();
    sched1.from_host(st, a.data(), a.size()); sched2.from_host(st, b.data(), b.size());
    stream_sync(st);    // the vectors die here
}
void Solver::computeOwnership() {
    if (part.regionCut.size() != (size_t)part.nranks + 1) part.regionCut.assign((size_t)part.nranks + 1, 0);   // no reduced regions
    ownK = rowsK(part.rank); ownP = rowsP(part.rank); ownC = rowsC(part.rank); ownE = rowsE(part.rank); ownSys = rowsSys(part.rank);
}

// Halo lists.  Matrices are replicated, so a rank derives BOTH directions locally and the two sides of a pair
// agree by construction: what I receive from h = columns of my rows that h owns; what I send to h = columns of
// h's rows that I own.  Lists are ascending in the global index.
void Solver::buildHalos() {
    PS_WHERE("buildHalos");
    haloX.reset(); haloW.reset();
    if (!part.multi()) return;
    const int64_t n = C.nSystemSize, nRows = C.nRowsExt;
    DBuf<uint8_t>& flag = scratch().haloFlag;
    flag.alloc((size_t)std::max(n, nRows) + 1);
    const int me = part.rank;
    const int peers[2] = {me > 0 ? me - 1 : -1, me + 1 < part.nranks ? me + 1 : -1};
    const OpArgs A = make_op(*this);
    auto listX = [&](int rowsOf, int colsOf, DBuf<int32_t>& out, int64_t off) {
        flag.zero(st, (size_t)n);
        k_mark_K_columns(st, A, rowsK(rowsOf), rowsSys(colsOf), flag.p);
        return select_flagged(st, n, flag.p, out, off);
    };
    auto listW = [&](int rowsOf, int colsOf, DBuf<int32_t>& out, int64_t off) {
        flag.zero(st, (size_t)nRows);
        k_mark_Kt_columns(st, A, rowsP(rowsOf), rowsE(rowsOf), rowsK(colsOf), flag.p);
        return select_flagged(st, nRows, flag.p, out, off);
    };
    for (int i = 0; i < 2; ++i) {
        haloX.peers[i] = haloW.peers[i] = peers[i];
        if (peers[i] < 0) continue;
        haloX.nRecv[i] = listX(me, peers[i], haloX.recvIdx, i ? haloX.nRecv[0] : 0);
        haloW.nRecv[i] = listW(me, peers[i], haloW.recvIdx, i ? haloW.nRecv[0] : 0);
        if (!part.local) {      // replicated matrices: the peer's rows are here too, derive the send side locally
            haloX.nSend[i] = listX(peers[i], me, haloX.sendIdx, i ? haloX.nSend[0] : 0);
            haloW.nSend[i] = listW(peers[i], me, haloW.sendIdx, i ? haloW.nSend[0] : 0);
        }
    }
    if (part.local) {
        // slab-local matrices: a rank only knows what it needs (columns of ITS rows that a neighbour owns).  The neighbours tell
        // each other: my send list towards h = h's receive list from me (ascending global indices on both sides).
        for (Halo* H : {&haloX, &haloW}) {
            std::vector<double> mine = {(double)H->nRecv[0], (double)H->nRecv[1]};
            const std::vector<double> all = hostAllgather(mine);
            for (int i = 0; i < 2; ++i) H->nSend[i] = peers[i] >= 0 ? (int64_t)std::llround(all[(size_t)peers[i] * 2 + (1 - i)]) : 0;     // what my lower peer wants from its upper side, and vice versa
            H->sendIdx.alloc((size_t)H->sendTotal() + 1);
            const void* sb[2] = {H->recvIdx.p, H->recvIdx.p + H->nRecv[0]};
            void* rb[2] = {H->sendIdx.p, H->sendIdx.p + H->nSend[0]};
            const size_t sby[2] = {(size_t)H->nRecv[0] * sizeof(int32_t), (size_t)H->nRecv[1] * sizeof(int32_t)};
            const size_t rby[2] = {(size_t)H->nSend[0] * sizeof(int32_t), (size_t)H->nSend[1] * sizeof(int32_t)};
            comm->sendrecv(2, peers, sb, sby, rb, rby, st);
        }
    }
    for (Halo* H : {&haloX, &haloW}) { H->sendBuf.alloc((size_t)H->sendTotal() + 1); H->recvBuf.alloc((size_t)H->recvTotal() + 1); H->sendIdx.alloc(1); H->recvIdx.alloc(1); }
}

// pack -> grouped send/recv with the z-neighbours -> scatter into the global-length vector
void Solver::exchange(Halo& H, double* v, const PcgScalars* S) {
    if (!part.multi() || !comm) return;
#ifndef PS_EMULATE
    if (peer.on) {
        // sender stores straight into the neighbour's receive buffer over NVLink and raises its flag; the receiver
        // waits on its own flag and scatters.  My lower neighbour sees me as its "above" side (1), the upper one as "below" (0).
        const int kind = (&H == &haloW) ? 1 : 0;
        const unsigned long long seq = ++peer.seqHalo[kind];
        const int par = (int)(seq & 1ull);
        for (int i = 0; i < 2; ++i) if ((size_t)H.nSend[i] > peer.cap || (size_t)H.nRecv[i] > peer.cap) throw Error("halo larger than the peer receive buffer");
        double* dst[2] = {nullptr, nullptr}; unsigned long long* dflag[2] = {nullptr, nullptr};
        const double* src[2] = {nullptr, nullptr}; const unsigned long long* sflag[2] = {nullptr, nullptr};
        for (int i = 0; i < 2; ++i) {
            const int pr = H.peers[i];
            if (pr < 0) continue;
            dst[i] = peer.recv(pr, kind, par, 1 - i); dflag[i] = &peer.sync(pr)->haloFlag[kind][par][1 - i];
            src[i] = peer.recv(part.rank, kind, par, i); sflag[i] = &peer.sync(part.rank)->haloFlag[kind][par][i];
        }
        k_halo_exchange_peer(st, H.nSend[0], H.nSend[1], H.sendIdx.p, dst[0], dst[1], dflag[0], dflag[1], H.nRecv[0], H.nRecv[1], H.recvIdx.p, src[0], src[1], sflag[0], sflag[1],
                             seq, v, scal.p, S != nullptr, &scal.p->ticket[4 + kind]);
        return;
    }
#endif
    k_halo_pack(st, H.sendTotal(), H.sendIdx.p, v, H.sendBuf.p, S);
    const void* sb[2] = {H.sendBuf.p, H.sendBuf.p + H.nSend[0]};
    void* rb[2] = {H.recvBuf.p, H.recvBuf.p + H.nRecv[0]};
    const size_t sbytes[2] = {(size_t)H.nSend[0] * sizeof(double), (size_t)H.nSend[1] * sizeof(double)};
    const size_t rbytes[2] = {(size_t)H.nRecv[0] * sizeof(double), (size_t)H.nRecv[1] * sizeof(double)};
    comm->sendrecv(2, H.peers, sb, sbytes, rb, rbytes, st);
    k_halo_unpack(st, H.recvTotal(), H.recvIdx.p, H.recvBuf.p, v, S);
}
// My boundary entries of w (kind 1), or of the p the coming update will produce (kind 0, `updateCtx` = the update's reduction context),
// straight into the neighbours' vectors.  The launch only stores; the returned link tells the NEXT launch which flags to raise.
VecLink Solver::pushDirect(Halo& H, int kind, const PeerCtx* updateCtx) {
    VecLink L;
#ifndef PS_EMULATE
    L.raiseSeq = ++peer.seqVec[kind];
    double* dst[2] = {nullptr, nullptr};
    for (int i = 0; i < 2; ++i) {
        const int pr = H.peers[i];
        if (pr < 0) continue;
        // w starts at the same offset in every rank's arena: it follows from the GLOBAL system size of THIS step (allocVectors), which
        // changes from step to step while the arenas stay where they are -- so it is recomputed, never remembered from the last exchange
        dst[i] = (double*)peer.vecBase[i] + (kind == 0 ? 0 : peer.vecOffW);
        L.raise[i] = &peer.sync(pr)->vecFlag[kind][1 - i];       // the lower neighbour sees this rank as its "above" side
    }
    if (kind == 0) k_halo_push_p(st, H.nSend[0], H.nSend[1], H.sendIdx.p, r.p, p.p, Ap.p, dst[0], dst[1], scal.p, *updateCtx);
    else k_halo_push_direct(st, H.nSend[0], H.nSend[1], H.sendIdx.p, w.p, dst[0], dst[1], scal.p);
#else
    (void)H; (void)kind; (void)updateCtx;
#endif
    return L;
}
void Solver::allreduce(double* devBuf, int n) { if (part.multi() && comm && !peer.on) comm->allreduce_sum(devBuf, n, st); }

static OpArgs make_op(const Solver& S) {
    OpArgs A;
    A.nRowsExt = S.C.nRowsExt; A.nActiveVs = S.C.nActiveVs; A.nP = S.C.nPressures; A.nT = S.C.nStresses; A.nC = S.C.nCenter;
    A.nE = S.C.nEdge[0] + S.C.nEdge[1] + S.C.nEdge[2];
    A.kcode = S.Op.kcode.p; A.kcol = S.Op.kcol.p; A.kmc = S.Op.kmc.p; A.mcInvLut = S.Op.mcInvLut.p;
    A.ccode = S.Op.ccode.p; A.ccol = S.Op.ccol.p; A.ecode = S.Op.ecode.p; A.ecol = S.Op.ecol.p;
    A.uInv = S.uInv.p; A.valScale = S.g.invDx / 64.;
    A.rowsK = S.ownK; A.rowsP = S.ownP; A.rowsE = S.ownE;
    A.s1 = S.sr1; A.s2 = S.sr2; A.sched1 = S.sched1.p; A.sched2 = S.sched2.p; A.nSched1 = S.nSched1; A.nSched2 = S.nSched2;
    return A;
}
OpArgs Solver::make_op_args() const { return make_op(*this); }

// pass 1 of an operator apply including the reduced term: w = [dt Mc^-1 K x ; c_f . B^-1 J x]
void Solver::pass1Apply(const OpArgs& A, const double* xin, const PcgScalars* S, const VecLink& V, bool withShared) {
    k_pass1(st, A, xin, w.p, g.dt, S, V);       // V: wait for the neighbours' entries of x at the head (direct halo stores)
    if (RG.count > 0) reduced_apply(st, g, RG, w.p + C.nActiveVs, 1.0, S);          // moments -> B^-1 -> expand, one CTA per region
    if (withShared) sharedApply(w.p + C.nActiveVs, nullptr, 0.0, 1.0, 1.0, nullptr, S);
}

// Shared regions: every rank forms the 3 x 10 moments of its own rows of them, the packed table [nShared][30] is summed over the
// ranks, then every rank solves the regions it takes part in and expands s_r onto its own rows.  The sum travels
//   * with the peer transport: straight into every rank's moment area of the symmetric blocks, summed in rank order by the waiting
//     finish kernel (time-outs set peerError like every other peer wait) -- two launches, no collective;
//   * otherwise, and in a step with more shared regions than that area holds (PEER_SH_CAP): ONE all-reduce of the communicator
//     (NCCL, or the host callbacks of the emulation twin), which hands every rank the same sums.
// Either way every rank forms the same s_r.  One more synchronisation point per apply, in every step with nShared > 0 (the same on
// all ranks); none otherwise.
void Solver::sharedApply(double* wRows, const double* extra, double extraScale, double tScale, double scale, double* sOut, const PcgScalars* S) {
    if (RG.nShared <= 0) return;
    bool solved = false;
    if (tScale != 0.) {
        shared_moments(st, g, RG, wRows, S);
#ifndef PS_EMULATE
        if (peer.on && (size_t)RG.nShared <= peer.shCap) {
            SharedPeer sp;
            sp.nranks = peer.nranks; sp.rank = peer.rank; sp.seq = ++peer.seqSh; sp.stride = peer.shCap * 30;
            for (int r = 0; r < peer.nranks; ++r) { sp.flag[r] = peer.shFlag(r); sp.val[r] = peer.shVal(r); }
            shared_exchange_peer(st, RG, sp, extra, extraScale, tScale, sOut, S, scal.p);
            ++sharedPeerExchanges;
            solved = true;
        }
#endif
        if (!solved) {
            shared_pack(st, RG);
            if (part.multi() && comm) comm->allreduce_sum(RG.shMoments.p, 30 * RG.nShared, st);
            ++sharedCommExchanges;
        }
    }
    if (!solved) shared_finish(st, RG, extra, extraScale, tScale, sOut, S);
    if (scale != 0.) shared_expand(st, g, RG, wRows, scale, S);
}

// assembleSystemPressureStressFactored (S_AS:432-470):
//   b = -[G^T; D] Mc^-1 rhs_u - (1/dt) [JG^T; DJ^T] B^-1 rhs_r + [rhs_p; rhs_tau]  =  -K_ext^T w + rhs_pt
//   with  w_active = Mc^-1 rhs_u,  w_reduced(f) = (1/dt) c_f . (B^-1 rhs_r)
void Solver::assemble() {
    const OpArgs A = make_op(*this);
    w.zero(st, (size_t)C.nRowsExt);
    if (part.local) {       // only the own rows of Mc^-1 / rhs_u exist here; the neighbours' arrive with the halo of w
        for (int a = 0; a < 3; ++a) {
            const int64_t lo = C.faceOff[a] + part.slotCut[SL_FACE + a][part.rank], hi = C.faceOff[a] + part.slotCut[SL_FACE + a][part.rank + 1];
            k_scale_rows(st, hi - lo, mcInv.p + lo, rhsU.p + lo, w.p + lo);
        }
    } else k_scale_rows(st, C.nActiveVs, mcInv.p, rhsU.p, w.p);
    if (RG.count > 0) {
        reduced_finish(st, g, RG, RG.rhsR.p, 1.0, 0.0, nullptr);                     // s = B^-1 rhs_r
        reduced_expand(st, g, RG, w.p + C.nActiveVs, g.invDt, nullptr);
        sharedApply(w.p + C.nActiveVs, RG.rhsR.p, 1.0, 0.0, g.invDt, nullptr, nullptr);     // rhs_r is replicated: no reduction
    }
    exchange(haloW, w.p, nullptr);            // the neighbours' coupled reduced rows (active rows are replicated above)
    k_pass2(st, A, w.p, nullptr, b.p, 0.0, rhsPT.p, nullptr, PeerCtx(), nullptr, 0);
    checkPeer("assemble");
}

// y = A x (ApplyPressureStressMatrix::applyMatrixVectorProducts, Apply.h:102-179)
void Solver::applyOperator(const double* xin, double* y, double* dotPart) {
    const OpArgs A = make_op(*this);
    pass1Apply(A, xin, nullptr);
    exchange(haloW, w.p, nullptr);
    k_pass2(st, A, w.p, xin, y, 0.5, nullptr, dotPart, PeerCtx(), nullptr, 0);
}

void Solver::timedOperator(int which) {
    const OpArgs A = make_op(*this);
    if (which == 0) { applyOperator(b.p, Ap.p, nullptr); return; }
    if (which == 1) pass1Apply(A, b.p, nullptr);                       // includes the reduced term (fused region epilogue)
    else if (which == 3) k_pass1(st, A, b.p, w.p, g.dt, nullptr);            // the sweep alone (raw products on the coupled reduced rows)
    else if (which == 6 && RG.count > 0) { reduced_apply(st, g, RG, w.p + C.nActiveVs, 1.0, nullptr); sharedApply(w.p + C.nActiveVs, nullptr, 0.0, 1.0, 1.0, nullptr, nullptr); }
    else if (which == 5) k_cg_update(st, ownSys, x.p, r.p, p.p, Ap.p, dotPartial.p, scal.p, PeerCtx());   // rank-local (timing only)
    else k_pass2(st, A, w.p, b.p, Ap.p, 0.5, nullptr, dotPartial.p, PeerCtx(), scal.p, which == 4 ? 3 : 0, r.p);      // 4: with the three fused dot products of the CG loop
}

// the caller's cancel callback, polled between iteration batches; with several ranks the decision is summed over the ranks so
// that all of them leave the loop at the same poll (a rank cancelled alone would leave the others spinning on its flags)
bool Solver::pollCancel() {
    if (!P.cancel_cb && !(part.multi() && comm && anyCancelCb)) return false;
    const double mine = (P.cancel_cb && P.cancel_cb(P.cancel_ctx)) ? 1. : 0.;
    return hostAllreduceSum(mine) > 0.5;
}

// solveSPDwithMatrixVectorPCG (S.cpp:734-812) -> pcg_external_matrix_A (pcg.h:268-340): identity
// preconditioner (Preconditioner.cpp:271-274), zero start, stop test min(rr, rr/xx) < tol^2.
int Solver::solve() {
    PS_WHERE("solve");
    StageTimer T(st, &stageMs[PS_STAGE_SOLVE]);
    // units.h:76-94: matrixSetup 0 = PRESSURE_STRESS; solverType 0 = PCG_MATRIX_VECTOR_PRODUCTS, 1 = EIGEN
    if (P.matrixSetup != 0 || (P.solverType != 0 && P.solverType != 1)) { result = R_UNSUPPORTED_SOLVER; return result; }
    if (P.solverType == 1) return solveEigenCG();
    const OpArgs A = make_op(*this);
    const int64_t n = C.nSystemSize;
    const int maxIt = P.maxSolverIterations;
    const int every = P.checkEvery > 0 ? P.checkEvery : 25;
    usedBiCGStab = 0;
    PcgScalars h; memset(&h, 0, sizeof h);
    if (n == 0) { solveIterations = 0; solveError = 0; result = R_SUCCESS; return result; }
    k_cg_init(st, ownSys, b.p, x.p, r.p, p.p, dotPartial.p, scal.p, P.tolerance, maxIt, reduceCtx(-1, 1));
    allreduce(scal.p->red + 3, 3);
    k_cg_begin(st, scal.p, reduceCtx(1, -1));
    bool cancelled = false;
    const bool fused = fusedHalo && peer.on;
#ifndef PS_EMULATE
    auto myFlag = [&](int kind, int side) -> const unsigned long long* {
        const int pr = side == 0 ? part.rank - 1 : part.rank + 1;
        return (pr < 0 || pr >= part.nranks) ? nullptr : &peer.sync(part.rank)->vecFlag[kind][side];
    };
#else
    auto myFlag = [&](int, int) -> const unsigned long long* { return nullptr; };
#endif
    // PS_TRACE=<iteration>: CUDA-event timeline of that CG iteration on stderr (diagnostic; events cost a few us each)
    static const int traceIter = getenv("PS_TRACE") ? atoi(getenv("PS_TRACE")) : -1;
    std::vector<std::pair<const char*, double>> trace;
#ifndef PS_EMULATE
    std::vector<cudaEvent_t> tev; std::vector<const char*> tname;
    auto mark = [&](bool on, const char* what) { if (!on) return; cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev.push_back(e); tname.push_back(what); };
#else
    auto mark = [&](bool, const char*) {};
#endif
    for (int it = 0; it < maxIt;) {
        const int batch = std::min(every, maxIt - it);
        for (int k = 0; k < batch; ++k) {
            const bool tr = (it + k == traceIter);
            mark(tr, "start");
            // halos: with the peer transport the boundary entries are stored straight into the neighbours' vectors by a short push launch
            // and the consuming kernel waits at its head (VecLink); only the very first p of a solve goes by the exchange kernel
            VecLink l1, l2;
            if (fused) {
                if (it + k > 0) { l1.wait[0] = myFlag(0, 0); l1.wait[1] = myFlag(0, 1); l1.waitSeq = peer.seqVec[0]; }
                else exchange(haloX, p.p, scal.p);
            } else exchange(haloX, p.p, scal.p);
            mark(tr, "halo p");
            pass1Apply(A, p.p, scal.p, l1, false);              mark(tr, "pass1 + regions");          // w = [dt Mc^-1 K p ; c_f . B^-1 J p]
            if (RG.nShared > 0) { sharedApply(w.p + C.nActiveVs, nullptr, 0.0, 1.0, 1.0, nullptr, scal.p); mark(tr, "shared regions"); }
            if (fused) { l2 = pushDirect(haloW, 1, nullptr); l2.wait[0] = myFlag(1, 0); l2.wait[1] = myFlag(1, 1); l2.waitSeq = peer.seqVec[1]; }
            else exchange(haloW, w.p, scal.p);
            mark(tr, "halo w");
            k_pass2(st, A, w.p, p.p, Ap.p, 0.5, nullptr, dotPartial.p, reduceCtx(-1, 0), scal.p, 3, r.p, l2);   // + this rank's p.Ap, r.Ap, Ap.Ap to every rank
            allreduce(scal.p->red, 3);                          mark(tr, "pass2 (+allreduce)");
            const PeerCtx uc = reduceCtx(0, 1, 1);              // global p.Ap.. and the previous r.r, x.p, p.p in; new r.r, x.p, p.p out
            VecLink l3;
            if (fused) l3 = pushDirect(haloX, 0, &uc);          // the boundary entries of the p this update is about to form, on their way while it runs
            k_cg_update(st, ownSys, x.p, r.p, p.p, Ap.p, dotPartial.p, scal.p, uc, l3);
            allreduce(scal.p->red + 3, 3);                      mark(tr, "update x,r,p (+allreduce)");
        }
        it += batch;
        copy_d2h(&h, scal.p, sizeof h, st);
#ifndef PS_EMULATE
        if (!tev.empty()) {
            fprintf(stderr, "[ps trace rank %d] CG iteration %d:", part.rank, traceIter);
            for (size_t i = 1; i < tev.size(); ++i) { float ms = 0; cudaEventElapsedTime(&ms, tev[i - 1], tev[i]); fprintf(stderr, "  %s %.1f us", tname[i], ms * 1e3); }
            float tot = 0; cudaEventElapsedTime(&tot, tev.front(), tev.back()); fprintf(stderr, "  | total %.1f us\n", tot * 1e3);
            for (auto e : tev) cudaEventDestroy(e);
            tev.clear(); tname.clear();
        }
#endif
        if (h.done || h.peerError) break;
        if (pollCancel()) { cancelled = true; break; }
    }
    copy_d2h(&h, scal.p, sizeof h, st);
    checkPeer("the CG loop");
    if (cancelled) { result = R_FAILED; peer.needResync = peer.on; g_lastError = "cancelled"; return result; }
    // b == 0: the reference would divide 0/0 (pcg.h:313); we return x = 0 after 0 iterations instead (DESIGN.md 7)
    solveIterations = (h.done == 1) ? h.iter : maxIt;
    solveError = std::sqrt(h.rre);
    solveXmag = h.xmag;
    // "have minres as a backup" (S.cpp:784-799): CG used up its iterations -> restart from x = 0 with BiCGSTAB
    if (solveIterations == maxIt && !cgOnly) return solveBiCGStab();
    result = (solveIterations == maxIt) ? R_NOCONVERGE : R_SUCCESS;
    return result;
}

// useWarmStart (PS.C:465-467): constructGuessVectors (S.cpp:521-531) + the copy into guessVector (S_AS:413-419)
//   pressureGuess = -G^T u_old - JG^T v*  = (-K_ext^T w)_p,   stressGuess = -2 mu^-1 (-D u_old - DJ^T v*) = -2 mu^-1 (-K_ext^T w)_tau
//   with w_active = u_old, w_f = c_f . v*_r on the coupled reduced rows.  The live solver never reads it: one GPU forms it in the
//   setup, several ranks only where it is read (ps_export, the global views of ps_api.cu), as a collective call.  Every rank forms
//   its own rows; v*_r (bestFit) exists for every region whose rows the rank holds (built for [bldLo, regHi)), and neither the
//   solve nor the write-back changes u_old or v*, so the guess formed after a step is the one of its setup.
void Solver::constructGuessVectors() {
    haveGuess = false;
    const int64_t n = C.nSystemSize;
    guess.alloc((size_t)std::max<int64_t>(n, 1));
    guess.zero(st, (size_t)n);
    if (!P.useWarmStart || n == 0) return;
    PS_WHERE("constructGuessVectors");
    const OpArgs A = make_op(*this);
    w.zero(st, (size_t)C.nRowsExt);
    for (int i = 0; i < ownK.n; ++i) {      // the owned active rows
        const int64_t lo = ownK.lo[i], hi = std::min(ownK.lo[i] + ownK.count(i), C.nActiveVs);
        if (hi > lo) copy_d2d(w.p + lo, oldVs.p + lo, (size_t)(hi - lo) * sizeof(double), st);
    }
    if (RG.count > 0) {
        k_sigma_from_s(st, RG.count, RG.bestFit.p, RG.sigma.p);
        reduced_expand(st, g, RG, w.p + C.nActiveVs, 1.0, nullptr);
        if (RG.nShared > 0) shared_expand(st, g, RG, w.p + C.nActiveVs, 1.0, nullptr);
    }
    exchange(haloW, w.p, nullptr);
    k_pass2(st, A, w.p, nullptr, guess.p, 0.0, nullptr, nullptr, PeerCtx(), nullptr, 0);
    k_guess_finish(st, A, guess.p);
    checkPeer("constructGuessVectors");
    haveGuess = true;
}

// diag(A) from the factors (ps_pcg.cu, k_diag_A)
void Solver::computeDiagonal() {
    if (haveDiag) return;
    diagA.alloc((size_t)std::max<int64_t>(C.nSystemSize, 1));
    diagA.zero(st, (size_t)C.nSystemSize);
    k_diag_A(st, g, make_op(*this), RG, diagA.p);
    haveDiag = true;
}

// solveEigenCG (S.cpp:814-862): Eigen::ConjugateGradient<SparseMatrix, Lower|Upper>, DiagonalPreconditioner,
// solveWithGuess(b, guessVector); iterations / error / Success as Eigen reports them (ConjugateGradient.h:28-93, :217-222).
// The reference needs the explicit A for this solver; here A stays factored and only its diagonal is formed, so the
// path also runs at sizes where the explicit matrix (dense region blocks) could not be stored.
int Solver::solveEigenCG() {
    if (part.multi()) { result = R_UNSUPPORTED_SOLVER; g_lastError = "solverType EIGEN runs on one GPU (diag(A) needs the neighbour's region blocks)"; return result; }
    const OpArgs A = make_op(*this);
    const int64_t n = C.nSystemSize;
    const int maxIt = P.maxSolverIterations;
    const int every = P.checkEvery > 0 ? P.checkEvery : 25;
    usedBiCGStab = 0;
    if (n == 0) { solveIterations = 0; solveError = 0; result = R_SUCCESS; return result; }
    computeDiagonal();
    if (haveGuess) copy_d2d(x.p, guess.p, (size_t)n * sizeof(double), st); else x.zero(st, (size_t)n);
    applyOperator(x.p, Ap.p, nullptr);
    k_eig_init(st, ownSys, b.p, Ap.p, r.p, dotPartial.p, scal.p, P.tolerance, maxIt);
    k_eig_stage(st, scal.p, 0);
    k_eig_first_p(st, ownSys, diagA.p, r.p, p.p, dotPartial.p, scal.p);
    k_eig_stage(st, scal.p, 1);
    PcgScalars h; memset(&h, 0, sizeof h);
    bool cancelled = false;
    for (int it = 0; it < maxIt;) {
        const int batch = std::min(every, maxIt - it);
        for (int k = 0; k < batch; ++k) {
            pass1Apply(A, p.p, scal.p);
            k_pass2(st, A, w.p, p.p, Ap.p, 0.5, nullptr, dotPartial.p, PeerCtx(), scal.p, 1);          // tmp = A p, p.tmp -> red[0]
            k_eig_update_xr(st, ownSys, diagA.p, x.p, r.p, p.p, Ap.p, dotPartial.p, scal.p);
            k_eig_stage(st, scal.p, 2);
            k_eig_update_p(st, ownSys, diagA.p, p.p, r.p, scal.p);
        }
        it += batch;
        copy_d2h(&h, scal.p, sizeof h, st);
        if (h.done) break;
        if (pollCancel()) { cancelled = true; break; }
    }
    copy_d2h(&h, scal.p, sizeof h, st);
    if (cancelled) { result = R_FAILED; g_lastError = "cancelled"; return result; }
    if (h.done == 3) x.zero(st, (size_t)n);                 // rhs == 0: x.setZero() (ConjugateGradient.h:47-53)
    solveIterations = h.iter;
    solveError = h.rre;
    result = (solveError <= P.tolerance) ? R_SUCCESS : R_NOCONVERGE;      // m_info (ConjugateGradient.h:222), S.cpp:853-859
    return result;
}

// bicgstab_external_matrix_A (pcg.h:134-200) on the factored operator: three applies per iteration (v = A p, t = A s and
// the explicit residual b - A x of the stop test), identity preconditioner, the reference's stop rule
// min(|err|^2, |err| / |x|) < tol.  Scalars stay on the device; the host polls the flag like the CG loop does.
int Solver::solveBiCGStab() {
    const OpArgs A = make_op(*this);
    const size_t n = (size_t)C.nSystemSize;
    const int maxIt = P.maxSolverIterations;
    const int every = P.checkEvery > 0 ? P.checkEvery : 25;
    usedBiCGStab = 1;
    bRhat.alloc(n); bV.alloc(n); bS.alloc(n); bT.alloc(n);
    auto applyTo = [&](double* xin, double* y) {
        exchange(haloX, xin, scal.p);
        pass1Apply(A, xin, scal.p);
        exchange(haloW, w.p, scal.p);
        k_pass2(st, A, w.p, xin, y, 0.5, nullptr, nullptr, PeerCtx(), scal.p, 0);
    };
    auto reduce = [&](int count) { if (part.multi() && comm) comm->allreduce_sum(scal.p->bred, count, st); };
    k_bicg_init(st, ownSys, b.p, x.p, r.p, bRhat.p, p.p, bV.p, scal.p, P.tolerance, maxIt);
    PcgScalars h; memset(&h, 0, sizeof h);
    bool cancelled = false;
    for (int it = 0; it < maxIt;) {
        const int batch = std::min(every, maxIt - it);
        for (int k = 0; k < batch; ++k) {
            k_bicg_dot(st, ownSys, bRhat.p, r.p, nullptr, nullptr, dotPartial.p, scal.p); reduce(1);      // rho = rhat . r
            k_bicg_stage(st, scal.p, 0);
            k_bicg_update_p(st, ownSys, p.p, r.p, bV.p, scal.p);
            applyTo(p.p, bV.p);                                                                           // v = A p
            k_bicg_dot(st, ownSys, bRhat.p, bV.p, nullptr, nullptr, dotPartial.p, scal.p); reduce(1);     // rhat . v
            k_bicg_stage(st, scal.p, 1);
            k_bicg_update_hs(st, ownSys, x.p, bS.p, r.p, p.p, bV.p, scal.p);
            applyTo(bS.p, bT.p);                                                                          // t = A s
            k_bicg_dot(st, ownSys, bT.p, bS.p, bT.p, bT.p, dotPartial.p, scal.p); reduce(2);              // t . s, t . t
            k_bicg_stage(st, scal.p, 2);
            k_bicg_update_x(st, ownSys, x.p, bS.p, dotPartial.p, scal.p);                                 // + x . x
            applyTo(x.p, Ap.p);
            k_bicg_err(st, ownSys, b.p, Ap.p, dotPartial.p, scal.p); reduce(2);                           // |b - A x|^2
            k_bicg_stage(st, scal.p, 3);
            k_bicg_update_r(st, ownSys, r.p, bS.p, bT.p, scal.p);
        }
        it += batch;
        copy_d2h(&h, scal.p, sizeof h, st);
        if (h.done || h.peerError) break;
        if (pollCancel()) { cancelled = true; break; }
    }
    copy_d2h(&h, scal.p, sizeof h, st);
    checkPeer("the BiCGSTAB loop");
    if (cancelled) { result = R_FAILED; peer.needResync = peer.on; g_lastError = "cancelled"; return result; }
    solveIterations = (h.done == 1) ? h.iter : maxIt;
    solveError = h.rre;                          // pcg.h:188-190: no square root on this path
    result = (solveIterations == maxIt) ? R_NOCONVERGE : R_SUCCESS;
    return result;
}

// recoverVelocityFromPressureStress (S.cpp:492-510)
void Solver::recoverVelocityFromPressureStress() {
    PS_WHERE("recoverVelocity");
    const OpArgs A = make_op(*this);
    exchange(haloX, x.p, nullptr);
    k_pass1(st, A, x.p, w.p, g.dt, nullptr);                         // active rows: dt Mc^-1 (G p + D^T tau); coupled reduced rows: raw (K_red x)_f
    RowSet act;                                                      // the owned active face rows
    for (int a = 0; a < 3; ++a) act.add(C.faceOff[a] + part.slotCut[SL_FACE + a][part.rank], C.faceOff[a] + part.slotCut[SL_FACE + a][part.rank + 1]);
    k_recover_active(st, g, act, w.p, mcInv.p, rhsU.p, velSol.p);
    if (RG.regHi > RG.regLo) {
        reduced_moments(st, g, RG, w.p + C.nActiveVs, nullptr);
        reduced_finish(st, g, RG, RG.rhsR.p, g.invDt, -1.0, nullptr);                            // B^-1 (rhs_r/dt - J x)
        k_copy_reduced_solution(st, (int64_t)(RG.regHi - RG.regLo) * RDOF, RG.s.p + (size_t)RG.regLo * RDOF, velSol.p + C.nActiveVs + (size_t)RG.regLo * RDOF);
    }
    sharedApply(w.p + C.nActiveVs, RG.rhsR.p, g.invDt, -1.0, 0.0, velSol.p + C.nActiveVs, nullptr);   // after the copy: it overwrites the shared regions
    checkPeer("the velocity recovery");
}

// buildValidFaces (S_Cls:4-54) + applySolutionToVelocity (S.cpp:937-1028)
// the voxels of a slot this rank delivers to the caller: its slab (the caller's arrays are full-grid; every rank fills its part, so ranks
// of one process can share them), everything on one GPU
void Solver::outRange(int slot, int64_t& lo, int64_t& hi) const {
    if (part.multi()) z_range(g, slot, g.zLo, g.zHi, lo, hi); else { lo = 0; hi = g.n[slot]; }
}

void Solver::applySolutionToVelocity(const ps_fields_out& out) {
    PS_WHERE("applySolutionToVelocity");
    const bool dev = out.memory == PS_MEM_DEVICE;
    const bool writeVel = (result == R_SUCCESS || P.keepNonConvergedResults);
#ifndef PS_EMULATE
    cudaEvent_t evLast = nullptr, evDone = nullptr;
#endif
    for (int a = 0; a < 3; ++a) {
        const size_t nf = (size_t)g.n[SL_FACE + a];
        int64_t oLo, oHi, kLo, kHi;
        outRange(SL_FACE + a, oLo, oHi);
        // the kernel also visits the plane above the slab: z-faces there can belong to a region of this rank (merged below)
        if (part.multi()) z_range(g, SL_FACE + a, g.zLo, std::min(g.nz, g.zHi + (a == 2 ? 1 : 0)), kLo, kHi); else { kLo = 0; kHi = (int64_t)nf; }
        float* velDev = nullptr; float* validDev = nullptr;
        // velocity staging starts as the input velocity: invalid faces are left untouched (S.cpp:975-978)
        if (out.velocity[a] && writeVel) {
            if (dev) { velDev = out.velocity[a]; if (velDev != dVel[a].p) copy_d2d(velDev + kLo, dVel[a].p + kLo, (size_t)(kHi - kLo) * sizeof(float), st); }
            else { outStage[a].alloc(nf); velDev = outStage[a].p; copy_d2d(velDev + kLo, dVel[a].p + kLo, (size_t)(kHi - kLo) * sizeof(float), st); }
        }
        if (out.valid[a] && !(validSent && !dev)) {
            if (dev) validDev = out.valid[a]; else { outStage[3 + a].alloc(nf); validDev = outStage[3 + a].p; }
        }
        FaceOwner own = {(int32_t)part.slotCut[SL_FACE + a][part.rank], (int32_t)part.slotCut[SL_FACE + a][part.rank + 1], RG.regLo, RG.regHi};
        if (RG.nShared > 0) { own.shared = RG.shFlag.p; own.zLo = g.zLo; own.zHi = g.zHi; own.nz = g.nz; }
        k_writeback_velocity(st, g, F, C, RG, velSol.p, a, velDev, validDev != nullptr, validDev, own, kLo, kHi, oLo, oHi);
        if (a == 2 && part.multi() && comm && velDev) {
            // the z-face plane on a slab cut carries DOFs of both neighbours (active: upper rank, reduced: lower rank's regions)
            const size_t plane = (size_t)g.nx * g.ny;
            DBuf<float>& planes = scratch().planes;
            planes.alloc(2 * plane);
            const int peers[2] = {part.rank > 0 ? part.rank - 1 : -1, part.rank + 1 < part.nranks ? part.rank + 1 : -1};
            const int kz[2] = {g.zLo, g.zHi};
            const void* sb[2] = {velDev + plane * kz[0], velDev + plane * kz[1]};
            void* rb[2] = {planes.p, planes.p + plane};
            const size_t bytes[2] = {peers[0] >= 0 ? plane * sizeof(float) : 0, peers[1] >= 0 ? plane * sizeof(float) : 0};
            comm->sendrecv(2, peers, sb, bytes, rb, bytes, st);
            for (int i = 0; i < 2; ++i) if (peers[i] >= 0) k_merge_face_plane(st, g, F, a, kz[i], planes.p + plane * i, velDev, own);
        }
        if (!dev) {
#ifndef PS_EMULATE
            // this axis crosses PCIe on the output stream while the next axis' kernel runs
            cudaEvent_t e; PS_CUDA(cudaEventCreate(&e));
            PS_CUDA(cudaEventRecord(e, st)); PS_CUDA(cudaStreamWaitEvent(stOut, e, 0));
            if (a == 2) evLast = e; else PS_CUDA(cudaEventDestroy(e));
            if (velDev) copy_d2any(out.velocity[a] + oLo, velDev + oLo, (size_t)(oHi - oLo) * sizeof(float), false, stOut);
            if (validDev) copy_d2any(out.valid[a] + oLo, validDev + oLo, (size_t)(oHi - oLo) * sizeof(float), false, stOut);
#else
            if (velDev) copy_d2any(out.velocity[a] + oLo, velDev + oLo, (size_t)(oHi - oLo) * sizeof(float), false, st);
            if (validDev) copy_d2any(out.valid[a] + oLo, validDev + oLo, (size_t)(oHi - oLo) * sizeof(float), false, st);
#endif
        }
    }
    stream_sync(st);
#ifndef PS_EMULATE
    if (!dev) {
        PS_CUDA(cudaEventCreate(&evDone)); PS_CUDA(cudaEventRecord(evDone, stOut));
        PS_CUDA(cudaEventSynchronize(evDone));
        float ms = 0; cudaEventElapsedTime(&ms, evLast, evDone); stageMs[PS_STAGE_DOWNLOAD] += ms;   // PCIe tail not hidden under kernels
        cudaEventDestroy(evLast); cudaEventDestroy(evDone);
    }
#endif
    validSent = false;
}

void Solver::setup() {
    unitLoad.clear(); unitCounts.clear();
    PS_WHERE("setup: peerResync");
    peerResync();
    // every rank must take part in the cancel all-reduce if any rank has a callback: agree on that once per setup
    anyCancelCb = part.multi() && comm ? hostAllreduceSum(P.cancel_cb ? 1. : 0.) > 0.5 : false;
    PS_WHERE("setup: weights");
    buildIntegrationWeightsAlt();
    {
        StageTimer T(st, &stageMs[PS_STAGE_CLASSIFY]);
        PS_WHERE("setup: classify");
        classifyCells();
        if (P.doReducedRegions) constructReducedRegions();
        classifyFaces();
        classifyEdges();
    }
    RG.count = 0; RG.regLo = RG.regHi = 0; RG.cellChunkLo = RG.cellChunkHi = 0; RG.rowChunkLo = RG.rowChunkHi = 0; RG.bldLo = 0;
    RG.nShared = RG.nShChunks = RG.nShMine = 0; RG.shRowLo = RG.shRowHi = 0;
    sharedPeerExchanges = sharedCommExchanges = 0;
    part.regionCut.assign((size_t)part.nranks + 1, 0);
    {
        StageTimer T(st, &stageMs[PS_STAGE_REDUCED]);
        PS_WHERE("setup: reduced indices");
        if (P.doReducedRegions) { constructCenterReducedIndices(); constructFacesReducedIndices(); constructEdgesReducedIndices(); }
    }
    PS_WHERE("setup: active indices");
    { StageTimer T(st, &stageMs[PS_STAGE_INDICES]); constructActiveIndices(); }
    PS_WHERE("setup: waitLateInputs");
    waitLateInputs();
    PS_WHERE("setup: region matrices");
    { StageTimer T(st, &stageMs[PS_STAGE_REGION_MATRICES]); if (P.doReducedRegions) computeReducedRegionMatrices(); }
    PS_WHERE("setup: matrix blocks");
    { StageTimer T(st, &stageMs[PS_STAGE_MATRIX_BLOCKS]); constructMatrixBlocks(); computeUnitLoads(); }
    PS_WHERE("setup: assemble");
    haveDiag = false; haveA = false;
    {
        StageTimer T(st, &stageMs[PS_STAGE_ASSEMBLE]);
        if (part.multi()) haveGuess = false;      // formed on demand (collective), a plain step pays nothing for it
        else constructGuessVectors();
        assemble();
    }
    haveSetup = true;
    result = R_INCOMPLETE;
}

// The work table of the setup (Solver::unitLoad): the active counts of the own units from the scans, the coupled reduced rows and the
// regions this rank owns counted by one kernel, all of it summed over the ranks by one all-gather (integers far below 2^53).
void Solver::computeUnitLoads() {
    PS_WHERE("setup: unit loads");
    const int unit = cutUnit(), nU = (int)unitActive[0].size();
    std::vector<double> mine((size_t)nU * UC_N, 0.);
    for (int s = 0; s < N_SLOTS; ++s) for (int u = 0; u < nU; ++u) mine[(size_t)u * UC_N + s] = (double)unitActive[s][u];
    const int64_t rLo = part.redRowCut[part.rank], rHi = part.redRowCut[part.rank + 1];
    if (RG.count > 0 && (rHi > rLo || RG.regHi > RG.regLo)) {
        DBuf<int>& cnt = scratch().rc;
        cnt.alloc((size_t)2 * nU); cnt.zero(st, (size_t)2 * nU);
        k_unit_counts(st, g, unit, nU, RG.rowXYZ.p, rLo, rHi, RG.cellList.p, RG.cellStart.p, RG.regLo, RG.regHi, cnt.p);
        const std::vector<int> h = cnt.to_host(st, (size_t)2 * nU);
        for (int u = 0; u < nU; ++u) { mine[(size_t)u * UC_N + UC_ROWS] = h[2 * u]; mine[(size_t)u * UC_N + UC_REGIONS] = h[2 * u + 1]; }
    }
    const std::vector<double> all = hostAllgather(mine);
    unitCounts.assign(mine.size(), 0);
    for (int k = 0; k < part.nranks; ++k) for (size_t i = 0; i < mine.size(); ++i) unitCounts[i] += std::llround(all[(size_t)k * mine.size() + i]);
    unitLoad.assign((size_t)nU, 0.);
    for (int u = 0; u < nU; ++u) {
        const int64_t* t = unitCounts.data() + (size_t)u * UC_N;
        OpCounts c;
        c.nCenter = t[SL_CENTER]; c.nActiveVs = t[SL_FACE] + t[SL_FACE + 1] + t[SL_FACE + 2]; c.nEdges = t[SL_EDGE] + t[SL_EDGE + 1] + t[SL_EDGE + 2];
        c.nRedRows = t[UC_ROWS]; c.nRegions = t[UC_REGIONS];
        unitLoad[u] = OpBytes(c).cgIteration;
    }
    loadUnit = unit;
}

// ps_set_partition: the cuts must be legal and the same on every rank; one all-gather of every rank's verdict and cuts decides for all
int Solver::setPartition(const int32_t* zCut) {
    const int N = part.nranks;
    std::vector<int> want;
    if (zCut) want.assign(zCut, zCut + N + 1);
    const bool ok = !zCut || valid_cuts(want, N, g.nz, cutUnit());
    std::vector<double> mine((size_t)N + 3, 0.);
    mine[0] = ok ? 1. : 0.; mine[1] = zCut ? 1. : 0.;
    for (int k = 0; zCut && k <= N; ++k) mine[2 + k] = want[k];
    const std::vector<double> all = hostAllgather(mine);
    bool agree = true;
    for (int r = 0; r < N; ++r) {
        if (all[(size_t)r * mine.size()] != 1.) agree = false;
        for (size_t i = 1; i < mine.size(); ++i) if (all[(size_t)r * mine.size() + i] != all[i]) agree = false;
    }
    if (!agree) {
        g_lastError = "ps_set_partition: the cuts must run 0 = zCut[0] < ... < zCut[nranks] = nz with interior cuts at multiples of " +
                      std::to_string(cutUnit()) + " layers, the same on every rank";
        return PS_INVALID;
    }
    userCut = want;
    if (comm) {
        const std::vector<int> old = part.zCut;
        computePartition(part.rank, N);
        if (part.zCut != old) haveSetup = false;
    }
    return PS_SUCCESS;
}

// ps_rebalance: the same deterministic choice on every rank (the unit loads are replicated), no communication
int Solver::rebalance(int32_t* zCut) {
    int rc = PS_NOCHANGE;
    if (unitLoad.empty() || loadUnit != cutUnit()) { g_lastError = "ps_rebalance: no unit loads of this tiling yet (call ps_setup or ps_step first)"; rc = PS_INVALID; }
    else if (part.multi() && comm) {
        const int N = part.nranks;
        std::vector<int> cur((size_t)N + 1);
        for (int k = 0; k <= N; ++k) cur[k] = (part.zCut[k] + loadUnit - 1) / loadUnit;
        const std::vector<int> best = balanced_cuts(unitLoad, N);
        if (max_slab_load(unitLoad, best) < max_slab_load(unitLoad, cur)) {
            userCut.assign((size_t)N + 1, g.nz);
            for (int k = 0; k < N; ++k) userCut[k] = best[k] * loadUnit;
            computePartition(part.rank, N);
            haveSetup = false;
            rc = PS_SUCCESS;
        }
    }
    if (zCut) std::copy(part.zCut.begin(), part.zCut.end(), zCut);
    return rc;
}

// inputs + setup; a slab-local attempt that meets work for the boundary fix-up is repeated with the setup replicated (collective: the
// decision comes from an all-reduce, every rank throws and restarts at the same point)
void Solver::setInputsAndSetup(const ps_fields_in& in) {
    try { setInputs(in); setup(); }
    catch (const NeedReplicatedSetup&) {
        stream_sync(stIn); stream_sync(st);
        lateInputsPending = false;
        replicatedSetup = true;
        computePartition(part.rank, part.nranks);
        setInputs(in);
        setup();
    }
}

int Solver::step(const ps_fields_in& in, const ps_fields_out* out, ps_stats* stats) {
    for (double& m : stageMs) m = 0;
    g_launches = 0;
    int res = R_INCOMPLETE;
    try {
        setInputsAndSetup(in);
        if (out) sendValidEarly(*out);
        if (P.doSolve) res = solve();
        else { x.alloc((size_t)std::max<int64_t>(C.nSystemSize, 1)); x.zero(st, (size_t)C.nSystemSize); result = R_INCOMPLETE; }     // solutionVector = 0 (S_AS:466), PS.C:513
        if (res == R_UNSUPPORTED_SOLVER) { stream_sync(stOut); validSent = false; if (stats) fillStats(stats); return res; }
        if (out) {
            {
                StageTimer T(st, &stageMs[PS_STAGE_WRITEBACK]);
                // PS.C:565-572: also without doSolve (the zero solution gives u = Mc^-1 rhs_u, v_r = B^-1 rhs_r / dt)
                if (res == R_SUCCESS || P.keepNonConvergedResults) recoverVelocityFromPressureStress();
                applySolutionToVelocity(*out);
            }
            stageMs[PS_STAGE_WRITEBACK] = std::max(0., stageMs[PS_STAGE_WRITEBACK] - stageMs[PS_STAGE_DOWNLOAD]);   // the PCIe tail is its own stage
        }
    } catch (...) {
        // no copy may still be reading / writing the caller's host buffers once the error is reported
        stream_sync(stIn); stream_sync(stOut);
        lateInputsPending = false; validSent = false;
        throw;
    }
    if (stats) fillStats(stats);
    return res;
}

// exportStats (S.cpp:574-606)
void Solver::fillStats(ps_stats* s) const {
    memset(s, 0, sizeof *s);
    const double d[27] = {(double)C.nCenter, (double)C.nFace[0], (double)C.nFace[1], (double)C.nFace[2],
                          (double)C.nEdge[0], (double)C.nEdge[1], (double)C.nEdge[2], (double)C.nActiveVs,
                          (double)C.nFace[0], (double)C.nFace[1], (double)C.nFace[2], (double)C.nReducedVs,
                          (double)C.nPressures, (double)C.nStresses, (double)C.nCenter, (double)C.nCenter, (double)C.nCenter,
                          (double)C.nEdge[0], (double)C.nEdge[1], (double)C.nEdge[2], (double)C.nTotalDOFs, (double)C.nSystemSize,
                          (double)smCount /* "thread count": SMs */, 0.0, (double)RG.count, g.dx, g.dt};
    for (int i = 0; i < 27; ++i) s->dimData[i] = d[i];
    double setupMs = 0;
    for (int i = PS_STAGE_WEIGHTS; i <= PS_STAGE_ASSEMBLE; ++i) setupMs += stageMs[i];
    s->solveData[0] = solveError; s->solveData[1] = solveIterations;
    s->solveData[2] = stageMs[PS_STAGE_SOLVE]; s->solveData[3] = stageMs[PS_STAGE_SOLVE];
    s->solveData[4] = setupMs; s->solveData[5] = setupMs;
    s->result = result; s->usedBiCGStab = usedBiCGStab;
    for (int i = 0; i < PS_NUM_STAGES; ++i) s->stage_ms[i] = stageMs[i];
    s->gpu_launches = g_launches;
}

}  // namespace ps
