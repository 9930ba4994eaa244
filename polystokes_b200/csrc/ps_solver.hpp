// ps_solver.hpp -- host-side Solver mirroring HDK_PolyStokes::Solver (exec/HDK_PolyStokesSolver.h:27-887):
// same stage names, same call order (exec/HDK_PolyStokes.C:344-584); every stage is one or a few CUDA
// kernels on the solver's stream, all state is device resident.
#pragma once
#include "ps_grid.hpp"
#include "ps_part.hpp"
#include "ps_comm.hpp"
#include "ps_peer.hpp"
#include "../../include/polystokes_b200.h"

namespace ps {

// Compact slot-major storage of K_ext = [G D^T] (face rows) and of its transpose (DOF rows).  Every entry of G / D^T is
// +-(faceFluidW * liquidW) / dx with both weights in eighths (S_CMB:408-411, 480-483, 568-571), i.e. an integer
// code in [-64, 64] times the constant 1/(64 dx): the value is rebuilt in the kernel as (double)code * (invDx / 64),
// which is the SAME double the reference forms (a power-of-two scaling commutes with the one rounding).  Columns:
//   face row   : pressure of cell(-), cell(+) [bits 30-31 of slot 0 = face axis], then the 4 edge stresses; the two
//                centre-stress columns are the pressure columns + nP + axis * nC and are not stored
//   cell row   : the 6 face rows (-x +x -y +y -z +z) serve the pressure row AND the xx / yy / zz stress rows of the cell
//                (same columns, opposite sign) -- one thread computes all four
//   edge row   : 4 face rows
// 33 B per face row, 32 B per cell, 20 B per edge instead of 96 / 144 / 48 B of fp64 + int32 ELL.  A slot with
// code 0 is empty: its column is never dereferenced.
struct CompactOp {
    int64_t nRows = 0, nCells = 0, nEdges = 0;
    DBuf<uint64_t> kcode;   // [nRows]   8 int8 codes: p-, p+, c-, c+, e0..e3
    DBuf<int32_t> kcol;     // [6][nRows]
    DBuf<uint8_t> kmc;      // [nActiveVs] faceFluidW * faceLiquidW (0..64): index of the M_c^-1 table
    DBuf<double> mcInvLut;  // [65] 1 / (rho * clamp(k / 64, 0.01, 1))
    DBuf<uint64_t> ccode;   // [nCells]  6 int8 codes of the pressure row
    DBuf<int32_t> ccol;     // [6][nCells]
    DBuf<uint32_t> ecode;   // [nEdges]  4 int8 codes
    DBuf<int32_t> ecol;     // [4][nEdges]
    void alloc(int64_t rows, int64_t nAct, int64_t cells, int64_t edges) {
        nRows = rows; nCells = cells; nEdges = edges;
        kcode.alloc((size_t)rows + 1); kcol.alloc((size_t)6 * rows + 1); kmc.alloc((size_t)nAct + 1); mcInvLut.alloc(65);
        ccode.alloc((size_t)cells + 1); ccol.alloc((size_t)6 * cells + 1); ecode.alloc((size_t)edges + 1); ecol.alloc((size_t)4 * edges + 1);
    }
};
PS_HD int op_code(uint64_t word, int k) { return (int)(int8_t)(uint8_t)(word >> (8 * k)); }
constexpr int32_t OP_COL_MASK = 0x3fffffff;

// Block schedule of a hot sweep.  The rows of K_ext come in four index ranges (x / y / z faces, coupled reduced rows),
// those of K_ext^T in four as well (cells, yz / xz / xy edges); each range is numbered in the reference's tile order, so
// equal FRACTIONS of two ranges cover the same part of the grid.  Sweeping range after range streams the gathered
// vector (132 MB at 256^3, more than the L2 holds) once per range; instead the 256-row blocks of all ranges are merged
// by fractional position, so that the blocks in flight at any moment gather from the same few MB of the vector.
//   entry = range << 28 | block index inside the range
constexpr int SCHED_BLOCK = 256;
struct SchedRanges {
    int n = 0;
    int64_t lo[4] = {0, 0, 0, 0}, hi[4] = {0, 0, 0, 0};
    int64_t items[4] = {-1, -1, -1, -1};     // >= 0: the range is a list of that many work items (lo = first item), not 256-row blocks
    void add(int64_t a, int64_t b) { lo[n] = a; hi[n] = b > a ? b : a; ++n; }
    void addItems(int64_t first, int64_t count) { lo[n] = first; hi[n] = first + (count > 0 ? count : 0); items[n] = count > 0 ? count : 0; ++n; }
    int64_t blocks(int k) const { return items[k] >= 0 ? items[k] : (hi[k] - lo[k] + SCHED_BLOCK - 1) / SCHED_BLOCK; }
};
std::vector<int32_t> merge_schedule(const SchedRanges& R);

struct RegionData {
    int32_t count = 0;
    DBuf<double> com;        // [R][3]
    DBuf<double> Mr, Visc, N, Binv;   // [R][26*26]
    DBuf<double> lsqRhs, bestFit, rhsR;  // [R][26]
    DBuf<double> moments;    // [R][400] polynomial moments the region matrices are expanded from (ps_reduced.cu)
    DBuf<double> tables;     // constant 26x10 / 26x4 images of the basis (generated once)
    DBuf<int32_t> cellList;  // REDUCED cells sorted by (region, tile order)
    DBuf<int32_t> cellStart; // [R+1]
    // coupled reduced face rows of K_ext, sorted by (region, axis, tile order)
    int64_t nRows = 0;
    DBuf<int32_t> rowFace;   // packed dense face index | axis << 29
    DBuf<uint32_t> rowXYZ;   // the same rows as x | y<<10 | z<<20 | axis<<30 (cheap decode in the hot kernels)
    DBuf<double> sigma;      // [R][3][10] polynomial coefficients of w_f per face axis
    DBuf<int32_t> rowRegion; // region of each row
    DBuf<int32_t> rowStart;  // [R+1] row range of each region (relative to nActiveVs)
    // chunk tables (fixed-size pieces of the sorted lists, each inside one region)
    int32_t nCellChunks = 0, nRowChunks = 0;
    DBuf<int32_t> cellChunk;   // [nChunks][3] = region, begin, end
    DBuf<int32_t> rowChunk;    // [nChunks][4] = region, begin, end, face axis (a chunk never mixes axes)
    DBuf<int32_t> cellChunkStart, rowChunkStart;  // [R+1] first chunk of each region
    DBuf<int32_t> rowAxisStart;  // [3R+1] first coupled reduced row of (region, face axis): the row ranges of reduced_region_kernel
    int32_t maxRegionRows = 0;   // largest number of coupled reduced rows of one region (decides fused vs chunked reduced kernels)
    int32_t maxRegionAxisRows = 0;                    // largest row count of one (region, face axis) built here (read-only count)
    int32_t maxRegionCells = 0, minRegionCells = 0;   // REDUCED cells of the largest / smallest owned region (read-only counts)
    DBuf<int32_t> regionOrder;   // [R] launch order of reduced_region_kernel: the owned regions by decreasing row count (longest CTA first)
    DBuf<double> partial;    // per-chunk partial sums
    DBuf<double> t, s;       // [R][26] per-apply moment / B^-1 t
    DBuf<unsigned int> regionTicket;   // [R] chunks of the region that have delivered their moments (self-resetting)
    int32_t ownRowLo = 0, ownRowHi = 0;   // coupled reduced rows of the owned regions
    // owned pieces of this rank (everything on one GPU): regions [regLo, regHi) and their chunk ranges
    int32_t regLo = 0, regHi = 0, cellChunkLo = 0, cellChunkHi = 0, rowChunkLo = 0, rowChunkHi = 0;
    int32_t bldLo = 0;       // region matrices are built for [bldLo, regHi): the owned regions, the shared ones this rank takes part in, and
                             // (one contiguous range) every region of lower ranks numbered between them
    // Shared regions (ps_part.hpp, Partition::spanning): reduced faces in more than one slab.  Their coupled rows follow the slab of
    // the face and sit after the rank's other coupled rows, [shRowLo, shRowHi); every apply sums their 3 x 10 moments over the ranks.
    int32_t nShared = 0;                 // global count (the same on every rank)
    int32_t nShChunks = 0, shRowLo = 0, shRowHi = 0, nShMine = 0;
    DBuf<int32_t> shRegion;              // [nShared] region id of every shared slot, ascending
    DBuf<int32_t> shChunk;               // [nShChunks][4] = region, begin, end, axis: this rank's rows of the shared regions
    DBuf<int32_t> shChunkStart;          // [nShared+1] first chunk of every slot
    DBuf<int32_t> shMine;                // [nShMine] slots this rank solves: it holds rows or reduced faces of the region, or owns it
    DBuf<uint8_t> shFlag;                // [R] 1 for a shared region (velocity write-back: faces are written by the slab that holds them)
    DBuf<double> shPartial, shMoments;   // per-chunk moments; [nShared][30] moments summed over the ranks
};

// halo of one distributed vector: entries this rank must send to / receive from its z-neighbours
// (global indices, ascending; the two peers' lists are concatenated [below | above])
struct Halo {
    int peers[2] = {-1, -1};
    int64_t nSend[2] = {0, 0}, nRecv[2] = {0, 0};
    DBuf<int32_t> sendIdx, recvIdx;
    DBuf<double> sendBuf, recvBuf;
    void reset() { for (int i = 0; i < 2; ++i) { peers[i] = -1; nSend[i] = nRecv[i] = 0; } }
    int64_t sendTotal() const { return nSend[0] + nSend[1]; }
    int64_t recvTotal() const { return nRecv[0] + nRecv[1]; }
};

struct Counts {
    int64_t nCenter = 0, nFace[3] = {0, 0, 0}, nEdge[3] = {0, 0, 0};
    int64_t nActiveVs = 0, nReducedVs = 0, nPressures = 0, nStresses = 0, nTotalDOFs = 0, nSystemSize = 0;
    int64_t faceOff[3] = {0, 0, 0};     // faceVelocityDOF offsets (S.h:628-642)
    int64_t stressOff[6] = {0, 0, 0, 0, 0, 0};   // XX,YY,ZZ,YZ,XZ,XY offsets inside the stress block (S.h:586-606)
    int64_t nRowsExt = 0;               // nActiveVs + coupled reduced rows
};

struct PcgScalars {   // device-resident CG state: no host round trip inside an iteration
    double rsold, pAp, alpha, beta, rsnew, xmag, rre;
    int iter, done, maxIter, pad;
    double tol2;
    unsigned int ticket[8];   // last-CTA-done tickets: 0 pass 2, 2 init, 3 x/r/p update, 4/5 halo push of p / w, 6 BiCGSTAB / Eigen sweeps
    int peerError, pad2;      // a peer-memory wait timed out (ps_peer.hpp); cleared when the host has reported it
    // rank-local sums handed to the all-reduces: [0..2] p.Ap, r.Ap, Ap.Ap (pass 2), [3..5] r.r, x.p, p.p (x/r/p update, or b.b, 0, b.b from init), [6] b.b
    double red[7];
    double xx;                // global x.x of the current iterate, advanced by |x + alpha p|^2 = x.x + 2 alpha x.p + alpha^2 p.p (ps_pcg.cu)
    // BiCGSTAB fallback (pcg.h:134-200): its own scalars; bred[] = rank-local dot products of the current stage
    double rhoCurr, rhoOld, omega, tol, bred[2];
    // solverType EIGEN (Eigen::ConjugateGradient, ConjugateGradient.h:28-93): |b|^2, max(tol^2 |b|^2, DBL_MIN), r.z
    double eigRhsNorm2, eigThreshold, eigAbsNew;
};

// explicit A of assembleSystemPressureStress (S_AS:351-430) as device CSR: export / parity only (ps_explicit.cu)
struct ExplicitA {
    int64_t n = 0, nnz = 0;
    DBuf<int64_t> ptr;      // [n+1]
    DBuf<int32_t> idx;      // sorted per row, explicit zeros kept
    DBuf<double> val;
};
struct OpArgs;
class Solver {
public:
    explicit Solver(const ps_params& p);
    ~Solver();
    ps_params P;
    Geom g;
    cudaStream_t st = nullptr;
    // host-memory callers (ps_fields_in/out::memory == PS_MEM_HOST): the PCIe copies run on their own streams underneath
    // the compute stream -- late inputs (viscosity, velocity, collision velocity: first read by the region matrices)
    // under weights + classification + numbering, the `valid` field (final once the faces are classified) under the CG
    // loop, each velocity axis under the write-back kernel of the next one
    cudaStream_t stIn = nullptr, stOut = nullptr;
    bool lateInputsPending = false, validSent = false;
    DBuf<float> outStage[6];            // device staging of velocity[3] / valid[3] for host outputs
    void waitLateInputs();
    void sendValidEarly(const ps_fields_out& out);
    Counts C;
    int result = R_INCOMPLETE;
    int solveIterations = -1;
    double solveError = -1;
    double solveXmag = 0;      // x.x as the CG stop test saw it at the last iteration (advanced by the recurrence of ps_pcg.cu)
    int usedBiCGStab = 0;
    bool cgOnly = false;                // ps_time_kernel("cg_iteration"): run exactly maxSolverIterations CG iterations, no fallback
    int fixLoops = 0;
    int smCount = 148;                  // SMs of the handle's device (the "thread count" of the exported statistics)
    double stageMs[PS_NUM_STAGES] = {0};

    // ---- the reference's per-step sequence (exec/HDK_PolyStokes.C:344-584) ----
    void setInputs(const ps_fields_in& in);
    void buildIntegrationWeightsAlt();
    void classifyCells();
    void constructReducedRegions();
    void classifyFaces();
    void classifyEdges();
    void constructCenterReducedIndices();
    void constructFacesReducedIndices();
    void constructEdgesReducedIndices();
    void constructActiveIndices();      // constructCenter/Faces/EdgesActiveIndices
    void computeReducedRegionMatrices();// computeCenterOfMasses, LeastSquaresFits, ReducedMassMatrices, ViscosityMatricesInteriorOnly
    void constructMatrixBlocks();
    void assemble();                    // assembleSystemPressureStressFactored
    int solve();                        // solveSPDwithMatrixVectorPCG
    int solveBiCGStab();                // its fallback when CG hits maxSolverIterations (S.cpp:784-799 -> pcg.h:134-200)
    int solveEigenCG();                 // solverType EIGEN (S.cpp:814-862): Jacobi-preconditioned Eigen CG from guessVector, on the factored operator
    void constructGuessVectors();       // useWarmStart (PS.C:465-467 -> S.cpp:521-531, S_AS:413-419)
    void computeDiagonal();             // diag(A) for Eigen's DiagonalPreconditioner (BasicPreconditioners.h:66-94), matrix free
    void buildValidFaces(const ps_fields_out& out);
    void recoverVelocityFromPressureStress();
    void applySolutionToVelocity(const ps_fields_out& out);
    void outRange(int slot, int64_t& lo, int64_t& hi) const;

    void setup();                       // weights .. assemble
    int step(const ps_fields_in& in, const ps_fields_out* out, ps_stats* stats);
    void fillStats(ps_stats* s) const;

    // ---- multi-GPU (one process per GPU; ps_part.hpp) ----
    Partition part;
    DBuf<int32_t> zCutDev;              // part.zCut on the device (Partition::spanning: slab of a face)
    Comm* comm = nullptr;
    void initComm(Comm* c);             // takes ownership; computes the z cuts
    void computePartition(int rank, int nranks);
    // Slab-local setup assumes that the boundary fix-up (S_Cls:1073-1172, a serial sweep) has nothing to do.  A step that finds a
    // candidate cell -- all ranks learn it from one all-reduce -- is restarted with the setup replicated (the round-1 form); the
    // handle stays there until the tiling / layer parameters change.
    struct NeedReplicatedSetup {};
    bool replicatedSetup = false;
    void setInputsAndSetup(const ps_fields_in& in);
    void setParams(const ps_params& p);
    void computeOwnership();            // owned row / DOF ranges of every rank from the (replicated or all-gathered) numbering
    // slab-local setup (Partition::local)
    struct LayerField { void* base; int slot; int elem; };
    void exchangeLayers(const std::vector<LayerField>& fields);      // halo layers of grid fields <- the neighbours' own layers
    void mergeSharedPlanes(int32_t* zFaceField);                     // z-face planes on the cuts: max of the two ranks' values
    std::vector<double> hostAllgather(const std::vector<double>& mine);   // [nranks][mine.size()], collective host sync
    void ownTileZ(int slot, int tz[2], int extraTop = 0) const;      // tile layers of the own slab for tile_order_scan
    std::vector<int64_t> cutsFromCounts(const std::vector<double>& all, int stride, int item) const;
    DBuf<uint8_t> xchgTmp;
    void buildHalos();                  // send / receive index lists of p (system vector) and w (K_ext rows)
    // direct halo stores (VecLink, ps_peer.hpp): p and w live in one arena that the z-neighbours map; masks of the entries they read
    DBuf<double> vecArena;
    VecLink pushDirect(Halo& H, int kind, const PeerCtx* updateCtx);   // my boundary entries of w (kind 1) / of the NEW p (kind 0) -> the neighbours' vectors; returns what the next launch must announce
    void allocVectors(size_t n, size_t nRows);      // p and w (in the arena when the peer transport is on)
    void exchangeVectorPointers();                  // collective: publish / map the arenas when any rank's moved
    void closeVectorMaps();
    bool fusedHalo = false;                         // agreed by all ranks in exchangeVectorPointers
    void* arenaGraveyard = nullptr;                 // the previous arena, alive until the neighbours have let go of it
    void exchange(Halo& H, double* v, const PcgScalars* S);
    void allreduce(double* devBuf, int n);   // host-enqueued NCCL all-reduce; a no-op when the peer transport fuses it into the kernels
    PeerLink peer;                      // NVLink peer-memory transport (ps_peer.hpp); off => NCCL for everything
    void setupPeer();                   // collective: allocate + exchange + map the symmetric blocks
    void closePeer();
    PeerCtx reduceCtx(int slotIn, int slotOut, int slotIn2 = -1);   // sequence numbers of the reductions one kernel consumes / produces
    void checkPeer(const char* where);  // throws (and schedules a resync) if a peer-memory wait timed out since the last check
    void peerResync();                  // collective, start of setup
    double hostAllreduceSum(double v);
    bool pollCancel();
    bool anyCancelCb = false;
    DBuf<double> hostRed;
    RowSet rowsK(int rank) const, rowsP(int rank) const, rowsC(int rank) const, rowsE(int rank) const;
    RangeSet rowsSys(int rank) const;
    RowSet ownK, ownP, ownC, ownE;
    RangeSet ownSys;
    Halo haloX, haloW;

    // operator y = A x on device vectors (Apply.h:102-179)
    void applyOperator(const double* x, double* y, double* pApPartial);
    void pass1Apply(const OpArgs& A, const double* x, const PcgScalars* S, bool reverse = false, const VecLink& V = VecLink(), bool withShared = true);   // pass 1 + the reduced term
    // the reduced term of the shared regions: s_r = B_r^-1 (extraScale extra_r + tScale t_r), t_r summed over the ranks (collective
    // when tScale != 0), then w_f = scale c_f . s_r on this rank's shared rows (scale 0: no expansion); sOut (region-indexed) receives s_r
    void sharedApply(double* wRows, const double* extra, double extraScale, double tScale, double scale, double* sOut, const PcgScalars* S);
    void classifySharedRegions();
    int64_t sharedPeerExchanges = 0, sharedCommExchanges = 0;      // moment sums of shared regions since the last setup, by transport      // Partition::spanning: region owners, shared list, build range (replicated classification, no communication)
    void timedOperator(int which);     // 0 = whole apply, 1 = pass 1 only, 2 = pass 2 only (on b -> Ap)

    // ---- device state ----
    Fields F;
    DBuf<float> dSurface, dCollision, dViscosity, dVel[3], dColVel[3];
    DBuf<uint8_t> dLiqW[N_SLOTS], dFluW[N_SLOTS];
    DBuf<int8_t> dLabel[N_SLOTS];
    DBuf<int32_t> dAidx[N_SLOTS], dRidx[N_SLOTS], dKrow[3];
    DBuf<uint8_t> scratch8[3];
    DBuf<int32_t> scratch32[4];
    DBuf<int32_t> tileCounts;
    DBuf<int> flags;             // small device flag / counter block
    RegionData RG;
    // matrices + vectors
    CompactOp Op;                 // K_ext and K_ext^T
    SchedRanges sr1, sr2;         // block schedules of pass 1 / pass 2 over the owned rows (merge_schedule)
    DBuf<int32_t> sched1, sched2, sched1a, sched1b;
    int nSched1 = 0, nSched2 = 0, nSched1a = 0, nSched1b = 0;
    void buildSchedules();
    DBuf<double> mcInv, mc, rhsU, oldVs, uInv, uDiag, rhsPT, b;
    DBuf<double> x, r, p, Ap, w, velSol;
    DBuf<double> bRhat, bV, bS, bT;     // BiCGSTAB work vectors, allocated when the fallback first fires
    DBuf<double> guess, diagA;          // guessVector (zero unless useWarmStart) and diag(A), built on demand
    bool haveGuess = false, haveDiag = false;
    ExplicitA Aexp;                     // built on demand by buildExplicitA (ps_get_csr("A"), Mat_A.mtx with solverType EIGEN)
    bool haveA = false;
    void buildExplicitA();
    OpArgs make_op_args() const;
    DBuf<double> dotPartial;
    DBuf<PcgScalars> scal;
    bool inputsOnDevice = false;
    bool haveSetup = false;
};

// ---- kernels (free functions; see the .cu files for the reference citations) ----
void k_build_weights(cudaStream_t, const Geom&, const Fields&, uint8_t* signX, uint8_t* signBox);
void k_classify_cells(cudaStream_t, const Geom&, const Fields&, bool genericToActive);
void k_air_layer_seed(cudaStream_t, const Geom&, const Fields&, uint8_t* stamp);
void k_layer_commit(cudaStream_t, const Geom&, const Fields&, const uint8_t* stamp, int layerStamp);
void k_air_layer_grow(cudaStream_t, const Geom&, const Fields&, uint8_t* stamp, int prevStamp);
void k_solid_layer_seed(cudaStream_t, const Geom&, const Fields&, uint8_t* stamp);
void k_solid_layer_grow(cudaStream_t, const Geom&, const Fields&, uint8_t* stamp, int prevStamp);
void k_tiles_and_reduce(cudaStream_t, const Geom&, const Fields&, bool doTile, int tileSize, int tilePadding);
void k_classify_faces(cudaStream_t, const Geom&, const Fields&);
void k_classify_edges(cudaStream_t, const Geom&, const Fields&);
void k_cc_init(cudaStream_t, const Geom&, const Fields&, int32_t* parent);
void k_cc_sweep(cudaStream_t, const Geom&, const Fields&, int32_t* parent, int* changed);
void k_cc_minkey(cudaStream_t, const Geom&, const int32_t* parent, int32_t* minKey);
void k_cc_first_flags(cudaStream_t, const Geom&, const int32_t* parent, const int32_t* minKey, uint8_t* flag);
void k_cc_publish(cudaStream_t, const Geom&, const int32_t* parent, const uint8_t* flag, const int32_t* firstRank, int32_t* rootId);
void k_cc_assign(cudaStream_t, const Geom&, const Fields&, const int32_t* parent, const int32_t* rootId);
void k_fix_candidates(cudaStream_t, const Geom&, const Fields&, uint8_t* cand, uint8_t* firedA, uint8_t* firedB, int* anyCand);
void k_fix_iterate(cudaStream_t, const Geom&, const Fields&, const uint8_t* cand, const uint8_t* firedIn, uint8_t* firedOut, int* changed);
void k_fix_apply(cudaStream_t, const Geom&, const Fields&, const uint8_t* fired, int* anyFired);
void k_region_bbox(cudaStream_t, const Geom&, const Fields&, int* bbMin, int* bbMax);
void k_region_remap(cudaStream_t, const Geom&, const Fields&, const int32_t* remap);
void k_faces_reduced(cudaStream_t, const Geom&, const Fields&);
void k_edges_reduced(cudaStream_t, const Geom&, const Fields&);
void k_generic_to_active_flags(cudaStream_t, const Geom&, int slot, int8_t* L, uint8_t* flag);
void k_valid_faces(cudaStream_t, const Geom&, const Fields&, float* const valid[3]);

// tile-order exclusive scan of a dense 0/1 flag field: out[q] = rank among flagged voxels in the
// reference's voxel iteration order, -1 where the flag is 0.  Returns the total (host sync).
// If `zCut` is given, cuts[k] receives the rank of the first flagged voxel with z >= zCut[k] (cuts multiple of 16).
// With `tileZ` only the tile layers [tileZ[0], tileZ[1]) are scanned (ranks start at 0 on the first of them; `out` is written there only).
int64_t tile_order_scan(cudaStream_t, const Geom&, int slot, const uint8_t* flag, int32_t* out, DBuf<int32_t>& tileCounts,
                        const std::vector<int>* zCut = nullptr, std::vector<int64_t>* cuts = nullptr, const int* tileZ = nullptr);
// out[k] = in[0] + ... + in[k-1] for k < n; returns the total (host sync)
int64_t exclusive_scan_i64(cudaStream_t, int64_t n, const int64_t* in, int64_t* out);
// stable sort of (key, value) pairs by key (keys < 2^keyBits)
void sort_pairs_by_key(cudaStream_t, int64_t n, int keyBits, DBuf<int32_t>& keys, DBuf<int32_t>& vals, DBuf<int32_t>& keysTmp, DBuf<int32_t>& valsTmp);

// ps_reduced.cu
void k_region_com(cudaStream_t, const Geom&, const Fields&, int32_t R, unsigned long long* sums, double* com);
void k_collect_region_keys(cudaStream_t, const Geom&, const int32_t* rank, const uint8_t* flag, const int32_t* region, int64_t lo, int64_t hi, int32_t tag, int32_t rankOffset, int32_t* keys, int32_t* vals);
void region_gram_partials(cudaStream_t, const Geom&, const Fields&, const RegionData&, double* partial);
void region_gram_finish(cudaStream_t, const Geom&, RegionData&, int nChunks);
void k_flag_coupled_faces(cudaStream_t, const Geom&, const Fields&, int axis, uint8_t* flag, int32_t regLo, int32_t regHi, int64_t lo, int64_t hi);

// ps_assemble.cu
void k_assemble_K(cudaStream_t, const Geom&, const Fields&, const Counts&, CompactOp& Op, double* mcInv, double* mc, double* rhsU, double* oldVs, const RowSet& ownRows);
void k_assemble_Kt(cudaStream_t, const Geom&, const Fields&, const Counts&, CompactOp& Op, double* uInv, double* uDiag, double* rhsPT, bool ownOnly);

// ps_pcg.cu
struct OpArgs {   // everything one operator apply touches
    int64_t nRowsExt, nActiveVs, nP, nT, nC, nE;
    SchedRanges s1, s2;           // pass 1: face rows x, y, z, coupled reduced rows; pass 2: cells, edges yz, xz, xy (edge numbering)
    const int32_t* sched1; const int32_t* sched2; int nSched1, nSched2;
    const int32_t* sched1a; const int32_t* sched1b; int nSched1a, nSched1b;   // pass 1 split: coupled reduced rows | active rows (same merged order)
    RowSet rowsK, rowsP, rowsE;   // rows this rank computes (all rows on one GPU); the centre-stress rows follow rowsP
    const uint64_t* kcode; const int32_t* kcol; const uint8_t* kmc; const double* mcInvLut;
    const uint64_t* ccode; const int32_t* ccol; const uint32_t* ecode; const int32_t* ecol;
    const double* uInv;
    double valScale;              // invDx / 64
};
void k_pass1(cudaStream_t, const OpArgs&, const double* x, double* w, double activeScale, const PcgScalars* scal, bool reverse = false, int part = 0, const VecLink& V = VecLink());
#ifndef PS_EMULATE
// pass 1 and the reduced term of one apply in two launches: coupled reduced rows, then active rows interleaved with the regions.
// false: not applicable (no tiled regions of this rank / PS_OVERLAP=0) -- nothing was launched, use k_pass1 + reduced_apply
bool k_pass1_regions(cudaStream_t, const OpArgs&, const double* x, double* w, double activeScale, const PcgScalars* scal, const Geom&, const RegionData&, double scale, const VecLink& V = VecLink());
#endif
// mode bit 0: dot(x, y) (p.Ap) -> red[0]; bit 1: also dot(r2, y), dot(y, y) (r.Ap, Ap.Ap) -> red[1], red[2]
void k_pass2(cudaStream_t, const OpArgs&, const double* w, const double* x, double* y, double muScale, const double* add, double* dotPartial, const PeerCtx& P, PcgScalars* scal, int mode,
             const double* r2 = nullptr, bool reverse = false, const VecLink& V = VecLink());
// moments of w_f per chunk; with `solve` the last chunk of every region also runs reduced_finish(nullptr, 0, 1) for it (one launch less)
void reduced_moments(cudaStream_t, const Geom&, const RegionData&, const double* wRows, const PcgScalars* scal, bool solve = false);
void reduced_finish(cudaStream_t, const Geom&, const RegionData&, const double* extraRhs, double extraScale, double tScale, const PcgScalars* scal);
void reduced_expand(cudaStream_t, const Geom&, const RegionData&, double* wRows, double scale, const PcgScalars* scal);
// the reduced term of one apply: w_f <- scale * c_f . B^-1 (sum_f c_f w_f); one fused launch for tiled regions, moments + expand otherwise
void reduced_apply(cudaStream_t, const Geom&, const RegionData&, double* wRows, double scale, const PcgScalars* scal);
int region_path(const OpArgs&, const RegionData&);      // the kernels reduced_apply / pass1Apply choose (ps_pcg.cu)
// shared regions (RegionData::nShared): moments of this rank's shared rows per chunk, their sum per slot in chunk order (shMoments,
// then summed over the ranks by the caller), the small solve of the slots this rank takes part in, the expansion onto its shared rows
void shared_moments(cudaStream_t, const Geom&, const RegionData&, const double* wRows, const PcgScalars* scal);
void shared_pack(cudaStream_t, const RegionData&);
void shared_finish(cudaStream_t, const RegionData&, const double* extra, double extraScale, double tScale, double* sOut, const PcgScalars* scal);
void shared_expand(cudaStream_t, const Geom&, const RegionData&, double* wRows, double scale, const PcgScalars* scal);
#ifndef PS_EMULATE
// peer transport: push this rank's packed moments into every rank's moment area, then wait, sum in rank order and solve (ps_pcg.cu)
void shared_exchange_peer(cudaStream_t, const RegionData&, const SharedPeer& P, const double* extra, double extraScale, double tScale, double* sOut,
                          const PcgScalars* scal, PcgScalars* err);
#endif
void k_cg_update(cudaStream_t, const RangeSet& own, double* x, double* r, double* p, const double* Ap, double* dotPartial, PcgScalars* scal, const PeerCtx& P, bool reverse = false, const VecLink& V = VecLink());
void k_cg_init(cudaStream_t, const RangeSet& own, const double* b, double* x, double* r, double* p, double* dotPartial, PcgScalars* scal, double tol, int maxIter, const PeerCtx& P);
void k_cg_begin(cudaStream_t, PcgScalars* scal, const PeerCtx& P);
// BiCGSTAB fallback (pcg.h:134-200).  Dot products land rank-local in scal->bred[], the host enqueues the all-reduce
// (NCCL) when there are several ranks, k_bicg_stage then advances the scalars exactly in the reference's order.
void k_bicg_init(cudaStream_t, const RangeSet& own, const double* b, double* x, double* r, double* rhat, double* p, double* v, PcgScalars* scal, double tol, int maxIter);
void k_bicg_dot(cudaStream_t, const RangeSet& own, const double* a0, const double* b0, const double* a1, const double* b1, double* dotPartial, PcgScalars* scal);
void k_bicg_stage(cudaStream_t, PcgScalars* scal, int stage);
void k_bicg_update_p(cudaStream_t, const RangeSet& own, double* p, const double* r, const double* v, const PcgScalars* scal);
void k_bicg_update_hs(cudaStream_t, const RangeSet& own, double* x, double* s, const double* r, const double* p, const double* v, const PcgScalars* scal);
void k_bicg_update_x(cudaStream_t, const RangeSet& own, double* x, const double* s, double* dotPartial, PcgScalars* scal);
void k_bicg_err(cudaStream_t, const RangeSet& own, const double* b, const double* Ax, double* dotPartial, PcgScalars* scal);
void k_bicg_update_r(cudaStream_t, const RangeSet& own, double* r, const double* s, const double* t, const PcgScalars* scal);
// solverType EIGEN (S.cpp:814-862): Eigen's CG loop with the Jacobi preconditioner, scalars on the device
void k_diag_A(cudaStream_t, const Geom&, const OpArgs&, const RegionData&, double* diag);
void k_sigma_from_s(cudaStream_t, int32_t R, const double* s, double* sigma);
void k_guess_finish(cudaStream_t, const OpArgs&, double* guess);
void k_eig_init(cudaStream_t, const RangeSet& own, const double* b, const double* Ax, double* r, double* dotPartial, PcgScalars* scal, double tol, int maxIter);
void k_eig_stage(cudaStream_t, PcgScalars* scal, int stage);
void k_eig_first_p(cudaStream_t, const RangeSet& own, const double* diag, const double* r, double* p, double* dotPartial, PcgScalars* scal);
void k_eig_update_xr(cudaStream_t, const RangeSet& own, const double* diag, double* x, double* r, const double* p, const double* Ap, double* dotPartial, PcgScalars* scal);
void k_eig_update_p(cudaStream_t, const RangeSet& own, const double* diag, double* p, const double* r, const PcgScalars* scal);
#ifndef PS_EMULATE
void k_halo_push_peer(cudaStream_t, int64_t n0, int64_t n1, const int32_t* idx, const double* v, double* dst0, double* dst1, unsigned long long* flag0, unsigned long long* flag1,
                      unsigned long long seq, PcgScalars* S, bool respectDone, unsigned int* ticket);
void k_halo_push_direct(cudaStream_t, int64_t n0, int64_t n1, const int32_t* idx, const double* v, double* dst0, double* dst1, const PcgScalars* S);
void k_halo_push_p(cudaStream_t, int64_t n0, int64_t n1, const int32_t* idx, const double* r, const double* p, const double* Ap, double* dst0, double* dst1, PcgScalars* S, const PeerCtx& P);
void k_halo_exchange_peer(cudaStream_t, int64_t ns0, int64_t ns1, const int32_t* sendIdx, double* dst0, double* dst1, unsigned long long* dflag0, unsigned long long* dflag1,
                          int64_t nr0, int64_t nr1, const int32_t* recvIdx, const double* src0, const double* src1, const unsigned long long* sflag0, const unsigned long long* sflag1,
                          unsigned long long seq, double* v, PcgScalars* S, bool respectDone, unsigned int* ticket);
void k_halo_unpack_peer(cudaStream_t, int64_t n0, int64_t n1, const int32_t* idx, const double* src0, const double* src1, const unsigned long long* flag0, const unsigned long long* flag1,
                        unsigned long long seq, double* v, PcgScalars* S, bool respectDone);
#endif
void k_recover_active(cudaStream_t, const Geom&, const RowSet& rows, const double* wAct, const double* mcInv, const double* rhsU, double* velSol);
// faces this rank writes: active faces with index in [aLo, aHi), reduced faces of regions [regLo, regHi), every face without a DOF;
// with `shared` (Partition::spanning) a reduced face of a shared region is written by the slab that holds it: z in [zLo, zHi)
// (the last slab also takes the top plane)
struct FaceOwner { int32_t aLo, aHi, regLo, regHi; const uint8_t* shared = nullptr; int32_t zLo = 0, zHi = 0, nz = 0; };
void k_writeback_velocity(cudaStream_t, const Geom&, const Fields&, const Counts&, const RegionData&, const double* velSol, int axis, float* velOut, bool writeValid, float* validOut, FaceOwner own,
                          int64_t lo, int64_t hi, int64_t validLo, int64_t validHi);
void k_merge_face_plane(cudaStream_t, const Geom&, const Fields&, int axis, int k, const float* peerPlane, float* velOut, FaceOwner own);
// halo plumbing
void k_halo_pack(cudaStream_t, int64_t n, const int32_t* idx, const double* v, double* buf, const PcgScalars* scal);
void k_halo_unpack(cudaStream_t, int64_t n, const int32_t* idx, const double* buf, double* v, const PcgScalars* scal);
// halo discovery: flag[c] = 1 for every column c (of a non-empty slot) of the given rows that `colsOwned` contains
void k_mark_K_columns(cudaStream_t, const OpArgs&, const RowSet& rows, const RangeSet& colsOwned, uint8_t* flag);
void k_mark_Kt_columns(cudaStream_t, const OpArgs&, const RowSet& cellRows, const RowSet& edgeRows, const RowSet& colsOwned, uint8_t* flag);
int64_t select_flagged(cudaStream_t, int64_t n, const uint8_t* flag, DBuf<int32_t>& out, int64_t outOffset);

extern thread_local std::string g_lastError;

}  // namespace ps
