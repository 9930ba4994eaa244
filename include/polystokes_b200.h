/* polystokes_b200.h -- C ABI of the B200-native PolyStokes per-step Stokes solve.
 *
 * This library replaces everything below the DOP node of the reference, i.e. class
 * HDK_PolyStokes::Solver (exec/HDK_PolyStokesSolver.h:27-887) and the lib/ linear algebra it calls,
 * behind plain-C entry points (no C++ / torch / HDK types in any signature).  The Houdini node
 * HDK_PolyStokes::solveGasSubclass (exec/HDK_PolyStokes.C:222-609) keeps its role as a thin
 * marshaller: it copies the SIM_RawField voxels into dense x-fastest arrays, fills ps_params from the
 * node's PRM accessors (exec/HDK_PolyStokes.h:23-43) and calls ps_step once per substep.
 * INTEGRATION.md shows that binding.
 *
 * Layout of every field: dense, x fastest, then y, then z, sized by sample type for an nx*ny*nz grid:
 *   centre (nx,ny,nz); face X (nx+1,ny,nz); face Y (nx,ny+1,nz); face Z (nx,ny,nz+1)
 *   (exec/HDK_PolyStokesSolver.h:193-222, 294-314).
 * Ownership of every pointer stays with the caller.  A handle is not thread safe.
 */
#ifndef POLYSTOKES_B200_H
#define POLYSTOKES_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* HDK_PolyStokes::Solver::SolverResult, exec/HDK_PolyStokesSolver.h:61-70 (same numeric values) */
enum {
    PS_UNSUPPORTED_SOLVER = -4, PS_INCOMPLETE = -3, PS_INVALID = -2, PS_FAILED = -1,
    PS_NOCONVERGE = 0, PS_SUCCESS = 1, PS_NOCHANGE = 2
};

enum { PS_MEM_HOST = 0, PS_MEM_DEVICE = 1 };

/* Node parameters: one field per PRM of the reference (exec/HDK_PolyStokes.h:23-43; defaults
 * exec/HDK_PolyStokes.C:123-206; README.md:33-45) plus the grid description the Solver
 * constructor receives (exec/HDK_PolyStokesSolver.cpp:18-68). */
typedef struct ps_params {
    int32_t nx, ny, nz;               /* velocityField->getTotalVoxelRes() */
    double dx, dt;                    /* PS.C:319-320 */
    double origin[3];                 /* field origin (enters no result, kept for the adaptor) */
    double constantDensity;           /* densityField constant value, PS.C:298-304 */
    double tolerance;                 /* SIM_NAME_TOLERANCE */
    int32_t maxSolverIterations;
    int32_t activeLiquidBoundaryLayerSize;
    int32_t activeSolidBoundaryLayerSize;
    int32_t doReducedRegions;
    int32_t doTile;
    int32_t tileSize;
    int32_t tilePadding;
    int32_t exportMatrices;
    int32_t exportComponentMatrices;
    int32_t exportStats;
    char exportDataPrefix[256];
    int32_t doSolve;
    int32_t keepNonConvergedResults;
    int32_t useWarmStart;             /* guessVector = constructGuessVectors (S.cpp:521-531); read by solverType 1 only --
                                       * the live solver (type 0) starts from zero whatever the guess (S.cpp:768) */
    int32_t matrixSetup;              /* 0 = pressurestress (units.h:76-83); others -> PS_UNSUPPORTED_SOLVER */
    int32_t solverType;               /* units.h:85-94: 0 = pcg_matrix_vector_products (solveSPDwithMatrixVectorPCG, S.cpp:734-812),
                                       * 1 = eigen (solveEigenCG, S.cpp:814-862: Eigen CG + Jacobi from guessVector; one GPU);
                                       * others -> PS_UNSUPPORTED_SOLVER */
    int32_t useInputSurfaceWeights;   /* validated, ignored by the live weights builder (PS.C:351-352) */
    int32_t useInputCollisionWeights;
    double minDensity, maxDensity;    /* stored, never used by the reference (S.cpp:55-56) */
    /* extensions (not in the reference) */
    int32_t device;                   /* CUDA device ordinal */
    int32_t checkEvery;               /* host polls the device-side convergence flag every N iterations (0 = default 25) */
    int (*cancel_cb)(void*);          /* UT_Interrupt::opInterrupt() stand-in, polled with the flag */
    void* cancel_ctx;
} ps_params;

/* Inputs of one step = the fields solveGasSubclass fetches (exec/HDK_PolyStokes.C:235-246). */
typedef struct ps_fields_in {
    int32_t memory;                   /* PS_MEM_HOST or PS_MEM_DEVICE */
    const float* surface;             /* liquid SDF, centre sampled, < 0 inside liquid */
    const float* collision;           /* solid SDF, centre sampled, < 0 inside solid */
    const float* viscosity;           /* centre sampled */
    const float* velocity[3];         /* face sampled */
    const float* collisionvel[3];     /* face sampled */
} ps_fields_in;

/* Outputs: velocity overwritten on valid faces + the `valid` vector field (PS.C:562-584). */
typedef struct ps_fields_out {
    int32_t memory;
    float* velocity[3];               /* must hold the input velocity on entry semantics: invalid faces are left untouched */
    float* valid[3];
} ps_fields_out;

enum {
    PS_STAGE_UPLOAD = 0, PS_STAGE_WEIGHTS, PS_STAGE_CLASSIFY, PS_STAGE_REDUCED, PS_STAGE_INDICES, PS_STAGE_REGION_MATRICES,
    PS_STAGE_MATRIX_BLOCKS, PS_STAGE_ASSEMBLE, PS_STAGE_SOLVE, PS_STAGE_WRITEBACK, PS_STAGE_DOWNLOAD, PS_NUM_STAGES
};

/* Mirrors exportStats' dimData / solveData vectors (exec/HDK_PolyStokesSolver.cpp:574-606). */
typedef struct ps_stats {
    double dimData[27];
    double solveData[6];              /* error, iterations, solve CPU ms, solve wall ms, setup CPU ms, setup wall ms */
    int32_t result;                   /* SolverResult */
    int32_t usedBiCGStab;             /* CG -> BiCGSTAB fallback taken (S.cpp:784-799) */
    double stage_ms[PS_NUM_STAGES];   /* CUDA-event time per stage (same stage split as PS.C:350-568) */
    int64_t gpu_launches;             /* kernels launched by this step */
} ps_stats;

typedef struct ps_solver* ps_handle;

/* Solver constructor (S.cpp:18-155).  Returns PS_SUCCESS or PS_FAILED/PS_INVALID. */
int ps_create(const ps_params* params, ps_handle* out);
void ps_destroy(ps_handle h);
/* New per-step parameters for an existing handle: everything but the grid (nx, ny, nz, dx) and the device may change -- a DOP
 * network calls the solver with a different dt every substep (PS.C:319), which must not rebuild streams and buffers. */
int ps_set_params(ps_handle h, const ps_params* params);
/* Page-locked host memory (cudaMallocHost) for callers that do not link CUDA themselves: host fields staged in it cross PCIe
 * asynchronously, under the solver's kernels.  NULL on failure. */
void* ps_alloc_pinned(size_t bytes);
void ps_free_pinned(void* p);
/* One solveGasSubclass body (PS.C:344-608): weights, classify, assemble, PCG, write-back.
 * Returns the SolverResult; `out` may be NULL (no write-back), `stats` may be NULL. */
int ps_step(ps_handle h, const ps_fields_in* in, ps_fields_out* out, ps_stats* stats);
/* The two halves of ps_step, separately callable (setup = PS.C:344-476, solve = PS.C:508-584). */
int ps_setup(ps_handle h, const ps_fields_in* in);
int ps_solve(ps_handle h, ps_fields_out* out, ps_stats* stats);
/* exportMatrices / exportComponentMatrices / exportStats (S.cpp:533-606): MatrixMarket files written with
 * Eigen's saveMarket format.  `what` is a bit mask: 1 = Mat_A + Vec_b + Vec_guess + solutionVector (Mat_A is the explicit
 * matrix with solverType 1 and the empty nSystemSize x nSystemSize matrix of the factored path otherwise, as in the
 * reference), 2 = component matrices, 4 = stats.  On a decomposed handle (one process per GPU, or ps_create_multi) ps_export is a
 * collective call: every rank calls it, rank 0 writes the whole file set under ITS prefix (the files of one GPU; dimData's "thread
 * count" is the SMs of all ranks, the solveData times are the slowest rank's) and the other ranks write nothing; every rank returns the
 * same code (PS_FAILED, naming the prefix, when a write failed).  ps_step's export through the ps_params toggles does the same. */
int ps_export(ps_handle h, const char* prefix, int what);
/* thread-local description of the last PS_FAILED / PS_INVALID */
const char* ps_last_error(void);

/* ---- several GPUs: one process per GPU, the grid slab-decomposed along z (SURVEY.md section 8e) ----
 * The reference is single-node shared-memory (TBB / OpenMP inside one Solver); the slab decomposition replaces that
 * intra-solver parallelism.  Call order: every rank creates its handle on its own device; rank 0 calls
 * ps_comm_unique_id and ships the 128 bytes to the others with any host transport (torch.distributed, MPI, a file);
 * every rank then calls ps_comm_init (collective).  Afterwards ps_step / ps_setup / ps_solve / ps_apply /
 * ps_time_kernel("cg_iteration") are collective calls: every rank passes pointers to the SAME full-grid input fields and
 * owns the z-slab reported by ps_get_partition.  With tilePadding >= 2 (or reduced regions off) the setup is slab-local: a rank
 * reads, classifies, numbers and assembles only its slab plus a halo of a few layers, the global numbering follows from an
 * all-gather of per-slab counts (ps_part.hpp); with tilePadding 1 every rank classifies the whole grid redundantly.  Output
 * contract: a rank writes velocity and `valid` on ITS SLAB of the output arrays (cells / faces / edges with z in [zLo, zHi), the
 * last rank also the top layer); the rest of the arrays is not touched.  Reduced regions that cross a cut (doTile off, or
 * tilePadding 0) are solved with a cross-rank reduction: each rank forms the moments of the region's rows in its slab, one
 * all-reduce per operator apply sums them, and every rank solves the region's small system; the setup stays replicated for
 * these configurations (ps_get_count "sharedRegions" counts such regions).  ps_set_params may switch doTile between steps: the
 * cuts follow (multiples of 16 without tiles, of lcm(16, tileSize) with them).  The cuts are even in layers unless the caller sets
 * them (ps_set_partition, ps_rebalance); caller-set cuts are kept by ps_set_params while they remain multiples of the unit, and
 * replaced by the even cuts when a new tileSize makes them illegal.
 * cancel_cb must answer identically on all ranks. */
/* ---- several GPUs behind ONE handle (SURVEY.md section 8b; the caller is one cook thread, exec/HDK_PolyStokes.C:222-345) ----
 * ps_create_multi builds the same slab decomposition inside one process: one rank per device devs[0..ndev) (NULL: devices
 * 0..ndev-1), one host thread per rank, NCCL + NVLink peer memory between them.  The handle is used exactly like a single-GPU
 * one: ps_step / ps_setup / ps_solve take the full-grid HOST fields of the caller, every rank uploads only its slab (+ halo) and
 * writes only its slab of velocity / valid, so after the call the caller's arrays are complete.  ps_get_count / ps_get_real /
 * ps_get_partition answer for the whole job; ps_export writes the file set of one GPU, and ps_get_vector / ps_get_csr / ps_apply
 * return the global vectors, matrices and A x, assembled from the ranks that own them.  The per-voxel introspection, diagA and the
 * explicit A need a single-GPU handle. */
int ps_create_multi(const ps_params* params, int ndev, const int* devs, ps_handle* out);
int ps_comm_unique_id(void* id128);
int ps_comm_init(ps_handle h, int rank, int nranks, const void* id128);
/* z cuts of all ranks: zCut[nranks+1] (may be NULL); returns nranks, this rank's slab in *zLo, *zHi */
int ps_get_partition(ps_handle h, int32_t* rank, int32_t* zLo, int32_t* zHi, int32_t* zCut);
/* Collective on a decomposed handle.  zCut[nranks+1]: 0 = zCut[0] < ... < zCut[nranks] = nz, interior cuts multiples of the unit
 * (lcm(16, tileSize) layers with tiles, 16 without); NULL = the even cuts.  PS_INVALID (the same on every rank, agreed by one
 * all-reduce) for cuts that break a rule or differ between ranks; the handle keeps its cuts then.  Takes effect at the next ps_setup /
 * ps_step.  On one GPU only NULL and {0, nz} are accepted (and change nothing). */
int ps_set_partition(ps_handle h, const int32_t* zCut);
/* Collective; needs a prior setup.  Every setup measures the work of each z-unit: the algorithmic bytes of one CG iteration
 * (ps_kernel_bytes "cg_iteration") of the rows the unit holds -- ps_get_vector "unitLoad", the same on every rank and independent of
 * the cuts; "unitCounts" is the table behind it, [unit][9]: active voxels of the 7 sample slots, coupled reduced rows (by the z of
 * their face), regions (by the z of their first cell).  ps_rebalance takes the cuts that minimise the largest slab's load (the
 * lexicographically smallest such cuts, every slab at least one unit) and applies them only if they lower that maximum:
 * PS_SUCCESS (applied; effective at the next ps_setup / ps_step), PS_NOCHANGE (kept; always on one GPU), PS_INVALID (no setup yet,
 * or the tiling changed since).  zCut (may be NULL) receives the cuts the handle holds afterwards. */
int ps_rebalance(ps_handle h, int32_t* zCut);

/* ---- introspection for parity tests (read-only views of the solver state, copied to HOST memory) ---- */
/* counters by name: nCenter nFaceX nFaceY nFaceZ nEdgeYZ nEdgeXZ nEdgeXY nActiveVs nReducedVs nPressures
 * nStresses nTotalDOFs nSystemSize regionCount iterations result usedBiCGStab nRowsExt */
int64_t ps_get_count(ps_handle h, const char* name);
double ps_get_real(ps_handle h, const char* name);     /* solveError, xmag (x.x of the CG stop test at the last iteration) */
/* kind: 0 labels (int8 widened), 1 active indices, 2 reduced indices; slot: 0 centre, 1-3 face x/y/z,
 * 4-6 edge YZ/XZ/XY.  `out` receives int32 values; returns the element count. */
int64_t ps_get_index_field(ps_handle h, int kind, int slot, int32_t* out);
/* liquid != 0: liquid weights, else fluid weights; values k/8 as float */
int64_t ps_get_weight_field(ps_handle h, int liquid, int slot, float* out);
/* CSR export of a block by name (G Dt JG JDt Mc McInv uInv u Mr B BInv A): call once with NULL arrays for
 * the sizes, then with arrays.  Column indices sorted per row, explicit zeros kept (Eigen semantics).  "A" is the explicit
 * system matrix of assembleSystemPressureStress (S_AS:351-430), built on the device on first request (one GPU; its region
 * blocks are dense, so it only fits for small / medium grids -- PS_FAILED beyond 2^31-1 entries or device memory). */
int ps_get_csr(ps_handle h, const char* name, int64_t* rows, int64_t* cols, int64_t* nnz, int64_t* rowptr, int32_t* colidx, double* vals);
/* dense vectors by name (activeRHS reducedRHS pressureRHS stressRHS b guess diagA solution velSolution com bestFit
 * MrDense ViscDense BinvDense unitLoad unitCounts); returns the length.  diagA = diag(A) formed from the factors (one GPU).  On a rank of a job with one
 * process per GPU, b / solution / guess / region data are zero outside the calling rank's share, so the sum over ranks is the global
 * vector; a ps_create_multi handle returns the global vector. */
int64_t ps_get_vector(ps_handle h, const char* name, double* out);
/* y = A x with host vectors of length nSystemSize (ApplyPressureStressMatrix::apply, Apply.h:182-184) */
int ps_apply(ps_handle h, const double* x, double* y);
/* Roofline support for bench.py.  `name` is one of
 *   "pass1"  w = dt Mc^-1 K x on the active face rows   (SpMV over the 8-wide face-row ELL)
 *   "reduced" the coupled reduced rows: K_red x -> moments -> B^-1 -> w_f  (3 small kernels)
 *   "pass2"  y = -K_ext^T w - 1/2 mu^-1 x    (SpMV over the 6/2/4-wide DOF-row ELL)
 *   "apply"  the whole operator (pass1 + reduced-region moments/expand + pass2)
 *   "cg_iteration"  one full CG iteration (apply + the two fused vector kernels)
 * ps_time_kernel runs it `reps` times back to back on the solver stream between CUDA events (after one
 * warm-up run) and returns the average milliseconds; ps_kernel_bytes returns the ALGORITHMIC bytes of one
 * run on the current system (DESIGN.md section 5).  Both need a prior ps_setup / ps_step. */
double ps_time_kernel(ps_handle h, const char* name, int reps);
double ps_kernel_bytes(ps_handle h, const char* name);
/* Stopwatch on the solver's own stream (all of a step's device work runs there; copies of host-memory callers are joined
 * to it by events): ps_timer(h, 0) records the start event, ps_timer(h, 1) records the stop event, waits for it and
 * returns the elapsed milliseconds between the two (< 0 on error).  No reference counterpart (the reference times
 * with UT_StopWatch around solveGasSubclass stages, S.cpp:578-602). */
double ps_timer(ps_handle h, int stop);

#ifdef __cplusplus
}
#endif
#endif
