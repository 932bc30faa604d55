/*
 * sipb200.h — C ABI of the B200-native PARSDMM projection iteration.
 *
 * Drop-in boundary for the hot path of slimgroup/SetIntersectionProjection.jl (pure Julia): the
 * Julia (or Python) host keeps the reference API and `ccall`s / `ctypes`-calls these entry points.
 * Every entry point cites the reference routine it replaces (paths relative to the reference's
 * src/).  Plain pointers and sizes only; no torch / C++ types cross the boundary.
 *
 * Conventions
 *   - every function returns SIPB_OK (0) or a negative error code and never throws;
 *     sipb_last_error() returns a thread-local message for the last failure;
 *   - `dtype`: SIPB_F32 (Float32) or SIPB_F64 (Float64) — the reference's TF;
 *   - vectors are column-major vec(model): linear index i + n1*(j + n2*k) (get_discrete_Grad.jl:63);
 *   - host arrays stay owned by the caller; device memory is owned by the ctx / problem;
 *   - one host thread drives one GPU (one process per GPU; multi-GPU slabs use sipb_comm_*).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     SIPB_E_CUDA.
 */
#ifndef SIPB200_H
#define SIPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIPB_ABI_VERSION 1

/* error codes */
#define SIPB_OK             0
#define SIPB_E_INVALID     -1   /* bad argument / inconsistent sizes                           */
#define SIPB_E_UNSUPPORTED -2   /* set / operator / option outside the device hot path          */
#define SIPB_E_CUDA        -3   /* CUDA runtime failure (incl. "no device")                      */
#define SIPB_E_NCCL        -4
#define SIPB_E_STATE       -5   /* call order violated (e.g. solve before finalize)              */
#define SIPB_E_MISSING_DIAG -6  /* CDS_scaled_add!.jl:18-20: diagonal of AtA_i missing in Q      */

#define SIPB_F32 0
#define SIPB_F64 1

/* projector / prox kinds (get_projector.jl:3-103, prox_l2s!.jl, prox_l1!.jl) */
#define SIPB_SET_BOUNDS_SCALAR 0   /* project_bounds!.jl:3-12   */
#define SIPB_SET_BOUNDS_VECTOR 1   /* project_bounds!.jl:14-25  */
#define SIPB_SET_L1            2   /* project_l1_Duchi!.jl:21-52 */
#define SIPB_SET_L2            3   /* project_l2!.jl:3-16       */
#define SIPB_SET_ANNULUS       4   /* project_annulus!.jl:3-21  */
#define SIPB_SET_CARDINALITY   5   /* project_cardinality!.jl:3-21 (vector mode) */
#define SIPB_SET_PROX_L1       6   /* prox_l1!.jl:8-10 (set_type "prox_l1", get_projector.jl:21-27) */
#define SIPB_SET_DISTANCE      7   /* prox_l2s!.jl:3-6: the 1/2||x-m||^2 term (PARSDMM_initialize.jl:64-71) */
#define SIPB_SET_BOUNDS_FIBER  8   /* project_bounds!.jl:38-88: per-fiber bounds, max then min, bounds indexed along the fiber */
#define SIPB_SET_CARD_FIBER    9   /* project_cardinality!.jl:23-113: k largest magnitudes of every fiber (stable ties) */
#define SIPB_SET_CARD_SLICE   10   /* project_cardinality!.jl:115-146: k largest magnitudes of every 2-D slice of a 3-D
                                      tensor; fiber_axis = the axis the slices are orthogonal to ("x","y","z" -> 0,1,2) */
#define SIPB_SET_HISTOGRAM    11   /* project_histogram_relaxed.jl:9-26: sorted values clamped by sorted bound vectors
                                      (min_vec / max_vec: TF[M], ascending); stable sort in Julia's isless order */
#define SIPB_SET_KIND_MAX     11

/* transform-domain operator kinds (get_TD_operator.jl:12-95, get_discrete_Grad.jl) */
#define SIPB_OP_IDENTITY 0
#define SIPB_OP_DX       1   /* first (fastest) axis  : offset 1        */
#define SIPB_OP_DY       2   /* second axis (3-D only): offset n1       */
#define SIPB_OP_DZ       3   /* last axis             : offset n1 (2-D) or n1*n2 (3-D) */
#define SIPB_OP_TV       4   /* vcat(D_z[,D_y],D_x)   (get_discrete_Grad.jl:33,69-72)  */
#define SIPB_OP_DXZ      5   /* D_z*D_x, 2-D only     (get_TD_operator.jl:69-73)       */
#define SIPB_OP_SPARSE   6   /* explicit sparse matrix: constraint.custom_TD_OP[1] (setup_constraints.jl:70-72) */

/* Minkowski block placement of an operator (PARSDMM_precompute_distribute_Minkowski.jl:78-88) */
#define SIPB_BLOCK_PLAIN 0   /* A       (N columns)  */
#define SIPB_BLOCK_LEFT  1   /* [A 0]   (2N columns) */
#define SIPB_BLOCK_RIGHT 2   /* [0 A]                */
#define SIPB_BLOCK_BOTH  3   /* [A A]                */

typedef struct sipb_ctx sipb_ctx;
typedef struct sipb_problem sipb_problem;

/* One term of the intersection: projector + operator.  Replaces one entry of the reference's
 * (P_sub[i], TD_OP[i], set_Prop.*[i]) triple (setup_constraints.jl:17-102). */
/* An explicit sparse transform-domain operator (SparseMatrixCSC of the reference) in both orientations, host
 * arrays, 0-based.  Products follow SparseArrays: (A*x)[r] is a left fold over the stored columns of row r in
 * ascending column order, (A'*v)[c] over the stored rows of column c in ascending row order. */
typedef struct sipb_sparse {
  int64_t rows, cols, nnz;
  const int64_t* rowptr;   /* [rows+1]  CSR of A                                  */
  const int32_t* colidx;   /* [nnz]     ascending inside a row                    */
  const void*    val;      /* [nnz]     TF                                        */
  const int64_t* colptr;   /* [cols+1]  CSC of A (colptr/rowval/nzval of Julia, minus 1) */
  const int32_t* rowidx;   /* [nnz]     ascending inside a column                 */
  const void*    valt;     /* [nnz]     TF                                        */
} sipb_sparse;

typedef struct sipb_set_desc {
  int32_t set_kind;        /* SIPB_SET_*                                                       */
  int32_t op_kind;         /* SIPB_OP_*                                                        */
  int32_t block_mode;      /* SIPB_BLOCK_*                                                     */
  int32_t ncvx;            /* set_Prop.ncvx[i] (setup_constraints.jl:89-97)                    */
  double  min;             /* scalar lower bound / annulus sigma_min                           */
  double  max;             /* scalar upper bound / l1 tau / l2 sigma / prox_l1 rho             */
  int64_t k;               /* cardinality                                                      */
  const void* min_vec;     /* host TF[M] for SIPB_SET_BOUNDS_VECTOR / SIPB_SET_HISTOGRAM, TF[td_n[fiber_axis]] for ..._FIBER, else NULL */
  const void* max_vec;
  int32_t fiber_axis;      /* fiber modes (app_mode ("fiber","x"|"y"|"z")): 0, 1 or 2 — axis of the transform-domain grid */
  int32_t reserved;
  int64_t td_n[3];         /* fiber modes: set_Prop.TD_n[i], the transform-domain grid (third entry 1 in 2-D)  */
  const sipb_sparse* sparse;  /* SIPB_OP_SPARSE: the matrix (copied to the device by sipb_problem_add_set), else NULL */
} sipb_set_desc;

/* Mirror of PARSDMM_options (SetIntersectionProjection.jl:110-128) after convert_options!. */
typedef struct sipb_options {
  int32_t maxit;
  int32_t rho_update_frequency;
  int32_t adjust_rho;
  int32_t adjust_gamma;
  int32_t adjust_feasibility_rho;
  int32_t zero_ini_guess;
  int32_t n_rho_ini;            /* 1 or p                                                       */
  int32_t profile_kernels;      /* 1: bracket every launch with CUDA events (kernel table below) */
  double  evol_rel_tol;         /* already rounded to TF by the host                            */
  double  feas_tol;
  double  obj_tol;
  double  gamma_ini;
  const double* rho_ini;        /* n_rho_ini values, already rounded to TF                      */
  int32_t fixed_iterations;     /* >0: ignore the stop rules and run exactly this many iterations (benchmarks) */
  int32_t return_ly;            /* 1: copy l and y back to the host arrays                      */
  int32_t resident_io;          /* 1: benchmark mode — m is taken from the device buffer left by the previous
                                   solve of this problem and x/l/y are not copied back (no H2D/D2H at all)   */
  int32_t warm_resident;        /* 1 (with zero_ini_guess == 0): the start vectors x, l, y already sit in the problem's
                                   device buffers (put there by sipb_problem_warm_from); nothing is uploaded for them */
} sipb_options;

#define SIPB_N_PHASES 7         /* TimerOutputs sections of PARSDMM.jl:40,100,105,113,152,163,229 */
#define SIPB_N_KERNEL_CLASSES 24

/* Mirror of log_type_PARSDMM (SetIntersectionProjection.jl:95-108).  The caller allocates every
 * array with `maxit` rows (row-major [maxit][p] / [maxit][pp]); the solver fills rows 0..iters-1
 * (set_feasibility rows 0..feas_rows-1), exactly the rows output_check_PARSDMM keeps
 * (PARSDMM.jl:261-278). */
typedef struct sipb_log {
  int32_t iters;                /* number of PARSDMM iterations performed (0 if input was feasible) */
  int32_t feas_rows;            /* rows of set_feasibility that are meaningful (= `counter`)        */
  int32_t stopped_feasible;     /* 1: PARSDMM_initialize found the input feasible (PARSDMM.jl:63-82) */
  int32_t p, pp;
  double* set_feasibility;      /* [maxit][pp] */
  double* r_dual;               /* [maxit][p]  */
  double* r_pri;                /* [maxit][p]  */
  double* r_dual_total;         /* [maxit]     */
  double* r_pri_total;
  double* obj;
  double* evol_x;
  double* rho;                  /* [maxit][p]  */
  double* gamma;                /* [maxit][p]  */
  int32_t* cg_it;               /* [maxit]     */
  double* cg_relres;
  double  phase_seconds[SIPB_N_PHASES];   /* DEVICE time per TimerOutputs section, same order: CUDA events on the
                                             solver's stream close every phase (the stopping-rule and adaptation
                                             sections are host scalar work: their entries hold the device idle gap) */
  double  solve_seconds;                  /* whole sipb_solve call incl. H2D/D2H                    */
  double  device_seconds;                 /* CUDA-event time of the whole solve on the stream, after the
                                             H2D of m is enqueued and before the D2H of x                 */
  /* kernel table (profile_kernels=1): launches and summed CUDA-event milliseconds per class */
  int64_t kernel_launches[SIPB_N_KERNEL_CLASSES];
  double  kernel_ms[SIPB_N_KERNEL_CLASSES];
  double  kernel_bytes[SIPB_N_KERNEL_CLASSES];  /* algorithmic bytes moved by the class (always counted): every array
                                             a kernel must read or write once, gathered vectors with perfect reuse;
                                             launches queued behind a finished CG count nothing                 */
  int64_t total_launches;                 /* all kernel launches inside sipb_solve (always counted) */
  int64_t h2d_bytes, d2h_bytes;
} sipb_log;

/* Environment switches (read when the object they affect is created; for A/B measurements and tests):
 *   SIPB_Q_CLASSES=0      sipb_problem_finalize keeps Q / AtA as CDS arrays (see sipb_problem_q_form)
 *   SIPB_SPMV_TILE=0      the CG uses the generic grid-stride SpMV instead of the tiled TMA-staged kernel
 *   SIPB_P2P=0            sipb_comm_init uses NCCL for the CG reductions and halos instead of peer memory
 *   SIPB_FUSE_STOP_OFF=1  sipb_solve reduces the obj / evol_x sums in a separate pass instead of inside the
 *                         distance term's y/l update
 *   SIPB_GRAPH_LOOPS=0    host-driven CG / l1-search loops instead of CUDA-graph WHILE nodes (same kernels)
 *   SIPB_SEL_SPEC=0       cardinality sets on one GPU: no speculative select levels inside pass 1 of the y/l
 *                         update and in-place tie zeroing (the search then runs all its histogram passes)
 *   SIPB_L1_SKIPV=0|2     l1 sets on one GPU: pass 1 of the y/l update always stores v (0) / never stores it and
 *                         leaves that to the device-gated second launch (2); default 1: skip while the ball was
 *                         inactive in the previous iteration
 *   SIPB_PEER_ALLREDUCE=0 slabs: NCCL instead of the small peer-memory all-reduces */

/* ---- library / context ------------------------------------------------------------------- */
int         sipb_abi_version(void);
const char* sipb_last_error(void);
const char* sipb_kernel_class_name(int cls);          /* name of kernel class 0..SIPB_N_KERNEL_CLASSES-1 */
int sipb_ctx_create(int device, sipb_ctx** out);      /* binds the calling process to `device`   */
int sipb_ctx_destroy(sipb_ctx* ctx);
int sipb_ctx_num_sms(sipb_ctx* ctx, int* out);

/* ---- multi-GPU slabs (one process per GPU).  Replaces the reference's Distributed/DArray
 *      set-parallelism (update_y_l_parallel.jl, adapt_rho_gamma_parallel.jl) by z-slab domain
 *      decomposition; the 128-byte NCCL unique id travels over the host's own transport
 *      (torch.distributed / MPI / Julia Distributed). ------------------------------------------ */
int sipb_comm_unique_id(void* out128);
int sipb_comm_init(sipb_ctx* ctx, int rank, int world, const void* uid128);
int sipb_comm_info(sipb_ctx* ctx, int* rank, int* world);
/* 1 when the CG's reductions and halo planes go through CUDA-IPC peer memory (NVLink loads/stores fused into
 * the kernels) instead of NCCL; set SIPB_P2P=0 before sipb_comm_init to force the NCCL path. */
int sipb_comm_peer_path(sipb_ctx* ctx, int* active);
/* planes [k0,k1) of the slowest grid axis owned by `rank`; after sipb_comm_init with world > 1 every
 * 3-D problem of the ctx is a slab problem: sipb_problem_create still takes the GLOBAL grid, while
 * sipb_problem_set_ata takes the rank's rows [n1*n2*k0, n1*n2*k1) of each diagonal and sipb_solve takes /
 * returns the rank's slab of m and x, and of every l[i], y[i] (per row block: the planes [k0,k1), for a
 * D_z block the planes [k0, min(k1, n3-1))). */
int sipb_slab_range(int64_t n_last, int rank, int world, int64_t* k0, int64_t* k1);

/* ---- problem set-up: replaces the device-relevant part of PARSDMM_precompute_distribute.jl:6-77
 *      and the allocation / Q assembly of PARSDMM_initialize.jl:117-230 ---------------------- */
int sipb_problem_create(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, const double* h,
                        int minkowski, int feasibility_only, sipb_problem** out);
/* sets must be added in TD_OP order; the distance term (SIPB_SET_DISTANCE) last. */
int sipb_problem_add_set(sipb_problem* pb, const sipb_set_desc* desc);
/* AtA[i] in CDS form exactly as mat2CDS (mat2CDS.jl:7-32) returns it: R is column-major
 * [rows x nd] host TF, offsets int64[nd] ascending. */
int sipb_problem_set_ata(sipb_problem* pb, int set_index, const void* R, int64_t rows,
                         const int64_t* offsets, int nd);
/* AtA[i] as one row per stencil class instead of the [rows x nd] array: tab is host TF[54][nd], tab[cls*nd + j] =
 * AtA[r, r + offsets[j]] for any row r of class cls = ((half*3 + c(k))*3 + c(j))*3 + c(i), c = 0 / 1 / 2 for the
 * first / an interior / the last index of the axis (half = second Minkowski half).  Every A'A the reference builds
 * from get_TD_operator.jl has this structure; passing the table skips forming, uploading and verifying the array
 * (PARSDMM_precompute_distribute.jl:44-55 costs 8 GB and ~7 s at 512^3).  All sets of a problem must then come as
 * tables (a problem with a custom sparse operator uses sipb_problem_set_ata for every set). */
int sipb_problem_set_ata_classes(sipb_problem* pb, int set_index, const void* tab, const int64_t* offsets, int nd);
/* uploads, builds Q_offsets in the reference's order (PARSDMM_initialize.jl:217-221). */
int sipb_problem_finalize(sipb_problem* pb);
int sipb_problem_num_q_offsets(sipb_problem* pb, int* nd);
int sipb_problem_q_offsets(sipb_problem* pb, int64_t* out);     /* Q_offsets, reference order */
/* How the device holds Q = sum rho_i AtA_i (PARSDMM_initialize.jl:223-229) after finalize:
 * 0 = CDS arrays [N x nd]; 1 = stencil-class tables (every AtA_i was verified to hold one value per diagonal
 * on all rows that agree on {first, interior, last} along each grid axis, so one row per class is kept and the
 * SpMV of cg.jl streams only the vectors; same multiply-adds in the same order -> bit-identical results).
 * The environment variable SIPB_Q_CLASSES=0 forces the array form. */
int sipb_problem_q_form(sipb_problem* pb, int* form);
int sipb_problem_destroy(sipb_problem* pb);

/* Multilevel warm start on the device: nearest-neighbour resampling of the coarse problem's x, l, y into the
 * fine problem's device buffers.  Replaces the Interpolations.jl calls of PARSDMM_multi_level.jl:61-67 and
 * interpolate_y_l.jl:32-91.  Each segment resamples one column-major box: `vec` = -1 for x, or the set index
 * for l and y (both are resampled); offsets are element offsets inside that vector; the sampling positions
 * are range(1, stop=n_src, length=n_dst) per axis with half-way positions rounded up.
 * Slab-decomposed problems (both levels on the same communicator): the segments are global — offsets and shapes
 * address the whole vector in the reference's row-block-major order — and the call is collective: every rank passes
 * the same segments, the coarse vectors are gathered whole on every rank (ncclSend / ncclRecv), and each rank
 * receives its own planes of the fine x, l, y.  Both problems must be slab-decomposed, or neither. */
typedef struct sipb_resample_seg {
  int32_t vec;
  int32_t reserved;
  int64_t src_off, dst_off;
  int64_t src_shape[3];
  int64_t dst_shape[3];
} sipb_resample_seg;
int sipb_problem_warm_from(sipb_problem* fine, sipb_problem* coarse, const sipb_resample_seg* segs, int nseg);

/* ---- the solve: replaces PARSDMM(m,AtA,TD_OP,set_Prop,P_sub,comp_grid,options[,x,l,y])
 *      (PARSDMM.jl:25-258).  m: host TF[N_model]; x: host TF[N] in/out (start guess when
 *      zero_ini_guess==0); l,y: arrays of p host pointers (may be NULL when zero_ini_guess==1 and
 *      return_ly==0). ------------------------------------------------------------------------- */
int sipb_solve(sipb_problem* pb, const void* m, void* x, void* const* l, void* const* y,
               const sipb_options* opt, sipb_log* log);

/* B independent projections at once: the per-channel / per-frame PARSDMM calls of examples/Constraint_examples_2D.jl:221-226
 * and PARSDMM used as the projector inside an outer loop (examples/Dykstra_parallel_vs_PARSDMM.jl:134,149).  pbs[b]
 * are finalized problems, EACH CREATED IN ITS OWN CONTEXT (sipb_ctx_create: a context owns one stream and its scratch);
 * m[b], x[b], l[b], y[b], logs[b] as in sipb_solve (l, y may be NULL).  One host thread per problem drives its solve,
 * the GPU overlaps the streams.  Results are those of B separate sipb_solve calls, bit for bit.  rcs (optional)
 * receives the return code of every problem; the function returns the first failure. */
int sipb_solve_batch(sipb_problem* const* pbs, int B, const void* const* m, void* const* x, void* const* const* l,
                     void* const* const* y, const sipb_options* opt, sipb_log* const* logs, int* rcs);

/* ---- unit entry points (host pointers; used by the parity tests and micro-benchmarks) ------ */
/* y = A*x for A in CDS form: replaces Ax_CDS_MT / CDS_MVp_MT (argmin_x.jl:72-78, CDS_MVp_MT.jl:9-25) */
int sipb_cds_spmv(sipb_ctx* ctx, int dtype, int64_t N, int nd, const void* R, const int64_t* offsets,
                  const void* x, void* y);
/* cg(A,b;tol,maxIter,x) with A in CDS form (cg.jl:44-128).  x in/out. */
int sipb_cds_cg(sipb_ctx* ctx, int dtype, int64_t N, int nd, const void* R, const int64_t* offsets,
                const void* b, void* x, double tol, int max_iter, int* flag, double* relres, int* iters);
/* in-place projector / prox on a host vector (P_sub[i](v), get_projector.jl). `m_vec` only for
 * SIPB_SET_DISTANCE (prox_l2s!(v,rho,m)), with rho passed in desc->max. */
int sipb_project(sipb_ctx* ctx, int dtype, const sipb_set_desc* desc, int64_t M, void* v, const void* m_vec);
/* s = TD_OP*x (forward) or t = TD_OP'*v (adjoint) for a matrix-free operator descriptor
 * (update_y_l.jl:43, rhs_compose.jl:28). */
int sipb_op_apply(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, const double* h, int op_kind,
                  int block_mode, int adjoint, const void* in, void* out);
int sipb_op_rows(int ndim, const int64_t* n, int op_kind, int64_t* rows);
/* the same for an explicit sparse operator (SIPB_OP_SPARSE) */
int sipb_sparse_apply(sipb_ctx* ctx, int dtype, const sipb_sparse* A, int adjoint, const void* in, void* out);
/* Q += alpha*B on matching diagonals (CDS_scaled_add!.jl:8-26). */
int sipb_cds_scaled_add(sipb_ctx* ctx, int dtype, int64_t N, int nd_a, void* A, const int64_t* a_offsets,
                        int nd_b, const void* B, const int64_t* b_offsets, double alpha);
/* micro-benchmark: device-resident CDS SpMV(+dot) on synthetic data, CUDA-event timed;
 * returns average milliseconds per launch over `reps` launches after `warmup`. */
int sipb_bench_spmv(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, int warmup, int reps,
                    int flush_l2, double* avg_ms, int64_t* algorithmic_bytes);

/* the same with a choice of matrix form (0 = CDS arrays, (nd+2)*N*s algorithmic bytes; 1 = stencil-class tables,
 * 2*N*s) and of kernel (tiled = 1: the TMA-staged plane sweep of spmv_tile.cuh; 0: the generic grid-stride kernel) */
int sipb_bench_spmv2(sipb_ctx* ctx, int dtype, int ndim, const int64_t* n, int warmup, int reps, int flush_l2,
                     int form, int tiled, double* avg_ms, int64_t* algorithmic_bytes);
/* y = A*x (CDS_MVp_MT.jl:9-25) for a CDS matrix living on a 3-D grid: takes the tiled kernel when the offsets are a
 * subset of {0, +-1, +-n1, +-n1*n2} and a grid line is a whole number of 16-byte vectors (*used_tiled = 1),
 * otherwise the generic kernel.  Unit-test entry point of the tiled SpMV. */
int sipb_cds_spmv_grid(sipb_ctx* ctx, int dtype, const int64_t* n, int nd, const void* R, const int64_t* offsets,
                       const void* x, void* y, int* used_tiled);
/* The SpMV of the CG exactly as the solver launches it, on a 3-D grid n with Q given either as a stencil-class table
 * `tab` (host TF[27][nd], row cls = (c(k)*3 + c(j))*3 + c(i) as in sipb_problem_set_ata_classes; R = NULL) or as CDS
 * arrays `R` (column-major [N x nd]; tab = NULL).  mode 1: y = Q*x (cg.jl:85, CDS_MVp_MT.jl:9-25) and sums[0] =
 * dot(x, y) (cg.jl:88); mode 2, the CG prologue (argmin_x.jl:33-37, cg.jl:47-61): r = b - Q*x, p = r, x_old = x,
 * sums[0] = dot(b,b), sums[1] = dot(r,r).  tiled = 1: the TMA-staged plane sweep of spmv_tile.cuh (SIPB_E_UNSUPPORTED
 * when the planner rejects the grid; mode 2 has a class-form body only), 0: the generic grid-stride kernels.
 * geom (optional) receives the plan: {ok, TJ, JT, KC, NS, grid, gpl, LPP}.  Unit-test entry point. */
int sipb_tile_probe(sipb_ctx* ctx, int dtype, const int64_t* n, int nd, const int64_t* offsets, const void* tab,
                    const void* R, const void* x, const void* b, int mode, int tiled, void* y, void* r, void* p,
                    void* x_old, double* sums, int* geom);
/* The single-GPU cardinality projection (project_cardinality!.jl:3-21) as the PARSDMM loop runs it: v (M entries) is
 * the input of the y/l update of a one-set problem with the identity operator, l = 0 and rho = gamma = 1 (so pass 1
 * produces s = 0 + v: v itself, except that a -0.0 becomes +0.0 as in the reference's A*x), and `guess`
 * is the previous threshold key the speculative levels are built around.  path 0 / 1: pass 1 without / with the
 * speculative select levels, the search, the tie counts and pass 2 zeroing the ties beyond the quota (deferred tie
 * handling); path 2: the sipb_project sequence (ties zeroed in place).  y receives the projection; stats (optional,
 * int64[8]) = {threshold magnitude key, tie quota, keys equal to the threshold, ties to resolve (0/1), histogram passes
 * that ran, per-chunk tie table valid (0/1), chunk length of the tie kernels, chunk settled in place (-1: none)}.
 * Unit-test entry point. */
int sipb_select_probe(sipb_ctx* ctx, int dtype, int64_t M, const void* v, int64_t k, uint64_t guess, int path, void* y,
                      int64_t* stats);
/* The two vector phases of PARSDMM iteration `it` (1-based) on a finalized single-GPU problem, exactly as sipb_solve
 * runs them: the rhs gather rhs = sum_i A_i'(rho_i y_i + l_i) (rhs_compose.jl), then the y/l update of every set
 * (update_y_l.jl:39-94) fused with the adaptation sums and snapshots (adapt_rho_gamma.jl:41-53, PARSDMM.jl:164-207),
 * the in-loop feasibility (it % 10 == 0), the dual residual and the stop sums (PARSDMM.jl:140-145).  do_adapt is the
 * loop's adaptation flag; it = 1 or do_adapt takes snapshots, do_adapt and it > 1 also reduces the six sums.
 * Inputs (TF arrays of the problem's dtype): m (prod(n)), x (the CG result) and x_old (N each); per set s: l[s], y[s]
 * (= y^k, in/out: y^{k+1} and l^{k+1} on return), y_prev[s] (= y^{k-1}), snapshots[4s..4s+3] = l_hat_0, s_0, l_0, y_0
 * (in/out), rho[s], gamma[s]; the state a previous iteration leaves: l1_inactive_prev[s] (l1 sets: the last sum|v| <=
 * tau), warm[2s..2s+1] (l1 warm thresholds: y update, feasibility), key_thr[s] (cardinality: previous threshold key).
 * Outputs: rhs (N); s[s] (optional, M; sets that keep s = A x: reduction-type and sparse-operator sets); slots (512
 * doubles: the scalar slot table, 16 per set from 0 and the global slots from 256); params[3s..] = theta, scale, fill
 * and iparams[6s..] = key_thr, quota, count_eq, keep_all, keep_none, need_ties of each set's y-update projector;
 * launches (SIPB_N_KERNEL_CLASSES) = launches per kernel class of this call; info[5] = {dual residual fused into the
 * rhs gather (0/1), the iteration the r_dual slots belong to (0: none), stop sums fused (0/1), slots per set, first
 * global slot}.  Overwrites the problem's device vectors.  SIPB_E_UNSUPPORTED on slab problems.  Unit-test entry. */
int sipb_iter_probe(sipb_problem* pb, int it, int do_adapt, const void* m, const void* x, const void* x_old,
                    const double* rho, const double* gamma, void* const* l, void* const* y, void* const* y_prev,
                    void* const* snapshots, const int* l1_inactive_prev, const double* warm, const uint64_t* key_thr,
                    void* rhs, void* const* s, double* slots, double* params, int64_t* iparams, int64_t* launches,
                    int* info);

#ifdef __cplusplus
}
#endif
#endif /* SIPB200_H */
