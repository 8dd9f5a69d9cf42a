/* libthb200 -- C ABI of the B200-native Theseus NLS hot path (linearize -> solve -> retract).
 *
 * This header is the drop-in boundary: plain C, device pointers + sizes + a cudaStream_t, no torch
 * types.  It replaces the pybind11 torch-extension modules of the reference's theseus/extlib and the
 * torch library calls on the per-iteration path.  Every entry point cites the reference interface it
 * replaces (file:line relative to facebookresearch/theseus v0.2.3).
 *
 * Conventions
 *  - All data pointers are DEVICE pointers owned by the caller (torch tensors in the Python host).
 *  - Batch-first, contiguous, row-major layouts identical to the reference's tensors:
 *      SE3 [B,3,4], SO3 [B,3,3], tangent/delta [B,n], A_val [B,nnz], b [B,m], AtA [B,n,n], Atb [B,n].
 *  - Suffix _f64 / _f32 = scalar type.  Index arrays are int32/int64 as stated.
 *  - Return value: 0 on success, <0 = invalid argument (THB_ERR_*), >0 = CUDA runtime error code.
 *    Numerical failure (non-positive pivot) is reported per batch item in an `info` array, like
 *    LAPACK; the Python host raises RuntimeError iff any(info != 0) -- the same exception type the
 *    reference loop catches (theseus/optimizer/nonlinear/nonlinear_least_squares.py:138-152).
 *  - Every kernel is enqueued on `stream`; no entry point synchronises the device (the reference's
 *    BaSpaCho wrappers call cudaDeviceSynchronize() after each kernel, baspacho_solver_cuda.cu:93,168,200).
 */
#ifndef THB200_H_
#define THB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* thb_stream_t; /* == cudaStream_t */

#define THB_OK 0
#define THB_ERR_BAD_ARG (-1)
#define THB_ERR_UNSUPPORTED (-2)
#define THB_ERR_ALLOC (-3)

/* Library identification: returns version (major*10000 + minor*100 + patch) and the compiled SM arch. */
int thb_version(void);
int thb_compiled_arch(void);
/* Number of CUDA kernels this library has launched in this process so far (bench.py's gpu_launches). */
int64_t thb_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Cost-function groups ("schemas").  One group = all cost functions of one type with the same
 * variable types and weight type -- what theseus/core/vectorizer.py:112-404 (Vectorize) builds by
 * torch.cat at every evaluation; here it is a precompiled table of device pointers and offsets.
 * ---------------------------------------------------------------------------------------------- */
enum thb_cost_kind {
  THB_COST_BETWEEN_SE3 = 0, /* theseus/embodied/measurements/between.py:34-45 with SE3 */
  THB_COST_LOCAL_SE3 = 1,   /* theseus/embodied/misc/local_cost_fn.py:40-61 (Local / Difference) with SE3 */
  THB_COST_BETWEEN_SO3 = 2,
  THB_COST_LOCAL_SO3 = 3,
  THB_COST_LOCAL_VECTOR = 4, /* Difference on Vector/Point: e = x - target, J = I (geometry/vector.py) */
  THB_COST_BETWEEN_SE2 = 6,  /* Between with SE2 [B,4] = [x,y,cos,sin] (theseus/geometry/se2.py) */
  THB_COST_LOCAL_SE2 = 7,    /* Difference / Local with SE2 */
  THB_COST_REPROJECTION = 5, /* theseus/embodied/measurements/reprojection.py:54-94: x0 = camera SE3, x1 = Point3,
                                aux = focal_length [Bf,1], aux2 = image_feature_point [Bi,2], aux3 = calib_k1, aux4 = calib_k2 */
  /* theseus/embodied/collision/collision.py: e = max(eps - sdf(xy), 0), dim 1, x0 = pose (Point2 [B,2] / SE2 [B,4]);
   * aux = sdf_origin [Bo,2], aux2 = sdf_data [Bs,sdf_rows,sdf_cols], aux3 = sdf_cell_size [Bc,1], aux4 = cost_eps [Be,1] */
  THB_COST_COLLISION2D_POINT2 = 8,
  THB_COST_COLLISION2D_SE2 = 9,
  /* theseus/embodied/motionmodel/double_integrator.py:16-95: e = [pose1.local(pose2) - dt vel1 ; vel2 - vel1], dim 2 dof;
   * x0 = pose1, x1 = vel1, x2 = pose2, x3 = vel2; aux = dt [Bd,1]; with THB_WEIGHT_GP aux2 = the weight's own dt [Bw,1].
   * VECTOR: poses of Vector kind with dof 2 or 3 (Point2, Point3, Vector); SE2: poses SE2, velocities Vector dof 3. */
  THB_COST_DOUBLE_INTEGRATOR_VECTOR = 10,
  THB_COST_DOUBLE_INTEGRATOR_SE2 = 11
};
enum thb_robust_kind { THB_ROBUST_NONE = 0, THB_ROBUST_WELSCH = 1, THB_ROBUST_HUBER = 2 };
enum thb_weight_kind {
  THB_WEIGHT_SCALE = 0,   /* theseus/core/cost_weight.py:60-93  (ScaleCostWeight, tensor [Bw,1]) */
  THB_WEIGHT_DIAGONAL = 1, /* theseus/core/cost_weight.py:98-139 (DiagonalCostWeight, tensor [Bw,dim]) */
  /* theseus/embodied/motionmodel/double_integrator.py:98-175 (GPCostWeight): w = Qc_inv [Bq,d,d], the weight's dt in aux2 [Bw,1].
   * Weighting is U e, U J with U = chol(W^T)^T, W = [[12/dt^3, -6/dt^2], [-6/dt^2, 4/dt]] (x) Qc_inv, formed in registers as
   * (chol(M) (x) chol(Qc_inv^T))^T (the Cholesky factor is unique).  Accepted by the DOUBLE_INTEGRATOR kinds only (d <= 3). */
  THB_WEIGHT_GP = 2
};
enum thb_var_kind { THB_VAR_SE3 = 0, THB_VAR_SO3 = 1, THB_VAR_VECTOR = 2, THB_VAR_SE2 = 3, THB_VAR_SO2 = 4 };

typedef struct thb_cost_group {
  int32_t kind;        /* enum thb_cost_kind */
  int32_t weight_kind; /* enum thb_weight_kind */
  int32_t K;           /* number of cost functions in the group */
  int32_t dim;         /* error dimension of each cost function (6 for SE3, 3 for SO3, k for Vector) */
  /* device arrays of length K holding DEVICE pointers to each cost function's tensors */
  const void* const* x0;  /* first optimisation variable  [Bx,...] */
  const void* const* x1;  /* second optimisation variable (Between) or NULL */
  const void* const* aux; /* measurement (Between) / target (Local) */
  const void* const* w;   /* cost-weight tensor */
  /* device int32 [K,4]: batch stride in ELEMENTS of x0,x1,aux,w (0 = batch-1 tensor broadcast to B,
   * the broadcasting rule of theseus/core/objective.py:708-724) */
  const int32_t* bstride;
  /* Placement in the reference's batched-CSR Jacobian (theseus/optimizer/sparse_linearization.py:34-84): */
  const int64_t* a_off;    /* device [K]   offset of the cost function's first row in A_val (cost_function_row_block_starts) */
  const int32_t* a_stride; /* device [K]   entries per row (cost_function_stride) */
  const int32_t* bp;       /* device [K,nv] column offset of each variable's block inside a row (cost_function_block_pointers);
                            * nv = 4 for the DOUBLE_INTEGRATOR kinds, 2 for every other kind (unused slots 0) */
  const int32_t* row0;     /* device [K]   first row of the cost function in b */
  /* further auxiliary tensors of schemas that need them (NULL otherwise) + their batch strides, device int32 [K,3] */
  const void* const* aux2;
  const void* const* aux3;
  const void* const* aux4;
  const int32_t* bstride2;
  /* Robust wrapper (theseus/core/robust_cost_function.py:87-135, robust_loss.py:33-52): 0 = none, 1 = Welsch, 2 = Huber.
   * log_radius: device [K] pointers to the log_loss_radius tensors [Br,1]; bstride_lr: device int32 [K]. */
  int32_t robust_kind;
  int32_t reserved0;
  const void* const* log_radius;
  const int32_t* bstride_lr;
  /* Fields appended after the ones above (whose offsets are unchanged):
   * third and fourth optimisation variable (DOUBLE_INTEGRATOR kinds: pose2, vel2) or NULL, their batch strides device int32 [K,2] */
  const void* const* x2;
  const void* const* x3;
  const int32_t* bstride3;
  /* grid shape [sdf_rows, sdf_cols] shared by every cost function of a COLLISION2D group (0 for other kinds) */
  int32_t sdf_rows;
  int32_t sdf_cols;
} thb_cost_group;

/* Fused residual + analytic Jacobian + weighting for every (cost function, batch item) of a group;
 * writes A_val[B,nnz] / b[B,m] (b = -weighted error) in the layout of SparseLinearization.
 * Replaces: Vectorize._vectorize (core/vectorizer.py:382-404), Between/Local.jacobians,
 * CostWeight.weight_jacobians_and_error (core/cost_weight.py:81-90,125-136),
 * SparseLinearization._linearize_jacobian_impl (optimizer/sparse_linearization.py:102-140). */
int thb_linearize_group_f64(const thb_cost_group* g, int64_t B, double* A_val, int64_t nnz, double* b, int64_t m,
                            thb_stream_t stream);
int thb_linearize_group_f32(const thb_cost_group* g, int64_t B, float* A_val, int64_t nnz, float* b, int64_t m,
                            thb_stream_t stream);

/* Residual-only pass: partial[c, b] = sum over the c-th chunk of cost functions of (w*e)^2 / 2.
 * `partial` has room for thb_error_num_chunks(K) rows of B.  The caller sums the rows in order
 * (thb_lm_control does) so the reduction is deterministic.
 * Replaces: Objective.error / error_metric (core/objective.py:562-641) through the vectorised
 * WEIGHTED_ERROR pass (core/vectorizer.py:406-407). */
int thb_error_num_chunks(int32_t K);
int thb_error_group_f64(const thb_cost_group* g, int64_t B, double* partial, thb_stream_t stream);
int thb_error_group_f32(const thb_cost_group* g, int64_t B, float* partial, thb_stream_t stream);
/* err[b] = sum_c partial[c,b] (fixed order). */
int thb_error_reduce_f64(const double* partial, int32_t num_chunks, int64_t B, double* err, thb_stream_t stream);
int thb_error_reduce_f32(const float* partial, int32_t num_chunks, int64_t B, float* err, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Retract: out_i[b] = X_i[b] * exp(step * delta[b, col_i : col_i+dof_i])   (Vector: x + step*delta)
 * for every optimisation variable; batch items with ignore[b] != 0 keep X_i[b].
 * Replaces: Objective.retract_vars_sequence (core/objective.py:873-914),
 * Vectorize._vectorized_retract_optim_vars (core/vectorizer.py:410-469), LieGroup._retract_impl
 * (geometry/lie_group.py:197-198), Variable.update masking (core/variable.py:65-69).
 * ---------------------------------------------------------------------------------------------- */
typedef struct thb_var_table {
  int32_t N;                 /* number of optimisation variables */
  const void* const* x;      /* device [N] pointers to current tensors  [B,...] */
  void* const* out;          /* device [N] pointers to output tensors   [B,...] */
  const int32_t* kind;       /* device [N] enum thb_var_kind */
  const int32_t* col;        /* device [N] first column in delta (Linearization.var_start_cols) */
  const int32_t* dof;        /* device [N] */
} thb_var_table;

int thb_retract_f64(const thb_var_table* vt, int64_t B, const double* delta, int64_t n, double step,
                    const uint8_t* ignore /* [B] or NULL */, thb_stream_t stream);
int thb_retract_f32(const thb_var_table* vt, int64_t B, const float* delta, int64_t n, float step,
                    const uint8_t* ignore, thb_stream_t stream);
/* x_i[b] <- out_i[b] where keep_old[b] == 0  (objective.update(..., batch_ignore_mask=reject),
 * nonlinear_least_squares.py:361; core/variable.py:65-69). */
int thb_commit_f64(const thb_var_table* vt, int64_t B, const uint8_t* keep_old, thb_stream_t stream);
int thb_commit_f32(const thb_var_table* vt, int64_t B, const uint8_t* keep_old, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Gram assembly from the batched-CSR Jacobian: AtA blocks and Atb without atomics.
 * The block structure is precomputed on the host (theseus_b200/structure.py): for every output
 * entry e (one scalar of one variable-pair block) a list of contributing cost functions.
 * Replaces: DenseLinearization._linearize_hessian_impl (optimizer/dense_linearization.py:58-62,
 * At.bmm(A) / At.bmm(b)); extlib mult_MtM / add_MtM / tmat_vec (extlib/mat_mult.cu:36-79,216-243,
 * extlib/baspacho_solver_cuda.cu:96-134).
 * ---------------------------------------------------------------------------------------------- */
typedef struct thb_gram_plan {
  int64_t num_entries;        /* NE: scalar entries of all (lower-triangular) variable-pair blocks */
  const int32_t* ent_blk;     /* device [NE] block id of the entry */
  const int16_t* ent_p;       /* device [NE] row inside the block */
  const int16_t* ent_q;       /* device [NE] col inside the block */
  const int64_t* blk_out;     /* device [NB] offset of block element (0,0) in one batch item's output */
  const int32_t* blk_ld;      /* device [NB] leading dimension of the block in the output */
  const int64_t* blk_mirror;  /* device [NB] offset of the transposed block's (0,0), or -1 */
  const int32_t* blk_cptr;    /* device [NB+1] CSR pointer into the contribution arrays */
  const int64_t* c_off;       /* device [NC] A_val offset of the contributing cost function's first row */
  const int32_t* c_stride;    /* device [NC] */
  const int32_t* c_rows;      /* device [NC] */
  const int32_t* c_bpa;       /* device [NC] block pointer of the block-row variable */
  const int32_t* c_bpb;       /* device [NC] block pointer of the block-col variable */
  /* Atb plan: one entry per column */
  int64_t n;                  /* num_cols */
  const int32_t* col_cptr;    /* device [n+1] */
  const int64_t* cc_off;      /* device [NCC] A_val offset of (first row, this column) */
  const int32_t* cc_stride;   /* device [NCC] */
  const int32_t* cc_rows;     /* device [NCC] */
  const int32_t* cc_row0;     /* device [NCC] first row in b */
  /* per-block view (block-per-thread kernels: thb_sparse_lane_gram_f64) */
  int64_t num_blocks;         /* NB */
  const int32_t* blk_rows;    /* device [NB] rows of the block (its columns are blk_ld for packed block storage) */
  const int32_t* blk_cols;    /* device [NB] columns of the block */
  /* block-per-thread Gram kernels (one thread = one whole block of one item): blocks grouped by shape.  num_segments == 0 (some block
   * shape outside {1,2,3,6} x {1,2,3,6}): the entry-per-thread kernel runs instead. */
  int64_t num_segments;
  const int32_t* segments;    /* HOST [num_segments,4] = (rows, cols, begin, end) into blk_order */
  const int32_t* blk_order;   /* device [NB] block ids sorted by shape */
} thb_gram_plan;

/* out[b*out_bstride + ...] receives the blocks (dense AtA: out_bstride = n*n, caller pre-zeroes via
 * thb_fill_zero); Atb[B,n]; diag[B,n] (optional, may be NULL) receives diag(AtA). */
int thb_gram_f64(const thb_gram_plan* p, int64_t B, const double* A_val, int64_t nnz, const double* b, int64_t m,
                 double* out, int64_t out_bstride, double* Atb, double* diag, thb_stream_t stream);
int thb_gram_f32(const thb_gram_plan* p, int64_t B, const float* A_val, int64_t nnz, const float* b, int64_t m,
                 float* out, int64_t out_bstride, float* Atb, float* diag, thb_stream_t stream);
int thb_fill_zero(void* ptr, int64_t bytes, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Batched dense Cholesky factor + solve with fused LM damping.
 *   M_b = AtA_b ; diag(M_b) <- diag(M_b) * (1 + alpha_b) + beta_b ; L_b L_b^T = M_b ; x_b = M_b^-1 rhs_b
 * (alpha,beta) follow theseus/optimizer/linear/utils.py:14-33; ellipsoidal: (lambda, eps), spherical (0, lambda).
 * AtA is read-only (LM needs its diagonal afterwards, levenberg_marquardt.py:185-190).
 * Workspace: thb_potrf_workspace_bytes(B, n).  info[b] = 0, or k>0 if the k-th pivot was not positive.
 * Replaces: DenseSolver._apply_damping (optimizer/linear/dense_solver.py:38-64) +
 * torch.linalg.cholesky + torch.cholesky_solve (dense_solver.py:159-161).
 * ---------------------------------------------------------------------------------------------- */
int64_t thb_potrf_workspace_bytes(int64_t B, int64_t n);
/* Factor only / solve only against the factor left in `workspace` by thb_potrf_f64 (any number of right-hand
 * sides, e.g. the backward pass of the solve, theseus/optimizer/autograd/: the factor is reused). */
int thb_potrf_f64(const double* AtA, const double* alpha, const double* beta, int32_t* info, int64_t B, int64_t n,
                  void* workspace, int64_t workspace_bytes, thb_stream_t stream);
int thb_potrs_f64(const double* rhs, double* x, int64_t B, int64_t n, const void* workspace, int64_t workspace_bytes,
                  thb_stream_t stream);
int thb_potrf_potrs_f64(const double* AtA, const double* rhs, const double* alpha, const double* beta, double* x,
                        int32_t* info, int64_t B, int64_t n, void* workspace, int64_t workspace_bytes,
                        thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Batched block-sparse Cholesky over a batch-shared symbolic plan (host analysis: theseus_b200/sparse.py).
 * Replaces theseus.extlib.baspacho_solver (SymbolicDecomposition / NumericDecomposition.{add_MtM,damp,factor,solve},
 * extlib/baspacho_solver.cpp:326-358, baspacho_solver_cuda.cu), cusolverRf refactor/solve
 * (extlib/cusolver_lu_solver.cpp:252-310) and the CHOLMOD per-item loop (optimizer/autograd/cholmod_sparse_autograd.py:25-61).
 *   factor storage  [B, data_size] fp64: per elimination column the diagonal block then its sub-diagonal blocks, row-major
 *                   (filled with the AtA blocks by thb_gram_f64 using a plan whose block offsets point into this storage)
 *   winv            [B, winv_size] fp64: inverse of every diagonal block of L (turns the triangular solves into mat-vecs)
 * All index arrays are device arrays shared by the whole batch.
 * ---------------------------------------------------------------------------------------------- */
typedef struct thb_sparse_plan {
  int32_t N;          /* number of variable blocks */
  int32_t num_levels; /* elimination-tree levels */
  int32_t max_dim;    /* largest block dimension (<= 16) */
  int32_t reserved;
  int64_t n;          /* scalar dimension */
  int64_t data_size;
  int64_t winv_size;
  const int32_t* dims;      /* [N] block size per elimination position */
  const int32_t* col_start; /* [N] first scalar column (ORIGINAL order) of the variable at this position */
  const int32_t* pstart;    /* [N] first scalar index in the permuted vector */
  const int64_t* winv_off;  /* [N] */
  const int64_t* diag_off;  /* [N] offset of the diagonal block */
  const int64_t* up_a;      /* update pairs: offset of L_ik */
  const int64_t* up_b;      /*               offset of L_jk */
  const int32_t* up_k;      /*               dk */
  const int64_t* u_ptr;     /* [L+1] work items of stage U per level */
  const int64_t* u_tgt; const int16_t* u_r; const int16_t* u_c; const int16_t* u_ld; const int64_t* u_p0; const int64_t* u_p1;
  const int64_t* f_ptr;     /* [L+1] stage F (diagonal blocks) */
  const int64_t* f_off; const int32_t* f_dim; const int64_t* f_w; const int32_t* f_col;
  const int64_t* t_ptr;     /* [L+1] stage T (block rows of sub-diagonal blocks) */
  const int64_t* t_off; const int16_t* t_r; const int16_t* t_dim; const int64_t* t_w;
  const int64_t* s_ptr;     /* [L+1] columns per level (solve) */
  const int32_t* s_col;
  const int64_t* fr_ptr; const int64_t* fr_off; const int32_t* fr_k; /* row lists (forward substitution) */
  const int64_t* bc_ptr; const int64_t* bc_off; const int32_t* bc_i; /* column lists (backward substitution) */
} thb_sparse_plan;

/* diag(M_b) <- diag(M_b) * (1 + alpha_b) + beta_b on the factor storage (NumericDecomposition.damp) */
int thb_sparse_damp_f64(const thb_sparse_plan* p, double* factor, const double* alpha, const double* beta, int64_t B,
                        thb_stream_t stream);
/* in-place L L^T = M (NumericDecomposition.factor); info[b] = 0 or 1 + permuted index of the first bad pivot */
int thb_sparse_factor_f64(const thb_sparse_plan* p, double* factor, double* winv, int32_t* info, int64_t B, thb_stream_t stream);
/* x = M^-1 rhs in the ORIGINAL variable order (NumericDecomposition.solve incl. scramble/unscramble); work: [B,n] scratch */
int thb_sparse_solve_f64(const thb_sparse_plan* p, const double* factor, const double* winv, const double* rhs, double* x,
                         double* work, int64_t B, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Symbolic analysis (host code, thb_symbolic.cu): ordering, fill, elimination-tree levels, factor layout and the work lists of
 * both numeric back ends.  Replaces SymbolicDecomposition(param_size i64[N], sparse_struct_ptrs i64[N+1], sparse_struct_inds i64,
 * device) of theseus/extlib/baspacho_solver.cpp:259-319 (and cusolver's symamd + csrluAnalysis, extlib/cusolver_lu_solver.cpp:95-196).
 * All three input arrays are HOST arrays, exactly what baspacho_sparse_solver.py:93-113 builds.  ordering: 0 = minimum degree,
 * 1 = natural.  The handle owns named host arrays (the fields of thb_sparse_plan / thb_sparse_lane_plan, the latter prefixed
 * "ln_", plus order / pos / level / struct_ptr / struct_idx / blk_off / blk_i / blk_j / blk_rows / blk_cols / up_ptr) and the
 * scalars N, n, data_size, winv_size, nnz_L, flops, levels, max_front, num_updates.  The caller uploads the arrays it needs.
 * ---------------------------------------------------------------------------------------------- */
typedef struct thb_symbolic thb_symbolic;
int thb_symbolic_create(const int64_t* param_size, int64_t N, const int64_t* blk_ptrs, const int64_t* blk_inds, int32_t ordering,
                        thb_symbolic** out);
void thb_symbolic_destroy(thb_symbolic* s);
int64_t thb_symbolic_array_count(const thb_symbolic* s, const char* name);      /* elements, -1 if unknown */
int32_t thb_symbolic_array_elem_bytes(const thb_symbolic* s, const char* name); /* 2, 4 or 8 */
int thb_symbolic_array_copy(const thb_symbolic* s, const char* name, void* dst, int64_t dst_bytes);
double thb_symbolic_stat(const thb_symbolic* s, const char* name);

/* ------------------------------------------------------------------------------------------------
 * Block-sparse Cholesky, batch-lane layout (thb_sparse_lane.cu): the same four BaSpaCho operations
 * (add_MtM / damp / factor / solve, extlib/baspacho_solver.cpp:93-257) for large batches.  The factor storage is
 * INTERLEAVED over the batch: element e of item b lives at factor[e * Bp + b], Bp = thb_sparse_lane_padded_batch(B)
 * (B rounded up to 32), so one warp runs one block operation for 32 batch items with coalesced accesses.
 *   factor [data_size, Bp] fp64   same per-item element order as thb_sparse_plan (blocks of L, row-major)
 *   diagl  [diag_size, Bp] fp64   Cholesky factors of the diagonal blocks (row-major d x d, RECIPROCAL diagonal)
 *   work   [n, Bp]         fp64   permuted right-hand side / solution
 * Block sizes must be in {1,2,3,6} (THB_ERR_UNSUPPORTED otherwise: use the thb_sparse_plan entry points).
 * `launches` is a HOST array [num_launches][5] = (kind, di, dj, begin, end) in execution order (level by level;
 * kinds below); every other pointer is a device array.  Elimination-tree levels are separate kernel launches.
 * ---------------------------------------------------------------------------------------------- */
enum { THB_LANE_U = 0, THB_LANE_T = 1, THB_LANE_S = 2, THB_LANE_UH = 3, THB_LANE_TU = 4 /* tiled external updates, below */ };
typedef struct thb_sparse_lane_plan {
  int64_t N;            /* number of variable blocks */
  int64_t n;            /* scalar dimension */
  int64_t data_size;    /* doubles per batch item in `factor` */
  int64_t diag_size;    /* doubles per batch item in `diagl` (sum of d^2) */
  int64_t num_launches;
  const int32_t* launches;  /* HOST [num_launches,5] */
  const int32_t* dims;      /* [N] block size per elimination position */
  const int32_t* col_start; /* [N] first scalar column (ORIGINAL order) */
  const int32_t* pstart;    /* [N] first scalar index in the permuted vector */
  const int64_t* dl_off;    /* [N] offset of the diagonal factor in diagl */
  const int64_t* diag_off;  /* [N] offset of the diagonal block in factor */
  const int64_t* up_a; const int64_t* up_b; const int32_t* up_k;    /* update pairs (offset of L_ik, of L_jk, dk) */
  const int64_t* u_tgt; const int64_t* u_p0; const int64_t* u_p1;   /* U items: target offset, pair range */
  const int64_t* t_off; const int64_t* t_diag; const int64_t* t_dl; /* T items: block, its column's diagonal block, diagl slot */
  const int32_t* t_pstart;                                          /*          first permuted scalar of the column (info) */
  const int32_t* s_col;                                             /* S items: columns */
  /* row lists (forward substitution): per column j the blocks L_jk: offset, first permuted scalar of k, dim of k */
  const int64_t* fr_ptr; const int64_t* fr_off; const int32_t* fr_p; const int32_t* fr_d;
  /* column lists (backward substitution): per column j the blocks L_ij: offset, first permuted scalar of i, dim of i */
  const int64_t* bc_ptr; const int64_t* bc_off; const int32_t* bc_p; const int32_t* bc_d;
} thb_sparse_lane_plan;

int64_t thb_sparse_lane_padded_batch(int64_t B);
/* add_MtM: AtA blocks -> factor (lane layout); the caller zero-fills factor first (fill-in blocks start at 0) */
int thb_sparse_lane_gram_f64(const thb_gram_plan* g, int64_t B, const double* A_val, int64_t nnz, double* factor, thb_stream_t stream);
int thb_sparse_lane_damp_f64(const thb_sparse_lane_plan* p, double* factor, const double* alpha, const double* beta, int64_t B,
                             thb_stream_t stream);
/* info[b] = 0 or 1 + permuted index of a non-positive pivot */
int thb_sparse_lane_factor_f64(const thb_sparse_lane_plan* p, double* factor, double* diagl, int32_t* info, int64_t B,
                               thb_stream_t stream);
/* Dense root of the elimination tree (sparse.py:root_split; opt-in `layout="lane_root"` of the Python solver, new in round 1 and
 * not yet profiled): the top chain of the tree is a dense trailing block [nt, nt]; the lane kernels run on the columns below the
 * cut (a thb_sparse_lane_plan whose launch list stops there and ends with the root's assembly updates), the root itself goes
 * through thb_potrf_f64 / thb_potrs_f64.  All pointers device arrays except `segments` (HOST, [num_segments,3] = block size, begin,
 * end into root_cols). */
typedef struct thb_sparse_lane_root {
  int64_t num_blocks;   /* blocks (i, j), i >= j >= cut, of the root */
  int64_t num_cols;     /* root columns */
  int64_t nt;           /* scalar size of the root */
  int64_t root_start;   /* first permuted scalar index of the root */
  int64_t num_segments;
  const int32_t* segments;  /* HOST */
  const int64_t* rb_off; const int32_t* rb_row; const int32_t* rb_col; const int32_t* rb_di; const int32_t* rb_dj; /* [num_blocks] */
  const int64_t* rf_p0; const int64_t* rf_p1;  /* [num_cols] bottom part of each root column's row list (indices into fr_*) */
  const int32_t* root_cols;                    /* [num_cols] elimination positions, grouped by block size (see segments) */
  const int32_t* root_dims;                    /* [num_cols] block sizes */
} thb_sparse_lane_root;
/* S [B, nt, nt] (batch-major, row-major; lower triangle = the assembled root, strict upper = 0) <- lane factor storage */
int thb_sparse_lane_root_gather_f64(const thb_sparse_lane_root* r, const double* factor, double* S, int64_t B, thb_stream_t stream);
/* forward / backward substitution of the columns in the plan's launch list only (thb_sparse_lane_solve_f64 = forward then backward) */
int thb_sparse_lane_forward_f64(const thb_sparse_lane_plan* p, const double* factor, const double* diagl, const double* rhs, double* work,
                                int64_t B, thb_stream_t stream);
int thb_sparse_lane_backward_f64(const thb_sparse_lane_plan* p, const double* factor, const double* diagl, double* work, double* x, int64_t B,
                                 thb_stream_t stream);
/* rhs_dense [B, nt] = permuted rhs of the root minus the contribution of the bottom columns (after thb_sparse_lane_forward_f64) */
int thb_sparse_lane_root_rhs_f64(const thb_sparse_lane_plan* p, const thb_sparse_lane_root* r, const double* factor, const double* rhs,
                                 const double* work, double* rhs_dense, int64_t B, thb_stream_t stream);
/* root solution x_dense [B, nt] -> work (for thb_sparse_lane_backward_f64) and x [B, n] (original order) */
int thb_sparse_lane_root_scatter_f64(const thb_sparse_lane_plan* p, const thb_sparse_lane_root* r, const double* x_dense, double* work, double* x,
                                     int64_t B, thb_stream_t stream);
/* Tiled external updates (opt-in layout `lane_tiled`; host lists: theseus_b200/sparse.py:tile_lane_lists).  The columns of a
 * fundamental supernode ("chain", cut into pieces of <= 4 columns) share their row structure, so the left-looking updates that reach
 * a piece from outside it (source column k before the piece: BaSpaCho's per-supernode "eliminateBoard" work, baspacho_solver_cuda.cu
 * via NumericDecomposition::factor, extlib/baspacho_solver.cpp:171-199) are done per TILE of 4 rows x 4 columns of 6x6 blocks by ONE
 * CTA of 16 warps (warp = one target block x 32 batch lanes, accumulators in registers): per source column k the <= 8 source blocks
 * L_(row),k and L_(column),k are staged ONCE in shared memory (cp.async, double buffered) and used by every target that has both,
 * instead of being streamed from L2/HBM once per update pair.  A launch row (THB_LANE_TU, 6, 6, begin, end) of the plan's launch
 * list runs tiles [begin, end).  All pointers device arrays. */
#define THB_TILE_ROWS 4
#define THB_TILE_COLS 4
typedef struct thb_sparse_lane_tiles {
  int64_t num_tiles, num_steps;
  const int64_t* tile_tgt;   /* [num_tiles, 16] offset of target block (row slot a, column slot b) at a*4+b, -1 if absent */
  const int64_t* step_ptr;   /* [num_tiles+1] k steps of a tile */
  const int64_t* step_src;   /* [num_steps, 8] offsets of L_(row slot 0..3),k then L_(column slot 0..3),k; -1 = structurally zero */
} thb_sparse_lane_tiles;
/* thb_sparse_lane_factor_f64 for a launch list that may contain THB_LANE_TU rows */
int thb_sparse_lane_factor_tiled_f64(const thb_sparse_lane_plan* p, const thb_sparse_lane_tiles* t, double* factor, double* diagl,
                                     int32_t* info, int64_t B, thb_stream_t stream);
/* Supernodal substitutions (opt-in; host lists: theseus_b200/sparse.py:piece_solve_lists).  A work item is a PIECE of <= 4 consecutive
 * columns of a fundamental supernode with equal block size: their external sums are independent (forward) or share every x_i (backward),
 * the dense triangle inside the piece is solved by one warp -- BaSpaCho's per-supernode solveL / solveLt (NumericDecomposition::solve,
 * extlib/baspacho_solver.cpp:201-246).  One launch per piece level and block size instead of one per elimination-tree level.
 * Same contract as thb_sparse_lane_forward_f64 / _backward_f64 (which they replace for the columns the pieces cover: all, or the columns
 * below a dense root).  Device arrays except `launches` (HOST, [num_launches, 3] = block size, begin, end into `order`). */
typedef struct thb_sparse_lane_pieces {
  int64_t num_pieces, num_launches;
  const int32_t* launches;      /* HOST */
  const int64_t* first;         /* [num_pieces] first column (elimination position) */
  const int32_t* width;         /* [num_pieces] 1..4 columns */
  const int64_t* fr_ext_end;    /* [N] end (index into fr_off) of the prefix of column j's row list that lies before its piece */
  const int64_t* bc_int_end;    /* [N] end (index into bc_off) of the prefix of column j's column list that lies inside its piece */
  const int64_t* order;         /* [num_pieces] pieces sorted by (level, block size) */
} thb_sparse_lane_pieces;
int thb_sparse_lane_piece_forward_f64(const thb_sparse_lane_plan* p, const thb_sparse_lane_pieces* pc, const double* factor, const double* diagl,
                                      const double* rhs, double* work, int64_t B, thb_stream_t stream);
int thb_sparse_lane_piece_backward_f64(const thb_sparse_lane_plan* p, const thb_sparse_lane_pieces* pc, const double* factor, const double* diagl,
                                       double* work, double* x, int64_t B, thb_stream_t stream);
/* rhs, x: [B, n] row-major in the ORIGINAL variable order (scramble / unscramble folded into the substitutions) */
int thb_sparse_lane_solve_f64(const thb_sparse_lane_plan* p, const double* factor, const double* diagl, const double* rhs,
                              double* x, double* work, int64_t B, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Levenberg-Marquardt control (device-resident accept/reject + damping update).
 *   den = 1/2 sum_j d_j (lam_eff_j d_j + Atb_j), d = step*delta, lam_eff = lam*diag(AtA) if ellipsoidal else lam
 *   rho = (err_prev - err_new)/den ; reject = rho <= damping_accept
 *   lam <- clamp(reject ? lam*up : lam/down, 1e-7, 1e7)
 * Replaces LevenbergMarquardt._check_accept (optimizer/nonlinear/levenberg_marquardt.py:172-201).
 * Also folds: err[b] <- reject ? err_prev : err_new; counts of rejected items -> stats[0].
 * ---------------------------------------------------------------------------------------------- */
int thb_lm_control_f64(const double* delta, const double* Atb, const double* diag, int64_t B, int64_t n, double step,
                       const double* err_prev, const double* err_new, double* lam, int32_t ellipsoidal,
                       double damping_accept, double down_ratio, double up_ratio, uint8_t* reject,
                       double* err_out, int32_t* stats, thb_stream_t stream);

int thb_lm_control_f32(const float* delta, const float* Atb, const float* diag, int64_t B, int64_t n, float step,
                       const float* err_prev, const float* err_new, float* lam, int32_t ellipsoidal, float damping_accept,
                       float down_ratio, float up_ratio, uint8_t* reject, float* err_out, int32_t* stats, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Dense batched Gram for GENUINELY dense Jacobians (AutoDiffCostFunction with dim >> dof):  AtA [B,n,n] = A^T A,  A [B,m,n] row-major.
 * Replaces `At.bmm(A)` of theseus/optimizer/dense_linearization.py:58-62 where the block-sparse Gram (thb_gram_f64) has nothing to skip.
 * TMA-staged tiles (one 3-D tensor map over [B,m,n], cp.async.bulk.tensor + mbarrier ring) feeding the FP64 tensor pipe (mma.sync DMMA;
 * tcgen05 has no fp64 kind); the full symmetric matrix is written.  n must be even and A 16-byte aligned (else THB_ERR_UNSUPPORTED:
 * the Python host then stays on thb_gram_f64).
 * ---------------------------------------------------------------------------------------------- */
int thb_gram_dense_f64(const double* A, double* AtA, int64_t B, int64_t m, int64_t n, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * MULTIFRONTAL (supernodal) batched block-sparse Cholesky -- layout "front" of the Python BaspachoSparseSolver.
 * Replaces BaSpaCho's batched supernodal factor / solve behind NumericDecomposition::factor / solve
 * (theseus/extlib/baspacho_solver_cuda.cu:203-214, 282-287; baspacho_solver.cpp:291) for batches that share one structure.
 * The symbolic side (theseus_b200/frontal.py: nested-dissection / minimum-degree ordering, relaxed supernode amalgamation ->
 * FRONTS, depth schedule) hands over flat per-front arrays; all pointers are device arrays.
 *   front t: w pivot scalars (contiguous in the permuted vector from f_first[t]), b border rows, r = w + b.
 *   factor storage of one item: per front a dense ROW-MAJOR r x w panel at f_panel_off[t] (leading dimension w):
 *     rows 0..w-1 the pivot block (lower triangle = L_tt), rows w.. the border rows L[border, pivots].
 *     add_MtM scatters AtA into the same panels (thb_gram_f64 with frontal.FrontPlan.gram_out_offsets, item-major
 *     [B, data_size]); the caller zero-fills first.  Damping (alpha, beta) is applied while a panel is loaded.
 *   update matrices (Schur complements) live for one depth step in arena [2][B][arena_size] (parity = depth & 1):
 *     small fronts: lower triangle of a b x b matrix at f_cb_off[t], leading dimension f_cb_ld[t];
 *     big fronts (f_class == 3): the whole padded front matrix F [np x np] at f_fr_off[t] (pivot columns padded to f_wpad[t],
 *     a multiple of 64, identity on the padding), factored in place by the DMMA dense kernel in partial mode
 *     (thb_potrf_partial_inplace_f64); its trailing block IS the update matrix (f_cb_off / f_cb_ld point into it).
 *   child -> parent maps: f_rel[rel_ptr[c] .. rel_ptr[c+1]) = local row index in the parent front of child c's border rows.
 * `launches` is a HOST array [num_launches][12] (int64) in factorisation order (deepest fronts first):
 *   (depth, class, begin, count [into sched], dynamic smem bytes of the factor kernel, largest front of the launch [np for class 3],
 *    largest panel (r * w) of the launch [pivot block columns for class 3], f_fr_off, f_first [info base], front index, w, b) -- the last six for class-3 launches (one front each).
 * No atomics on data: results are bitwise reproducible and independent of the batch size.
 * ---------------------------------------------------------------------------------------------- */
typedef struct thb_front_plan {
  int64_t S;            /* number of fronts */
  int64_t n;            /* scalar dimension */
  int64_t data_size;    /* doubles per item in `factor` */
  int64_t arena_size;   /* doubles per item and parity in `arena` */
  int64_t varena_size;  /* doubles per item and parity in `varena` (border vectors of the forward substitution) */
  const int32_t* f_w; const int32_t* f_b; const int32_t* f_first; const int32_t* f_class;
  const int32_t* f_wpad; const int32_t* f_np; const int32_t* f_cb_ld; const int32_t* f_depth;
  const int64_t* f_panel_off; const int64_t* f_cb_off; const int64_t* f_fr_off; const int64_t* f_u_off;
  const int32_t* child_ptr; const int32_t* child_list;   /* children of front t: child_list[child_ptr[t] .. child_ptr[t+1]) */
  const int64_t* rel_ptr; const int32_t* f_rel;
  const int64_t* rows_ptr; const int32_t* f_rows;        /* border rows of front t as permuted scalar indices */
  const int32_t* sched;                                  /* [S] fronts in launch order */
  const int32_t* perm;                                   /* [n] original scalar column of permuted scalar p */
  /* per CHILD front t of parent p: c_jw[t] = number of t's border rows that are pivots of p; c_sp[c_sp_ptr[t] + s] = first border row
   * of t whose image lies at or after border row 32 s of p (s = 0 .. ceil(b_p / 32)): what the kernels would otherwise binary-search */
  const int32_t* c_jw; const int64_t* c_sp_ptr; const int32_t* c_sp;
  /* per CHILD front t of parent p: c_inv[c_inv_ptr[t] + l] = border row of t whose image is row l of p's front (l < r_p), or -1:
   * the shared-memory kernel GATHERS the children's update matrices through it (no scatter, no barriers) */
  const int64_t* c_inv_ptr; const int32_t* c_inv;
  /* flat descriptors of the shared-memory kernel: fd[q] (q = position in sched) = (front, w, b, f_first, f_panel_off, f_cb_off, f_cb_ld,
   * child_begin | nchildren << 32);  pc[child_begin + k] = (f_cb_off, f_cb_ld | b << 32, first and last front row reached, offset of the inverse
   * map in c_inv, f_u_off) of the front's k-th child */
  const int64_t* fd; const int64_t* pc;
  /* panel map: pmap[o] for offset o of one item's factor storage = offset of that AtA entry in the COMPACT block storage written by
   * thb_gram_f64 (frontal.FrontPlan.gram_compact_offsets), or -1 for fill-in.  With it the factorisation reads AtA where it is
   * non-zero and the panels need no zero fill. */
  const int32_t* pmap;
} thb_front_plan;

#define THB_FRONT_LAUNCH_COLS 12
/* dynamic shared memory (bytes) the shared-memory factor kernel needs for a front with w pivots, b border rows and nchildren children
 * (the padded panel + the children's inverse maps) */
int64_t thb_front_small_smem_bytes(int32_t w, int32_t b, int32_t nchildren);
/* factor: `factor` [B, data_size] receives L.  Input: either ata != NULL = compact AtA blocks [B, ata_stride] read through p->pmap (no zero
 * fill, no scatter into the panels), or ata == NULL = the panels of `factor` already hold AtA + zeros (the extlib flow); dense_ws: workspace of
 * thb_potrf_partial_workspace_bytes(B, max np) bytes (may be NULL when there is no class-3 front);
 * info[b] = 0 or 1 + permuted index of a non-positive pivot (cleared here). */
int thb_front_factor_f64(const thb_front_plan* p, const int64_t* launches, int64_t num_launches, double* factor, const double* ata,
                         int64_t ata_stride, const double* alpha, const double* beta, double* arena, void* dense_ws, int64_t dense_ws_bytes,
                         int32_t* info, int64_t B, thb_stream_t stream);
/* x = (L L^T)^-1 rhs; rhs, x [B, n] in ORIGINAL column order; work [B, n], varena [2, B, varena_size] scratch */
int thb_front_solve_f64(const thb_front_plan* p, const int64_t* launches, int64_t num_launches, const double* factor, const double* rhs,
                        double* x, double* work, double* varena, int64_t B, thb_stream_t stream);
int64_t thb_potrf_partial_workspace_bytes(int64_t B, int64_t np);
int thb_potrf_partial_inplace_f64(double* F, int64_t bstride, int64_t np, int32_t nb_piv, int32_t w_real, int32_t n_real, int32_t info_base,
                                  int32_t* info, int64_t B, void* workspace, int64_t workspace_bytes, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Batched CSR helpers (same semantics as theseus/extlib/mat_mult.cu:359-400, int64 indices):
 *   thb_mat_vec : y[b,row]  = sum_k A_val[b,k] v[b,col_k]          (mat_vec,  mat_mult.cu:134-214)
 *   thb_tmat_vec: y[b,col] += A_val[b,k] v[b,row]  (deterministic) (tmat_vec, mat_mult.cu:216-295)
 * ---------------------------------------------------------------------------------------------- */
int thb_mat_vec_f64(int64_t B, int64_t num_rows, int64_t num_cols, const int64_t* row_ptr, const int64_t* col_ind,
                    const double* A_val, const double* v, double* y, thb_stream_t stream);
int thb_tmat_vec_f64(int64_t B, int64_t num_rows, int64_t num_cols, const int64_t* row_ptr, const int64_t* col_ind,
                     const double* A_val, const double* v, double* y, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Backward of the linear solve x = (AtA + D)^-1 At b with respect to A_val [B,nnz] and b [B,m]
 * (optimizer/autograd/common.py:11-48 compute_A_grad -- a Python loop over the m rows in the reference -- and
 * the backward() of baspacho_sparse_autograd.py:117-168 / cholmod_sparse_autograd.py:64-110 / lu_cuda_sparse_autograd.py:86-155).
 * H [B,n] = (AtA + D)^-1 grad_x is obtained by the caller with the factor of the forward pass (thb_potrs_f64 /
 * thb_sparse_solve_f64 / thb_sparse_lane_solve_f64).  Then
 *   b_grad[b,r]  = (A H)[r]
 *   A_grad[b,k]  = (b - A x)[r] H[c] - (A H)[r] x[c] - 2 alpha_b H[c] x[c] A[k]        (entry k = (r,c))
 * detach_hessian != 0 : A_grad[b,k] = b[r] H[c]  (the reference's _detach_hessian GN step).
 * alpha may be NULL (no multiplicative damping); A_grad or b_grad may be NULL.
 * ---------------------------------------------------------------------------------------------- */
int thb_solve_backward_f64(int64_t B, int64_t num_rows, int64_t num_cols, const int64_t* row_ptr, const int64_t* col_ind,
                           const double* A_val, const double* b, const double* x, const double* H, const double* alpha,
                           int32_t detach_hessian, double* A_grad, double* b_grad, thb_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Stand-alone Lie-group kernels (torchlie.functional SE3 namespace, torchlie/functional/lie_group.py:332-366).
 * Shapes: tangent [N,6], group [N,3,4], jacobian [N,6,6].
 * ---------------------------------------------------------------------------------------------- */
int thb_se3_exp_f64(const double* tangent, double* group, int64_t N, thb_stream_t stream);
int thb_se3_log_f64(const double* group, double* tangent, double* jlog /* may be NULL */, int64_t N, thb_stream_t stream);
int thb_se3_adjoint_f64(const double* group, double* adj, int64_t N, thb_stream_t stream);
int thb_se3_inverse_f64(const double* group, double* out, int64_t N, thb_stream_t stream);
int thb_se3_compose_f64(const double* g0, const double* g1, double* out, int64_t N, thb_stream_t stream);
int thb_se3_exp_f32(const float* tangent, float* group, int64_t N, thb_stream_t stream);
int thb_se3_log_f32(const float* group, float* tangent, float* jlog, int64_t N, thb_stream_t stream);
int thb_se3_adjoint_f32(const float* group, float* adj, int64_t N, thb_stream_t stream);
int thb_se3_inverse_f32(const float* group, float* out, int64_t N, thb_stream_t stream);
int thb_se3_compose_f32(const float* g0, const float* g1, float* out, int64_t N, thb_stream_t stream);

/* SO3 (torchlie/functional/so3_impl.py:220-261 exp, :390-433 log, :442-479 jlog, :669-672 compose, :561-563 inverse; adjoint = R)
 * and SE2 (theseus/geometry/se2.py:239-300 exp_map, :165-228 log_map + Jacobian, :309-316 adjoint, :318-332 compose, :334-339 inverse).
 * Shapes: SO3 tangent [N,3], group [N,3,3], jacobian [N,3,3]; SE2 tangent [N,3] = [ux,uy,theta], group [N,4] = [x,y,cos,sin]. */
int thb_so3_exp_f64(const double* tangent, double* group, int64_t N, thb_stream_t stream);
int thb_so3_log_f64(const double* group, double* tangent, double* jlog /* may be NULL */, int64_t N, thb_stream_t stream);
int thb_so3_adjoint_f64(const double* group, double* adj, int64_t N, thb_stream_t stream);
int thb_so3_inverse_f64(const double* group, double* out, int64_t N, thb_stream_t stream);
int thb_so3_compose_f64(const double* g0, const double* g1, double* out, int64_t N, thb_stream_t stream);
int thb_se2_exp_f64(const double* tangent, double* group, int64_t N, thb_stream_t stream);
int thb_se2_log_f64(const double* group, double* tangent, double* jlog /* may be NULL */, int64_t N, thb_stream_t stream);
int thb_se2_adjoint_f64(const double* group, double* adj, int64_t N, thb_stream_t stream);
int thb_se2_inverse_f64(const double* group, double* out, int64_t N, thb_stream_t stream);
int thb_se2_compose_f64(const double* g0, const double* g1, double* out, int64_t N, thb_stream_t stream);
int thb_so3_exp_f32(const float* tangent, float* group, int64_t N, thb_stream_t stream);
int thb_so3_log_f32(const float* group, float* tangent, float* jlog /* may be NULL */, int64_t N, thb_stream_t stream);
int thb_so3_adjoint_f32(const float* group, float* adj, int64_t N, thb_stream_t stream);
int thb_so3_inverse_f32(const float* group, float* out, int64_t N, thb_stream_t stream);
int thb_so3_compose_f32(const float* g0, const float* g1, float* out, int64_t N, thb_stream_t stream);
int thb_se2_exp_f32(const float* tangent, float* group, int64_t N, thb_stream_t stream);
int thb_se2_log_f32(const float* group, float* tangent, float* jlog /* may be NULL */, int64_t N, thb_stream_t stream);
int thb_se2_adjoint_f32(const float* group, float* adj, int64_t N, thb_stream_t stream);
int thb_se2_inverse_f32(const float* group, float* out, int64_t N, thb_stream_t stream);
int thb_se2_compose_f32(const float* g0, const float* g1, float* out, int64_t N, thb_stream_t stream);

/* Exponential map together with its right Jacobian d exp(t) / d t (torchlie/functional/so3_impl.py:270-320 _jexp_impl,
 * se3_impl.py:225-330 _jexp_impl_helper / _jexp_impl; what LieGroup.exp_map(tangent, jacobians=[...]) returns, lie_group.py:84-93).
 * Shapes: SO3 tangent [N,3], group [N,3,3], jexp [N,3,3]; SE3 tangent [N,6], group [N,3,4], jexp [N,6,6].  `group` may be NULL. */
int thb_so3_jexp_f64(const double* tangent, double* group /* may be NULL */, double* jexp, int64_t N, thb_stream_t stream);
int thb_se3_jexp_f64(const double* tangent, double* group /* may be NULL */, double* jexp, int64_t N, thb_stream_t stream);
int thb_so3_jexp_f32(const float* tangent, float* group /* may be NULL */, float* jexp, int64_t N, thb_stream_t stream);
int thb_se3_jexp_f32(const float* tangent, float* group /* may be NULL */, float* jexp, int64_t N, thb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* THB200_H_ */
