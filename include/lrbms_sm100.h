/*
 * lrbms_sm100.h -- C ABI of the B200 (sm_100a) LRBMS hot path.
 *
 * The reference (dune-community/pylrbms) has no FFI for this path: its arithmetic runs inside a pyMOR fork
 * (Python loops + NumPy) that calls dune-xt-la one vector at a time.  Each entry point below therefore names
 * the reference call site it replaces (paths relative to the reference's python/dune/pylrbms/), and
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - every function returns 0 on success or a negative lrbms_status; lrbms_last_error(h) has the message.
 *     Nothing throws or aborts across this boundary.
 *   - all numeric data is FP64, indices are int32, pointers marked "device" are CUDA device pointers owned by
 *     the caller (the host side passes torch data_ptr()s).  The library frees nothing it did not allocate.
 *     Plans own a small amount of device metadata (descriptor tables, schedules) plus, for projection plans,
 *     a partial-sum scratch buffer; they release it in lrbms_plan_destroy.
 *   - all work is enqueued on the cudaStream_t passed as `stream` (void* here) and is asynchronous.
 *   - one handle per device; calls on one handle must be serialised by the caller.
 *   - "dof-major" VectorArray storage: element (dof d, vector a) of an array lives at data[d * ld + a].
 *     (pyMOR's (len, dim) layout is the transpose; the host side converts at to_numpy()/from_numpy().)
 *   - there is no CPU fallback: on a machine without an sm_100 device lrbms_create fails.
 */
#ifndef LRBMS_SM100_H
#define LRBMS_SM100_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRBMS_VERSION 101

typedef enum {
  LRBMS_OK = 0,
  LRBMS_ERR_INVALID = -1,    /* bad argument */
  LRBMS_ERR_CUDA = -2,       /* CUDA runtime error */
  LRBMS_ERR_NO_DEVICE = -3,  /* no usable sm_100 device */
  LRBMS_ERR_ALLOC = -4,      /* allocation failed */
  LRBMS_ERR_UNSUPPORTED = -5,/* size outside what the kernels are instantiated for */
  LRBMS_ERR_NOT_SPD = -6     /* a reduced system was not positive definite */
} lrbms_status;

typedef struct lrbms_context* lrbms_handle_t;
typedef struct lrbms_plan* lrbms_plan_t;
typedef struct lrbms_symbolic* lrbms_symbolic_t;

/* ---------------------------------------------------------------------------------------------------- */
/*  context                                                                                             */
/* ---------------------------------------------------------------------------------------------------- */
int lrbms_version(void);
int lrbms_create(int device, lrbms_handle_t* out);
int lrbms_destroy(lrbms_handle_t h);
const char* lrbms_last_error(lrbms_handle_t h);       /* h may be NULL: error of the last failed create */
int lrbms_device_sm_count(lrbms_handle_t h, int* out);
/* Run-time switches of a context (there are no environment variables in the library).
 * LRBMS_OPT_SINGLE_STREAM: 1 = offline plans launch all their kernels on the caller's stream (profiling); 0 (default) =
 * the independent launches of one plan run are spread over the caller's stream and three side streams of the context.
 * LRBMS_OPT_PCG_MULTI_LAUNCH: 1 = lrbms_pcg_solve issues three launches per iteration; 0 (default) = 25 iterations per
 * cooperative launch with grid-wide barriers (same arithmetic; used automatically only where the whole grid is resident). */
enum { LRBMS_OPT_SINGLE_STREAM = 1, LRBMS_OPT_PCG_MULTI_LAUNCH = 2 };
int lrbms_set_option(lrbms_handle_t h, int32_t option, int32_t value);
/* Test hook: fills the shared memory of every SM with NaNs (a kernel that relied on stale shared memory being finite
 * or zero then fails its parity test instead of passing by luck). */
int lrbms_debug_poison_shared(lrbms_handle_t h, void* stream);

/* ---------------------------------------------------------------------------------------------------- */
/*  GPU VectorArray backing                                                                              */
/*  replaces: DuneXTVectorSpace / ListVectorArray of IstlDenseVectorDouble, one Python object and one   */
/*  C++ dot/axpy/scal per vector (discretize_elliptic_block_swipdg.py:11,51; estimators.py:15).         */
/* ---------------------------------------------------------------------------------------------------- */
/* y[:, a] = alpha[a] * y[:, a]                      (VectorArray.scal) */
int lrbms_va_scal(lrbms_handle_t h, int64_t dim, int32_t len, const double* alpha_host, int32_t n_alpha,
                  double* y, int32_t ldy, void* stream);
/* y[:, a] += alpha[a] * x[:, a]  (x may have len 1: broadcast)   (VectorArray.axpy) */
int lrbms_va_axpy(lrbms_handle_t h, int64_t dim, int32_t len, const double* alpha_host, int32_t n_alpha,
                  const double* x, int32_t ldx, int32_t len_x, double* y, int32_t ldy, void* stream);
/* out[a] = sum_d x[d, a] * y[d, a]                   (VectorArray.pairwise_dot); out is device, length len */
int lrbms_va_pairwise_dot(lrbms_handle_t h, int64_t dim, int32_t len, const double* x, int32_t ldx,
                          const double* y, int32_t ldy, double* out, void* stream);
/* y[:, 0:n_out] = x[:, 0:len] @ C  with C (len x n_out, row-major, device)   (VectorArray.lincomb / reconstruct) */
int lrbms_va_lincomb(lrbms_handle_t h, int64_t dim, int32_t len, int32_t n_out, const double* x, int32_t ldx,
                     const double* coeff, int32_t ldc, double* y, int32_t ldy, void* stream);
/* y[:, dst0 + k] = x[:, src[k]]   k < n_cols          (append / copy / indexing); src is a host int32 array or NULL (= 0..n) */
int lrbms_va_copy_cols(lrbms_handle_t h, int64_t dim, int32_t n_cols, const int32_t* src_host, const double* x,
                       int32_t ldx, double* y, int32_t ldy, int32_t dst0, void* stream);
/* (len, dim) row-major host-layout array <-> dof-major (dim, ld): out-of-place transposes on the device */
int lrbms_va_transpose_in(lrbms_handle_t h, int64_t dim, int32_t len, const double* rowmajor_len_dim,
                          double* dofmajor, int32_t ld, void* stream);
int lrbms_va_transpose_out(lrbms_handle_t h, int64_t dim, int32_t len, const double* dofmajor, int32_t ld,
                           double* rowmajor_len_dim, void* stream);

/* ---------------------------------------------------------------------------------------------------- */
/*  Offline: batched block-CSR SpMM  W = A V   (K1)                                                      */
/*  replaces: DuneXTMatrixOperator.apply -> IstlRowMajorSparseMatrixDouble.mv once per basis vector      */
/*  (discretize_elliptic_block_swipdg.py:333,353,375,473,502,670,679,689,725), and the per-vector grid    */
/*  walks of OswaldInterpolationErrorOperator.apply / FluxReconstructionOperator.apply (:83-122,:148-176) */
/*  as consumed at reductor.py:43,60.                                                                    */
/* ---------------------------------------------------------------------------------------------------- */
typedef struct {
  const int32_t* rowptr;   /* device, n_rows + 1 */
  const int32_t* colind;   /* device, nnz */
  const double* values;    /* device, nnz */
  int32_t n_rows, n_cols;
  const double* V;         /* device, dof-major n_cols x N */
  int32_t ldv;
  int32_t N;               /* number of vectors */
  double* W;               /* device, dof-major n_rows x N (written, not accumulated) */
  int32_t ldw;
} lrbms_spmm_desc_t;

int lrbms_spmm_plan_create(lrbms_handle_t h, int32_t n_desc, const lrbms_spmm_desc_t* descs_host, lrbms_plan_t* out);

/* ---------------------------------------------------------------------------------------------------- */
/*  Offline: batched fused Galerkin projection  G = alpha * VL^T (A VR)   (K1 + K2)                      */
/*  replaces: GenericRBSystemReductor._reduce -> project_system -> op.apply2(RB, SB) per block, i.e. the  */
/*  N_R mv calls + N_L * N_R dots of reductor.py:70 for d.operator, d.rhs, d.products and every           */
/*  estimator operator (nc_i, r_fd_i, r_dd_i, df_aa_i, df_bb_i, df_ab_i; discretize...:733-770).          */
/*  rowptr == NULL selects the identity operator: G = VL^T VR (VectorArray.dot / Gram matrices).          */
/* ---------------------------------------------------------------------------------------------------- */
typedef struct {
  const int32_t* rowptr;   /* device, n_rows + 1, or NULL for A = I (then n_cols == n_rows) */
  const int32_t* colind;   /* device */
  const double* values;    /* device */
  int32_t n_rows, n_cols;
  const double* VL;        /* device, dof-major n_rows x NL */
  int32_t ldl, NL;
  const double* VR;        /* device, dof-major n_cols x NR */
  int32_t ldr, NR;
  double* out;             /* device, row-major NL x NR: out[a * ldo + b] (overwritten) */
  int32_t ldo;
  double alpha;
  int32_t symmetric;       /* caller asserts A = A^T and VL, VR are the same array: only the lower-triangular output
                              chunks are computed and mirrored (estimator Grams nc_i, r_dd_i, df_bb_i, products) */
  int32_t reserved;
} lrbms_project_desc_t;

int lrbms_project_plan_create(lrbms_handle_t h, int32_t n_desc, const lrbms_project_desc_t* descs_host,
                              lrbms_plan_t* out);
/* The same with caller-provided scratch (SURVEY.md section 8b: "the library allocates nothing except an explicitly sized
 * workspace handed in by the caller").  Descriptors too wide for the fused kernel (NL or NR > 40 with a sparse operator) are
 * computed as W = A VR into scratch followed by a dense Gram; lrbms_project_plan_scratch_bytes says how much scratch a
 * descriptor list needs, lrbms_project_plan_create_ws carves the W arrays out of `scratch` (device, 256-byte aligned, must
 * outlive the plan; plans that never run concurrently may share it) instead of allocating them. */
int lrbms_project_plan_scratch_bytes(int32_t n_desc, const lrbms_project_desc_t* descs_host, size_t* bytes);
/* unit_rows_hint > 0: the amount of work (sum over descriptors of output chunks x rows, 3x for the wide dense Grams) the
 * row partition is sized for, instead of the sum over this plan's own descriptors.  A rank that projects only its share of a
 * descriptor list passes the figure of the WHOLE list: the rows of every descriptor are then cut exactly as in the
 * unsharded plan and the results are bit-identical to it (the partial sums of a block are added in partition order). */
int lrbms_project_plan_create_ws(lrbms_handle_t h, int32_t n_desc, const lrbms_project_desc_t* descs_host, void* scratch,
                                 size_t scratch_bytes, int64_t unit_rows_hint, lrbms_plan_t* out);

/* Incremental re-projection after an enrichment (SURVEY.md section 8f rank 2).  The reference re-runs the whole        */
/* reductor.reduce() after every enrichment (online_enrichment.py:49-51); only the rows / columns that belong to the      */
/* appended basis vectors change.  One descriptor assembles one new reduced block:                                       */
/*   dst[r][c] = prev[row_map[r]][col_map[c]]                    both old                                                */
/*             = cols_new[r][-col_map[c]-1]                      column c is new   (cols_new = alpha L^T A R[:, new])     */
/*             = rows_new[c][-row_map[r]-1]                      row r is new      (rows_new = alpha R^T A^T L[:, new];   */
/*                                                               rows_new == NULL: symmetric block, cols_new is used)    */
typedef struct {
  double* dst;             /* device, row-major NL x NR */
  int32_t NL, NR;
  const double* prev;      /* device, previous block, row-major with pNR columns (may be NULL if every row or column is new) */
  int32_t pNR, n_cn;
  const double* cols_new;  /* device, row-major NL x n_cn, or NULL when no column is new */
  const double* rows_new;  /* device, row-major NR x n_rn, or NULL */
  int32_t n_rn, reserved;
  const int32_t* row_map;  /* device [NL] */
  const int32_t* col_map;  /* device [NR] */
} lrbms_remap_desc_t;
int lrbms_remap_blocks(lrbms_handle_t h, int32_t n, const lrbms_remap_desc_t* descs_host, void* stream);

/* Multi-GPU exchange of the sharded offline results over peer memory (replaces the Allreduce(SUM) of zero-padded
 * blocks at reference src/reductor.py:93).  Stores `n_bytes` at `src` (device, 16-byte aligned) to each of the `n_dst`
 * device addresses in `dst_host` -- peer pointers of the other ranks' buffers mapped into this process (NVLink P2P), or,
 * with multicast != 0, ONE NVSwitch multicast address (n_dst == 1) that the switch replicates to every GPU.  Stream
 * ordered; the caller follows it with a cross-rank barrier (signal pads of the symmetric allocation) before reading. */
#define LRBMS_MAX_PEERS 16
int lrbms_peer_push(lrbms_handle_t h, const void* src, int64_t n_bytes, int32_t n_dst, const uint64_t* dst_host,
                    int32_t multicast, void* stream);

/* run / destroy / introspect any plan */
int lrbms_plan_run(lrbms_plan_t plan, void* stream);
int lrbms_plan_destroy(lrbms_plan_t plan);
/* what: 0 = kernel launches per run, 1 = CTAs of the main kernel, 2 = algorithmic bytes per run (tight count),
 *       3 = algorithmic flops per run, 4 = device bytes owned by the plan, 5 = algorithmic bytes (SURVEY formula);
 *       online plans: 6 = solve kernel the plan selected (LRBMS_SOLVER_WINDOW or LRBMS_SOLVER_BANDED), 7 = factor flops
 *       per parameter that kernel executes, 8 = scalar half bandwidth of the reduced operator, 9 = parameters per CTA of
 *       the estimator kernel (64, 32, 16 or 8; 0 without estimator terms) */
int lrbms_plan_info(lrbms_plan_t plan, int32_t what, double* out);

/* ---------------------------------------------------------------------------------------------------- */
/*  Online: mu-batched assemble + factor + solve + estimate of the block-sparse reduced system (K3-K5)   */
/*  replaces: rd.solve(mu) = LincombOperator.assemble(mu) + numpy.linalg.solve on the unblocked dense     */
/*  matrix (online_enrichment.py:72, scripts/online_adaptive_lrbms.py:141) and rd.estimate(U, mu) =       */
/*  EstimatorBase._estimate_elliptic (estimators.py:45-112), one mu per call in the reference.            */
/* ---------------------------------------------------------------------------------------------------- */

/* Host-only symbolic phase: 8x8-tile sparse Cholesky of the reduced block pattern (no GPU needed). */
int lrbms_symbolic_create(int32_t n_sub, const int32_t* basis_sizes, int32_t n_blocks, const int32_t* block_i,
                          const int32_t* block_j, lrbms_symbolic_t* out);
int lrbms_symbolic_destroy(lrbms_symbolic_t s);
/* Elimination order (what online plans do once the shared-memory window kernel is selected): re-plan the schedule of s,
 * built in the given subdomain order, in the cheapest of the given order, the Cuthill-McKee level-set order of the
 * subdomain graph and its reverse, by a column-period model of the window kernel.  A candidate is only taken if it keeps
 * the staggered schedule variant of the given order and its kernel shared memory for Q operator terms stays within
 * smem_budget bytes; the given order wins ties.  Fails with LRBMS_ERR_INVALID if s was already re-planned. */
int lrbms_symbolic_reorder(lrbms_symbolic_t s, int32_t Q, int64_t smem_budget);
/* what: 0 n_red, 1 padded n, 2 tile columns, 3 L tiles, 4 A tiles, 5 update pairs, 6 factor flops per mu,
 *       7 max targets per tile column, 8 shared-memory window slots (live off-diagonal L tiles, peak),
 *       11 schedule variant of the shared-memory kernel: 1 = early updates stop at source column J - 3 and the pair with
 *          source column J - 2 rides with the late update (every such pair has a carrier tile), 0 = barrier schedule,
 *       12 elimination order (0 given, 1 Cuthill-McKee, 2 reverse Cuthill-McKee), 13 / 14 / 15 modelled SM cycles per
 *          parameter of the given / CM / RCM order (after lrbms_symbolic_reorder; 0 = not evaluated) */
int lrbms_symbolic_info(lrbms_symbolic_t s, int32_t what, int64_t* out);
/* copy out schedule arrays (for tests): which: 0 col_ptr[ntc+1], 1 row_idx[n_tiles], 2 pair_ptr[n_tiles+ntc+1],
 * 3 pair_a, 4 pair_b, 5 a_map[n_tiles], 6 win_slot[n_tiles], 7 late_ptr[n_tiles+ntc], 8 win_a[pairs], 9 win_b[pairs],
 * 10 xo_ptr[ntc+1], 11 xo_idx[n_tiles+ntc], 12 cnext[n_tiles+ntc], 13 chas[ntc], 14 cord[n_tiles+ntc],
 * 15 perm[n_sub] (subdomain eliminated k-th), 16 iperm[n_sub], 17 row_map[n_red] (given row of every permuted row);
 * returns number of int32 written (<= cap) or a negative status */
int64_t lrbms_symbolic_get(lrbms_symbolic_t s, int32_t which, int32_t* out, int64_t cap);

/* one estimator term:  out[kind][sub][mu] += coef * theta[qa](mu) * theta[qb](mu) * xl^T M xr  */
enum { LRBMS_VEC_ONE = 0, LRBMS_VEC_UI = 1, LRBMS_VEC_UN = 2, LRBMS_VEC_UR = 3 };
enum { LRBMS_OUT_NC = 0, LRBMS_OUT_R = 1, LRBMS_OUT_DF = 2 };
typedef struct {
  int32_t subdomain;
  int32_t out_kind;        /* LRBMS_OUT_* */
  int32_t left_kind;       /* LRBMS_VEC_*: 1 (linear form), u_i, u over N(i), or U_r = [theta_q u_k]_{k in N(i), q} */
  int32_t right_kind;
  int32_t rows, cols;      /* of M; must match the vector kinds */
  int32_t qa, qb;          /* theta indices multiplied in, -1 = none */
  double coef;
  int64_t matrix_offset;   /* into the estimator matrix buffer, in doubles; M row-major, ld = cols */
} lrbms_estimator_term_t;

/* Solve kernel of an online plan.  AUTO: WINDOW, the shared-memory-window kernel (one SM per parameter, live factor window
 * in shared memory), when the window fits one SM, else BANDED, the block-banded out-of-HBM Cholesky (whole GPU per chunk).
 * WINDOW / BANDED force one of them (WINDOW fails with LRBMS_ERR_UNSUPPORTED when the window does not fit).  Any other
 * value fails with LRBMS_ERR_INVALID. */
enum { LRBMS_SOLVER_AUTO = 0, LRBMS_SOLVER_WINDOW = 1, LRBMS_SOLVER_BANDED = 3 };

typedef struct {
  int32_t n_sub;
  const int32_t* basis_sizes;          /* host [n_sub] */
  int32_t Q;                           /* affine terms of the reduced operator */
  int32_t Qf;                          /* affine terms of the reduced rhs */
  int32_t n_blocks;
  const int32_t* block_i;              /* host [n_blocks]; only blocks with i >= j are read: the operator MUST be symmetric
                                          (block (j, i) = block (i, j)^T); this is not validated */
  const int32_t* block_j;
  const int64_t* block_offset;         /* host [Q * n_blocks]: offset (doubles) of block b of term q: [q * n_blocks + b] */
  const double* lhs_blocks;            /* device: packed row-major N_i x N_j blocks */
  const double* rhs;                   /* device: [Qf][n_red] */
  /* estimator */
  const int32_t* nbh_ptr;              /* host [n_sub + 1] */
  const int32_t* nbh_idx;              /* host: neighbourhoods (contain i) */
  int32_t n_terms;
  const lrbms_estimator_term_t* terms; /* host */
  const double* est_matrices;          /* device */
  const double* rf_squared;            /* host [n_sub]: local_eta_rf_squared */
  const double* r_scale;               /* host [n_sub]: (1/pi^2) / min_diffusion_ev * h^2  (estimators.py:88-91) */
  const double* theta_bar;             /* host [Q] theta_q(mu_bar) */
  const double* theta_hat;             /* host [Q] theta_q(mu_hat) */
  int32_t alpha_returns_first;         /* 1 reproduces estimators.py:114-121 (alpha = theta_0 ratio only) */
  int32_t solver;                      /* LRBMS_SOLVER_* (0 = AUTO) */
} lrbms_reduced_system_t;

int lrbms_online_plan_create(lrbms_handle_t h, const lrbms_reduced_system_t* sys, lrbms_plan_t* out);
int lrbms_online_workspace_bytes(lrbms_plan_t plan, int64_t n_mu, size_t* bytes);
/* theta: device, row-major n_mu x (Q + Qf).  u: device n_mu x n_red (pyMOR (len, dim) layout).
 * info: device int32 [n_mu], 0 or 1 + index of the first non-positive pivot. */
int lrbms_online_solve(lrbms_plan_t plan, int64_t n_mu, const double* theta, double* u, int32_t* info,
                       void* workspace, size_t workspace_bytes, void* stream);
/* parts: device [3][n_sub][n_mu] (nc, r, df) or NULL; indicators: device [n_sub][n_mu] or NULL; eta: device [n_mu] */
int lrbms_online_estimate(lrbms_plan_t plan, int64_t n_mu, const double* theta, const double* u, double* eta,
                          double* parts, double* indicators, void* workspace, size_t workspace_bytes, void* stream);
/* solve + estimate in one call (the unit of work of BASELINE.json's metric) */
int lrbms_online_sweep(lrbms_plan_t plan, int64_t n_mu, const double* theta, double* u, double* eta, double* parts,
                       double* indicators, int32_t* info, void* workspace, size_t workspace_bytes, void* stream);
/* Developer aid, only in libraries compiled with -DLRBMS_DEVTOOLS (the shipped build returns LRBMS_ERR_UNSUPPORTED):
 * with LRBMS_SOLVE_TIMING=1 in the environment at plan creation the shared-memory solve kernel records,
 * for CTA 0, SM-clock cycles per warp and phase ([16 warps][8 phases]: 0 metadata staging, 1 diagonal tile, 2 early
 * updates, 3 barrier, 4 triangular solve + late update, 5 barrier, 6 backward substitution, 7 store).  Copies up to n
 * counters to out_host and returns how many were written, or a negative status. */
int lrbms_online_debug_timing(lrbms_plan_t plan, int64_t* out_host, int32_t n);
/* max and argmax of eta (device outputs: max_out[1], argmax_out[1]); the per-GPU leg of the estimator-max gather */
int lrbms_eta_max(lrbms_handle_t h, int64_t n_mu, const double* eta, double* max_out, int64_t* argmax_out, void* stream);

/* ---------------------------------------------------------------------------------------------------- */
/*  Fine-scale neighbourhood solve of the local corrector problems (SURVEY.md section 8f rank 4)          */
/*  replaces: lhs.apply_inverse(rhs.as_source_array(mu), mu, inverse_options) on the neighbourhood system   */
/*  assembled by solve_for_local_correction (discretize_elliptic_block_swipdg.py:227-316; dune-istl in the   */
/*  reference), called from LRBMSReductor.enrich_local (reductor.py:75-78).                                 */
/*  Jacobi-preconditioned CG on a device CSR matrix; x holds the initial guess on entry and the solution on  */
/*  exit; stops when ||b - A x||_2 <= rtol ||b||_2 or after max_iter iterations (not an error: inspect       */
/*  relres_out).  Returns LRBMS_ERR_NOT_SPD when p^T A p <= 0 is met.  iters_out / relres_out are host.      */
/* ---------------------------------------------------------------------------------------------------- */
int lrbms_pcg_workspace_bytes(lrbms_handle_t h, int64_t n, size_t* bytes);
int lrbms_pcg_solve(lrbms_handle_t h, int32_t n, const int32_t* rowptr, const int32_t* colind, const double* values,
                    const double* b, double* x, double rtol, int32_t max_iter, int32_t* iters_out, double* relres_out,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Fine-scale solve of an affine operator for a batch of parameters (replaces d.solve(mu): LincombOperator.assemble(mu)
 * + apply_inverse, dune-istl in the reference).  A(mu) = sum_q theta[mu][q] A_q on ONE CSR pattern (values: [Q][nnz],
 * 1 <= Q <= 4, else LRBMS_ERR_UNSUPPORTED), b(mu) = sum_f theta[mu][Q + f] rhs[f] (rhs: [Qf][n]).  theta: device,
 * row-major n_mu x (Q + Qf) -- the layout of the online plans.  x: device, dof-major n x ldx, column k = parameter k;
 * initial guess on entry, solution on exit.  Jacobi-preconditioned CG, 32 parameters per warp-row; a parameter's result
 * is bit-identical whatever the batch it is solved in (size, position, chunking).  A parameter whose recurrence residual
 * reaches rtol restarts from its iterate with the true residual b - A x, at most max_restarts times and only while each
 * restart halves the true residual; then it is frozen (its columns are no longer written).
 * Per parameter (host arrays [n_mu]): iterations, TRUE relative residual ||b - A x|| / ||b||, status
 * 0 = converged (true residual <= rtol), 1 = not converged within max_iter / restarts, 2 = p^T A p <= 0 met.
 * Runs as a cooperative launch only (one CTA of 1024 threads per SM); a device that cannot gets LRBMS_ERR_UNSUPPORTED.
 * lrbms_affine_pcg_workspace_bytes: device workspace for n_mu parameters (about 6 n doubles each); split larger batches. */
int lrbms_affine_pcg_workspace_bytes(lrbms_handle_t h, int64_t n, int64_t n_mu, size_t* bytes);
int lrbms_affine_pcg_solve(lrbms_handle_t h, int32_t n, int32_t Q, const int32_t* rowptr, const int32_t* colind,
                           const double* values, int32_t Qf, const double* rhs, int64_t n_mu, const double* theta,
                           double* x, int32_t ldx, double rtol, int32_t max_iter, int32_t max_restarts,
                           int32_t* iters_out, double* relres_out, int32_t* status_out,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------- */
/*  Reduction error of a parameter batch (reduction_error_analysis; the reference's "max discretization    */
/*  error" loop, scripts/online_adaptive_lrbms.py:49-53,141-143: reductor.reconstruct(rd.solve(mu)), the   */
/*  difference to d.solve(mu) and its norm, one mu and one subdomain at a time).                          */
/* ---------------------------------------------------------------------------------------------------- */
/* One subdomain of the reconstruction: rows row_offset .. row_offset + n_rows of u_h / e, the local basis V (device,
 * dof-major n_rows x ldv, len vectors) and the first N of its vectors (N = block_dims[i] of the reduced solution, which may
 * be smaller than len for a solution of an older reduced model; N > len is LRBMS_ERR_INVALID), whose coefficients sit in
 * columns red_offset .. red_offset + N of u_N.  Blocks are in ascending, disjoint row order. */
typedef struct {
  const double* V;
  int32_t ldv;
  int32_t len;
  int32_t N;
  int32_t red_offset;
  int64_t row_offset;
  int32_t n_rows;
  int32_t reserved;
} lrbms_recon_block_t;
/* e[r][m] = u_h[r][m] - sum_{k < N_i} V_i[r - row_offset_i][k] * u_N[m][red_offset_i + k], k ascending, for every row of
 * every block and every m < n_mu, in one launch.  u_h: device, dof-major rows x ldu (the buffer of d.solve_batch, column =
 * parameter; columns n_mu .. ldu are not read); u_N: device, row-major n_mu x ldn, n_red used columns (the reduced
 * solutions); e: device, dof-major rows x lde, written for m < n_mu only (it may not alias u_h).  ldu, lde < n_mu or
 * ldn < n_red are LRBMS_ERR_INVALID.  A block with N = 0 gets e = u_h.  Every entry is one sequential fma chain: a
 * parameter's bits do not depend on the batch.  lrbms_recon_error_workspace_bytes: device workspace for n_mu parameters of
 * n_red reduced coefficients (a transposed copy of u_N, the block table and the row partition). */
int lrbms_recon_error_workspace_bytes(lrbms_handle_t h, int32_t n_sub, const lrbms_recon_block_t* blocks_host, int64_t n_mu,
                                      int32_t n_red, size_t* bytes);
int lrbms_recon_error(lrbms_handle_t h, int32_t n_sub, const lrbms_recon_block_t* blocks_host, int64_t n_mu,
                      const double* u_h, int32_t ldu, const double* u_N, int32_t n_red, int32_t ldn, double* e, int32_t lde,
                      void* workspace, size_t workspace_bytes, void* stream);
/* Segmented affine quadratic form: out[s][m] = sum_{seg_ptr[s] <= r < seg_ptr[s+1]} x[r][m] sum_c (sum_q theta[m][q]
 * A_q[r][c]) x[c][m] for the n_seg row segments (host seg_ptr [n_seg + 1], non-decreasing within [0, n]).  The Q
 * components share ONE CSR pattern (rowptr [n + 1], colind [nnz], values [Q][nnz]; 1 <= Q <= 4, else
 * LRBMS_ERR_UNSUPPORTED); theta: device, row-major n_mu x ldt, the first Q columns read (ldt < Q is LRBMS_ERR_INVALID), or
 * NULL for theta = 1 with Q = 1 (a plain product matrix).  x: device, dof-major n x ldx (ldx >= n_mu); out: device, n_seg x
 * ldo (ldo >= n_mu).  Used with the block-diagonal local energy products (segments = subdomains: local squared norms) and
 * with the affine system operator (one segment: |||x|||_mu^2; per-subdomain row partials of a coupled operator are not
 * norms).  Row sums run in CSR order inside one lane, rows are added per warp, warp and CTA in a fixed order over a row
 * partition set by the segment sizes and the SM count only: a parameter's bits do not depend on the batch.  No atomics.
 * lrbms_segmented_form_workspace_bytes: device workspace (CTA partials of 256 parameters and the partition). */
int lrbms_segmented_form_workspace_bytes(lrbms_handle_t h, int32_t n_seg, const int32_t* seg_ptr_host, size_t* bytes);
int lrbms_segmented_form(lrbms_handle_t h, int32_t n, int32_t Q, const int32_t* rowptr, const int32_t* colind,
                         const double* values, int64_t nnz, int32_t n_seg, const int32_t* seg_ptr_host, int64_t n_mu,
                         const double* theta, int32_t ldt, const double* x, int32_t ldx, double* out, int32_t ldo,
                         void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LRBMS_SM100_H */
