/*
 * demethify_b200.h — C ABI of libdemethify_sm100.so, the sm_100a kernel library behind the
 * DeMethify NMF-deconvolution hot path (X ~ [R|U]·alpha, accelerated projected gradient).
 *
 * The reference (cortes-ciriano-lab/DeMethify) is pure Python + numba and has NO FFI of its own
 * (SURVEY.md §8 b1/b2); every entry point below therefore cites the reference FUNCTION whose
 * arithmetic it replaces (file:line under demethify/), and INTEGRATION.md shows the ctypes stub a
 * maintainer would add to demethify/deconvolution.py to bind it.
 *
 * Conventions
 *   - plain C, raw DEVICE pointers + sizes, caller owns every buffer (allocate with torch / cudaMalloc),
 *     no ownership transfer, every function returns 0 on success or a DMF_E_* code
 *     (text via dmf_last_error()).  All matrices row-major.  All base pointers 16-byte aligned.
 *   - stream arguments are cudaStream_t passed as void* (0 = legacy default stream).
 *   - a "batch" is a set of independent fits of identical shape (M,N,K,n_u): bootstrap resamples,
 *     restarts, BCV folds (bootstrap.py:26, demethify.py:167-203, ic.py:67).  The n_u sweep of
 *     ic.py:192 is one batch per n_u.  Fits never exchange data; each owns its U, alpha and state.
 *   - floating-point reductions over CpG rows are fp64 with a fixed order (run-to-run deterministic for
 *     a given grid), so the |cf - cf_0| < tol test of deconvolution.py:220 is reproducible.
 */
#ifndef DEMETHIFY_B200_H
#define DEMETHIFY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMF_ABI_VERSION 4

enum { DMF_OK = 0, DMF_E_ARG = 1, DMF_E_CUDA = 2, DMF_E_SHAPE = 3, DMF_E_STATE = 4 };

/* arithmetic/storage type of X, Rk, U, alpha */
enum { DMF_F64 = 0, DMF_F32 = 1 };
/* storage of the coverage weights d_x: same float type as X, or narrow unsigned integers
 * (exact for integer coverage; SURVEY.md §7.1 #6) */
enum { DMF_W_FLOAT = 0, DMF_W_U16 = 1 };
/* solver variant */
enum {
    DMF_MODE_PARTIAL = 0,      /* mdwbssmf_deconv      deconvolution.py:190-223 */
    DMF_MODE_PURITY = 1,       /* mdwbssmf_deconv_p    deconvolution.py:305-337 */
    DMF_MODE_UNSUPERVISED = 2  /* unsupervised_deconv  deconvolution.py:107-184 (K = 0; U-gradient at u, :163) */
};

/* how the inner iterations are executed (results agree to ~1e-15 on alpha; both are pinned by the same golden vectors)
 *   STREAM: one launch per reference inner iteration, each a streaming pass over X, d_x (dmf_pass_u / _alpha / _fw / _cost)
 *   GRAM  : per outer iteration two streaming passes build the sufficient statistics of the U step (per CpG row) and of the
 *           alpha step (per sample); the n_iter2 inner iterations then run on those (dmf_gram_*).  n_u <= 4, or n_u <= 8 with K <= 6.
 *   FUSED : ONE streaming pass per outer iteration (dmf_fused_outer): a row tile goes through row statistics -> the n_iter2
 *           update_u iterations -> the Gram panel with the new u on a single visit; the cost of the incoming iterate is taken on
 *           the same visit and the U step is committed only if the fit did not just terminate.  FP64 storage, n_u <= 2, K <= 8,
 *           N <= 256, n_iter2 <= 64, four U slots (dmf_shape_t.u_slots); the default where it applies. */
enum { DMF_ENGINE_STREAM = 0, DMF_ENGINE_GRAM = 1, DMF_ENGINE_FUSED = 2 };

typedef struct dmf_shape {
    int64_t M;      /* CpG rows                         */
    int32_t N;      /* samples                          */
    int32_t K;      /* known cell types (0 allowed)     */
    int32_t n_u;    /* unknown cell types (>= 1)        */
    int32_t dtype;  /* DMF_F64 | DMF_F32                */
    int32_t wtype;  /* DMF_W_FLOAT | DMF_W_U16          */
    int32_t mode;   /* DMF_MODE_*                       */
    int32_t n_fits; /* fits in the batch                */
    int32_t max_ctas_per_fit; /* 0 = let the library choose (multiple of the SM count overall) */
    /* Row pitches in elements.  ALL PITCHES MUST BE EVEN and the padding entries MUST BE ZERO: the kernels
     * fetch every matrix as aligned two-element vectors and rely on zero padding instead of bounds tests.
     * A row tile reaches shared memory as one bulk copy and keeps its pitch there; the FUSED engine walks four rows per warp
     * instruction, which is free of bank conflicts when the pitch of X is 32 bytes and the pitch of u16 weights 16 bytes
     * beyond a multiple of 128 bytes (e.g. N = 256 fp64: ldx = 260, ldd = 264 for u16).  Any even pitch is correct. */
    int64_t ldx;    /* row pitch of X  (>= N, even)      */
    int64_t ldd;    /* row pitch of D  (>= N, even)      */
    int64_t ldr;    /* row pitch of Rk (>= K, even)      */
    int64_t ldu;    /* row pitch of U  (>= n_u, even)    */
    int64_t u_slot; /* elements between consecutive slots of U (>= M*ldu, u_slot*sizeof(T) % 16 == 0) */
    int32_t u_slots; /* slots of U behind dmf_fit_desc_t.U: 2 (or 0), or 4 - the FUSED engine writes the new (u, u_) pair next to
                        the current one and needs 4; slots 2 and 3 must start zeroed */
    int32_t reserved;
} dmf_shape_t;

/* Per-fit buffers (host array of n_fits of these is passed to dmf_batch_create). */
typedef struct dmf_fit_desc {
    const void* X;         /* M x N   methylation frequencies (meth_frequency)                 */
    const void* D;         /* M x N   coverage weights d_x                                      */
    const void* Rk;        /* M x K   known reference profiles R_trunc (NULL when K = 0)        */
    const int32_t* rows;   /* optional gather: fit row p reads source row rows[p] of X, D, Rk
                              (bootstrap.py:28 resample); NULL = identity.  U stays position-indexed.
                              With mult / offs (below): the sorted position -> source row map, nothing is gathered */
    void* U;               /* shape.u_slots slots of M x n_u (pitch ldu), shape.u_slot elements apart; slots 0 and 1 BOTH hold the initial u */
    void* A;               /* [2][Kt][N]; BOTH slots hold the initial alpha (alpha_ = alpha.copy())    */
    const double* purity;  /* [N] internal purity vector (DMF_MODE_PURITY) else NULL            */
    double* cost_trace;    /* optional [trace_cap] cost after every outer iteration, or NULL    */
    int32_t trace_cap;
    int32_t reserved;
    /* Bootstrap resample in MULTIPLICITY FORM (all fits of a batch or none).  X, D, Rk are the SOURCE matrices (shape.M source
     * rows, typically shared by all fits); source row m was drawn mult[m] times and owns the u rows offs[m] .. offs[m+1]-1
     * (offs has M + 1 entries, offs[M] == M: the resample has as many rows as the source, sklearn.utils.resample,
     * bootstrap.py:28).  u is thus ordered by source row, and `rows` must hold the nondecreasing source row of every position
     * (the sorted resample index).  The streaming passes then read X, D, Rk contiguously instead of gathering rows.
     * Device pointers, int32; mult 16-byte aligned. */
    const int32_t* mult;
    const int32_t* offs;
} dmf_fit_desc_t;

/* Per-fit result block, filled by dmf_batch_read_state (host memory). */
typedef struct dmf_fit_state {
    double cost;       /* cost_f_w at the returned iterate                           */
    double cost_prev;
    double l_w, l_h;   /* current step constants (deconvolution.py:198-201,212,216)  */
    double a1, a2;     /* extrapolation scalars (deconvolution.py:84,96)              */
    double dmax;       /* max d_x over the fit's rows                                 */
    int32_t n_outer;   /* outer iterations executed                                   */
    int32_t done;      /* 1 once |cf-cf_0| < tol fired                                */
    int32_t u_slot;    /* which slot of U (0..3) / A (0..1) holds the current iterate   */
    int32_t a_slot;
} dmf_fit_state_t;

typedef struct dmf_handle_s* dmf_handle_t;
typedef struct dmf_batch_s* dmf_batch_t;

/* library / device ----------------------------------------------------------------------------- */
int dmf_abi_version(void);
const char* dmf_last_error(void);
int dmf_create(int device, dmf_handle_t* out);
int dmf_destroy(dmf_handle_t h);
int dmf_sm_count(dmf_handle_t h, int* out);

/* batch set-up --------------------------------------------------------------------------------- */
/* bytes of device workspace a batch of this shape needs (partials, tickets, per-fit state) */
int dmf_batch_workspace_bytes(dmf_handle_t h, const dmf_shape_t* shape, size_t* bytes);
int dmf_batch_create(dmf_handle_t h, const dmf_shape_t* shape, const dmf_fit_desc_t* fits_host,
                     void* workspace_dev, size_t workspace_bytes, void* stream, dmf_batch_t* out);
int dmf_batch_destroy(dmf_batch_t b);
/* launch geometry chosen for the batch (for roofline accounting) */
int dmf_batch_geometry(dmf_batch_t b, int32_t* ctas_per_fit, int32_t* tile_rows, int32_t* smem_bytes);

/* reference-shaped single steps: ONE launch each, all live fits of the batch -------------------- */
/* cost_f_w + ||R||_F^2 + max d_x, initialises l_w, l_h, cf (deconvolution.py:192-204 / :308-318) */
int dmf_pass_init(dmf_batch_t b, void* stream);
/* one inner iteration of update_u (deconvolution.py:82-89) */
int dmf_pass_u(dmf_batch_t b, void* stream);
/* one inner iteration of update_alpha incl. projection_simplex_sort_2d (deconvolution.py:94-101, :21-37) */
int dmf_pass_alpha(dmf_batch_t b, void* stream);
/* one Frank-Wolfe iteration k of frank_wolfe_nmf (deconvolution.py:285-299) */
int dmf_pass_fw(dmf_batch_t b, int32_t k_inner, void* stream);
/* cost_f_w + termination test |cf - cf_0| < tol (deconvolution.py:218-221) */
int dmf_pass_cost(dmf_batch_t b, double tol, void* stream);
/* Set the extrapolation state of every fit before dmf_pass_u (which = 0: a1, l_w, l_w_old) or dmf_pass_alpha
 * (which = 1: a2, l_h, l_h_old).  Host arrays of n_fits values each.  Nothing else in the state changes. */
int dmf_batch_set_step_state(dmf_batch_t b, int32_t which, const double* a, const double* l, const double* l_old, void* stream);

/* Gram-form engine: the same outer iteration (deconvolution.py:206-221 / :320-335) on sufficient statistics ------- */
int dmf_batch_set_engine(dmf_batch_t b, int32_t engine);
int dmf_batch_get_engine(dmf_batch_t b, int32_t* engine);
/* streaming pass 1: cost_f_w of the current iterate (set-up when initial != 0, else termination test against tol,
 * deconvolution.py:192-204 / :218-221) + per-row statistics b_m = (d o (x - R_trunc a_k)) a_u^T, H_m = a_u diag(d_m) a_u^T */
int dmf_gram_rowgram(dmf_batch_t b, int32_t initial, double tol, void* stream);
/* n_iter2 update_u iterations (deconvolution.py:82-89) per row on (b_m, H_m) */
int dmf_gram_u_inner(dmf_batch_t b, int32_t n_iter2, void* stream);
/* streaming pass 2: blocks of G_j = R^T diag(d_.j) R and R^T (d_.j o x_.j) that involve u (known_block = 0, every outer
 * iteration) or only R_trunc (known_block = 1, once at set-up) */
int dmf_gram_panels(dmf_batch_t b, int32_t known_block, void* stream);
/* n_iter2 update_alpha iterations incl. simplex projection (deconvolution.py:94-101, :21-37), or Frank-Wolfe iterations
 * (deconvolution.py:285-299) for purity batches, per sample on (G_j, bx_j) */
int dmf_gram_alpha_inner(dmf_batch_t b, int32_t n_iter2, void* stream);
/* CpG rows sharded over several GPUs (one process per GPU, each batch holds its own row range of X, d_x, R_trunc, u and a
 * replica of alpha).  Every shape a batch can run can be sharded; the engine is chosen by shape: fused where it applies, then
 * the Gram form, then the stream engine.  With sharding on, the steps publish THIS GPU's sums in the `local` statistics block
 * of every fit and leave the fit state alone; the caller copies local -> global, all-reduces `global` over the GPUs (sum; max
 * for scal[3]) and then runs the step that reads `global`.  scal (8) = [cost, ||R_trunc||^2, ||u||^2 at set-up, max d_x,
 * ||u||^2 after the U step, unused].  Every rank ends up with the identical state and alpha.  Fits are doubles_per_fit apart
 * in both blocks.
 *   Gram form: blocks [G (Kt*Kt*N) | bx (Kt*N) | scal].  dmf_gram_rowgram -> scalars -> dmf_gram_finalize_cost;
 *     dmf_gram_u_inner + dmf_gram_panels -> blocks -> dmf_gram_alpha_inner.
 *   Stream engine (shapes without the Gram form): blocks [alpha gradient (Kt*N) | scal].  dmf_pass_init / dmf_pass_cost ->
 *     scalars -> dmf_gram_finalize_cost; n_iter2 x dmf_pass_u -> scalars -> dmf_pass_u_commit (l_h from the reduced ||u||^2);
 *     n_iter2 x (dmf_pass_alpha or dmf_pass_fw(k) -> blocks -> dmf_pass_alpha_commit(k)), the projected-gradient or Frank-Wolfe
 *     step on the reduced gradient.  dmf_enqueue_outer / dmf_fit_batched refuse such batches; the dmf_pass_* calls and the two commits
 * refuse sharded batches on the fused or Gram-form engine. */
int dmf_batch_set_sharded(dmf_batch_t b, int32_t on, void* stream);
int dmf_batch_stats_buffers(dmf_batch_t b, void** local_dev, void** global_dev, int64_t* doubles_per_fit, int64_t* scal_offset);
int dmf_gram_finalize_cost(dmf_batch_t b, int32_t initial, double tol, void* stream);
int dmf_pass_u_commit(dmf_batch_t b, void* stream);
int dmf_pass_alpha_commit(dmf_batch_t b, int32_t k_inner, void* stream);
/* Row-sharded runs, all-reduce over NVLink PEER MEMORY instead of NCCL: every rank provides a zero-initialised symmetric buffer of
 * dmf_batch_peer_bytes() bytes that all ranks of the box have mapped (peer_bases[r] = rank r's buffer as addressable from THIS
 * process, e.g. torch symmetric memory's buffer_ptrs).  dmf_gram_exchange is then ONE kernel per rank that pushes this rank's sums
 * into every rank's buffer, signals, waits for all ranks and adds the slots in rank order into the `global` statistics block
 * (which: 0 whole blocks before dmf_gram_alpha_inner; 1 the cost scalars before dmf_gram_finalize_cost; 2 the same at set-up, where
 * max d_x is max-reduced).  Every rank must issue the same sequence of exchanges. */
int dmf_batch_peer_bytes(dmf_batch_t b, int32_t world, size_t* bytes);
int dmf_batch_set_peers(dmf_batch_t b, int32_t rank, int32_t world, const void* const* peer_bases, size_t bytes_per_peer, void* stream);
int dmf_gram_exchange(dmf_batch_t b, int32_t which, void* stream);
/* The extrapolation weights of deconvolution.py:83-85 are data independent; the library keeps them in a device table that
 * grows on demand (growth allocates and synchronises).  Reserving n_inner_total inner iterations up front makes every later
 * dmf_gram_* call allocation- and sync-free, so that an outer iteration can be captured into a CUDA graph. */
int dmf_batch_reserve_momentum(dmf_batch_t b, int64_t n_inner_total, void* stream);
/* set-up (rowgram initial + known panels) and one whole outer iteration (u_inner, panels, alpha_inner, rowgram) */
int dmf_gram_init(dmf_batch_t b, void* stream);
int dmf_gram_outer(dmf_batch_t b, int32_t n_iter2, double tol, void* stream);

/* Fused engine: one outer iteration of deconvolution.py:206-221 / :320-335 as ONE streaming pass + the per-sample kernel.
 * dmf_fused_outer = [cost_f_w of the incoming iterate and, when that iterate closes an outer iteration, the |cf - cf_0| < tol
 * test (:218-221); update_u x n_iter2 (:82-89); Gram panel with the new u] + dmf_gram_alpha_inner.  Set-up is dmf_gram_init.
 * After the last dmf_fused_outer the cost of the final iterate is still pending: dmf_fused_finish evaluates it (one cost-only
 * pass; counts the outer iteration, runs the test).  dmf_fit_batched does all of this.  fused_pass alone (no alpha step) is
 * exposed for timing. */
int dmf_fused_pass(dmf_batch_t b, int32_t n_iter2, double tol, void* stream);
int dmf_fused_outer(dmf_batch_t b, int32_t n_iter2, double tol, void* stream);
int dmf_fused_finish(dmf_batch_t b, double tol, void* stream);
/* Row-sharded batches (dmf_batch_set_sharded): dmf_fused_pass publishes THIS GPU's cost, ||u||^2 and panel in the `local`
 * statistics block and leaves the fit state alone; after the blocks are all-reduced into `global` (dmf_gram_exchange(0) or
 * NCCL) dmf_fused_alpha_commit runs the termination test, commits the U step and runs the alpha iterations - identically on
 * every rank.  ONE collective per outer iteration.  dmf_fused_finish is then dmf_gram_rowgram + scalar all-reduce +
 * dmf_gram_finalize_cost as for the Gram engine. */
int dmf_fused_alpha_commit(dmf_batch_t b, int32_t n_iter2, double tol, void* stream);

/* whole loops --------------------------------------------------------------------------------- */
/* enqueue n_outer outer iterations (n_iter2 U steps, n_iter2 alpha/FW steps, cost) without host sync;
 * fits that reach termination skip their remaining launches on the device. */
int dmf_enqueue_outer(dmf_batch_t b, int32_t n_outer, int32_t n_iter2, double tol, void* stream);
/* mdwbssmf_deconv / mdwbssmf_deconv_p / unsupervised_deconv for every fit of the batch: init pass,
 * then outer iterations until every fit terminated or n_iter1 is reached.  Blocks the calling thread. */
int dmf_fit_batched(dmf_batch_t b, int32_t n_iter1, int32_t n_iter2, double tol, void* stream);
/* copy per-fit state to host (synchronises the stream) */
int dmf_batch_read_state(dmf_batch_t b, dmf_fit_state_t* out_host, int32_t n, void* stream);
/* number of kernel launches issued through this batch since creation */
int dmf_batch_launch_count(dmf_batch_t b, int64_t* out);

/* reference-based fit ---------------------------------------------------------------------------- */
/* wls_intercept (init_func.py:8-14) for every sample column at once:
 *   out[:, j] = c_j / max(sum c_j, 1e-10),  c_j = argmin_{c >= 0, b} sum_m D[m,j] (y[m,j] - [R1|R2][m,:] c - b)^2
 * with y = X (y_is_dx = 0; the `uniform` / SVD inits, deconvolution.py:51, init_func.py:23) or y = D o X
 * (y_is_dx = 1; the nbunknown = 0 path, demethify.py:212 and bootstrap.py:42).  R2 (M x K2, pitch ldr2) is an
 * optional second block of regressors (the unknown profiles u in deconvolution.py:51), NULL when K2 = 0.
 * Same pitch rules as dmf_shape_t (even, zero padded).  out is a DEVICE buffer of (K + K2) x N doubles. */
typedef struct dmf_wls_desc {
    int64_t M;
    int32_t N, K, K2;
    int32_t dtype, wtype;
    int32_t y_is_dx, reserved;
    int64_t ldx, ldd, ldr, ldr2;
    const void* X;
    const void* D;
    const void* R1;
    const void* R2;
    double* out;
} dmf_wls_desc_t;
int dmf_wls_workspace_bytes(dmf_handle_t h, const dmf_wls_desc_t* d, size_t* bytes);
int dmf_wls_fit(dmf_handle_t h, const dmf_wls_desc_t* d, void* workspace_dev, size_t workspace_bytes, void* stream);
/* dmf_wls_fit in two halves, for CpG rows sharded over several GPUs.  dmf_wls_moments streams the caller's M rows and writes the
 * weighted moment matrix  mom[(p Kz + q) N + j] = sum_m D[m,j] z_p z_q,  z = [1, y, R1 row, R2 row],  Kz = K + K2 + 2  (DEVICE
 * buffer of Kz Kz N doubles; all zero when M = 0).  dmf_wls_solve runs the per-sample NNLS on a moment matrix the caller may have
 * summed over GPUs: it reads M (the GLOBAL row count: the NNLS tolerance depends on it), N, K, K2 and out from the descriptor and
 * needs 256 bytes of workspace.  Moments then solve on one GPU give dmf_wls_fit's result bit for bit. */
int dmf_wls_moments(dmf_handle_t h, const dmf_wls_desc_t* d, double* mom, void* workspace_dev, size_t workspace_bytes, void* stream);
int dmf_wls_solve(dmf_handle_t h, const dmf_wls_desc_t* d, const double* mom, void* workspace_dev, size_t workspace_bytes, void* stream);

/* NNDSVD of the floored residual over row-sharded rows (init_func.py:17-93) ------------------------------------------------ */
/* r_mj = max(X[m,j] - sum_k R[m,k] H1[k,j], 1e-8) for K > 0 (the partial / purity SVD init), r_mj = X[m,j] for K = 0 (the
 * reference-free SVD init).  X (M x ldx) and R (M x ldr) are fp64 with even, zero-padded pitches; H1 is K x N row-major;
 * N <= 512.  The residual is formed on the fly and never written to memory.  M = 0 is allowed (a GPU without rows). */
typedef struct dmf_resid_desc {
    int64_t M;
    int32_t N, K;
    int64_t ldx, ldr;
    const double* X;
    const double* R;
    const double* H1;
} dmf_resid_desc_t;
int dmf_resid_workspace_bytes(dmf_handle_t h, const dmf_resid_desc_t* d, size_t* bytes);
/* G = sum_m r_m r_m^T over the caller's rows (N x N, DEVICE, fp64 on the tensor cores; bit-reproducible for a given device and
 * shape).  *has_negative (DEVICE int32) becomes 1 when K = 0 and X has a negative entry, else 0. */
int dmf_resid_gram(dmf_handle_t h, const dmf_resid_desc_t* d, double* G, int32_t* has_negative, void* workspace_dev,
                   size_t workspace_bytes, void* stream);
/* U = r Vh^T diag(inv_sigma) for the caller's rows (M x rank row-major; Vh is rank x N row-major, rank <= 32), and
 * sums[i] = sum_m max(U[m,i], 0)^2, sums[rank + i] = sum_m max(-U[m,i], 0)^2 over the caller's rows (DEVICE, 2 rank doubles). */
int dmf_resid_project(dmf_handle_t h, const dmf_resid_desc_t* d, const double* Vh, const double* inv_sigma, int32_t rank, double* U,
                      double* sums, void* workspace_dev, size_t workspace_bytes, void* stream);
/* dmf_nndsvd_split's rule on the caller's rows of U with the norms of U taken from `sums` (dmf_resid_project's sums added over
 * all GPUs): W (M x rank, the caller's rows) and H (rank x N), both row-major. */
int dmf_nndsvd_apply(const double* U, int64_t M, const double* Vh, const double* S, const double* sums, int32_t N, int32_t rank,
                     double* W, double* H, void* stream);

/* utilities ------------------------------------------------------------------------------------ */
/* narrow fp64/fp32/int64 coverage to u16 with range/integrality check; *bad receives the number of
 * entries that are not integers in [0, 65535] (device int32) */
int dmf_pack_weights_u16(const void* src, int32_t src_kind /*0 f64, 1 f32, 2 i64*/, int64_t count,
                         uint16_t* dst, int32_t* bad_dev, void* stream);
/* dst[p, :] = src[rows[p], :] row gather (sklearn.utils.resample, bootstrap.py:28), elem_bytes in {1,2,4,8} */
int dmf_gather_rows(const void* src, const int32_t* rows, int64_t n_rows, int64_t row_elems,
                    int32_t elem_bytes, void* dst, void* stream);

/* the steps right before / after the path (SURVEY.md 8 f4) ------------------------------------------ */
/* NNDSVD (init_func.py:40-69) on the factors of a thin SVD (device pointers; U is M x ldu row-major, Vh is r x ldv):
 * W (M x rank) and H (rank x N) row-major; component 0 = sqrt(S_0) |u_0|, |v_0|; component i >= 1 = the sign pattern with the
 * larger product of norms, scaled by sqrt(S_i term) / norm; entries < 1e-11 are set to 0 (flag = 0 of the reference). */
int dmf_nndsvd_split(const double* U, int64_t ldu, const double* S, const double* Vh, int64_t ldv, int64_t M, int32_t N, int32_t rank,
                     double* W, double* H, void* stream);
/* np.percentile(stack, [q_lo, q_hi], axis=0), default linear rule (bootstrap.py:53-54, :77-78): stack is B x P row-major (one row
 * per resample), q in percent.  Selection per entry, no sort; needs floor((B-1) q_lo/100) + 2 and B - floor((B-1) q_hi/100) to be
 * at most dmf_percentile_max_keep() (DMF_E_SHAPE otherwise). */
int dmf_percentile_max_keep(void);
int dmf_percentile_bounds(const double* stack, int32_t B, int64_t P, double q_lo, double q_hi, double* out_lo, double* out_hi, void* stream);
/* The legacy numpy streams a bootstrap resample draws (SURVEY.md 8 f2), bit for bit, one warp per stream.  For stream b, with
 * seed = seeds[b] (DEVICE array of n_streams uint32):
 *   idx   != NULL:  idx[b * ld_idx + i]  = RandomState(seed).randint(0, M, size=M)[i]      (sklearn.utils.resample, bootstrap.py:28)
 *   u     != NULL:  u[b * ld_u + i]      = RandomState(seed).uniform(size=n_dbl)[i]        (set_seed + rd.uniform, deconvolution.py:9-11, :54-55)
 *   state != NULL:  state[b * 625 ..]    = the 624 key words and pos of that generator AFTER the n_dbl doubles, so that the host can
 *                                          continue the stream (RandomState.set_state) with the small draws that follow (dirichlet).
 * MT19937 as numpy seeds and steps it; randint = masked rejection on 32-bit outputs; uniform = ((a >> 5) 2^26 + (b >> 6)) / 2^53. */
int dmf_rng_legacy_streams(const uint32_t* seeds, int32_t n_streams, int64_t M, int32_t* idx, int64_t ld_idx, int64_t n_dbl, double* u,
                           int64_t ld_u, uint32_t* state, void* stream);
/* compute_consensus_matrix (ic.py:24-37): alpha_runs is n_runs x Kt x N, labels_ws n_runs x N int32 scratch, consensus N x N. */
int dmf_consensus(const double* alpha_runs, int32_t n_runs, int32_t Kt, int32_t N, int32_t* labels_ws, double* consensus, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DEMETHIFY_B200_H */
