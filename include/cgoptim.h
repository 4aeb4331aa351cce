/*
 * cgoptim.h — C ABI of libcgoptim.so: the B200-native (sm_100a) per-iteration hot path of
 * ConjugateGradientOptim.jl (reference citations are file:line under /root/reference).
 *
 * The reference is pure Julia and has no FFI; these entry points are what a Julia host would
 * `ccall` (see INTEGRATION.md and julia/) to replace every vector-touching line of
 * `minimizeobjective` (src/engine/optim.jl:6-171).  All scalar logic (line-search state
 * machines, β formulas, statuses, restarts) stays in the host language.
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on a CUDA / NCCL / argument error;
 *    cgo_last_error() then returns a thread-local message.  Numerical trouble (NaN, Inf) is
 *    DATA, returned as-is for the host to classify exactly like optim.jl:53,108 do.
 *  - host pointers are borrowed for the duration of one call; device memory is owned by the
 *    opaque handles.  One host thread drives one ctx; distinct ctxs are independent.
 *  - every call is synchronous at return (its kernels ran on the ctx stream and the scalar
 *    pack was read back).
 *  - FP64 only (the reference's `a_initial = NaN` literal pins T = Float64, SURVEY.md §7.4-8).
 *
 * Canonical reduction order (what makes every dot product run-to-run and launch-config
 * independent, and bit-reproducible by oracle/cgo_oracle.c in ORC_SUM_CGO mode):
 *   items are visited in index order; item i belongs to lane t = q % 256 of virtual CTA
 *   c = (q / (256*U)) % G with q = i / V.  BLAS-1 kernels read 128-bit double2 (V=2, U=4);
 *   row-per-lane CSR kernels use V=1, U=1.  Each (c,t) accumulates its terms sequentially from
 *   +0.0; the 256 lanes of a virtual CTA are combined by a xor-butterfly (16,8,4,2,1) inside
 *   each warp, then sequentially over the 8 warps; the min(G, ntiles) CTA partials are combined
 *   by the last-arriving block in exactly the same way (lane t takes partials t, t+256, ...).
 *   Long rows (logistic regression from a host CSR, cgo_obj_logreg_create_csr, on the k_spmv_direct family): a row
 *   of A or Aᵀ with more than CGO_LONG_ROW entries is summed in this order too — its products val_k · x[col_k], k in
 *   storage order, are the items, with V=1, U=4 and the ctx's G.  The softmax objective (cgo_obj_softmax_create_csr)
 *   applies the rule to A ⊗ I_K: for each class k, the items of a long row are val_k · x[col_k·K + k].  An intercept
 *   (cgo_obj_logreg_create_csr_ex / cgo_obj_softmax_create_csr_ex) has the unit row: a row of Aᵀ that is not stored,
 *   with entry 1.0 at every sample.  Its items are 1.0 · c_i (1.0 · c_ik for class k), summed in the long-row order
 *   (V=1, U=4, the ctx's G) whatever N is.  Every other row of every CSR matrix is summed sequentially in storage order.
 *   CSR matrices whose gathers do not coalesce (the synthetic least-squares matrix with coh_log2 < 4; a host
 *   CSR whose warp-level gathers touch more than four lines on average: cgo_obj_reduction_site tells) are
 *   multiplied by a kernel without reductions, and their dots come from BLAS-1 passes (V=2, U=4).
 *   G defaults to 296 (= 2 persistent CTAs on each of a B200's 148 SMs, whatever the device: one
 *   sweep over the data by the whole grid) and is a property of the ctx.  With R ranks every rank
 *   reduces its contiguous shard this way; the R shard results are all-gathered and added in
 *   rank order on every rank.
 */
#ifndef CGOPTIM_H
#define CGOPTIM_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cgo_ctx cgo_ctx;
typedef struct cgo_obj cgo_obj;
typedef struct cgo_state cgo_state;

#define CGO_PACK_LEN 16

/* scalar pack written by cgo_eval_trial*, with g⁺ = df_xp, g = df_x, y = g⁺ − g (elementwise) */
enum {
    CGO_P_PHI = 0,   /* ϕ(a) = f(x + a u)                                 cg_utils.jl:18 */
    CGO_P_DPHI = 1,  /* g⁺·u                                              cg_utils.jl:20 */
    CGO_P_GPGP = 2,  /* g⁺·g⁺  (norm(info.df_xp)² optim.jl:107)                          */
    CGO_P_YY = 3,    /* y·y                                               cg_flavours.jl:67,73,102 */
    CGO_P_UY = 4,    /* u·y                                               cg_flavours.jl:66,98,167 */
    CGO_P_YGP = 5,   /* y·g⁺                                              cg_flavours.jl:67,166 */
    CGO_P_GPG = 6,   /* g⁺·g                                              cg_flavours.jl:141 */
    CGO_P_UG = 7,    /* u·g   (= dϕ(0), nocedal.jl:56; cg_flavours.jl:145) */
    CGO_P_UU = 8,    /* u·u   (cg_flavours.jl:65)                                              */
    /* reduced by the BLAS-1 kernel that wrote u (the same numbers as slots 7/8 for one-kernel
     * objectives; for CSR objectives a different canonical-order site):                       */
    CGO_P_DIR_GU = 9,   /* g·u = dϕ(0) of the NEXT line search (nocedal.jl:56, wolfe.jl:40, geometric.jl:43) */
    CGO_P_DIR_UU = 10,  /* u·u  (wolfe.jl:240, geometric.jl:52)                               */
    CGO_P_XPXP = 11     /* xp·xp (ℓ2 regulariser of the logistic-regression objective)        */
};
/* pack written by cgo_update_dir / cgo_reset_direction / cgo_lbfgs_update_dir */
enum { CGO_D_GU = 0 /* g·u, the next dϕ(0) */, CGO_D_UU = 1 /* u·u */ };

/* status Symbols of the reference as integers (batched on-device solver; host code uses the
 * same numbering).  SURVEY.md §5 lists the file:line of each. */
enum {
    CGO_ST_INCOMPLETE = 0, CGO_ST_SUCCESS = 1, CGO_ST_INCREASING_OBJECTIVE = 2,
    CGO_ST_MAX_ITERS_REACHED = 3, CGO_ST_NON_FINITE_PROPOSED = 4, CGO_ST_NON_DESCENT = 5,
    CGO_ST_A_MAX_OVERFLOW = 6, CGO_ST_LS_MAX_ITERS = 7, CGO_ST_ZOOM_MAX_ITERS = 8,
    CGO_ST_ACCEPTED_NON_FINITE = 9, CGO_ST_NO_INITIAL_FEASIBLE = 10, CGO_ST_MAX_STEP_LENGTH = 11,
    CGO_ST_NO_FEASIBLE_STEP = 12, CGO_ST_NON_FINITE_STEP = 13, CGO_ST_SAME_STEP = 14,
    CGO_ST_BRACKET_PRECISION = 15, CGO_ST_LINESEARCH_FAILED = 16 /* solve_system.jl:140 */,
    CGO_ST_INFEASIBLE_START = 17, CGO_ST_CENTERING_STEP_ISSUE = 18 /* primal_barrier.jl:189, :223 */
};

/* ---------------------------------------------------------------- context ---------------- */
const char *cgo_last_error(void);
int cgo_version(void);
/* `cuda_stream`: a cudaStream_t to launch on, or NULL to let the ctx create its own. */
int cgo_ctx_create(int device, void *cuda_stream, cgo_ctx **out);
int cgo_ctx_destroy(cgo_ctx *ctx);
int cgo_ctx_stream(cgo_ctx *ctx, void **cuda_stream_out);
int cgo_ctx_set_reduction_ctas(cgo_ctx *ctx, int G);        /* canonical-order G (default 296) */
/* objectives whose gathers range over a vector larger than this are stored column-blocked and
 * evaluated one block per pass, so that the gathered window stays L2-resident (default 40 MiB;
 * 0 = never block).  Column blocks apply to the k_spmv_direct family (cgo_ctx_set_csr_mode): an
 * objective forced onto k_csr_rows runs single-pass.  Applies to objectives created afterwards;
 * results are bit-identical. */
int cgo_ctx_set_gather_block_bytes(cgo_ctx *ctx, int64_t bytes);
/* which SpMV kernel family CSR objectives created afterwards use: 0 = per matrix (default: k_spmv_direct + BLAS-1
 * dots when its gathers do not coalesce, the fused k_csr_rows otherwise), 1 = always k_csr_rows, 2 = always
 * k_spmv_direct (environment CGO_CSR_MODE).  Changes the canonical order of the dots (cgo_obj_reduction_site),
 * not the row sums. */
int cgo_ctx_set_csr_mode(cgo_ctx *ctx, int mode);
/* the ctx keeps the vectors of destroyed states for the next state of the same size (cudaMalloc / cudaFree of GB-sized
 * blocks cost milliseconds and synchronise the device): up to 24 GB.  This gives them back to the driver. */
int cgo_ctx_trim_pools(cgo_ctx *ctx, int64_t *freed_bytes);
int cgo_ctx_sm_count(cgo_ctx *ctx, int *sms);
int cgo_ctx_kernel_launches(cgo_ctx *ctx, int64_t *count);  /* kernels launched so far */
/* optional per-launch CUDA-event timing on the ctx stream, by kernel class:
 * 0 trial (fused evalϕdϕ!), 1 direction, 2 axpy(+dir), 3 SpMV, 4 SpMVᵀ, 5 L-BFGS, 6 other, 7 batched */
int cgo_ctx_timing(cgo_ctx *ctx, int enable);
int cgo_ctx_timing_read(cgo_ctx *ctx, double ms[8], int64_t counts[8], int reset);
/* multi-GPU: one process per GPU.  Rank 0 calls cgo_comm_get_unique_id and the host broadcasts
 * the 128 bytes (torch.distributed / MPI / files); every rank then calls cgo_ctx_comm_init.  */
int cgo_comm_get_unique_id(void *id128);
int cgo_ctx_comm_init(cgo_ctx *ctx, int nranks, int rank, const void *id128);
int cgo_ctx_barrier(cgo_ctx *ctx);
/* 1 when the ranks mapped each other's device memory (CUDA IPC over NVLink / NVSwitch): halo
 * exchanges are then stores fused into the producing kernels plus a flag hand-off, instead of
 * NCCL point-to-point transfers.  Environment CGO_NO_PEER=1 forces the NCCL path. */
int cgo_ctx_peer_memory(cgo_ctx *ctx, int *enabled);
/* page-locked host memory (Results.minimizer / Results.gradient land in it at PCIe speed; x_initial
 * may live in it too).  Plain pageable pointers are accepted everywhere, just slower. */
int cgo_host_alloc(size_t bytes, void **out);
int cgo_host_free(void *ptr);
/* contiguous shard [lo,hi) of n items for `rank` of `nranks`, boundaries multiples of `align` */
int cgo_shard_range(int64_t n, int nranks, int rank, int64_t align, int64_t *lo, int64_t *hi);

/* ---------------------------------------------------------------- objectives --------------
 * Device-resident replacements of the user callback fdf!(g, x) -> f (optim.jl:25,
 * cg_utils.jl:18).  With a communicator on the ctx the constructors build this rank's shard. */
/* ANY objective: the device form of the reference's user callback fdf!(g, x) -> f.  `fdf` is called once per trial
 * on the host thread that drives the ctx and must ENQUEUE on `cuda_stream` (a cudaStream_t, the ctx stream) the
 * work that, from the trial point xp_dev[0..n_local) (this rank's shard, global offset `offset`), writes the
 * gradient to g_dev[0..n_local) and this rank's part of f to *f_dev (one device double; the ranks' parts are added
 * in rank order).  It returns 0, or non-zero to abort the trial (reported as an error of cgo_eval_trial).  It must
 * not synchronise the stream.  Everything else of evalϕdϕ! / getβ (xp = x + a u, dϕ, ‖g⁺‖², the β dots) is the
 * library's.  n_global even (pad an odd problem with one fixed coordinate). */
typedef int (*cgo_user_fdf)(void *user, void *cuda_stream, int64_t n_local, int64_t offset,
                            const double *xp_dev, double *g_dev, double *f_dev);
int cgo_obj_user_create(cgo_ctx *ctx, int64_t n_global, cgo_user_fdf fdf, void *user, cgo_obj **out);
/* extended Rosenbrock (pairs) f = Σ 100 (x_{2i} − x_{2i−1}²)² + (1 − x_{2i−1})², n_global even */
int cgo_obj_rosenbrock_create(cgo_ctx *ctx, int64_t n_global, cgo_obj **out);
/* the reference's own chained Rosenbrock, rosenbrockfunc of examples/helpers/test_funcs.jl:50-57 with its
 * hand-derived gradient (SURVEY.md §8d cfg 1): f = Σ_{i<n} (1 − x_i)² + 100 (x_{i+1} − x_i²)²; sharded runs keep a
 * ±1 halo of the trial point, pushed over peer memory by the kernel that forms it.  n_global even. */
int cgo_obj_rosenbrock_chained_create(cgo_ctx *ctx, int64_t n_global, cgo_obj **out);
/* ½‖Ax − b‖², A n×n banded-random CSR generated on device (generator spec: DESIGN.md §objectives;
 * restated in oracle/cgo_oracle.c orc_obj_sparse_ls_synth), b = A x_true. */
int cgo_obj_sparse_ls_create_synthetic(cgo_ctx *ctx, int64_t n_global, int32_t nnz_per_row,
                                       int64_t W, uint64_t seed, int32_t coh_log2, cgo_obj **out);
/* ½‖Ax − b‖² from a host CSR (int64 row pointers, int32 columns), single GPU */
int cgo_obj_sparse_ls_create_csr(cgo_ctx *ctx, int64_t nrows, int64_t ncols, const int64_t *rowptr,
                                 const int32_t *col, const double *val, const double *b,
                                 cgo_obj **out);
/* (1/N) Σ log(1 + exp(−y_i a_i·w)) + (λ/2)‖w‖², synthetic CSR.  With R ranks the samples (rows of A)
 * and the features (state vectors) are both sharded contiguously (cgo_shard_range, align 2): per
 * trial the shards of xp are all-gathered, every rank forms Aᵀ_r c_r over all features, the shard
 * slices are exchanged all-to-all and added in rank order (deterministic for a fixed R). */
int cgo_obj_logreg_create_synthetic(cgo_ctx *ctx, int64_t nsamples, int64_t nfeat,
                                    int32_t nnz_per_row, uint64_t seed, double lambda,
                                    cgo_obj **out);
/* rows of more than CGO_LONG_ROW entries (an intercept's column of ones is a row of Aᵀ with nsamples entries) are
 * summed by the whole grid in the canonical order instead of on one lane (see the canonical reduction order above) */
#define CGO_LONG_ROW 1024
/* (1/N) Σ log(1 + exp(−y_i a_i·w)) + (λ/2)‖w‖² from a host CSR (int64 row pointers, int32 columns, 0-based), labels
 * y_i ∈ {−1, +1}; single GPU.  A column of ones is an intercept that λ penalises like every other weight
 * (cgo_obj_logreg_create_csr_ex fits one that it does not penalise).  Every
 * matrix with a row longer than CGO_LONG_ROW runs on k_spmv_direct; forced onto k_csr_rows (cgo_ctx_set_csr_mode 1)
 * it keeps sequential row sums, exact but slow on long rows. */
int cgo_obj_logreg_create_csr(cgo_ctx *ctx, int64_t nsamples, int64_t nfeat, const int64_t *rowptr,
                              const int32_t *col, const double *val, const double *y, double lambda, cgo_obj **out);
/* (1/N) Σ_i [log Σ_k exp(z_ik) − z_{i,y_i}] + (λ/2)‖W‖², z_i = a_i W, from a host CSR (0-based int64 row pointers,
 * int32 columns) and labels y_i ∈ [0, K); single GPU.  The state vector is W (nfeat × nclasses) feature-major:
 * w[j·K + k], n = nfeat·nclasses.  2 <= K <= 256.  Z = A W is the SpMV of A ⊗ I_K on the flat W, and every row sum
 * follows that matrix's order (long rows included).  Runs on the K-column SpMM whatever cgo_ctx_set_csr_mode says,
 * except mode 1, which is rejected.  No Hessian-vector product or quadratic-aware line search.  The CSR test hooks
 * return A / Aᵀ; cgo_obj_spmv takes and returns K-wide vectors (Z = A W, d·K → N·K; Aᵀ C, N·K → d·K). */
int cgo_obj_softmax_create_csr(cgo_ctx *ctx, int64_t nsamples, int64_t nfeat, int32_t nclasses,
                               const int64_t *rowptr, const int32_t *col, const double *val,
                               const int32_t *labels, double lambda, cgo_obj **out);
/* The two objectives above with per-sample weights and an intercept that λ does not penalise:
 *   binary   f(w, b) = (1/S) Σ_i s_i log(1 + exp(−y_i (a_i·w + b))) + (λ/2)‖w‖²
 *   softmax  f(W, b) = (1/S) Σ_i s_i [logsumexp(a_i W + b) − (a_i W + b)_{y_i}] + (λ/2)‖W‖²
 * with S = Σ_i s_i, correctly rounded on the host.  sample_weight: N finite weights >= 0 with S > 0, or NULL for unit
 * weights (S = N).  fit_intercept 0 or 1.  The intercept is feature nfeat: the binary state is (w, b), n = nfeat + 1,
 * x[nfeat] = b; the softmax state is feature-major W with b as its last row, n = (nfeat + 1)·K, b_k = x[nfeat·K + k].
 * It is the layout of an explicit ones column appended as feature nfeat, which A no longer needs to store.
 * Arithmetic: the margins are the row sums of A plus b (b_k); the loss op reduces s_i ℓ_i and writes c_i = s_i·(−y_i σ_i)
 * (c_ik = s_i·(p_ik − [k = y_i])); the intercept's gradient is the sum of the unit row (see the canonical order above)
 * times 1/S; a feature's gradient is (Aᵀc)_j / S + λ w_j; f = Σ/S + (λ/2) P, where P is xp·xp reduced by K_a with +0.0
 * in place of every intercept coordinate's square.  With (NULL, 0) these are the constructors above.  Otherwise the
 * objective runs on k_spmv_direct (binary) or the SpMM (softmax) and rejects cgo_ctx_set_csr_mode 1.  Single GPU; no
 * Hessian-vector product or quadratic-aware line search.  cgo_obj_spmv(transposed = 1) returns all n entries: Aᵀc
 * followed by the intercept's sums; transposed = 0 multiplies A by the feature part; the CSR download returns A. */
int cgo_obj_logreg_create_csr_ex(cgo_ctx *ctx, int64_t nsamples, int64_t nfeat, const int64_t *rowptr,
                                 const int32_t *col, const double *val, const double *y, const double *sample_weight,
                                 int32_t fit_intercept, double lambda, cgo_obj **out);
int cgo_obj_softmax_create_csr_ex(cgo_ctx *ctx, int64_t nsamples, int64_t nfeat, int32_t nclasses,
                                  const int64_t *rowptr, const int32_t *col, const double *val,
                                  const int32_t *labels, const double *sample_weight, int32_t fit_intercept,
                                  double lambda, cgo_obj **out);
/* t·f0(x) − Σ log(ubs − x) − Σ log(x − lbs) around `inner` (which must outlive it): evalbarrier!
 * (src/engine/primal_barrier.jl:112-133) with the box constraints of examples/constrained.jl:17-47;
 * lbs / ubs are this rank's shard.  cgo_obj_barrier_set_t changes t between centering steps (:246);
 * cgo_obj_barrier_infeasible counts the coordinates of x (host, this rank's shard; all ranks' counts
 * are added) with fi >= 0, the feasibility test of :187-198. */
int cgo_obj_box_barrier_create(cgo_ctx *ctx, cgo_obj *inner, const double *lbs_host, const double *ubs_host,
                               double t, cgo_obj **out);
int cgo_obj_barrier_set_t(cgo_obj *obj, double t);
int cgo_obj_barrier_infeasible(cgo_obj *obj, const double *x_host, int64_t *count);
int cgo_obj_destroy(cgo_obj *obj);
int cgo_obj_dims(cgo_obj *obj, int64_t *n_local, int64_t *n_global, int64_t *offset);
/* canonical-order mapping (V, U) of the kernels that reduce this objective's trial dots: (2, 4) when a BLAS-1
 * kernel does (Rosenbrock, the barrier, gather-bound CSR matrices), (1, 1) for the row-per-lane CSR kernels */
int cgo_obj_reduction_site(cgo_obj *obj, int32_t *V, int32_t *U);
int cgo_obj_bytes_per_eval(cgo_obj *obj, double *bytes);   /* algorithmic HBM bytes of one fdf! on this rank */
/* synthetic start / truth vectors (this rank's shard), for hosts and tests */
int cgo_obj_default_x0(cgo_obj *obj, uint64_t seed, double perturb, double *x0_host);
/* test hooks: CSR download (transposed = 0/1) and y = A x / Aᵀ x on device, single GPU */
int cgo_obj_csr_nnz(cgo_obj *obj, int transposed, int64_t *nrows, int64_t *nnz);
int cgo_obj_csr_blocks(cgo_obj *obj, int transposed, int32_t *nblocks);   /* passes per SpMV (1 = unblocked) */
int cgo_obj_csr_download(cgo_obj *obj, int transposed, int64_t *rowptr, int32_t *col, double *val,
                         double *b);
int cgo_obj_spmv(cgo_obj *obj, int transposed, const double *x_host, double *y_host);

/* ---------------------------------------------------------------- solver state ------------
 * Device-side LineSearchContainer (types.jl:84-100: xp, df_xp, x, u) plus df_x, and the
 * L-BFGS history when lbfgs_m > 0.  cgo_state_create does optim.jl:20-26 (copies x0, evaluates
 * f and g there): out[CGO_P_PHI] = f(x0), out[CGO_P_GPGP] = ‖g‖². */
int cgo_state_create(cgo_ctx *ctx, cgo_obj *obj, const double *x0_host, int32_t lbfgs_m,
                     cgo_state **out_state, double out[CGO_PACK_LEN]);
/* the same with x0 = vector `which` (0 x, 1 g, 2 u, 3 xp, 4 g⁺) of a live state of the same dimension: the restart
 * of minimizeobjectivererun (optim.jl:191-201: the next attempt starts from rets[end].minimizer) and the centering
 * steps of primalbarriermethod! (primal_barrier.jl:215-247) without a host round trip — one D2D copy, no H2D.
 * `obj` may differ from the source state's objective (the barrier objective changes t between steps). */
int cgo_state_create_from_state(cgo_ctx *ctx, cgo_obj *obj, cgo_state *src, int32_t which, int32_t lbfgs_m,
                                cgo_state **out_state, double out[CGO_PACK_LEN]);
int cgo_state_destroy(cgo_state *st);
/* initializeLineSearchContainer! (cg_flavours.jl:22-35) and wolfe.jl:129: u = −g.
 * out[CGO_D_GU], out[CGO_D_UU]. */
int cgo_reset_direction(cgo_state *st, double out[CGO_PACK_LEN]);
/* evalϕdϕ! (cg_utils.jl:3-22) fused with every dot the β flavours need: xp = x + a u,
 * g⁺ = ∇f(xp); fills the CGO_P_* pack. */
int cgo_eval_trial(cgo_state *st, double a, double out[CGO_PACK_LEN]);
/* updatedir! (cg_flavours.jl:2-15) fused into the first trial of the next line search:
 * u = −g + β u, then as cgo_eval_trial.  CGO_P_UG / CGO_P_UU refer to the NEW u. */
int cgo_eval_trial_fused_dir(cgo_state *st, double beta, double a, double out[CGO_PACK_LEN]);
/* optim.jl:136-140: x ← xp, df_x ← df_xp, info.x ← x (pointer swaps, no kernel) */
int cgo_accept(cgo_state *st);
/* updatedir! (cg_flavours.jl:2-15): u = −g + β u.  out[CGO_D_GU], out[CGO_D_UU]. */
int cgo_update_dir(cgo_state *st, double beta, double out[CGO_PACK_LEN]);
/* cg_flavours.jl:71-76 / :100-105 as written: Σ (y_i − m u_i)(g⁺_i / R), y = g⁺ − g */
int cgo_beta_literal(cgo_state *st, double R, double m, double *beta_out);
/* norm(u + df_x)² (wolfe.jl:123) */
int cgo_norm_sq_u_plus_g(cgo_state *st, double *out);
/* L-BFGS (new flavour, N&W Alg 7.4/7.5): s = xp − x, y = g⁺ − g into the slot after the newest
 * pair; out[0] = s·y, out[1] = y·y.  `commit` != 0 makes it the newest pair with ρ = 1/s·y. */
int cgo_lbfgs_stage_pair(cgo_state *st, double out[CGO_PACK_LEN]);
int cgo_lbfgs_commit_pair(cgo_state *st, int32_t commit, double rho, double gamma);
/* two-loop recursion on the device: u = −H g.  out[CGO_D_GU], out[CGO_D_UU]. */
int cgo_lbfgs_update_dir(cgo_state *st, double out[CGO_PACK_LEN]);
/* solvesystem (src/engine/solve_system.jl:64-239, CG for nonlinear systems g(x) = 0).  The line
 * search (:29-55) is cgo_eval_trial; these are its three other vector steps:
 *  begin    x_next = copy(x) (:82);
 *  project  updateiteratesolvesys! (:237-253): x_next = base + m·df_xp, then f_x_next = fdf!(df_xp,
 *           x_next) (:179) with the usual pack (CGO_P_PHI = f(x_next), CGO_P_GPGP = ‖g(x_next)‖², getβ
 *           dots against the old df_x and u).  base = x_next as the reference writes it (which from
 *           the 2nd iteration on is the iterate BEFORE x), or x when fix_stale_iterate != 0;
 *  accept   x, x_next = x_next, x; df_x = df_xp; info.x = x (:196, :207-208). */
int cgo_solvesys_begin(cgo_state *st);
int cgo_solvesys_project(cgo_state *st, double m, int32_t fix_stale_iterate, double out[CGO_PACK_LEN]);
int cgo_solvesys_accept(cgo_state *st, int32_t fix_stale_iterate);
/* Quadratic-aware line search (SURVEY.md §8f N1) for ½‖Ax − b‖²: along x + a u the residual is r + a·Au,
 * so after ONE SpMV every trial of linesearch! (nocedal.jl:33-209, wolfe.jl:13-165) is scalar arithmetic:
 * ϕ(a) = ½ r·r + a r·v + ½ a² v·v, dϕ(a) = r·v + a v·v, v = A u.
 *   cgo_quad_begin   v = A u;  out[0] = r·v, out[1] = v·v, out[2] = r·r   (r: residual at x)
 *   cgo_quad_accept  the accepted step: xp = x + a u, r += a v, g⁺ = Aᵀ r and the pack of cgo_eval_trial
 *                    (CGO_P_PHI = ½ Σ r²), after which cgo_accept adopts (xp, g⁺) as usual.
 * One SpMV + one SpMVᵀ per iteration whatever the number of trials; decisions agree with the plain
 * path up to rounding of ϕ (tests/test_gpu_sparse_ls.py). */
int cgo_quad_begin(cgo_state *st, double out[CGO_PACK_LEN]);
int cgo_quad_accept(cgo_state *st, double a, double out[CGO_PACK_LEN]);
/* Hessian-vector product along the current direction, hv = ∇²f(x) u (CSR least squares: Aᵀ(A u), two
 * SpMV launches; the curvature a quadratic-aware line search needs — the reference engine itself
 * never forms one, src/engine/optim.jl:83-145).  out[0] = u·Hu (as ‖Au‖²), out[1] = u·hv, out[2] = hv·hv;
 * hv is readable with cgo_download_vector(st, 5, …). */
int cgo_hessvec_dir(cgo_state *st, double out[CGO_PACK_LEN]);
/* Results.minimizer / Results.gradient (types.jl:107-114): one D2H each; NULL skips */
int cgo_download(cgo_state *st, double *x_host, double *g_host);
/* test hook: 0 x, 1 g, 2 u, 3 xp, 4 g⁺, 5 hv */
int cgo_download_vector(cgo_state *st, int32_t which, double *host);

/* ---------------------------------------------------------------- batched solver ----------
 * SURVEY.md §8 cfg 5: many independent small problems, the whole of minimizeobjective
 * (optim.jl:6-171) + any of the three line searches (nocedal.jl, wolfe.jl, geometric.jl) + getβ
 * (cg_flavours.jl) on the device, one CTA per problem, all five n-vectors in registers.     */
typedef struct {
    double eps;             /* CGConfig.ϵ            types.jl:161 */
    int64_t max_iters;      /* CGConfig.max_iters    types.jl:164 */
    int32_t flavour;        /* 0 HagerZhang, 1 YuanWangSheng, 2 SallehAlhawarat, 3 LiuStorrey */
    int32_t linesearch;     /* 0 StrongWolfeBisection (nocedal.jl), 1 WolfeBisection{Wolfe}, 2 WolfeBisection{YuanWeiLuWolfe}
                               (wolfe.jl), 3 Backtracking{Armijo} (geometric.jl) */
    double mu;              /* YuanWangSheng.μ */
    double c1, c2, growth;  /* c1 (all), c2 (0-2), a_max_growth_factor (0)   nocedal.jl:3-11, wolfe.jl:213-262, geometric.jl:159 */
    int64_t ls_max_iters, zoom_max_iters;
    double delta1;          /* YuanWeiLuWolfe.δ1                 wolfe.jl:216 */
    double max_step_size;   /* WolfeBisection.max_step_size      wolfe.jl:9   */
    double discount;        /* Backtracking.discount_factor      geometric.jl:17 */
    int64_t feas_max_iters; /* feasibility_max_iters             wolfe.jl:10, geometric.jl:19 */
} cgo_batched_config;
/* lanes per problem of the batched kernel: the fewest warps (1, 2, 4, 8) that keep at most eight
 * element pairs per lane; its reductions follow the canonical order with B = 32·nwarp lanes, one tile */
int cgo_batched_layout(int32_t n, int32_t *nwarp, int32_t *pairs_per_lane);
/* extended Rosenbrock problems of dimension n (even, <= 4096); x0 is nprob×n row-major on the
 * host.  Outputs (host, any may be NULL): objective[nprob], iters_ran[nprob], status[nprob],
 * fdf_evals[nprob], minimizer[nprob×n], grad_norm[nprob]. */
int cgo_batched_minimize_rosenbrock(cgo_ctx *ctx, int64_t nprob, int32_t n, const double *x0,
                                    const cgo_batched_config *cfg, double *objective,
                                    int64_t *iters_ran, int32_t *status, int64_t *fdf_evals,
                                    double *minimizer, double *grad_norm);

#ifdef __cplusplus
}
#endif
#endif
