// internal.cuh — shared declarations of libcgoptim.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <map>
#include <string>
#include <vector>

#include "../../include/cgoptim.h"

// ------------------------------------------------------------------ errors
void cgo_set_error(const char *fmt, ...);
#define CGO_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            cgo_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__,    \
                          __LINE__);                                                            \
            return 1;                                                                           \
        }                                                                                       \
    } while (0)
#define CGO_CHECK(cond, ...)                                                                    \
    do {                                                                                        \
        if (!(cond)) {                                                                          \
            cgo_set_error(__VA_ARGS__);                                                         \
            return 2;                                                                           \
        }                                                                                       \
    } while (0)
#define CGO_TRY(call)                                                                           \
    do {                                                                                        \
        int r__ = (call);                                                                       \
        if (r__) return r__;                                                                    \
    } while (0)

// ------------------------------------------------------------------ canonical reduction
constexpr int CGO_B = 256;        // lanes per (virtual) CTA
constexpr int CGO_NW = CGO_B / 32;
constexpr int CGO_U_VEC = 4;      // double2 loads per lane per tile, BLAS-1 kernels (V = 2)
constexpr int CGO_MAXK = 12;      // widest pack any kernel reduces

struct RedArgs {
    double *partial;        // [K][G] CTA partials
    unsigned int *ticket;   // arrival counter, self-resetting
    double *out;            // K results: mapped pinned host memory (1 rank) or device (R ranks)
    int G;                  // virtual CTAs of the canonical order
    // cross-GPU hand-off over peer memory (halo pushes fused into the producing kernel): the
    // last CTA release-stores sig_val to sig0/sig1 (flags in the neighbours' memory) once every
    // CTA's peer stores are fenced; a consuming kernel spins until its local wait0/wait1 reach
    // wait_val before it touches its halos.  nullptr = not used.
    unsigned long long *sig0 = nullptr, *sig1 = nullptr;
    const unsigned long long *wait0 = nullptr, *wait1 = nullptr;
    unsigned long long sig_val = 0, wait_val = 0;
    // all-ranks variant (sample-sharded logistic regression): the last CTA release-stores sig_val
    // to slot sig_all_slot + me of EVERY rank's flag block (flags_all[r], device table); a consumer
    // waits until its local slots wait_all[0 .. nranks) reach wait_val.
    void *const *flags_all = nullptr;
    const unsigned long long *wait_all = nullptr;
    int sig_all_slot = -1, nranks = 1, me = 0;
};

// ------------------------------------------------------------------ context
struct NcclApi;
// kernel classes for the optional per-launch CUDA-event timing (bench.py roofline)
enum { CGO_T_TRIAL = 0, CGO_T_DIR = 1, CGO_T_AXPY = 2, CGO_T_SPMV = 3, CGO_T_SPMVT = 4,
       CGO_T_LBFGS = 5, CGO_T_OTHER = 6, CGO_T_BATCHED = 7, CGO_T_N = 8 };
struct CgoPendingTimer { int cls; cudaEvent_t e0, e1; };
struct cgo_ctx {
    int device = 0;
    int sms = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int G = 296;
    size_t gather_block_bytes = (size_t)40 << 20;   // column-block size of large random gathers (csr.cu)
    int64_t launches = 0;
    int csr_mode = 0;        // 0: per matrix (sliced layout + k_spmv_direct when its gathers do not coalesce); 1: never; 2: always (CGO_CSR_MODE)
    unsigned long long *d_progress = nullptr;   // [1..3] set-up scratch; [4] k_spmv_direct's slice queue
    // reduction scratch
    double *d_partial = nullptr;     // CGO_MAXK * Gmax
    unsigned int *d_ticket = nullptr;
    double *h_pack = nullptr;        // pinned + mapped, CGO_PACK_LEN
    double *d_pack_map = nullptr;    // device alias of h_pack
    double *d_pack = nullptr;        // device pack (multi-rank)
    double *d_gather = nullptr;      // nranks * CGO_PACK_LEN
    double *d_scal = nullptr;        // device scalars for chained kernels (L-BFGS dots)
    // optional timing
    bool timing = false;
    std::vector<CgoPendingTimer> pending;
    std::vector<cudaEvent_t> ev_pool;
    double t_ms[CGO_T_N] = {0};
    int64_t t_cnt[CGO_T_N] = {0};
    // communicator
    int nranks = 1, rank = 0;
    void *comm = nullptr;            // ncclComm_t
    NcclApi *nccl = nullptr;
    // peer memory (CUDA IPC between the ranks of one node): flags[r] is rank r's flag block
    bool peer_ok = false;
    unsigned long long *flags_local = nullptr;
    std::vector<void *> flags_peer;  // nranks entries ([rank] = flags_local)
    unsigned long long epoch = 0;    // advances in lockstep on every rank
    // scalar-pack exchange over peer memory: gather_peer[r] is rank r's [2][nranks][CGO_PACK_LEN]
    // block (double-buffered by the parity of pack_epoch)
    double *gather_local = nullptr;
    std::vector<void *> gather_peer;
    void **d_gather_peer = nullptr, **d_flags_peer = nullptr;   // device copies of the pointer tables
    unsigned long long pack_epoch = 0;
    std::map<size_t, std::vector<std::vector<void *>>> peer_pool;   // released blocks by size
    std::map<void *, size_t> peer_bytes;                            // size of every live block
    size_t peer_pool_bytes = 0;
    // plain device blocks of destroyed states, by size: the next state of the same problem reuses them
    // (cudaMalloc / cudaFree of 1.6 GB vectors cost milliseconds each and cudaFree synchronises the device)
    std::map<size_t, std::vector<void *>> dev_pool;
    size_t dev_pool_bytes = 0;
};
bool cgo_ctx_alive(cgo_ctx *ctx);                               // false once cgo_ctx_destroy ran (GC-ordered finalisers)
int cgo_dev_alloc(cgo_ctx *ctx, size_t bytes, void **out);     // zero-filled (stream-ordered)
void cgo_dev_free(cgo_ctx *ctx, void *ptr, size_t bytes);
// flag slots of a rank's block
// (CGO_F_PACK + r: rank r's scalar pack of the current exchange has landed in my gather block)
constexpr int CGO_MAX_RANKS = 64;
// (CGO_F_XPALL + r: rank r's shard of xp has landed in my all-gathered copy; CGO_F_CALL + r: rank r's shard of
// c = −y σ has landed in my all-gathered c)
enum { CGO_F_XP_FROM_PREV = 0, CGO_F_XP_FROM_NEXT = 1, CGO_F_R_FROM_PREV = 2, CGO_F_R_FROM_NEXT = 3, CGO_F_PACK = 8,
       CGO_F_XPALL = 8 + CGO_MAX_RANKS, CGO_F_CALL = 8 + 2 * CGO_MAX_RANKS, CGO_F_N = 8 + 3 * CGO_MAX_RANKS };
// allocate `bytes` of device memory on every rank (collective) and map every peer's block:
// peers[r] is rank r's block in this process's address space (peers[rank] == *local).
int cgo_peer_alloc(cgo_ctx *ctx, size_t bytes, void **local, std::vector<void *> &peers);
// collective: barrier before the peers unmap and before the owner frees (all ranks call it at the
// same point of the host program); non-collective only at process teardown
int cgo_peer_free(cgo_ctx *ctx, void *local, std::vector<void *> &peers, bool collective);
constexpr int CGO_GMAX = 8192;
constexpr int CGO_NSCAL = 256;     // device scalar slots (L-BFGS dots), last one reserved
constexpr int CGO_LBFGS_MAX_M = 64;

// launch the pack finalisation for the current kernel sequence: after the producing kernel
// wrote K sums to ctx->red_out(), make them visible on the host in out[0..K).
// `slot`: first pack slot the kernel's K sums land in (kernels of one trial fill disjoint slots)
RedArgs cgo_red_args(cgo_ctx *ctx, int slot = 0);
void cgo_timer_begin(cgo_ctx *ctx, int cls);   // records an event on the ctx stream (if enabled)
void cgo_timer_end(cgo_ctx *ctx);
void cgo_timer_collect(cgo_ctx *ctx);          // after a stream sync: fold pending timers
int cgo_finish_pack(cgo_ctx *ctx, int K, double *out_host);
int cgo_combine_ranks(cgo_ctx *ctx, int K, double *out_dev);   // multi-rank: Σ_r d_pack[0..K) in rank order → out_dev
int cgo_sendrecv_ring(cgo_ctx *ctx, const double *send_to_prev, double *recv_from_next,
                      const double *send_to_next, double *recv_from_prev, int64_t count);
int cgo_allgatherv_f64(cgo_ctx *ctx, const double *mine, double *full, const int64_t *lo);

// ------------------------------------------------------------------ objective interface
struct cgo_state;
struct cgo_obj {
    cgo_ctx *ctx = nullptr;
    int64_t n_global = 0, n_local = 0, offset = 0;
    int64_t halo = 0;                 // elements of padding each side of every state vector
    int64_t n_alloc = 0;              // rank-independent allocation length of peer-mapped vectors (0: n_local)
    virtual ~cgo_obj() {}
    // xp = x + a u (optionally u = −g + β u first), g⁺ = ∇f(xp), fills the device pack and
    // finishes it into out_host.
    virtual int eval_trial(cgo_state *st, double a, bool fused_dir, double beta,
                           double *out_host) = 0;
    // Hessian-vector product along the current direction: hv = ∇²f(x) u; out[0] = u·Hu (as ‖Au‖² for
    // least squares), out[1] = u·hv, out[2] = hv·hv.  Objectives without one return an error.
    virtual int hessvec_dir(cgo_state *st, double *out_host);
    // quadratic-aware line search (SURVEY.md §8f N1): for f = ½‖Ax − b‖², r(x + a u) = r + a·Au, so
    // ϕ(a) = ½(r·r) + a (r·v) + ½ a² (v·v) and dϕ(a) = r·v + a (v·v) with v = A u: every trial of one line
    // search is scalar arithmetic after ONE SpMV.  quad_begin: v = A u, out = {r·v, v·v, r·r};
    // quad_accept: xp = x + a u, r += a v, g⁺ = Aᵀ r and the usual pack (CGO_P_PHI = ½ Σ r²).
    virtual int quad_begin(cgo_state *st, double *out_host);
    virtual int quad_accept(cgo_state *st, double a, double *out_host);
    // cgo_accept(st) adopted (xp, g⁺) as (x, g): objectives that keep per-trial state (the residual) take note
    virtual void on_accept(cgo_state *) {}
    virtual double bytes_per_eval() const = 0;
    // canonical-order mapping (V, U) of the kernels that reduce this objective's trial dots (include/cgoptim.h)
    virtual void reduction_site(int32_t *V, int32_t *U) const = 0;
    virtual int default_x0(uint64_t seed, double perturb, double *x0_host) = 0;
};

struct cgo_state {
    cgo_ctx *ctx = nullptr;
    cgo_obj *obj = nullptr;
    int64_t n = 0;                    // local length
    int64_t halo = 0;
    double *base[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // allocations
    double *x = nullptr, *g = nullptr, *u = nullptr, *xp = nullptr, *gp = nullptr;  // base + halo
    // sharded CSR objectives with peer memory: the two x / xp allocations are mapped by the ring
    // neighbours, which push their boundary elements of xp straight into this rank's halos
    bool peer_x = false;
    std::vector<void *> xpeers[2];   // per allocation (0: base[0]'s, 1: base[3]'s at creation)
    int xp_alloc = 1;                // which of the two allocations is xp right now (flips on accept)
    double *hv = nullptr;             // Hessian-vector product scratch (cgo_hessvec_dir), allocated on first use
    double *xn = nullptr;             // solvesystem's x_next (solve_system.jl:78), allocated by cgo_solvesys_begin
    // L-BFGS history
    int m = 0, count = 0, head = 0, staged = -1;
    std::vector<double *> S, Y;
    std::vector<double> rho;
    double gamma = 1.0;
    double *q = nullptr;
};

// BLAS-1 kernels shared by objectives (blas1.cu)
// xp = x + a u (optionally after u = −g + βu); {g·u, u·u, xp·xp} land in pack slots
// CGO_P_DIR_GU, CGO_P_DIR_UU, CGO_P_XPXP
// `push`: also store the first / last `halo` elements of xp into the ring neighbours' halos
// (peer memory) and signal their flags with `epoch` when the kernel's stores are fenced
struct HaloPush {
    double *prev_right = nullptr;    // previous rank's xp + its n (its right halo)
    double *next_left = nullptr;     // next rank's xp − halo (its left halo)
    unsigned long long *sig_prev = nullptr, *sig_next = nullptr;
    unsigned long long epoch = 0;
    // all-gather variant: my whole shard goes to dst_all[r] (rank r's all-gathered xp at my offset;
    // device table of nranks pointers), then flag CGO_F_XPALL + me of every rank
    void *const *dst_all = nullptr;
};
int cgo_blas1_axpy_dir(cgo_state *st, double a, bool fused_dir, double beta, const HaloPush *push = nullptr);
int cgo_blas1_residual_axpy(cgo_ctx *ctx, double *r, const double *v, double a, int64_t nrows, int slot);
int cgo_blas1_sumsq(cgo_ctx *ctx, const double *a, int64_t n, int slot);                        // Σ a²
int cgo_blas1_dots3(cgo_ctx *ctx, const double *a, const double *b, int64_t n, int slot);       // {a·b, b·b, a·a}
// margins → c = −y σ in place, Σ loss → pack slot; dst_all != NULL: also all-gather c over peer memory (flag CGO_F_CALL)
int cgo_blas1_logit(cgo_ctx *ctx, double *zc, const double *y, int64_t n, int slot, void *const *dst_all, unsigned long long epoch);
// softmax regression: Z (n × nclass, row-major) → C = P − Y in place (labels y as doubles), Σ loss → pack slot
int cgo_blas1_softmax(cgo_ctx *ctx, double *zc, const double *y, int64_t n, int nclass, int slot);
int cgo_blas1_grad_dots(cgo_state *st);     // the eight dots of EpiGrad over (g⁺, g, u) → pack slots CGO_P_DPHI…
// logistic regression on k_spmv_direct: g⁺ = g⁺ · invN + λ xp in place (g⁺ holds Aᵀc), fused with the dot pack of
// EpiGrad (slots CGO_P_DPHI .. CGO_P_UU)
int cgo_blas1_grad_combine(cgo_state *st, double invN, double lambda);
// the GLM objectives with weights or an intercept (coordinates [npen, n) unpenalised): K_a with P, the penalised part
// of xp·xp, in slot CGO_P_XPXP; the loss ops with weights wt (NULL: unit) and the intercept at bias (NULL: none);
// the combine pass without λ w on the intercept coordinates
int cgo_blas1_axpy_dir_pen(cgo_state *st, double a, bool fused_dir, double beta, int64_t npen);
int cgo_blas1_logit_glm(cgo_ctx *ctx, double *zc, const double *y, const double *wt, const double *bias, int64_t n, int slot);
int cgo_blas1_softmax_glm(cgo_ctx *ctx, double *zc, const double *y, const double *wt, const double *bias, int64_t n,
                          int nclass, int slot);
int cgo_blas1_grad_combine_pen(cgo_state *st, double invS, double lambda, int64_t npen);

// ------------------------------------------------------------------ CSR (csr.cu)
struct CsrMat {
    int64_t nrows = 0, nnz = 0;
    int64_t *rowptr = nullptr;   // nrows + 1
    int32_t *col = nullptr;      // index into the gathered vector (may be negative: left halo)
    double *val = nullptr;
    // sliced: inside every 32-row slice [rowptr[32s], rowptr[32s+32]) the entries are stored level-major
    // (all first entries of the slice's rows in row order, then all second entries, …) instead of row-major
    int32_t sliced = 0;
    int32_t ragged = 0;          // sliced: more than one slice in 16 has rows of different lengths (picks the batch width)
};
