/*
 * cgo_oracle.c — CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).  See cgo_oracle.h.
 *
 * Restates, in plain C and in the reference's own (unfused, temporary-allocating) shape:
 *   src/engine/optim.jl:6-208      minimizeobjective / minimizeobjectivererun
 *   src/cg_utils.jl:3-22           evalϕdϕ!
 *   src/cg_flavours.jl:2-170       updatedir!, getβ for YuanWangSheng / HagerZhang /
 *                                  SallehAlhawarat / LiuStorrey
 *   src/linesearch/nocedal.jl      StrongWolfeBisection linesearch! + zoom!
 *   src/linesearch/wolfe.jl        WolfeBisection linesearch!, findfeasiblestepsize!, conditions
 *   src/linesearch/geometric.jl    Backtracking linesearch!, geometricsearch!, Armijo
 * plus a textbook L-BFGS flavour (Nocedal & Wright Alg. 7.4/7.5; no reference counterpart, the
 * reference's src/qn_flavours.jl is a dense no-op update, SURVEY.md §0) and the synthetic
 * objectives / generators of SURVEY.md §8(d).
 *
 * Build with -O2 -ffp-contract=off (no FMA contraction: Julia does not contract a*b+c).
 * PARITY UNPINNED (see header).
 */
#include "cgo_oracle.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------------------------------
 * counter-based hash (generator spec, SURVEY.md §8d: "counter-based hash keyed (seed,row,k)")
 * ---------------------------------------------------------------------------------------- */
static inline uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
static inline uint64_t hash3(uint64_t seed, uint64_t i, uint64_t k) {
    uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ULL);
    h = mix64(h ^ (i + 0x9E3779B97F4A7C15ULL));
    h = mix64(h ^ (k + 0x632BE59BD9B4E019ULL));
    return h;
}
static inline double u01(uint64_t seed, uint64_t i, uint64_t k) {
    return (double)(hash3(seed, i, k) >> 11) * (1.0 / 9007199254740992.0);
}
double orc_hash_u01(uint64_t seed, uint64_t i, uint64_t k) { return u01(seed, i, k); }

/* ------------------------------------------------------------------------------------------
 * reductions.  The reference calls LinearAlgebra.dot / norm (OpenBLAS ddot/dnrm2, order
 * unspecified, SURVEY.md §8c).  Three orders are offered; threads split [0,n) into contiguous
 * chunks that are combined in chunk order, so every mode is deterministic.
 * ---------------------------------------------------------------------------------------- */
static double dot_seq(const double *a, const double *b, int64_t n) {
    double s = 0.0;
    for (int64_t i = 0; i < n; ++i) s += a[i] * b[i];
    return s;
}
static double dot_pair(const double *a, const double *b, int64_t n) {
    if (n <= 128) return dot_seq(a, b, n);
    int64_t h = n / 2;
    return dot_pair(a, b, h) + dot_pair(a + h, b + h, n - h);
}
static double dot_comp(const double *a, const double *b, int64_t n) { /* Neumaier */
    double s = 0.0, c = 0.0;
    for (int64_t i = 0; i < n; ++i) {
        double p = a[i] * b[i];
        double t = s + p;
        if (fabs(s) >= fabs(p)) c += (s - t) + p; else c += (p - t) + s;
        s = t;
    }
    return s + c;
}
/* ---- canonical "CGO" order: the reduction order the CUDA kernels implement (include/cgoptim.h,
 * "Canonical reduction order").  Items are visited in index order; item i is owned by lane
 * t = q % B of virtual CTA c = (q / (B*U)) % G with q = i / V.  Each (c,t) accumulates its items
 * sequentially from +0.0; a CTA combines its B lanes by a xor-butterfly (16,8,4,2,1) inside each
 * warp and then sequentially over warps; the grid combines the min(G, ntiles) CTA partials the
 * same way (lane t takes partials t, t+B, ...).  Shards (ranks) each reduce their contiguous
 * slice this way and the shard results are added in rank order.                            */
enum { CGO_BMAX = 256 };
static int g_cgo_G = 296, g_cgo_shards = 1;
/* lanes per virtual CTA: 256 everywhere except the batched on-device solver, whose CTA is as small
 * as eight element pairs per lane allow (32, 64, 128 or 256 lanes; include/cgoptim.h) */
static int CGO_B = 256;
void orc_set_cgo_order(int G, int shards) { g_cgo_G = G > 0 ? G : 296; g_cgo_shards = shards > 0 ? shards : 1; }
/* items per lane and tile of the BLAS-1 mapping: 4 double2 loads (k_blas1), 8 in the batched solver */
static int g_blas1_U = 4;
static int g_site_V = 2, g_site_U = 4;
void orc_set_cgo_lanes(int B) {
    CGO_B = (B == 32 || B == 64 || B == 128) ? B : 256;
    g_blas1_U = 4; g_site_V = 2; g_site_U = 4;
}
void orc_set_cgo_batched(int B) {       /* the batched solver's order: B lanes, every item in ONE tile */
    CGO_B = (B == 32 || B == 64 || B == 128) ? B : 256;
    g_blas1_U = 8; g_site_V = 2; g_site_U = 8;
}
static double cgo_cta_combine(double *lane /* CGO_B, clobbered */) {
    double wsum[CGO_BMAX / 32] = {0};
    for (int w = 0; w < CGO_B / 32; ++w) {
        double *v = lane + 32 * w, t[32];
        for (int off = 16; off >= 1; off >>= 1) {
            for (int l = 0; l < 32; ++l) t[l] = v[l] + v[l ^ off];
            for (int l = 0; l < 32; ++l) v[l] = t[l];
        }
        wsum[w] = v[0];
    }
    double s = wsum[0];
    for (int w = 1; w < CGO_B / 32; ++w) s = s + wsum[w];
    return s;
}
typedef double (*term_fn)(const void *ctx, int64_t i);
static double cgo_reduce_slice(term_fn f, const void *ctx, int64_t lo, int64_t count, int V, int U) {
    int G = g_cgo_G;
    int64_t nq = (count + V - 1) / V;
    int64_t ntiles = (nq + (int64_t)CGO_B * U - 1) / ((int64_t)CGO_B * U);
    int nact = (int)(ntiles < G ? ntiles : G);
    if (nact < 1) nact = 1;
    double *acc = (double *)calloc((size_t)nact * CGO_B, sizeof(double));
    for (int64_t i = 0; i < count; ++i) {
        int64_t q = i / V;
        int64_t c = (q / ((int64_t)CGO_B * U)) % G;
        int t = (int)(q % CGO_B);
        acc[c * CGO_B + t] = acc[c * CGO_B + t] + f(ctx, lo + i);
    }
    double *P = (double *)calloc((size_t)nact, sizeof(double));
    for (int c = 0; c < nact; ++c) P[c] = cgo_cta_combine(acc + (size_t)c * CGO_B);
    double lane[CGO_BMAX];
    for (int t = 0; t < CGO_B; ++t) {
        double s2 = 0.0;
        for (int k = t; k < nact; k += CGO_B) s2 = s2 + P[k];
        lane[t] = s2;
    }
    double r = cgo_cta_combine(lane);
    free(acc); free(P);
    return r;
}
/* contiguous shard partition used by the product (cgo_shard_range in include/cgoptim.h):
 * boundaries at multiples of `align` items */
static int64_t shard_lo(int64_t n, int r, int N, int64_t align) {
    int64_t units = n / align;
    int64_t b = (units * r / N) * align;
    return r == N ? n : b;
}
static double cgo_reduce(term_fn f, const void *ctx, int64_t count, int V, int U, int64_t align) {
    int N = g_cgo_shards;
    if (N <= 1) return cgo_reduce_slice(f, ctx, 0, count, V, U);
    double s = 0.0;
    for (int r = 0; r < N; ++r) {
        int64_t lo = shard_lo(count, r, N, align), hi = shard_lo(count, r + 1, N, align);
        double p = cgo_reduce_slice(f, ctx, lo, hi - lo, V, U);
        s = (r == 0) ? p : s + p;
    }
    return s;
}
typedef struct { const double *a, *b; } dot_ctx;
static double dot_term(const void *c, int64_t i) { const dot_ctx *d = (const dot_ctx *)c; return d->a[i] * d->b[i]; }
static double sum_term(const void *c, int64_t i) { return ((const double *)c)[i]; }
/* BLAS-1 kernels read vectors as 128-bit double2 (V=2) with U=4 loads per lane per tile;
 * row-per-lane (CSR) kernels use V=1, U=1.  g_site_V/U select the mapping of the kernel that
 * computes the reduction at the current call site (see DESIGN.md "reduction sites"). */
void orc_set_site(int V, int U) { g_site_V = V; g_site_U = U; }
static double dot_cgo(const double *a, const double *b, int64_t n) {
    dot_ctx d = {a, b};
    return cgo_reduce(dot_term, &d, n, g_site_V, g_site_U, 2);
}

static double dot_mode(const double *a, const double *b, int64_t n, int mode) {
    switch (mode) {
    case ORC_SUM_PAIRWISE: return dot_pair(a, b, n);
    case ORC_SUM_COMP: return dot_comp(a, b, n);
    case ORC_SUM_CGO: return dot_cgo(a, b, n);
    default: return dot_seq(a, b, n);
    }
}
double orc_dot(const double *a, const double *b, int64_t n, int mode, int threads) {
    if (threads <= 1 || n < 4096 || mode == ORC_SUM_CGO) return dot_mode(a, b, n, mode);
    double *part = (double *)calloc((size_t)threads, sizeof(double));
#pragma omp parallel for num_threads(threads) schedule(static, 1)
    for (int t = 0; t < threads; ++t) {
        int64_t lo = n * t / threads, hi = n * (t + 1) / threads;
        part[t] = dot_mode(a + lo, b + lo, hi - lo, mode);
    }
    double s = 0.0;
    for (int t = 0; t < threads; ++t) s += part[t];
    free(part);
    return s;
}
static double sum_mode_(const double *a, int64_t n, int mode) {
    if (mode == ORC_SUM_PAIRWISE) {
        if (n <= 128) { double s = 0; for (int64_t i = 0; i < n; ++i) s += a[i]; return s; }
        int64_t h = n / 2;
        return sum_mode_(a, h, mode) + sum_mode_(a + h, n - h, mode);
    }
    if (mode == ORC_SUM_COMP) {
        double s = 0.0, c = 0.0;
        for (int64_t i = 0; i < n; ++i) {
            double p = a[i], t = s + p;
            if (fabs(s) >= fabs(p)) c += (s - t) + p; else c += (p - t) + s;
            s = t;
        }
        return s + c;
    }
    double s = 0;
    for (int64_t i = 0; i < n; ++i) s += a[i];
    return s;
}
/* per-item terms (one per pair / per row): V=1; U as the owning kernel family defines it */
double orc_sum_cgo(const double *a, int64_t n, int U, int64_t align) {
    return cgo_reduce(sum_term, a, n, 1, U, align);
}
double orc_sum(const double *a, int64_t n, int mode, int threads) {
    if (mode == ORC_SUM_CGO) return orc_sum_cgo(a, n, g_blas1_U, 1);
    if (threads <= 1 || n < 4096) return sum_mode_(a, n, mode);
    double *part = (double *)calloc((size_t)threads, sizeof(double));
#pragma omp parallel for num_threads(threads) schedule(static, 1)
    for (int t = 0; t < threads; ++t) {
        int64_t lo = n * t / threads, hi = n * (t + 1) / threads;
        part[t] = sum_mode_(a + lo, hi - lo, mode);
    }
    double s = 0.0;
    for (int t = 0; t < threads; ++t) s += part[t];
    free(part);
    return s;
}

/* ------------------------------------------------------------------------------------------
 * objectives: fdf!(g, x) -> f   (user callback of the reference, optim.jl:25, cg_utils.jl:18)
 * ---------------------------------------------------------------------------------------- */
typedef double (*fdf_fn)(orc_objective *, double *g, const double *x);
struct orc_objective {
    int64_t n;          /* dimension of x */
    fdf_fn fdf;
    int sum_mode, threads;
    /* CSR payload (sparse LS: A nrows x n ; logreg: A nsamples x n) */
    int64_t nrows, nnz;
    int64_t *rowptr; int32_t *col; double *val;
    int64_t *rowptrT; int32_t *colT; double *valT;
    double *b;          /* rhs or labels */
    double *scratch;    /* nrows */
    double *scratch2;   /* n (per-element f terms) */
    double *scratch2rows; /* nrows */
    double lambda;
    int owns;
    int trial_V, trial_U;   /* canonical-order mapping of this objective's trial kernels */
    /* box-constraint log barrier around another objective (primal_barrier.jl) */
    orc_objective *inner;
    double *lbs, *ubs;
    double t;
};

/* Booth, examples/helpers/test_funcs.jl:3-12 */
static double booth_fdf(orc_objective *o, double *g, const double *p) {
    (void)o;
    double x = p[0], y = p[1];
    double t1 = x + 2 * y - 7, t2 = 2 * x + y - 5;
    double f = t1 * t1 + t2 * t2;
    g[0] = 2 * t1 + 2 * t2 * 2;
    g[1] = 2 * t1 * 2 + 2 * t2;
    return f;
}

/* extended Rosenbrock (pairs), SURVEY.md §8d cfg 1/2:
 * f = Σ_pairs 100 (x2 − x1²)² + (1 − x1)².  The expression order below is the spec the CUDA
 * kernel follows bit for bit: t = x2 − x1*x1; om = 1 − x1;
 * f_pair = (100*t)*t + om*om; g1 = (−400*x1)*t − 2*om; g2 = 200*t.                         */
static double rosen_fdf(orc_objective *o, double *g, const double *x) {
    int64_t np = o->n / 2;
    double *fp = o->scratch2;
#pragma omp parallel for num_threads(o->threads) schedule(static) if (o->threads > 1)
    for (int64_t p = 0; p < np; ++p) {
        double x1 = x[2 * p], x2 = x[2 * p + 1];
        double t = x2 - x1 * x1;
        double om = 1.0 - x1;
        fp[p] = (100.0 * t) * t + om * om;
        g[2 * p] = (-400.0 * x1) * t - 2.0 * om;
        g[2 * p + 1] = 200.0 * t;
    }
    return orc_sum(fp, np, o->sum_mode, o->threads);
}

/* chained Rosenbrock, value from examples/helpers/test_funcs.jl:50-57, hand-derived gradient */
static double rosen_chained_fdf(orc_objective *o, double *g, const double *x) {
    int64_t d = o->n;
    double *fp = o->scratch2;
    for (int64_t i = 0; i < d; ++i) g[i] = 0.0;
    for (int64_t i = 0; i < d - 1; ++i) {
        double om = 1.0 - x[i];
        double t = x[i + 1] - x[i] * x[i];
        fp[i] = om * om + (100.0 * t) * t;
        g[i] += -2.0 * om - (400.0 * x[i]) * t;
        g[i + 1] += 200.0 * t;
    }
    /* canonical order: the device kernel (blas1.cu RosenChainedEval) reads double2 and adds the terms of both
     * elements lane by lane (V = 2, U = 4), one term per ELEMENT with a +0.0 for the last one, so that the shards
     * of the sum are the shards of the vector */
    if (o->sum_mode == ORC_SUM_CGO) {
        fp[d - 1] = 0.0;
        return cgo_reduce(sum_term, fp, d, 2, g_blas1_U, 2);
    }
    return orc_sum(fp, d - 1, o->sum_mode, 1);
}

/* log-barrier box objective: non-finite outside |x_i|<1 (exercises the feasibility back-off
 * of wolfe.jl:171-207 / geometric.jl:62-75 and the non-finite exits of optim.jl:108-121).  */
static double barrier_fdf(orc_objective *o, double *g, const double *x) {
    int64_t n = o->n;
    double *fp = o->scratch2;
    for (int64_t i = 0; i < n; ++i) {
        double c = 2.0;
        double w = 1.0 - x[i] * x[i];
        double d = x[i] - c;
        fp[i] = -log(w) + 0.5 * d * d;
        g[i] = (2.0 * x[i]) / w + d;
    }
    return orc_sum(fp, n, o->sum_mode, 1);
}

/* y = A x (row sums in storage order, unfused mul+add) */
static void csr_mv(int64_t nrows, const int64_t *rp, const int32_t *ci, const double *v,
                   const double *x, double *y, int threads) {
#pragma omp parallel for num_threads(threads) schedule(static) if (threads > 1)
    for (int64_t i = 0; i < nrows; ++i) {
        double acc = 0.0;
        for (int64_t p = rp[i]; p < rp[i + 1]; ++p) acc += v[p] * x[ci[p]];
        y[i] = acc;
    }
}

/* f = ½‖Ax − b‖², g = Aᵀ(Ax − b)    (SURVEY.md §8d cfg 3) */
static double sparse_ls_fdf(orc_objective *o, double *g, const double *x) {
    double *r = o->scratch;
    csr_mv(o->nrows, o->rowptr, o->col, o->val, x, r, o->threads);
#pragma omp parallel for num_threads(o->threads) schedule(static) if (o->threads > 1)
    for (int64_t i = 0; i < o->nrows; ++i) r[i] = r[i] - o->b[i];
    double f;
    if (o->sum_mode == ORC_SUM_CGO) {   /* K_b reduces r_i² row-per-lane (V=1, U=1); for gather-bound matrices
                                         * a BLAS-1 pass does (V=2, U=4): csr.cu k_spmv_direct */
        double *rr = o->scratch2rows;
        for (int64_t i = 0; i < o->nrows; ++i) rr[i] = r[i] * r[i];
        f = 0.5 * (o->trial_V == 2 ? cgo_reduce(sum_term, rr, o->nrows, 2, g_blas1_U, 2) : orc_sum_cgo(rr, o->nrows, 1, 2));
    } else {
        f = 0.5 * orc_dot(r, r, o->nrows, o->sum_mode, o->threads);
    }
    /* Aᵀ r through the explicit transpose, whose rows are sorted by source row: the same
     * accumulation order as the sequential scatter g[col] += val*r[i], i ascending. */
    csr_mv(o->n, o->rowptrT, o->colT, o->valT, r, g, o->threads);
    return f;
}

/* logistic regression (SURVEY.md §8d cfg 4):
 * f = (1/N) Σ softplus(−y_i a_i·w) + (λ/2)‖w‖²;  g = (1/N) Aᵀc + λ w,
 * with t = −y z, e = exp(−|t|), softplus(t) = max(t,0) + log1p(e),
 * σ(t) = t ≥ 0 ? 1/(1+e) : e/(1+e),  c_i = −y_i σ(t_i).                                    */
static double logreg_fdf(orc_objective *o, double *g, const double *w) {
    double *c = o->scratch;
    int64_t N = o->nrows;
    csr_mv(N, o->rowptr, o->col, o->val, w, c, o->threads);
    double *lp = (double *)malloc(sizeof(double) * (size_t)N);
#pragma omp parallel for num_threads(o->threads) schedule(static) if (o->threads > 1)
    for (int64_t i = 0; i < N; ++i) {
        double y = o->b[i];
        double t = -y * c[i];
        double e = exp(-fabs(t));
        lp[i] = (t > 0.0 ? t : 0.0) + log1p(e);
        double sg = t >= 0.0 ? 1.0 / (1.0 + e) : e / (1.0 + e);
        c[i] = -y * sg;
    }
    /* row-per-lane epilogue (V=1, U=1), or the BLAS-1 logit kernel of the k_spmv_direct path (V=2, U=4) */
    double loss = (o->sum_mode == ORC_SUM_CGO ? (o->trial_V == 2 ? cgo_reduce(sum_term, lp, N, 2, g_blas1_U, 2) : orc_sum_cgo(lp, N, 1, 2))
                                              : orc_sum(lp, N, o->sum_mode, o->threads)) / (double)N;
    free(lp);
    csr_mv(o->n, o->rowptrT, o->colT, o->valT, c, g, o->threads);
    int sv = g_site_V, su = g_site_U;
    g_site_V = 2; g_site_U = g_blas1_U;         /* w·w is reduced by the BLAS-1 kernel K_a */
    double ww = orc_dot(w, w, o->n, o->sum_mode, o->threads);
    g_site_V = sv; g_site_U = su;
    double invN = 1.0 / (double)N;
#pragma omp parallel for num_threads(o->threads) schedule(static) if (o->threads > 1)
    for (int64_t j = 0; j < o->n; ++j) g[j] = g[j] * invN + o->lambda * w[j];
    return loss + (0.5 * o->lambda) * ww;
}

/* evalbarrier! (src/engine/primal_barrier.jl:112-133) with the box constraints of
 * examples/constrained.jl:17-47: fi = [x − ubs; lbs − x], dfi = [+e_d; −e_d].
 *   f0 = fdf!(df_x, x)                                                     :121
 *   evalconstraints! (:63-91): clamp!(fi, −Inf, 0) (:77); ψ = −Σ log(−fi) (:78);
 *     dψ[d] −= dfi[i][d]/fi[i] over all constraints (:80-85): for a box, dψ[d] = (0 − 1/fu_d) − (−1/fl_d)
 *     (the other terms subtract ±0).  Not restated: with fi[i] = 0 (a point on or outside the box) the
 *     reference's dense loop makes EVERY entry of dψ NaN (0/0); here only entry d is non-finite.
 *     Either way ‖g‖ and g·u are non-finite and ϕ = +Inf, which is all the line searches test.
 *   df_x = t .* df_x .+ dψ (:130);  return t*f0 + ψ (:132)
 * ORC_SUM_CGO: ψ's 2n log terms are added element by element (upper, lower) by the BLAS-1
 * barrier kernel (V = 2, U = 4); otherwise in the reference's order (all uppers, then all lowers). */
static double box_barrier_fdf(orc_objective *o, double *g, const double *x) {
    orc_objective *in = o->inner;
    int64_t n = o->n;
    in->sum_mode = o->sum_mode; in->threads = o->threads;
    double f0 = in->fdf(in, g, x);
    double *tu = o->scratch2, *tl = o->scratch;
    for (int64_t d = 0; d < n; ++d) {
        double fu = x[d] - o->ubs[d], fl = o->lbs[d] - x[d];
        if (fu > 0.0) fu = 0.0;             /* clamp!(fi_evals, -Inf, 0): NaN stays NaN */
        if (fl > 0.0) fl = 0.0;
        tu[d] = log(-fu);
        tl[d] = log(-fl);
        double dpsi = 0.0 - 1.0 / fu;
        dpsi = dpsi - (-1.0) / fl;
        g[d] = o->t * g[d] + dpsi;
    }
    double sum;
    if (o->sum_mode == ORC_SUM_CGO) {
        for (int64_t d = 0; d < n; ++d) tu[d] = tu[d] + tl[d];
        int sv = g_site_V, su = g_site_U;
        g_site_V = 2; g_site_U = g_blas1_U;
        sum = cgo_reduce(sum_term, tu, n, 2, g_blas1_U, 2);
        g_site_V = sv; g_site_U = su;
    } else {
        sum = 0.0;
        for (int64_t d = 0; d < n; ++d) sum += tu[d];
        for (int64_t d = 0; d < n; ++d) sum += tl[d];
    }
    return o->t * f0 + (-sum);
}

static orc_objective *obj_new(int64_t n, fdf_fn f) {
    orc_objective *o = (orc_objective *)calloc(1, sizeof(*o));
    o->n = n; o->fdf = f; o->sum_mode = ORC_SUM_SEQ; o->threads = 1;
    o->trial_V = 2; o->trial_U = 4;
    o->scratch2 = (double *)malloc(sizeof(double) * (size_t)(n > 0 ? n : 1));
    return o;
}
orc_objective *orc_obj_booth(void) { return obj_new(2, booth_fdf); }
orc_objective *orc_obj_rosenbrock(int64_t n) { return (n % 2) ? NULL : obj_new(n, rosen_fdf); }
orc_objective *orc_obj_rosenbrock_chained(int64_t n) { return obj_new(n, rosen_chained_fdf); }
orc_objective *orc_obj_quartic_barrier(int64_t n) { return obj_new(n, barrier_fdf); }
int64_t orc_obj_dim(const orc_objective *o) { return o->n; }
/* the inner objective stays owned by the caller and must outlive the barrier objective */
orc_objective *orc_obj_box_barrier(orc_objective *inner, const double *lbs, const double *ubs, double t) {
    orc_objective *o = obj_new(inner->n, box_barrier_fdf);
    o->inner = inner; o->t = t; o->owns = 1;
    o->lbs = (double *)malloc(sizeof(double) * (size_t)inner->n);
    o->ubs = (double *)malloc(sizeof(double) * (size_t)inner->n);
    o->scratch = (double *)malloc(sizeof(double) * (size_t)inner->n);
    memcpy(o->lbs, lbs, sizeof(double) * (size_t)inner->n);
    memcpy(o->ubs, ubs, sizeof(double) * (size_t)inner->n);
    o->trial_V = 2; o->trial_U = 4;     /* the barrier kernel (BLAS-1) reduces the trial's dots */
    return o;
}
void orc_obj_barrier_set_t(orc_objective *o, double t) { o->t = t; }
void orc_obj_set_sum_mode(orc_objective *o, int mode, int threads) { o->sum_mode = mode; if (threads > 0) o->threads = threads; }
void orc_obj_trial_site(const orc_objective *o, int *V, int *U) { *V = o->trial_V; *U = o->trial_U; }
/* which kernels reduce the trial's dots is a property of the device objective (cgo_obj_reduction_site) */
void orc_obj_set_trial_site(orc_objective *o, int V, int U) { o->trial_V = V; o->trial_U = U; }

/* stable counting-sort transpose: rows of Aᵀ come out sorted by source row */
static void build_transpose(orc_objective *o) {
    int64_t nr = o->nrows, nc = o->n, nnz = o->nnz;
    o->rowptrT = (int64_t *)calloc((size_t)nc + 1, sizeof(int64_t));
    o->colT = (int32_t *)malloc(sizeof(int32_t) * (size_t)(nnz > 0 ? nnz : 1));
    o->valT = (double *)malloc(sizeof(double) * (size_t)(nnz > 0 ? nnz : 1));
    for (int64_t p = 0; p < nnz; ++p) o->rowptrT[o->col[p] + 1]++;
    for (int64_t j = 0; j < nc; ++j) o->rowptrT[j + 1] += o->rowptrT[j];
    int64_t *cur = (int64_t *)malloc(sizeof(int64_t) * (size_t)(nc > 0 ? nc : 1));
    memcpy(cur, o->rowptrT, sizeof(int64_t) * (size_t)nc);
    for (int64_t i = 0; i < nr; ++i)
        for (int64_t p = o->rowptr[i]; p < o->rowptr[i + 1]; ++p) {
            int64_t q = cur[o->col[p]]++;
            o->colT[q] = (int32_t)i;
            o->valT[q] = o->val[p];
        }
    free(cur);
}

void orc_sparse_ls_xtrue(int64_t n, uint64_t seed, double *out) {
    for (int64_t i = 0; i < n; ++i) out[i] = 2.0 * u01(seed + 1, (uint64_t)i, 0) - 1.0;
}

/* banded-random generator, SURVEY.md §8d cfg 3 (made explicit here; this text is the spec):
 *  entry 0: col = i, val = 4 + u01(seed,i,0)
 *  entry k = 1..K-1: S = K-1 strata of width w = 2W/S over offsets [-W, W); lo = -W + (k-1) w;
 *     δ = lo + hash3(seed ^ 0xA5A5A5A5A5A5A5A5, i >> coh_log2, k) % w;  δ == 0 -> (lo+w > 1 ? 1 : -1);
 *     col = (i + δ) mod n;  val = 0.3 (2 u01(seed,i,k) − 1)
 *  x_true_i = 2 u01(seed+1,i,0) − 1;  b = A x_true;  requires n > 2W and 2W >= 2S.          */
orc_objective *orc_obj_sparse_ls_synth(int64_t n, int32_t K, int64_t W, uint64_t seed,
                                       int32_t coh_log2, int32_t threads) {
    int64_t S = K - 1;
    if (K < 1 || (S > 0 && (2 * W < 2 * S || n <= 2 * W))) return NULL;
    orc_objective *o = obj_new(n, sparse_ls_fdf);
    o->trial_V = 1; o->trial_U = 1;
    /* offsets redrawn at least every 8 rows: the device treats the matrix as gather-bound and reduces the
     * trial's dots in BLAS-1 passes (include/cgoptim.h, canonical reduction order) */
    if (coh_log2 < 4 && K > 1) { o->trial_V = 2; o->trial_U = 4; }
    o->threads = threads < 1 ? 1 : threads;
    o->nrows = n; o->nnz = n * (int64_t)K; o->owns = 1;
    o->rowptr = (int64_t *)malloc(sizeof(int64_t) * (size_t)(n + 1));
    o->col = (int32_t *)malloc(sizeof(int32_t) * (size_t)o->nnz);
    o->val = (double *)malloc(sizeof(double) * (size_t)o->nnz);
    o->b = (double *)malloc(sizeof(double) * (size_t)n);
    o->scratch = (double *)malloc(sizeof(double) * (size_t)n);
    o->scratch2rows = (double *)malloc(sizeof(double) * (size_t)n);
    int64_t w = S > 0 ? (2 * W) / S : 0;
#pragma omp parallel for num_threads(o->threads) schedule(static) if (o->threads > 1)
    for (int64_t i = 0; i < n; ++i) {
        int64_t p = i * K;
        o->rowptr[i] = p;
        o->col[p] = (int32_t)i;
        o->val[p] = 4.0 + u01(seed, (uint64_t)i, 0);
        for (int64_t k = 1; k < K; ++k) {
            int64_t lo = -W + (k - 1) * w;
            int64_t d = lo + (int64_t)(hash3(seed ^ 0xA5A5A5A5A5A5A5A5ULL,
                                             (uint64_t)(i >> coh_log2), (uint64_t)k) % (uint64_t)w);
            if (d == 0) d = (lo + w > 1) ? 1 : -1;
            int64_t c = i + d;
            if (c < 0) c += n;
            if (c >= n) c -= n;
            o->col[p + k] = (int32_t)c;
            o->val[p + k] = 0.3 * (2.0 * u01(seed, (uint64_t)i, (uint64_t)k) - 1.0);
        }
    }
    o->rowptr[n] = o->nnz;
    double *xt = (double *)malloc(sizeof(double) * (size_t)n);
    orc_sparse_ls_xtrue(n, seed, xt);
    csr_mv(n, o->rowptr, o->col, o->val, xt, o->b, o->threads);
    free(xt);
    build_transpose(o);
    return o;
}

orc_objective *orc_obj_sparse_ls_csr(int64_t nrows, int64_t ncols, const int64_t *rowptr,
                                     const int32_t *col, const double *val, const double *b,
                                     int32_t threads) {
    orc_objective *o = obj_new(ncols, sparse_ls_fdf);
    o->trial_V = 1; o->trial_U = 1;
    o->threads = threads < 1 ? 1 : threads;
    o->nrows = nrows; o->nnz = rowptr[nrows]; o->owns = 1;
    o->rowptr = (int64_t *)malloc(sizeof(int64_t) * (size_t)(nrows + 1));
    o->col = (int32_t *)malloc(sizeof(int32_t) * (size_t)(o->nnz > 0 ? o->nnz : 1));
    o->val = (double *)malloc(sizeof(double) * (size_t)(o->nnz > 0 ? o->nnz : 1));
    o->b = (double *)malloc(sizeof(double) * (size_t)(nrows > 0 ? nrows : 1));
    o->scratch = (double *)malloc(sizeof(double) * (size_t)(nrows > 0 ? nrows : 1));
    o->scratch2rows = (double *)malloc(sizeof(double) * (size_t)(nrows > 0 ? nrows : 1));
    memcpy(o->rowptr, rowptr, sizeof(int64_t) * (size_t)(nrows + 1));
    memcpy(o->col, col, sizeof(int32_t) * (size_t)o->nnz);
    memcpy(o->val, val, sizeof(double) * (size_t)o->nnz);
    memcpy(o->b, b, sizeof(double) * (size_t)nrows);
    build_transpose(o);
    return o;
}

/* logistic-regression generator (SURVEY.md §8d cfg 4; this text is the spec):
 *  entry k = 0..K-1: stratum width w = d / K; col = k w + hash3(seed,i,k) % w;
 *     val = 2 u01(seed+7,i,k) − 1
 *  w_true_j = 2 u01(seed+2,j,0) − 1; noise_i = 2 u01(seed+3,i,0) − 1;
 *  y_i = (a_i·w_true + 0.1 noise_i >= 0) ? +1 : −1                                          */
orc_objective *orc_obj_logreg_synth(int64_t N, int64_t d, int32_t K, uint64_t seed, double lambda,
                                    int32_t threads) {
    if (K < 1 || d / K < 1) return NULL;
    orc_objective *o = obj_new(d, logreg_fdf);
    o->trial_V = 1; o->trial_U = 1;
    o->threads = threads < 1 ? 1 : threads;
    o->nrows = N; o->nnz = N * (int64_t)K; o->owns = 1; o->lambda = lambda;
    o->rowptr = (int64_t *)malloc(sizeof(int64_t) * (size_t)(N + 1));
    o->col = (int32_t *)malloc(sizeof(int32_t) * (size_t)o->nnz);
    o->val = (double *)malloc(sizeof(double) * (size_t)o->nnz);
    o->b = (double *)malloc(sizeof(double) * (size_t)N);
    o->scratch = (double *)malloc(sizeof(double) * (size_t)N);
    int64_t w = d / K;
    double *wt = (double *)malloc(sizeof(double) * (size_t)d);
    for (int64_t j = 0; j < d; ++j) wt[j] = 2.0 * u01(seed + 2, (uint64_t)j, 0) - 1.0;
#pragma omp parallel for num_threads(o->threads) schedule(static) if (o->threads > 1)
    for (int64_t i = 0; i < N; ++i) {
        int64_t p = i * K;
        o->rowptr[i] = p;
        double acc = 0.0;
        for (int64_t k = 0; k < K; ++k) {
            int64_t c = k * w + (int64_t)(hash3(seed, (uint64_t)i, (uint64_t)k) % (uint64_t)w);
            double v = 2.0 * u01(seed + 7, (uint64_t)i, (uint64_t)k) - 1.0;
            o->col[p + k] = (int32_t)c;
            o->val[p + k] = v;
            acc += v * wt[c];
        }
        double noise = 2.0 * u01(seed + 3, (uint64_t)i, 0) - 1.0;
        o->b[i] = (acc + 0.1 * noise >= 0.0) ? 1.0 : -1.0;
    }
    o->rowptr[N] = o->nnz;
    free(wt);
    build_transpose(o);
    return o;
}

void orc_obj_destroy(orc_objective *o) {
    if (!o) return;
    free(o->rowptr); free(o->col); free(o->val);
    free(o->rowptrT); free(o->colT); free(o->valT);
    free(o->b); free(o->scratch); free(o->scratch2); free(o->scratch2rows);
    free(o->lbs); free(o->ubs);
    free(o);
}
int64_t orc_csr_nnz(const orc_objective *o) { return o->nnz; }
int64_t orc_csr_nrows(const orc_objective *o) { return o->nrows; }
const int64_t *orc_csr_rowptr(const orc_objective *o) { return o->rowptr; }
const int32_t *orc_csr_col(const orc_objective *o) { return o->col; }
const double *orc_csr_val(const orc_objective *o) { return o->val; }
const double *orc_csr_b(const orc_objective *o) { return o->b; }
const int64_t *orc_csrT_rowptr(const orc_objective *o) { return o->rowptrT; }
const int32_t *orc_csrT_col(const orc_objective *o) { return o->colT; }
const double *orc_csrT_val(const orc_objective *o) { return o->valT; }
void orc_spmv(const orc_objective *o, int transposed, const double *x, double *y) {
    if (!transposed) csr_mv(o->nrows, o->rowptr, o->col, o->val, x, y, o->threads);
    else csr_mv(o->n, o->rowptrT, o->colT, o->valT, x, y, o->threads);
}
double orc_fdf(orc_objective *o, double *g, const double *x) { return o->fdf(o, g, x); }

/* x0 = (−1.2, 1, −1.2, 1, …) + perturb·(2 u01(seed,i,0) − 1)   (SURVEY.md §8d cfg 1/2) */
void orc_rosenbrock_x0(int64_t n, uint64_t seed, double perturb, double *x0) {
    for (int64_t i = 0; i < n; ++i) {
        double base = (i % 2 == 0) ? -1.2 : 1.0;
        x0[i] = perturb != 0.0 ? base + perturb * (2.0 * u01(seed, (uint64_t)i, 0) - 1.0) : base;
    }
}

/* ------------------------------------------------------------------------------------------
 * solver state
 * ---------------------------------------------------------------------------------------- */
typedef struct { /* LineSearchContainer, src/types.jl:84-100 */
    double *xp, *df_xp, *x, *u;
    int64_t n;
} ls_container;

typedef struct { /* L-BFGS history (new flavour; N&W Alg 7.4/7.5): a ring of m + 1 slots, at most m pairs live */
    int m, count, head;     /* head = slot of the newest pair */
    double **S, **Y;
    double *rho, *alpha;
    double gamma;
} lbfgs_hist;

typedef struct {
    orc_objective *obj;
    const orc_config *cfg;
    ls_container info;
    lbfgs_hist hist;
    int64_t evals_total;
} solver;

/* reduction sites (only matter in ORC_SUM_CGO mode): SITE_BLAS1 = reduced by an elementwise
 * BLAS-1 kernel (V=2,U=4); SITE_TRIAL = reduced inside the objective's trial kernels */
enum { SITE_BLAS1 = 0, SITE_TRIAL = 1 };
static inline double vdot_site(const solver *s, const double *a, const double *b, int site) {
    if (site == SITE_TRIAL) { g_site_V = s->obj->trial_V; g_site_U = s->obj->trial_V == 2 ? g_blas1_U : s->obj->trial_U; }
    else { g_site_V = 2; g_site_U = g_blas1_U; }
    double r = orc_dot(a, b, s->info.n, s->cfg->sum_mode, s->cfg->threads);
    g_site_V = 2; g_site_U = g_blas1_U;
    return r;
}
static inline double vdot(const solver *s, const double *a, const double *b) {
    return vdot_site(s, a, b, SITE_BLAS1);
}
static inline double tdot(const solver *s, const double *a, const double *b) {
    return vdot_site(s, a, b, SITE_TRIAL);
}
/* LinearAlgebra.norm → dnrm2; restated as sqrt(Σ x²) (no overflow rescaling) */
static inline double vnorm(const solver *s, const double *a) { return sqrt(vdot(s, a, a)); }
static inline double tnorm(const solver *s, const double *a) { return sqrt(tdot(s, a, a)); }

/* evalϕdϕ!, src/cg_utils.jl:3-22 */
static void eval_phi_dphi(solver *s, double a, double *phi, double *dphi) {
    ls_container *I = &s->info;
    for (int64_t i = 0; i < I->n; ++i) I->xp[i] = I->x[i] + a * I->u[i];   /* :13-15 */
    *phi = s->obj->fdf(s->obj, I->df_xp, I->xp);                            /* :18 */
    *dphi = tdot(s, I->df_xp, I->u);                                        /* :20 */
    s->evals_total++;
}

/* ---------------- StrongWolfeBisection, src/linesearch/nocedal.jl ---------------- */
/* zoom!, nocedal.jl:162-209 */
static int zoom(solver *s, double a_lb, double a_ub, double phi_lb, double phi0, double dphi0,
                double c1, double c2, int64_t evals, int64_t max_iters, double *phi_out,
                double *a_out, int64_t *evals_out) {
    double a = 0.0, phi_a = 0.0, dphi_a = 0.0;
    for (int64_t it = 0; it < max_iters; ++it) {
        a = (a_lb + a_ub) / 2;                                              /* :187 */
        eval_phi_dphi(s, a, &phi_a, &dphi_a);                               /* :190 */
        evals += 1;
        if ((phi_a > phi0 + c1 * a * dphi0) || (phi_a >= phi_lb)) {         /* :193 */
            a_ub = a;
        } else {
            if (fabs(dphi_a) <= -c2 * dphi0) {                              /* :196 */
                *phi_out = phi_a; *a_out = a; *evals_out = evals;
                return ORC_SUCCESS;
            }
            if (dphi_a * (a_ub - a_lb) >= 0) a_ub = a_lb;                   /* :200 */
            a_lb = a;
            phi_lb = phi_a;
        }
    }
    *phi_out = phi_a; *a_out = a; *evals_out = evals;
    return ORC_ZOOM_MAX_ITERS;                                              /* :208 */
}

/* linesearch!, nocedal.jl:33-158 */
static int ls_strong_wolfe(solver *s, double f_x, const double *df_x, double a_initial,
                           double *phi_out, double *a_out, int64_t *evals_out) {
    const orc_config *c = s->cfg;
    double c1 = c->c1, c2 = c->c2, growth = c->growth;
    if (!(0.0 < a_initial && isfinite(a_initial))) a_initial = 1.0;         /* :49-52 */
    double phi0 = f_x;
    double dphi0 = vdot(s, df_x, s->info.u);                                /* :56 */
    if (dphi0 > 0.0) {                                                      /* :57-63 */
        *phi_out = phi0; *a_out = 0.0; *evals_out = 0;
        return ORC_NON_DESCENT;
    }
    double a_prev = 0.0, phi_prev = phi0;
    double a = a_initial, phi_a = phi0, dphi_a = dphi0;
    double a_max = a * growth;
    int64_t evals = 0;
    int non_initial = 0;
    for (int64_t it = 0; it < c->ls_max_iters; ++it) {                      /* :76 */
        eval_phi_dphi(s, a, &phi_a, &dphi_a);                               /* :78 */
        evals += 1;
        int chk1 = phi_a > phi0 + c1 * a * dphi0;                           /* :81 */
        int chk2 = phi_a >= phi_prev;                                       /* :82 */
        if (chk1 || (chk2 && non_initial))                                  /* :83-105 */
            return zoom(s, a_prev, a, phi_prev, phi0, dphi0, c1, c2, evals, c->zoom_max_iters,
                        phi_out, a_out, evals_out);
        if (fabs(dphi_a) <= -c2 * dphi0) {                                  /* :107-110 */
            *phi_out = phi_a; *a_out = a; *evals_out = evals;
            return ORC_SUCCESS;
        }
        if (dphi_a >= 0)                                                    /* :112-134 */
            return zoom(s, a, a_prev, phi_a, phi0, dphi0, c1, c2, evals, c->zoom_max_iters,
                        phi_out, a_out, evals_out);
        a_prev = a; phi_prev = phi_a; non_initial = 1;                      /* :137-139 */
        a_max = a * growth;                                                 /* :143 */
        if (a > a_max) {                                                    /* :144-149 */
            *phi_out = phi_a; *a_out = a; *evals_out = evals;
            return ORC_A_MAX_OVERFLOW;
        }
        a = (a_max + a) / 2;                                                /* :150 */
    }
    *phi_out = phi_a; *a_out = a; *evals_out = evals;
    return ORC_LS_MAX_ITERS;                                                /* :157 */
}

/* ---------------- WolfeBisection, src/linesearch/wolfe.jl ---------------- */
enum { FEAS_OK = 0, FEAS_INFEASIBLE = 1, FEAS_LB_LARGER = 2 };
/* findfeasiblestepsize!, wolfe.jl:171-207 */
static int find_feasible(solver *s, int64_t *evals, double *a_io, double reduction, double lb,
                         int64_t max_iters, double *phi_out, double *dphi_out) {
    double a = *a_io;
    if (lb > a) { *phi_out = 0.0; *dphi_out = 0.0; return FEAS_LB_LARGER; } /* :186-188 */
    double phi_a, dphi_a;
    eval_phi_dphi(s, a, &phi_a, &dphi_a);                                   /* :191 */
    *evals += 1;
    int64_t iter = 1;
    while (a > lb && iter < max_iters) {                                    /* :195 */
        if (isfinite(phi_a) && isfinite(dphi_a)) {
            *phi_out = phi_a; *dphi_out = dphi_a; *a_io = a;
            return FEAS_OK;
        }
        a = a * reduction;                                                  /* :200 */
        eval_phi_dphi(s, a, &phi_a, &dphi_a);
        *evals += 1;
        iter += 1;
    }
    *phi_out = phi_a; *dphi_out = dphi_a; *a_io = a;
    return FEAS_INFEASIBLE;                                                 /* :206 */
}

static inline double jl_min(double a, double b) { /* Julia min: NaN-propagating */
    if (a != a) return a;
    if (b != b) return b;
    return a < b ? a : b;
}
/* evalwolfeconditions, wolfe.jl:219-251 (YuanWeiLuWolfe) and :264-294 (Wolfe) */
static void eval_wolfe(solver *s, double phi_a, double dphi_a, double a, double phi0, double dphi0,
                       int *valid_large, int *valid_small) {
    const orc_config *c = s->cfg;
    if (c->ls_kind == ORC_LS_YWL) {
        double nu = vdot(s, s->info.u, s->info.u);                          /* :240 */
        double t1 = -c->delta1 * dphi0, t2 = c->c1 * a * nu / 2;
        double rhs1 = phi0 + c->c1 * a * dphi0 + a * jl_min(t1, t2);
        *valid_large = phi_a <= rhs1;                                       /* :243-244 */
        double t3 = c->c1 * a * nu;
        double rhs2 = c->c2 * dphi0 + jl_min(t1, t3);
        *valid_small = dphi_a >= rhs2;                                      /* :247-248 */
    } else {
        *valid_large = phi_a <= phi0 + c->c1 * a * dphi0;                   /* :285-286 */
        *valid_small = dphi_a >= c->c2 * dphi0;                             /* :289-290 */
    }
}

/* linesearch!, wolfe.jl:13-165 */
static int ls_wolfe_bisection(solver *s, double f_x, const double *df_x, double a_initial,
                              double *phi_out, double *a_out, int64_t *evals_out) {
    const orc_config *c = s->cfg;
    ls_container *I = &s->info;
    const double reduction = 0.5, growth = 2.0;                             /* :23-24 */
    double max_step = c->max_step_size;
    if (!(max_step > a_initial && a_initial > 0.0))                         /* :30-32 */
        a_initial = fmin(1.0, max_step / 2);
    double phi0 = f_x;
    if (!isfinite(phi0)) { *phi_out = phi0; *a_out = 0; *evals_out = 0; return ORC_ACCEPTED_NON_FINITE; }
    double dphi0 = vdot(s, df_x, I->u);                                     /* :40 */
    if (dphi0 > 0.0) { *phi_out = phi0; *a_out = 0; *evals_out = 0; return ORC_NON_DESCENT; }
    double a = a_initial;
    int64_t evals = 0;
    double lb = 0.0, ub = INFINITY;
    double phi_a, dphi_a;
    int st = find_feasible(s, &evals, &a, reduction, 0.0, c->feas_max_iters, &phi_a, &dphi_a);
    if (st != FEAS_OK) { *phi_out = phi0; *a_out = 0; *evals_out = 0; return ORC_NO_INITIAL_FEASIBLE; }
    for (int64_t it = 0; it < c->ls_max_iters; ++it) {                      /* :67 */
        int vl, vs;
        eval_wolfe(s, phi_a, dphi_a, a, phi0, dphi0, &vl, &vs);             /* :70-78 */
        if (!vl || !vs) {
            if (!vl) {
                ub = a;                                                     /* :86 */
                a = (lb + ub) / 2;                                          /* :95 */
            } else {
                lb = a;                                                     /* :98 */
                if (!isfinite(ub)) {
                    a = growth * a;                                         /* :102 */
                    if (a > max_step) {                                     /* :104-112 */
                        *phi_out = phi0; *a_out = 0; *evals_out = 0;
                        return ORC_MAX_STEP_LENGTH;
                    }
                } else {
                    a = (lb + ub) / 2;                                      /* :114 */
                }
            }
            if (!(lb < a && a < ub)) {                                      /* :122 */
                /* !isapprox(norm(u+df_x), 0): with rtol=√eps, atol=0 this is norm != 0 (or NaN) */
                double *tmp = (double *)malloc(sizeof(double) * (size_t)I->n);
                for (int64_t i = 0; i < I->n; ++i) tmp[i] = I->u[i] + df_x[i];
                double nrm = vnorm(s, tmp);
                free(tmp);
                if (!(nrm == 0.0)) {                                        /* :123-129 */
                    lb = 0.0; ub = INFINITY;
                    a = a_initial;
                    for (int64_t i = 0; i < I->n; ++i) I->u[i] = -df_x[i];
                }
                /* else: wolfe.jl:131 builds a tuple but does not return it — falls through */
            }
            st = find_feasible(s, &evals, &a, reduction, lb, c->feas_max_iters, &phi_a, &dphi_a);
            if (st != FEAS_OK) {                                            /* :153-158 */
                *phi_out = phi0; *a_out = 0; *evals_out = 0;
                return ORC_NO_FEASIBLE_STEP;
            }
        } else {
            *phi_out = phi_a; *a_out = a; *evals_out = evals;               /* :160 */
            return ORC_SUCCESS;
        }
    }
    *phi_out = phi_a; *a_out = a; *evals_out = evals;
    return ORC_LS_MAX_ITERS;                                                /* :164 */
}

/* ---------------- Backtracking, src/linesearch/geometric.jl ---------------- */
/* evalbacktrackcondition (Armijo), geometric.jl:164-186 */
static int eval_armijo(double c1, double phi_a, double a, double phi0, double dphi0) {
    if (!isfinite(phi0) || !isfinite(phi_a) || !isfinite(a)) return 0;      /* :177-179 */
    return (phi0 - phi_a) >= -c1 * a * dphi0;                               /* :182-183 */
}
/* geometricsearch!, geometric.jl:102-152; divide=1 → a/ρ, else a·ρ (:7-13) */
static int geometric_search(solver *s, double a, int divide, int64_t evals, double phi_a,
                            double phi0, double dphi0, double *phi_out, double *a_out,
                            int64_t *evals_out) {
    const orc_config *c = s->cfg;
    double a_prev = a, phi_prev = phi_a, dummy;
    for (int64_t it = 0; it < c->ls_max_iters; ++it) {
        a = divide ? a / c->discount : a * c->discount;                     /* :127 */
        if (!isfinite(a)) { *phi_out = phi_prev; *a_out = a_prev; *evals_out = evals; return ORC_NON_FINITE_STEP; }
        if (a == a_prev) { *phi_out = phi_prev; *a_out = a_prev; *evals_out = evals; return ORC_SAME_STEP; }
        eval_phi_dphi(s, a, &phi_a, &dummy);                                /* :137 */
        evals += 1;
        if (!eval_armijo(c->c1, phi_a, a, phi0, dphi0)) {                   /* :140-144 */
            /* returns the PREVIOUS (ϕ, a) while info.xp/df_xp hold this rejected trial */
            *phi_out = phi_prev; *a_out = a_prev; *evals_out = evals;
            return ORC_SUCCESS;
        }
        a_prev = a; phi_prev = phi_a;
    }
    *phi_out = phi_a; *a_out = a; *evals_out = evals;
    return ORC_LS_MAX_ITERS;                                                /* :151 */
}
/* linesearch!, geometric.jl:22-100 */
static int ls_backtracking(solver *s, double f_x, const double *df_x, double a_initial,
                           double *phi_out, double *a_out, int64_t *evals_out) {
    const orc_config *c = s->cfg;
    ls_container *I = &s->info;
    double phi0 = f_x;
    if (!isfinite(phi0)) { *phi_out = phi0; *a_out = 0; *evals_out = 0; return ORC_ACCEPTED_NON_FINITE; }
    double dphi0 = vdot(s, df_x, I->u);                                     /* :43 */
    if (dphi0 > 0.0) { *phi_out = phi0; *a_out = 0; *evals_out = 0; return ORC_NON_DESCENT; }
    int64_t evals = 0;
    double a = a_initial;
    if (!isfinite(a)) a = fabs(phi0) / vdot(s, I->u, I->u);                 /* :50-53 */
    if (!isfinite(a)) a = 1.0;                                              /* :54-57 */
    double phi_a, dphi_a;
    int st = find_feasible(s, &evals, &a, 0.5, 0.0, c->feas_max_iters, &phi_a, &dphi_a);
    if (st != FEAS_OK) { *phi_out = phi0; *a_out = 0; *evals_out = 0; return ORC_NO_INITIAL_FEASIBLE; }
    eval_phi_dphi(s, a, &phi_a, &dphi_a);                                   /* :78 (redundant) */
    evals += 1;
    int valid = eval_armijo(c->c1, phi_a, a, phi0, dphi0);                  /* :81 */
    return geometric_search(s, a, valid ? 1 : 0, evals, phi_a, phi0, dphi0, phi_out, a_out,
                            evals_out);                                     /* :83-97 */
}

static int linesearch(solver *s, double f_x, const double *df_x, double a_initial, double *phi_out,
                      double *a_out, int64_t *evals_out) {
    switch (s->cfg->ls_kind) {
    case ORC_LS_WOLFE:
    case ORC_LS_YWL: return ls_wolfe_bisection(s, f_x, df_x, a_initial, phi_out, a_out, evals_out);
    case ORC_LS_BACKTRACK: return ls_backtracking(s, f_x, df_x, a_initial, phi_out, a_out, evals_out);
    default: return ls_strong_wolfe(s, f_x, df_x, a_initial, phi_out, a_out, evals_out);
    }
}

/* ---------------- β flavours, src/cg_flavours.jl ---------------- */
static inline double jl_max(double a, double b) { /* Julia max: NaN-propagating */
    if (a != a) return a;
    if (b != b) return b;
    return a > b ? a : b;
}
static double *vtmp(int64_t n) { return (double *)malloc(sizeof(double) * (size_t)(n > 0 ? n : 1)); }

/* getβ(::YuanWangSheng) cg_flavours.jl:51-79 and getβ(::HagerZhang) :87-108 */
static double beta_hz_family(solver *s, const double *g_next, const double *g, const double *u,
                             int yws) {
    int64_t n = s->info.n;
    double *y = vtmp(n), *tmp1 = vtmp(n), *tmp2 = vtmp(n);
    for (int64_t i = 0; i < n; ++i) y[i] = g_next[i] - g[i];                /* :63 / :96 */
    double R;
    if (yws) {
        double R1 = s->cfg->mu * tnorm(s, u) * tnorm(s, y);                 /* :65 */
        double R2 = tdot(s, u, y);                                          /* :66 */
        double R3 = 2 * tdot(s, y, y) * tdot(s, u, g_next) / tdot(s, y, g_next); /* :67 */
        R = jl_max(jl_max(R1, R2), R3);                                     /* :68 */
    } else {
        R = tdot(s, u, y);                                                  /* :98 */
    }
    double m = 2 * tdot(s, y, y) / R;                                       /* :73 / :102 */
    double beta;
    if (s->cfg->beta_form == ORC_BETA_FUSED) {
        /* algebraically equal single-pass form used by the fused GPU path:
         * Σ (y_i − m u_i)(g⁺_i / R) = (y·g⁺ − m u·g⁺) / R */
        beta = (tdot(s, y, g_next) - m * tdot(s, u, g_next)) / R;
    } else {
        for (int64_t i = 0; i < n; ++i) tmp2[i] = g_next[i] / R;            /* :71 / :100 */
        for (int64_t i = 0; i < n; ++i) tmp1[i] = y[i] - m * u[i];          /* :74 / :103 */
        beta = vdot(s, tmp1, tmp2);                                         /* :76 / :105 */
    }
    free(y); free(tmp1); free(tmp2);
    return beta;
}
/* getβ(::SallehAlhawarat) cg_flavours.jl:133-151 */
static double beta_sa(solver *s, const double *g_next, const double *g, const double *u) {
    double nrm = tnorm(s, g_next);
    double norm_sq = nrm * nrm;                                             /* :140 */
    double tmp = tdot(s, g_next, g);                                        /* :141 */
    if (norm_sq > tmp) {
        double num = norm_sq - tmp;
        double den = tdot(s, u, g_next) - tdot(s, u, g);                    /* :145 */
        return num / den;
    }
    return 0.0;
}
/* getβ(::LiuStorrey) cg_flavours.jl:157-170 */
static double beta_ls(solver *s, const double *g_next, const double *g, const double *u) {
    int64_t n = s->info.n;
    double *y = vtmp(n);
    for (int64_t i = 0; i < n; ++i) y[i] = g_next[i] - g[i];                /* :164 */
    double num = tdot(s, g_next, y);                                        /* :166 */
    double den = -tdot(s, u, y);                                            /* :167 */
    free(y);
    return num / den;
}

/* L-BFGS "getβ": push (s = xp − x, y = g⁺ − g) if s·y > 0.  Called at optim.jl:130, i.e.
 * before x ← xp, so info.x still holds the old iterate. */
static void lbfgs_push(solver *s, const double *g_next, const double *g) {
    lbfgs_hist *H = &s->hist;
    ls_container *I = &s->info;
    int slot = (H->head + 1) % (H->m + 1);
    double *S = H->S[slot], *Y = H->Y[slot];
    /* write into the slot after the newest, which no live pair occupies; only commit (advance head)
     * when curvature holds.  A rejected pair leaves the history unchanged. */
    for (int64_t i = 0; i < I->n; ++i) S[i] = I->xp[i] - I->x[i];
    for (int64_t i = 0; i < I->n; ++i) Y[i] = g_next[i] - g[i];
    double sy = vdot(s, S, Y);
    double yy = vdot(s, Y, Y);
    if (sy > 0.0) {
        H->head = slot;
        if (H->count < H->m) H->count++;
        H->rho[slot] = 1.0 / sy;
        H->gamma = sy / yy;
    }
}
/* L-BFGS updatedir!: two-loop recursion, N&W Alg 7.4; u = −H g */
static void lbfgs_updatedir(solver *s, double *u, const double *g) {
    lbfgs_hist *H = &s->hist;
    int64_t n = s->info.n;
    if (H->count == 0) {
        for (int64_t i = 0; i < n; ++i) u[i] = -g[i];
        return;
    }
    double *q = vtmp(n);
    for (int64_t i = 0; i < n; ++i) q[i] = g[i];
    for (int k = 0; k < H->count; ++k) {                /* newest → oldest */
        int slot = ((H->head - k) % (H->m + 1) + H->m + 1) % (H->m + 1);
        double al = H->rho[slot] * vdot(s, H->S[slot], q);
        H->alpha[slot] = al;
        const double *Y = H->Y[slot];
        for (int64_t i = 0; i < n; ++i) q[i] = q[i] - al * Y[i];
    }
    for (int64_t i = 0; i < n; ++i) q[i] = H->gamma * q[i];
    for (int k = H->count - 1; k >= 0; --k) {           /* oldest → newest */
        int slot = ((H->head - k) % (H->m + 1) + H->m + 1) % (H->m + 1);
        double be = H->rho[slot] * vdot(s, H->Y[slot], q);
        double cf = H->alpha[slot] - be;
        const double *S = H->S[slot];
        for (int64_t i = 0; i < n; ++i) q[i] = q[i] + S[i] * cf;
    }
    for (int64_t i = 0; i < n; ++i) u[i] = -q[i];
    free(q);
}

/* ------------------------------------------------------------------------------------------
 * minimizeobjective, src/engine/optim.jl:6-171
 * ---------------------------------------------------------------------------------------- */
int orc_minimize(orc_objective *obj, const double *x0, const orc_config *cfg, double *x_out,
                 double *g_out, orc_result *res, double *tr_f, double *tr_gnorm, double *tr_step,
                 int64_t *tr_evals) {
    if (!(0.0 < cfg->eps && cfg->eps < 1.0)) return -1;                     /* types.jl:187 */
    if (cfg->ls_kind == ORC_LS_STRONGWOLFE &&
        !(0.0 < cfg->c1 && cfg->c1 < cfg->c2 && cfg->c2 < 1.0 && cfg->growth > 1.0)) return -2; /* nocedal.jl:22-26 */
    int64_t D = obj->n;
    solver S;
    memset(&S, 0, sizeof(S));
    S.obj = obj; S.cfg = cfg;
    obj->sum_mode = cfg->sum_mode;
    if (cfg->threads > 0) obj->threads = cfg->threads;
    double *df_x = vtmp(D), *x = vtmp(D);                                   /* :20-21 */
    memcpy(x, x0, sizeof(double) * (size_t)D);
    S.info.n = D;
    S.info.xp = vtmp(D); S.info.df_xp = vtmp(D); S.info.x = vtmp(D); S.info.u = vtmp(D); /* :45 */
    ls_container *I = &S.info;
    if (cfg->flavour == ORC_LBFGS) {
        int m = cfg->lbfgs_m > 0 ? cfg->lbfgs_m : 1;
        S.hist.m = m;
        S.hist.S = (double **)calloc((size_t)m + 1, sizeof(double *));
        S.hist.Y = (double **)calloc((size_t)m + 1, sizeof(double *));
        for (int k = 0; k <= m; ++k) { S.hist.S[k] = vtmp(D); S.hist.Y[k] = vtmp(D); }
        S.hist.rho = (double *)calloc((size_t)m + 1, sizeof(double));
        S.hist.alpha = (double *)calloc((size_t)m + 1, sizeof(double));
    }

    double f_x = obj->fdf(obj, df_x, x);                                    /* :25 */
    S.evals_total++;
    double norm_df_x = tnorm(&S, df_x);                                     /* :26 */
    double norm_df_xp = NAN;
    double f_x0 = f_x;                                                      /* :31 */
    /* initializeLineSearchContainer!, cg_flavours.jl:22-35 */
    for (int64_t i = 0; i < D; ++i) I->u[i] = -df_x[i];
    memcpy(I->x, x, sizeof(double) * (size_t)D);
    memcpy(I->xp, x, sizeof(double) * (size_t)D);
    memcpy(I->df_xp, df_x, sizeof(double) * (size_t)D);
    double a_initial = NAN;                                                 /* :47 */

    int status = ORC_INCOMPLETE;
    int64_t iters_ran = 0;
    int64_t n_it;
    for (n_it = 1; n_it <= cfg->max_iters; ++n_it) {                        /* :50 */
        if (isfinite(f_x) && isfinite(norm_df_x)) {                         /* :53 */
            if (norm_df_x < cfg->eps) {
                status = (f_x <= f_x0) ? ORC_SUCCESS : ORC_INCREASING_OBJECTIVE; /* :56-80 */
                iters_ran = n_it - 1;
                goto done;
            }
        }
        double f_xp, a_star; int64_t evals;
        int st = linesearch(&S, f_x, df_x, a_initial, &f_xp, &a_star, &evals); /* :83 */
        a_initial = a_star;                                                 /* :92 */
        if (st != ORC_SUCCESS) { status = st; iters_ran = n_it - 1; goto done; } /* :93-104 */
        norm_df_xp = tnorm(&S, I->df_xp);                                   /* :107 */
        if (!isfinite(f_xp) || !isfinite(norm_df_xp)) {                     /* :108-121 */
            status = ORC_NON_FINITE_PROPOSED; iters_ran = n_it - 1; goto done;
        }
        double beta = 0.0;
        switch (cfg->flavour) {                                             /* :130-135 */
        case ORC_YWS: beta = beta_hz_family(&S, I->df_xp, df_x, I->u, 1); break;
        case ORC_SA: beta = beta_sa(&S, I->df_xp, df_x, I->u); break;
        case ORC_LS: beta = beta_ls(&S, I->df_xp, df_x, I->u); break;
        case ORC_LBFGS: lbfgs_push(&S, I->df_xp, df_x); break;
        default: beta = beta_hz_family(&S, I->df_xp, df_x, I->u, 0); break;
        }
        memcpy(x, I->xp, sizeof(double) * (size_t)D);                       /* :136 */
        f_x = f_xp;                                                         /* :138 */
        memcpy(df_x, I->df_xp, sizeof(double) * (size_t)D);                 /* :139 */
        memcpy(I->x, x, sizeof(double) * (size_t)D);                        /* :140 */
        norm_df_x = norm_df_xp;                                             /* :141 */
        if (cfg->flavour == ORC_LBFGS) lbfgs_updatedir(&S, I->u, df_x);
        else
            for (int64_t i = 0; i < D; ++i) I->u[i] = -df_x[i] + beta * I->u[i]; /* :145, cg_flavours.jl:10-12 */
        if (tr_f) {                                                         /* :152-159 */
            tr_f[n_it - 1] = f_x; tr_gnorm[n_it - 1] = norm_df_x;
            tr_step[n_it - 1] = a_star; tr_evals[n_it - 1] = evals;
        }
    }
    status = ORC_MAX_ITERS_REACHED;                                         /* :162-170 */
    iters_ran = cfg->max_iters;
done:
    res->objective = f_x;
    res->iters_ran = iters_ran;
    res->status = status;
    res->trace_len = iters_ran;                                             /* types.jl:148 */
    res->fdf_evals_total = S.evals_total;
    memcpy(x_out, x, sizeof(double) * (size_t)D);
    memcpy(g_out, df_x, sizeof(double) * (size_t)D);
    free(df_x); free(x);
    free(I->xp); free(I->df_xp); free(I->x); free(I->u);
    if (cfg->flavour == ORC_LBFGS) {
        for (int k = 0; k <= S.hist.m; ++k) { free(S.hist.S[k]); free(S.hist.Y[k]); }
        free(S.hist.S); free(S.hist.Y); free(S.hist.rho); free(S.hist.alpha);
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * solvesystem: CG for a nonlinear system g(x) = 0 (Yuan, Wang & Sheng 2019, Alg. 3.1),
 * src/engine/solve_system.jl.  `fdf!` returns some merit value f and writes g(x) into its first
 * argument.  Restated with its quirks:
 *  - linesearch! (:29-55) returns the 0-based trial index i as its "evaluation count" (:50);
 *  - its failure return (:54) reads the loop variable `i` outside the loop: in Julia that is an
 *    UndefVarError, so the :linesearch_failed branch of solvesystem (:131-142) is never reached
 *    by the reference itself.  The evident intent is restated here: status ORC_LINESEARCH_FAILED;
 *  - updateiteratesolvesys! (:237-253, called at :171-177) adds the projection step to `x_next`, which
 *    after the first swap (:196) holds the iterate BEFORE the current one, not the current one:
 *    from the second iteration on the method no longer follows Alg. 3.1 and in practice diverges
 *    (Booth, dev/solve_sys.jl settings: 1000 iterations to x ≈ (−683, −686)).  This is the
 *    default (bit-for-bit drop-in); ls->fix_stale_iterate = 1 projects from the current iterate.
 * a = s·ρ^i uses C pow (Julia's Float64^Int is its own accurate power; the two can differ in the
 * last place — third-party arithmetic, version unpinned, SURVEY.md §8c).
 * ---------------------------------------------------------------------------------------- */
int orc_solvesystem(orc_objective *obj, const double *x0, const orc_config *cfg,
                    const orc_solvesys_ls *ls, double *x_out, double *g_out, orc_result *res,
                    double *tr_f, double *tr_gnorm, double *tr_step, int64_t *tr_evals) {
    if (!(0.0 < cfg->eps && cfg->eps < 1.0)) return -1;                     /* types.jl:187 */
    if (!(0.0 < ls->rho && ls->rho < 1.0 && ls->s > 0.0)) return -2;        /* solve_system.jl:21-23 */
    if (cfg->flavour == ORC_LBFGS) return -3;                               /* BT <: CGβConfig (:69) */
    int64_t D = obj->n;
    solver S;
    memset(&S, 0, sizeof(S));
    S.obj = obj; S.cfg = cfg;
    obj->sum_mode = cfg->sum_mode;
    if (cfg->threads > 0) obj->threads = cfg->threads;
    double *df_x = vtmp(D), *x = vtmp(D), *x_next = vtmp(D);                /* :80-82 */
    memcpy(x, x0, sizeof(double) * (size_t)D);
    memcpy(x_next, x0, sizeof(double) * (size_t)D);
    S.info.n = D;
    S.info.xp = vtmp(D); S.info.df_xp = vtmp(D); S.info.x = vtmp(D); S.info.u = vtmp(D);
    ls_container *I = &S.info;
    double f_x = obj->fdf(obj, df_x, x);                                    /* :86 */
    S.evals_total++;
    double norm_df_x = tnorm(&S, df_x);                                     /* :87 */
    for (int64_t i = 0; i < D; ++i) I->u[i] = -df_x[i];                     /* :105, cg_flavours.jl:22-35 */
    memcpy(I->x, x, sizeof(double) * (size_t)D);
    memcpy(I->xp, x, sizeof(double) * (size_t)D);
    memcpy(I->df_xp, df_x, sizeof(double) * (size_t)D);
    int status = ORC_INCOMPLETE;
    int64_t iters_ran = 0, trace_len = 0, n_it;
    const double *xr = x, *gr = df_x;                                       /* what updateresult! copies */
    for (n_it = 1; n_it <= cfg->max_iters; ++n_it) {                        /* :109 */
        if (norm_df_x < cfg->eps) {                                         /* :112-123 */
            status = ORC_SUCCESS; iters_ran = trace_len = n_it - 1;
            goto done;
        }
        /* linesearch!, :29-55 */
        double norm_u_sq = vdot(&S, I->u, I->u);                            /* :39 */
        double f_xp = 0.0, norm_df_xp = NAN, a_star = NAN;
        int64_t evals = 0;
        int ok = 0;
        for (int64_t i = 0; i < ls->max_iters; ++i) {                       /* :41 */
            double a = ls->s * pow(ls->rho, (double)i);                     /* :42 */
            double dphi;
            eval_phi_dphi(&S, a, &f_xp, &dphi);                             /* :44 */
            norm_df_xp = tnorm(&S, I->df_xp);                               /* :47 */
            if (!(-dphi < ls->sigma * a * norm_df_xp * norm_u_sq)) {        /* :48 */
                a_star = a; evals = i; ok = 1;
                break;
            }
        }
        if (!ok) {                                                          /* :131-142 */
            status = ORC_LINESEARCH_FAILED; iters_ran = trace_len = n_it - 1;
            goto done;
        }
        if (norm_df_xp < cfg->eps) {                                        /* :146-168 */
            status = ORC_SUCCESS; iters_ran = trace_len = n_it;
            f_x = f_xp; xr = I->xp; gr = I->df_xp;
            if (tr_f) {
                tr_f[n_it - 1] = f_xp; tr_gnorm[n_it - 1] = tnorm(&S, I->df_xp);
                tr_step[n_it - 1] = a_star; tr_evals[n_it - 1] = evals;
            }
            goto done;
        }
        /* updateiteratesolvesys!, :237-253 (m :246, loop :248-250) */
        double m = a_star * tdot(&S, I->df_xp, I->u) / (norm_df_xp * norm_df_xp);
        if (ls->fix_stale_iterate)      /* Alg. 3.1 as published: project from the CURRENT iterate */
            for (int64_t i = 0; i < D; ++i) x_next[i] = x[i] + m * I->df_xp[i];
        else                            /* as written (:171-177, :249): x_next still holds the iterate before x */
            for (int64_t i = 0; i < D; ++i) x_next[i] = x_next[i] + m * I->df_xp[i];
        double f_x_next = obj->fdf(obj, I->df_xp, x_next);                  /* :179 */
        S.evals_total++;
        double nrm_next = tnorm(&S, I->df_xp);
        if (!isfinite(f_x_next) || !isfinite(nrm_next)) {                   /* :180-194 */
            status = ORC_NON_FINITE_PROPOSED; iters_ran = trace_len = n_it - 1;
            goto done;
        }
        { double *t = x; x = x_next; x_next = t; }                          /* :196 */
        xr = x;
        f_x = f_x_next;
        double beta = 0.0;                                                  /* :201-206 */
        switch (cfg->flavour) {
        case ORC_YWS: beta = beta_hz_family(&S, I->df_xp, df_x, I->u, 1); break;
        case ORC_SA: beta = beta_sa(&S, I->df_xp, df_x, I->u); break;
        case ORC_LS: beta = beta_ls(&S, I->df_xp, df_x, I->u); break;
        default: beta = beta_hz_family(&S, I->df_xp, df_x, I->u, 0); break;
        }
        memcpy(df_x, I->df_xp, sizeof(double) * (size_t)D);                 /* :207 */
        memcpy(I->x, x, sizeof(double) * (size_t)D);                        /* :208 */
        norm_df_x = nrm_next;                                               /* :209 (same vector, same order) */
        for (int64_t i = 0; i < D; ++i) I->u[i] = -df_x[i] + beta * I->u[i];   /* :212 */
        if (tr_f) {                                                         /* :215-222 */
            tr_f[n_it - 1] = f_x; tr_gnorm[n_it - 1] = norm_df_x;
            tr_step[n_it - 1] = a_star; tr_evals[n_it - 1] = evals;
        }
    }
    status = ORC_MAX_ITERS_REACHED;                                         /* :225-233 */
    iters_ran = trace_len = cfg->max_iters;
done:
    res->objective = f_x;
    res->iters_ran = iters_ran;
    res->status = status;
    res->trace_len = trace_len;
    res->fdf_evals_total = S.evals_total;
    memcpy(x_out, xr, sizeof(double) * (size_t)D);
    memcpy(g_out, gr, sizeof(double) * (size_t)D);
    free(df_x); free(x); free(x_next);
    free(I->xp); free(I->df_xp); free(I->x); free(I->u);
    return 0;
}

/* minimizeobjectivererun, optim.jl:173-208 */
int orc_minimize_rerun(orc_objective *obj, const double *x0, const orc_config *cfgs, int ncfg,
                       double *x_out, double *g_out, orc_result *res, int64_t tr_stride,
                       double *tr_f, double *tr_gnorm, double *tr_step, int64_t *tr_evals) {
    int64_t n = obj->n;
    int rc = orc_minimize(obj, x0, &cfgs[0], x_out, g_out, &res[0], tr_f, tr_gnorm, tr_step, tr_evals);
    if (rc) return rc;
    int nret = 1;
    for (int k = 1; k < ncfg; ++k) {
        if (res[nret - 1].status != ORC_SUCCESS) {                          /* :191 */
            const double *start = x_out + (int64_t)(nret - 1) * n;          /* :197 */
            rc = orc_minimize(obj, start, &cfgs[k], x_out + (int64_t)nret * n,
                              g_out + (int64_t)nret * n, &res[nret], tr_f + nret * tr_stride,
                              tr_gnorm + nret * tr_stride, tr_step + nret * tr_stride,
                              tr_evals + nret * tr_stride);
            if (rc) return rc;
            nret++;
        } else {
            return nret;                                                    /* :203 */
        }
    }
    return nret;
}
