// blas1.cu — the fused BLAS-1 chain of the CG iteration and the solver-state C ABI.
//
// One templated streaming kernel (k_blas1) drives every elementwise op: 128-bit coalesced
// loads (U = 4 in flight per input vector per lane), unfused IEEE arithmetic (-fmad=false: the
// reference's Julia loops do not contract a*b+c, SURVEY.md §3.5), canonical-order reductions
// (reduce.cuh).  Ops:
//   RosenTrial<FUSED>  evalϕdϕ! (src/cg_utils.jl:3-22) for the extended Rosenbrock objective,
//                      fused with norm(df_xp) (src/engine/optim.jl:107) and every dot of getβ
//                      (src/cg_flavours.jl:51-170); FUSED also does updatedir! (:2-15) first.
//   DirUpdate          updatedir! u = −g + βu (cg_flavours.jl:2-15) + next dot(df_x,u)
//                      (nocedal.jl:56, wolfe.jl:40, geometric.jl:43) + dot(u,u) (wolfe.jl:240)
//   ResetDir           u = −g (cg_flavours.jl:28, wolfe.jl:129)
//   BetaLiteral        Σ (y_i − m u_i)(g⁺_i / R)  (cg_flavours.jl:71-76, :100-105, as written)
//   NormUPlusG         ‖u + df_x‖² (wolfe.jl:123)
//   AxpyDir            xp = x + a u [after u = −g + βu] for multi-kernel (CSR) objectives
//   L-BFGS ops         stage (s,y), two-loop recursion steps (N&W Alg 7.4)
#include "internal.cuh"
#include "reduce.cuh"

// ------------------------------------------------------------------ generic streaming kernel
template <class Op>
__global__ void __launch_bounds__(CGO_B, Op::OCC) k_blas1(Op op, int64_t n, RedArgs red) {
    constexpr int K = Op::K;
    __shared__ double sm[K * CGO_NW];
    const int64_t nq = (n + 1) >> 1;
    constexpr int64_t tileq = (int64_t)CGO_B * CGO_U_VEC;
    const int64_t ntiles = (nq + tileq - 1) / tileq;
    const int nact = (int)(ntiles < (int64_t)red.G ? ntiles : (int64_t)red.G);
    cgo_wait_flags(red, BarAll());
    op.prologue();
    for (int v = blockIdx.x; v < nact; v += gridDim.x) {
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.0;
        for (int64_t tile = v; tile < ntiles; tile += red.G) {
            const int64_t q0 = tile * tileq + threadIdx.x;
            typename Op::In in[CGO_U_VEC];
#pragma unroll
            for (int j = 0; j < CGO_U_VEC; ++j) {
                const int64_t q = q0 + (int64_t)j * CGO_B;
                if (q < nq) in[j] = op.load(q);
            }
#pragma unroll
            for (int j = 0; j < CGO_U_VEC; ++j) {
                const int64_t q = q0 + (int64_t)j * CGO_B;
                if (q < nq) op.apply(q, in[j], acc, 2 * q + 1 < n);
            }
        }
        cgo_cta_combine<K>(acc, sm);
        cgo_publish<K>(red, v, acc);
    }
    cgo_grid_finish<K>(red, nact, sm);
}

template <class Op>
static int launch_blas1(cgo_ctx *c, const Op &op, int64_t n, const RedArgs &red) {
    const int64_t nq = (n + 1) >> 1;
    const int64_t tileq = (int64_t)CGO_B * CGO_U_VEC;
    int64_t ntiles = (nq + tileq - 1) / tileq;
    int64_t nact = ntiles < red.G ? ntiles : red.G;
    int64_t phys = (int64_t)c->sms * Op::OCC;
    int grid = (int)(nact < phys ? nact : phys);
    if (grid < 1) grid = 1;
    cgo_timer_begin(c, Op::TCLASS);
    k_blas1<Op><<<grid, CGO_B, 0, c->stream>>>(op, n, red);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    return 0;
}

__device__ __forceinline__ double2 ld2rw(const double2 *p) {   // vectors updated in place
    double2 r;
    asm volatile("ld.global.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p) : "memory");
    return r;
}

// ------------------------------------------------------------------ ops
// extended Rosenbrock trial.  Elementwise spec (bit-for-bit the oracle's rosen_fdf):
//   t = x2 − x1*x1; om = 1 − x1; f = (100 t) t + om om; g1 = (−400 x1) t − 2 om; g2 = 200 t
template <bool FUSED>
struct RosenTrial {
    static constexpr int TCLASS = CGO_T_TRIAL;
    static constexpr int K = 9;
    static constexpr int OCC = 2;
    struct In { double2 x, u, g; };
    const double2 *x, *g;
    double2 *u;
    double2 *xp, *gp;
    double a, beta;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.x = cgo_ld2(x + q);
        r.g = cgo_ld2(g + q);
        r.u = FUSED ? ld2rw(u + q) : cgo_ld2(u + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool) const {
        double2 uu = in.u;
        if (FUSED) {                                   // updatedir!, cg_flavours.jl:10-12
            uu.x = -in.g.x + beta * in.u.x;
            uu.y = -in.g.y + beta * in.u.y;
            cgo_st2(u + q, uu);
        }
        double2 p;                                     // cg_utils.jl:13-15
        p.x = in.x.x + a * uu.x;
        p.y = in.x.y + a * uu.y;
        cgo_st2(xp + q, p);
        const double t = p.y - p.x * p.x;
        const double om = 1.0 - p.x;
        const double f = (100.0 * t) * t + om * om;
        double2 gn;
        gn.x = (-400.0 * p.x) * t - 2.0 * om;
        gn.y = 200.0 * t;
        cgo_st2(gp + q, gn);
        const double y1 = gn.x - in.g.x, y2 = gn.y - in.g.y;
        acc[CGO_P_PHI] = acc[CGO_P_PHI] + f;
        acc[CGO_P_DPHI] = acc[CGO_P_DPHI] + gn.x * uu.x;   acc[CGO_P_DPHI] = acc[CGO_P_DPHI] + gn.y * uu.y;
        acc[CGO_P_GPGP] = acc[CGO_P_GPGP] + gn.x * gn.x;   acc[CGO_P_GPGP] = acc[CGO_P_GPGP] + gn.y * gn.y;
        acc[CGO_P_YY] = acc[CGO_P_YY] + y1 * y1;           acc[CGO_P_YY] = acc[CGO_P_YY] + y2 * y2;
        acc[CGO_P_UY] = acc[CGO_P_UY] + uu.x * y1;         acc[CGO_P_UY] = acc[CGO_P_UY] + uu.y * y2;
        acc[CGO_P_YGP] = acc[CGO_P_YGP] + y1 * gn.x;       acc[CGO_P_YGP] = acc[CGO_P_YGP] + y2 * gn.y;
        acc[CGO_P_GPG] = acc[CGO_P_GPG] + gn.x * in.g.x;   acc[CGO_P_GPG] = acc[CGO_P_GPG] + gn.y * in.g.y;
        acc[CGO_P_UG] = acc[CGO_P_UG] + uu.x * in.g.x;     acc[CGO_P_UG] = acc[CGO_P_UG] + uu.y * in.g.y;
        acc[CGO_P_UU] = acc[CGO_P_UU] + uu.x * uu.x;       acc[CGO_P_UU] = acc[CGO_P_UU] + uu.y * uu.y;
    }
};

// u = −g + βu (RESET: u = −g); pack {g·u, u·u}
template <bool RESET>
struct DirUpdate {
    static constexpr int TCLASS = CGO_T_DIR;
    static constexpr int K = 2;
    static constexpr int OCC = 4;
    struct In { double2 g, u; };
    const double2 *g;
    double2 *u;
    double beta;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.g = cgo_ld2(g + q);
        if (!RESET) r.u = ld2rw(u + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 un;
        if (RESET) { un.x = -in.g.x; un.y = -in.g.y; }
        else { un.x = -in.g.x + beta * in.u.x; un.y = -in.g.y + beta * in.u.y; }
        if (!v2) un.y = 0.0;
        cgo_st2(u + q, un);
        acc[CGO_D_GU] = acc[CGO_D_GU] + in.g.x * un.x;
        acc[CGO_D_UU] = acc[CGO_D_UU] + un.x * un.x;
        if (v2) {
            acc[CGO_D_GU] = acc[CGO_D_GU] + in.g.y * un.y;
            acc[CGO_D_UU] = acc[CGO_D_UU] + un.y * un.y;
        }
    }
};

// Σ (y_i − m u_i)(g⁺_i / R) with y = g⁺ − g: tmp2 = g_next ./ R; tmp1 = y − m .* u; dot(tmp1,tmp2)
struct BetaLiteral {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 1;
    static constexpr int OCC = 2;
    struct In { double2 gp, g, u; };
    const double2 *gp, *g, *u;
    double R, m;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.gp = cgo_ld2(gp + q); r.g = cgo_ld2(g + q); r.u = cgo_ld2(u + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t, const In &in, double (&acc)[K], bool v2) const {
        const double y1 = in.gp.x - in.g.x;
        const double t2a = in.gp.x / R;
        const double t1a = y1 - m * in.u.x;
        acc[0] = acc[0] + t1a * t2a;
        if (v2) {
            const double y2 = in.gp.y - in.g.y;
            const double t2b = in.gp.y / R;
            const double t1b = y2 - m * in.u.y;
            acc[0] = acc[0] + t1b * t2b;
        }
    }
};

struct NormUPlusG {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 1;
    static constexpr int OCC = 4;
    struct In { double2 g, u; };
    const double2 *g, *u;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.g = cgo_ld2(g + q); r.u = cgo_ld2(u + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t, const In &in, double (&acc)[K], bool v2) const {
        const double t1 = in.u.x + in.g.x;
        acc[0] = acc[0] + t1 * t1;
        if (v2) { const double t2 = in.u.y + in.g.y; acc[0] = acc[0] + t2 * t2; }
    }
};

// xp = x + a u, optionally after u = −g + βu; pack {g·u, u·u, xp·xp}.  PUSH: the first / last
// `hq` double2 of xp are also stored into the ring neighbours' halos (peer memory, NVLink) —
// the halo exchange of the sharded CSR objectives, fused into the kernel that produces xp.
template <bool FUSED, int PUSH>      // PUSH: 0 none, 1 ring halos, 2 whole shard to every rank
struct AxpyDir {
    static constexpr int TCLASS = CGO_T_AXPY;
    static constexpr int K = 3;
    static constexpr int OCC = 2;
    struct In { double2 x, u, g; };
    const double2 *x, *g;
    double2 *u, *xp;
    double a, beta;
    double2 *prev_right, *next_left;     // PUSH 1
    int64_t hq, nq;                      // PUSH 1: halo and local length in double2
    void *const *dst_all;                // PUSH 2: nranks destinations (device table)
    int nranks;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.x = cgo_ld2(x + q);
        r.g = cgo_ld2(g + q);
        r.u = FUSED ? ld2rw(u + q) : cgo_ld2(u + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 uu = in.u;
        if (FUSED) {
            uu.x = -in.g.x + beta * in.u.x;
            uu.y = v2 ? -in.g.y + beta * in.u.y : 0.0;
            cgo_st2(u + q, uu);
        }
        double2 p;
        p.x = in.x.x + a * uu.x;
        p.y = v2 ? in.x.y + a * uu.y : 0.0;
        cgo_st2(xp + q, p);
        if (PUSH == 1) {
            if (q < hq) cgo_st2(prev_right + q, p);
            if (q >= nq - hq) cgo_st2(next_left + (q - (nq - hq)), p);
        }
        if (PUSH == 2) {
            for (int r = 0; r < nranks; ++r) cgo_st2((double2 *)dst_all[r] + q, p);
        }
        acc[0] = acc[0] + in.g.x * uu.x;
        acc[1] = acc[1] + uu.x * uu.x;
        acc[2] = acc[2] + p.x * p.x;
        if (v2) {
            acc[0] = acc[0] + in.g.y * uu.y;
            acc[1] = acc[1] + uu.y * uu.y;
            acc[2] = acc[2] + p.y * p.y;
        }
    }
};

// Sample-sharded logistic regression (multi-rank): every rank's Aᵀ_r c_r partial gradient slice
// of this rank's feature shard sits in q[r·stride ..]; add them in rank order, scale, add the
// regulariser, and reduce the same eight dots as the single-rank SpMVᵀ epilogue (csr.cu EpiGrad).
struct GradCombine {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 8;
    static constexpr int OCC = 2;
    struct In { double2 s, u, g, w; };
    const double2 *q, *u, *g, *w;
    double2 *gp;
    int nparts;
    int64_t stride2;            // part stride in double2 units
    double invN, lambda;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t i) const {
        In r;
        r.s = ld2rw(q + i);          // coherent loads: peers deliver q while this kernel waits for their flags
        for (int p = 1; p < nparts; ++p) {
            const double2 t = ld2rw(q + (int64_t)p * stride2 + i);
            r.s.x = r.s.x + t.x;
            r.s.y = r.s.y + t.y;
        }
        r.u = cgo_ld2(u + i); r.g = cgo_ld2(g + i); r.w = cgo_ld2(w + i);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t i, const In &in, double (&acc)[K], bool v2) const {
        double2 gn;
        gn.x = in.s.x * invN + lambda * in.w.x;
        gn.y = v2 ? in.s.y * invN + lambda * in.w.y : 0.0;
        cgo_st2(gp + i, gn);
        const double ux = in.u.x, uy = v2 ? in.u.y : 0.0, gx = in.g.x, gy = v2 ? in.g.y : 0.0;
        const double y1 = gn.x - gx, y2 = gn.y - gy;
        acc[CGO_P_DPHI - 1] = acc[CGO_P_DPHI - 1] + gn.x * ux;
        acc[CGO_P_GPGP - 1] = acc[CGO_P_GPGP - 1] + gn.x * gn.x;
        acc[CGO_P_YY - 1] = acc[CGO_P_YY - 1] + y1 * y1;
        acc[CGO_P_UY - 1] = acc[CGO_P_UY - 1] + ux * y1;
        acc[CGO_P_YGP - 1] = acc[CGO_P_YGP - 1] + y1 * gn.x;
        acc[CGO_P_GPG - 1] = acc[CGO_P_GPG - 1] + gn.x * gx;
        acc[CGO_P_UG - 1] = acc[CGO_P_UG - 1] + ux * gx;
        acc[CGO_P_UU - 1] = acc[CGO_P_UU - 1] + ux * ux;
        if (v2) {
            acc[CGO_P_DPHI - 1] = acc[CGO_P_DPHI - 1] + gn.y * uy;
            acc[CGO_P_GPGP - 1] = acc[CGO_P_GPGP - 1] + gn.y * gn.y;
            acc[CGO_P_YY - 1] = acc[CGO_P_YY - 1] + y2 * y2;
            acc[CGO_P_UY - 1] = acc[CGO_P_UY - 1] + uy * y2;
            acc[CGO_P_YGP - 1] = acc[CGO_P_YGP - 1] + y2 * gn.y;
            acc[CGO_P_GPG - 1] = acc[CGO_P_GPG - 1] + gn.y * gy;
            acc[CGO_P_UG - 1] = acc[CGO_P_UG - 1] + uy * gy;
            acc[CGO_P_UU - 1] = acc[CGO_P_UU - 1] + uy * uy;
        }
    }
};

// Dots of the gather-bound CSR objectives (csr.cu k_spmv_direct keeps no reduction): Σ r² after K_b; after K_c
// the eight dots of EpiGrad — norm(df_xp)² (optim.jl:107), dϕ = g⁺·u (cg_utils.jl:20) and the getβ dots
// (cg_flavours.jl:63-76, 96-105, 140-145, 164-167) — in the BLAS-1 canonical order.
struct VecSumSq {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 1;
    static constexpr int OCC = 4;
    struct In { double2 a; };
    const double2 *a;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const { return In{cgo_ld2(a + q)}; }
    __device__ __forceinline__ void apply(int64_t, const In &in, double (&acc)[K], bool v2) const {
        acc[0] = acc[0] + in.a.x * in.a.x;
        if (v2) acc[0] = acc[0] + in.a.y * in.a.y;
    }
};
struct Dots3 {                 // {a·b, b·b, a·a}
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 3;
    static constexpr int OCC = 4;
    struct In { double2 a, b; };
    const double2 *a, *b;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const { return In{cgo_ld2(a + q), cgo_ld2(b + q)}; }
    __device__ __forceinline__ void apply(int64_t, const In &in, double (&acc)[K], bool v2) const {
        acc[0] = acc[0] + in.a.x * in.b.x; acc[1] = acc[1] + in.b.x * in.b.x; acc[2] = acc[2] + in.a.x * in.a.x;
        if (v2) { acc[0] = acc[0] + in.a.y * in.b.y; acc[1] = acc[1] + in.b.y * in.b.y; acc[2] = acc[2] + in.a.y * in.a.y; }
    }
};
struct GradDots {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 8;
    static constexpr int OCC = 2;
    struct In { double2 gp, g, u; };
    const double2 *gp, *g, *u;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const { return In{cgo_ld2(gp + q), cgo_ld2(g + q), cgo_ld2(u + q)}; }
    __device__ __forceinline__ void one(double gn, double gg, double uu, double (&acc)[K]) const {
        const double y = gn - gg;
        acc[CGO_P_DPHI - 1] = acc[CGO_P_DPHI - 1] + gn * uu;
        acc[CGO_P_GPGP - 1] = acc[CGO_P_GPGP - 1] + gn * gn;
        acc[CGO_P_YY - 1] = acc[CGO_P_YY - 1] + y * y;
        acc[CGO_P_UY - 1] = acc[CGO_P_UY - 1] + uu * y;
        acc[CGO_P_YGP - 1] = acc[CGO_P_YGP - 1] + y * gn;
        acc[CGO_P_GPG - 1] = acc[CGO_P_GPG - 1] + gn * gg;
        acc[CGO_P_UG - 1] = acc[CGO_P_UG - 1] + uu * gg;
        acc[CGO_P_UU - 1] = acc[CGO_P_UU - 1] + uu * uu;
    }
    __device__ __forceinline__ void apply(int64_t, const In &in, double (&acc)[K], bool v2) const {
        one(in.gp.x, in.g.x, in.u.x, acc);
        if (v2) one(in.gp.y, in.g.y, in.u.y, acc);
    }
};

// logistic loss and its derivative from the margins (csr.cu EpiLogit, oracle logreg_fdf), in place: z → c = −y σ;
// Σ ℓ.  PUSH: this rank's shard of c also goes into every rank's all-gathered copy (peer memory), then flag
// CGO_F_GPART + me of every rank
template <bool PUSH>
struct LogitLoss {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 1;
    static constexpr int OCC = 2;
    struct In { double2 z, y; };
    double2 *zc;
    const double2 *y;
    void *const *dst_all;
    int nranks;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const { return In{ld2rw(zc + q), cgo_ld2(y + q)}; }
    __device__ __forceinline__ double one(double z, double yy, double (&acc)[K]) const {
        const double t = -yy * z;
        const double e = exp(-fabs(t));
        const double l = (t > 0.0 ? t : 0.0) + log1p(e);
        const double sg = t >= 0.0 ? 1.0 / (1.0 + e) : e / (1.0 + e);
        acc[0] = acc[0] + l;
        return -yy * sg;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 c;
        c.x = one(in.z.x, in.y.x, acc);
        c.y = v2 ? one(in.z.y, in.y.y, acc) : 0.0;
        cgo_st2(zc + q, c);
        if (PUSH) for (int r = 0; r < nranks; ++r) cgo_st2((double2 *)dst_all[r] + q, c);
    }
};

// updateiteratesolvesys! (src/engine/solve_system.jl:237-253): x_next[i] = base[i] + m*df_xp[i]
// (base = x_next itself as the reference writes it, or x for Alg. 3.1 as published)
struct SolveSysProject {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 1;
    static constexpr int OCC = 4;
    struct In { double2 b, g; };
    const double2 *base, *gp;
    double2 *xn;
    double m;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.b = ld2rw(base + q); r.g = cgo_ld2(gp + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 o;
        o.x = in.b.x + m * in.g.x;
        o.y = v2 ? in.b.y + m * in.g.y : 0.0;
        cgo_st2(xn + q, o);
        acc[0] = acc[0] + o.x * o.x;        // (‖x_next‖², unused: the kernel template reduces K >= 1 sums)
        if (v2) acc[0] = acc[0] + o.y * o.y;
    }
};

// L-BFGS: S = xp − x, Y = g⁺ − g; pack {s·y, y·y}
struct LbfgsStage {
    static constexpr int TCLASS = CGO_T_LBFGS;
    static constexpr int K = 2;
    static constexpr int OCC = 2;
    struct In { double2 xp, x, gp, g; };
    const double2 *xp, *x, *gp, *g;
    double2 *S, *Y;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.xp = cgo_ld2(xp + q); r.x = cgo_ld2(x + q); r.gp = cgo_ld2(gp + q); r.g = cgo_ld2(g + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 s, y;
        s.x = in.xp.x - in.x.x; y.x = in.gp.x - in.g.x;
        s.y = v2 ? in.xp.y - in.x.y : 0.0; y.y = v2 ? in.gp.y - in.g.y : 0.0;
        cgo_st2(S + q, s); cgo_st2(Y + q, y);
        acc[0] = acc[0] + s.x * y.x; acc[1] = acc[1] + y.x * y.x;
        if (v2) { acc[0] = acc[0] + s.y * y.y; acc[1] = acc[1] + y.y * y.y; }
    }
};

// Two-loop recursion steps.  Scalars produced by the previous kernel are read from device
// memory (no host round trip inside the recursion).
//  MODE 0: q = g;                              dot = S·q          (first step of loop 1)
//  MODE 1: q = q − (ρp·dp) Yp;                 dot = S·q          (loop 1)
//  MODE 2: q = q − (ρp·dp) Yp; q = γ q;        dot = Y·q          (end of loop 1, start of loop 2)
//  MODE 3: q = q + Sp (αp − ρp·dp);            dot = Y·q          (loop 2)
//  MODE 4: q = q + Sp (αp − ρp·dp); u = −q;    pack {g·u, u·u}    (end of loop 2)
// with αp = ρp·(loop-1 dot of that pair) read from alpha_slot.
template <int MODE>
struct LbfgsStep {
    static constexpr int TCLASS = CGO_T_LBFGS;
    static constexpr int K = (MODE == 4) ? 2 : 1;
    static constexpr int OCC = 2;
    struct In { double2 q, a, b; };
    double2 *q;             // in/out
    const double2 *A;       // Yp (modes 1,2) or Sp (modes 3,4) or g (mode 0)
    const double2 *B;       // vector dotted with the new q (modes 0-3) or g (mode 4)
    double2 *uout;          // mode 4
    const double *dprev;    // device scalar: previous kernel's dot
    const double *alpha_dot;// device scalar: loop-1 dot of the pair applied in modes 3,4
    double rho_prev, gamma;
    double coef;
    __device__ __forceinline__ void prologue() {
        if (MODE == 1 || MODE == 2) coef = rho_prev * __ldcg(dprev);
        if (MODE == 3 || MODE == 4) coef = rho_prev * __ldcg(alpha_dot) - rho_prev * __ldcg(dprev);
    }
    __device__ __forceinline__ In load(int64_t i) const {
        In r;
        if (MODE != 0) r.q = ld2rw(q + i);
        r.a = cgo_ld2(A + i);
        r.b = cgo_ld2(B + i);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t i, const In &in, double (&acc)[K], bool v2) const {
        double2 qn;
        if (MODE == 0) { qn = in.a; }
        else if (MODE == 1 || MODE == 2) { qn.x = in.q.x - coef * in.a.x; qn.y = in.q.y - coef * in.a.y; }
        else { qn.x = in.q.x + in.a.x * coef; qn.y = in.q.y + in.a.y * coef; }
        if (MODE == 2) { qn.x = gamma * qn.x; qn.y = gamma * qn.y; }
        if (!v2) qn.y = 0.0;
        if (MODE == 4) {
            double2 un; un.x = -qn.x; un.y = v2 ? -qn.y : 0.0;
            cgo_st2(uout + i, un);
            acc[0] = acc[0] + in.b.x * un.x; acc[1] = acc[1] + un.x * un.x;
            if (v2) { acc[0] = acc[0] + in.b.y * un.y; acc[1] = acc[1] + un.y * un.y; }
        } else {
            cgo_st2(q + i, qn);
            acc[0] = acc[0] + in.b.x * qn.x;
            if (v2) acc[0] = acc[0] + in.b.y * qn.y;
        }
    }
};

// ------------------------------------------------------------------ Rosenbrock objective
static inline uint64_t h_mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
double cgo_host_u01(uint64_t seed, uint64_t i, uint64_t k) {
    uint64_t h = h_mix64(seed + 0x9E3779B97F4A7C15ULL);
    h = h_mix64(h ^ (i + 0x9E3779B97F4A7C15ULL));
    h = h_mix64(h ^ (k + 0x632BE59BD9B4E019ULL));
    return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}

struct RosenObj : cgo_obj {
    int eval_trial(cgo_state *st, double a, bool fused, double beta, double *out) override {
        RedArgs red = cgo_red_args(ctx);
        if (fused) {
            RosenTrial<true> op;
            op.x = (const double2 *)st->x; op.g = (const double2 *)st->g; op.u = (double2 *)st->u;
            op.xp = (double2 *)st->xp; op.gp = (double2 *)st->gp; op.a = a; op.beta = beta;
            CGO_TRY(launch_blas1(ctx, op, st->n, red));
        } else {
            RosenTrial<false> op;
            op.x = (const double2 *)st->x; op.g = (const double2 *)st->g; op.u = (double2 *)st->u;
            op.xp = (double2 *)st->xp; op.gp = (double2 *)st->gp; op.a = a; op.beta = 0.0;
            CGO_TRY(launch_blas1(ctx, op, st->n, red));
        }
        CGO_TRY(cgo_finish_pack(ctx, 9, out));
        out[CGO_P_DIR_GU] = out[CGO_P_UG];     // same kernel, same (V=2,U=4) site
        out[CGO_P_DIR_UU] = out[CGO_P_UU];
        return 0;
    }
    // fused minimum (SURVEY.md §8d): R x,g,u ; W (u,) xp, g⁺
    double bytes_per_eval() const override { return 8.0 * 5.0 * (double)n_local; }
    void reduction_site(int32_t *V, int32_t *U) const override { *V = 2; *U = CGO_U_VEC; }
    int default_x0(uint64_t seed, double perturb, double *x0) override {
        for (int64_t i = 0; i < n_local; ++i) {
            int64_t gi = offset + i;
            double base = (gi % 2 == 0) ? -1.2 : 1.0;
            x0[i] = perturb != 0.0 ? base + perturb * (2.0 * cgo_host_u01(seed, (uint64_t)gi, 0) - 1.0) : base;
        }
        return 0;
    }
};

// ------------------------------------------------------------------ user objective
// The reference takes ANY fdf!(g, x) -> f (src/engine/optim.jl:6-11, :25; src/cg_utils.jl:18).  On the device that
// callback is a host function that ENQUEUES, on the ctx stream, whatever computes g⁺ = ∇f(xp) and f from the
// trial point (its own kernels, cuBLAS / cuSPARSE calls, a framework's ops): cgo_user_fdf.  The library does the
// rest of evalϕdϕ! and of getβ around it: K_a xp = x + a u [after updatedir!], then the callback, then one BLAS-1
// pass for dϕ = g⁺·u, ‖g⁺‖² and the getβ dots (GradDots).  Two kernels of the library per trial + the user's.
__global__ void k_scalar_to_pack(const double *src, double *dst) { *dst = *src; }
struct UserObj : cgo_obj {
    cgo_user_fdf fn = nullptr;
    void *user = nullptr;
    double *d_f = nullptr;
    ~UserObj() override {
        if (ctx && cgo_ctx_alive(ctx)) cudaSetDevice(ctx->device);
        cudaFree(d_f);
    }
    int eval_trial(cgo_state *st, double a, bool fused, double beta, double *out) override {
        CGO_TRY(cgo_blas1_axpy_dir(st, a, fused, beta));                                  // K_a
        const int rc = fn(user, (void *)ctx->stream, st->n, offset, st->xp, st->gp, d_f);
        CGO_CHECK(rc == 0, "user objective callback returned %d", rc);
        k_scalar_to_pack<<<1, 1, 0, ctx->stream>>>(d_f, cgo_red_args(ctx, CGO_P_PHI).out);  // this rank's part of f
        ctx->launches++;
        CGO_CUDA(cudaGetLastError());
        CGO_TRY(cgo_blas1_grad_dots(st));
        return cgo_finish_pack(ctx, 12, out);
    }
    double bytes_per_eval() const override { return 8.0 * 6.0 * (double)n_local; }   // K_a 24n + dots 24n (+ the user's)
    void reduction_site(int32_t *V, int32_t *U) const override { *V = 2; *U = CGO_U_VEC; }
    int default_x0(uint64_t, double, double *x0) override {
        for (int64_t i = 0; i < n_local; ++i) x0[i] = 0.0;
        return 0;
    }
};
extern "C" int cgo_obj_user_create(cgo_ctx *ctx, int64_t n_global, cgo_user_fdf fdf, void *user, cgo_obj **out) {
    CGO_CHECK(ctx && fdf && out, "NULL argument");
    CGO_CHECK(n_global >= 2 && n_global % 2 == 0, "user objective: need an even n >= 2 (got %lld; pad with a fixed coordinate)", (long long)n_global);
    CGO_CUDA(cudaSetDevice(ctx->device));
    int64_t lo, hi;
    CGO_TRY(cgo_shard_range(n_global, ctx->nranks, ctx->rank, 2, &lo, &hi));
    UserObj *o = new UserObj();
    o->ctx = ctx; o->fn = fdf; o->user = user;
    o->n_global = n_global; o->offset = lo; o->n_local = hi - lo;
    if (cudaMalloc(&o->d_f, sizeof(double)) != cudaSuccess) { delete o; cgo_set_error("cudaMalloc failed"); return 1; }
    *out = o;
    return 0;
}

// ------------------------------------------------------------------ chained Rosenbrock
// The reference's own Rosenbrock, rosenbrockfunc (examples/helpers/test_funcs.jl:50-57):
//   f = Σ_{i<d} (1 − x_i)² + 100 (x_{i+1} − x_i²)²,
//   g_i = 200 (x_i − x_{i−1}²) [i > 1] − 2 (1 − x_i) − 400 x_i (x_{i+1} − x_i²) [i < d]      (SURVEY.md §8d cfg 1).
// Elements couple to both neighbours, so one trial is two kernels, like the CSR objectives: K_a xp = x + a u
// (AxpyDir; sharded: pushes the two boundary elements into the ring neighbours' halos) and this one, which reads
// xp with its ±1 neighbours and reduces f, dϕ, ‖g⁺‖² and the getβ dots.  Arithmetic as oracle rosen_chained_fdf.
struct RosenChainedEval {
    static constexpr int TCLASS = CGO_T_TRIAL;
    static constexpr int K = 9;
    static constexpr int OCC = 2;
    struct In { double2 p, u, g; double pm, pn; };
    const double *xp;               // local origin; xp[−1] and xp[n] are halo (sharded) or never read (the ends)
    const double2 *u, *g;
    double2 *gp;
    int64_t offset, n_global, n_local;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.p = cgo_ld2((const double2 *)xp + q);
        r.u = cgo_ld2(u + q); r.g = cgo_ld2(g + q);
        const int64_t i0 = 2 * q, i1 = 2 * q + 1;
        r.pm = offset + i0 > 0 ? __ldg(xp + i0 - 1) : 0.0;
        r.pn = offset + i1 + 1 < n_global ? __ldg(xp + i1 + 1) : 0.0;
        return r;
    }
    __device__ __forceinline__ void dots(double gn, double gg, double uu, double (&acc)[K]) const {
        const double y = gn - gg;
        acc[CGO_P_DPHI] = acc[CGO_P_DPHI] + gn * uu;
        acc[CGO_P_GPGP] = acc[CGO_P_GPGP] + gn * gn;
        acc[CGO_P_YY] = acc[CGO_P_YY] + y * y;
        acc[CGO_P_UY] = acc[CGO_P_UY] + uu * y;
        acc[CGO_P_YGP] = acc[CGO_P_YGP] + y * gn;
        acc[CGO_P_GPG] = acc[CGO_P_GPG] + gn * gg;
        acc[CGO_P_UG] = acc[CGO_P_UG] + uu * gg;
        acc[CGO_P_UU] = acc[CGO_P_UU] + uu * uu;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        const int64_t gi0 = offset + 2 * q, gi1 = gi0 + 1;
        const double x0 = in.p.x, x1 = in.p.y;
        const double tm = x0 - in.pm * in.pm;               // t_{i0−1}
        const double t0 = x1 - x0 * x0;                     // t_{i0}
        const double t1 = in.pn - x1 * x1;                  // t_{i1}
        const double om0 = 1.0 - x0, om1 = 1.0 - x1;
        double2 gn;
        double g0 = 0.0, f0 = 0.0;
        if (gi0 > 0) g0 = g0 + 200.0 * tm;
        if (gi0 < n_global - 1) { g0 = g0 + (-2.0 * om0 - (400.0 * x0) * t0); f0 = om0 * om0 + (100.0 * t0) * t0; }
        gn.x = g0;
        acc[CGO_P_PHI] = acc[CGO_P_PHI] + f0;
        dots(g0, in.g.x, in.u.x, acc);
        gn.y = 0.0;
        if (v2) {
            double g1 = 0.0, f1 = 0.0;
            g1 = g1 + 200.0 * t0;                           // gi1 > 0 always
            if (gi1 < n_global - 1) { g1 = g1 + (-2.0 * om1 - (400.0 * x1) * t1); f1 = om1 * om1 + (100.0 * t1) * t1; }
            gn.y = g1;
            acc[CGO_P_PHI] = acc[CGO_P_PHI] + f1;
            dots(g1, in.g.y, in.u.y, acc);
        }
        cgo_st2(gp + q, gn);
    }
};

struct RosenChainedObj : cgo_obj {
    int eval_trial(cgo_state *st, double a, bool fused, double beta, double *out) override {
        const int R = ctx->nranks, me = ctx->rank;
        RedArgs red = cgo_red_args(ctx, CGO_P_PHI);
        if (R > 1 && st->peer_x) {
            const int prev = (me + R - 1) % R, next = (me + 1) % R;
            const unsigned long long e = ++ctx->epoch;
            unsigned long long *fprev = (unsigned long long *)ctx->flags_peer[(size_t)prev];
            unsigned long long *fnext = (unsigned long long *)ctx->flags_peer[(size_t)next];
            int64_t plo, phi;
            CGO_TRY(cgo_shard_range(n_global, R, prev, 2, &plo, &phi));
            HaloPush hp;
            hp.prev_right = (double *)st->xpeers[st->xp_alloc][(size_t)prev] + halo + (phi - plo);
            hp.next_left = (double *)st->xpeers[st->xp_alloc][(size_t)next];
            hp.sig_prev = fprev + CGO_F_XP_FROM_NEXT;
            hp.sig_next = fnext + CGO_F_XP_FROM_PREV;
            hp.epoch = e;
            CGO_TRY(cgo_blas1_axpy_dir(st, a, fused, beta, &hp));                         // K_a + halo push
            red.wait0 = ctx->flags_local + CGO_F_XP_FROM_PREV; red.wait1 = ctx->flags_local + CGO_F_XP_FROM_NEXT;
            red.wait_val = e;
        } else {
            CGO_TRY(cgo_blas1_axpy_dir(st, a, fused, beta));                              // K_a
            if (R > 1) CGO_TRY(cgo_sendrecv_ring(ctx, st->xp, st->xp + st->n, st->xp + st->n - halo, st->xp - halo, halo));
        }
        RosenChainedEval op;
        op.xp = st->xp; op.u = (const double2 *)st->u; op.g = (const double2 *)st->g; op.gp = (double2 *)st->gp;
        op.offset = offset; op.n_global = n_global; op.n_local = st->n;
        CGO_TRY(launch_blas1(ctx, op, st->n, red));
        return cgo_finish_pack(ctx, 12, out);
    }
    // K_a R x,u W xp (+ R g, W u on the first trial of an iteration) | R xp,u,g W g⁺
    double bytes_per_eval() const override { return 8.0 * 7.0 * (double)n_local; }
    void reduction_site(int32_t *V, int32_t *U) const override { *V = 2; *U = CGO_U_VEC; }
    int default_x0(uint64_t seed, double perturb, double *x0) override {
        for (int64_t i = 0; i < n_local; ++i) {
            int64_t gi = offset + i;
            double base = (gi % 2 == 0) ? -1.2 : 1.0;
            x0[i] = perturb != 0.0 ? base + perturb * (2.0 * cgo_host_u01(seed, (uint64_t)gi, 0) - 1.0) : base;
        }
        return 0;
    }
};
extern "C" int cgo_obj_rosenbrock_chained_create(cgo_ctx *ctx, int64_t n_global, cgo_obj **out) {
    CGO_CHECK(ctx && out, "NULL argument");
    CGO_CHECK(n_global >= 2 && n_global % 2 == 0, "chained Rosenbrock: need an even n >= 2 (got %lld)", (long long)n_global);
    CGO_CHECK(ctx->nranks == 1 || n_global >= 4 * ctx->nranks, "chained Rosenbrock: %d ranks need n >= %d", ctx->nranks, 4 * ctx->nranks);
    int64_t lo, hi;
    CGO_TRY(cgo_shard_range(n_global, ctx->nranks, ctx->rank, 2, &lo, &hi));
    RosenChainedObj *o = new RosenChainedObj();
    o->ctx = ctx;
    o->n_global = n_global;
    o->offset = lo;
    o->n_local = hi - lo;
    o->halo = ctx->nranks > 1 ? 2 : 0;           // ±1 neighbour, kept even (16-byte alignment)
    for (int q = 0; q < ctx->nranks; ++q) {
        int64_t a, b;
        cgo_shard_range(n_global, ctx->nranks, q, 2, &a, &b);
        if (b - a > o->n_alloc) o->n_alloc = b - a;
    }
    *out = o;
    return 0;
}

extern "C" int cgo_obj_rosenbrock_create(cgo_ctx *ctx, int64_t n_global, cgo_obj **out) {
    CGO_CHECK(ctx && out, "NULL argument");
    CGO_CHECK(n_global >= 2 && n_global % 2 == 0, "extended Rosenbrock needs an even n >= 2 (got %lld)", (long long)n_global);
    RosenObj *o = new RosenObj();
    o->ctx = ctx;
    o->n_global = n_global;
    int64_t lo, hi;
    CGO_TRY(cgo_shard_range(n_global, ctx->nranks, ctx->rank, 2, &lo, &hi));
    o->offset = lo;
    o->n_local = hi - lo;
    *out = o;
    return 0;
}
int cgo_obj::hessvec_dir(cgo_state *, double *) {
    cgo_set_error("this objective has no Hessian-vector product (CSR least squares has)");
    return 2;
}
int cgo_obj::quad_begin(cgo_state *, double *) {
    cgo_set_error("this objective has no quadratic-aware line search (CSR least squares has)");
    return 2;
}
int cgo_obj::quad_accept(cgo_state *, double, double *) {
    cgo_set_error("this objective has no quadratic-aware line search (CSR least squares has)");
    return 2;
}
extern "C" int cgo_quad_begin(cgo_state *st, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    return st->obj->quad_begin(st, out);
}
extern "C" int cgo_quad_accept(cgo_state *st, double a, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    return st->obj->quad_accept(st, a, out);
}
// r = r + a v, Σ r²  (the residual of the accepted step of a quadratic-aware line search)
struct ResidualAxpy {
    static constexpr int TCLASS = CGO_T_AXPY;
    static constexpr int K = 1;
    static constexpr int OCC = 4;
    struct In { double2 r, v; };
    double2 *r;
    const double2 *v;
    double a;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In o;
        o.r = ld2rw(r + q); o.v = cgo_ld2(v + q);
        return o;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 o;
        o.x = in.r.x + a * in.v.x;
        o.y = v2 ? in.r.y + a * in.v.y : 0.0;
        cgo_st2(r + q, o);
        acc[0] = acc[0] + o.x * o.x;
        if (v2) acc[0] = acc[0] + o.y * o.y;
    }
};
int cgo_blas1_residual_axpy(cgo_ctx *c, double *r, const double *v, double a, int64_t nrows, int slot) {
    ResidualAxpy op;
    op.r = (double2 *)r; op.v = (const double2 *)v; op.a = a;
    return launch_blas1(c, op, nrows, cgo_red_args(c, slot));
}
extern "C" int cgo_hessvec_dir(cgo_state *st, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    if (!st->hv) {
        CGO_CUDA(cudaMalloc(&st->hv, sizeof(double) * (size_t)(st->n + 4)));
        CGO_CUDA(cudaMemsetAsync(st->hv, 0, sizeof(double) * (size_t)(st->n + 4), st->ctx->stream));
    }
    return st->obj->hessvec_dir(st, out);
}
extern "C" int cgo_obj_destroy(cgo_obj *o) {
    delete o;
    return 0;
}
extern "C" int cgo_obj_dims(cgo_obj *o, int64_t *nl, int64_t *ng, int64_t *off) {
    CGO_CHECK(o != nullptr, "NULL objective");
    if (nl) *nl = o->n_local;
    if (ng) *ng = o->n_global;
    if (off) *off = o->offset;
    return 0;
}
extern "C" int cgo_obj_reduction_site(cgo_obj *o, int32_t *V, int32_t *U) {
    CGO_CHECK(o && V && U, "NULL argument");
    o->reduction_site(V, U);
    return 0;
}
extern "C" int cgo_obj_bytes_per_eval(cgo_obj *o, double *bytes) {
    CGO_CHECK(o && bytes, "NULL argument");
    *bytes = o->bytes_per_eval();
    return 0;
}
extern "C" int cgo_obj_default_x0(cgo_obj *o, uint64_t seed, double perturb, double *x0) {
    CGO_CHECK(o && x0, "NULL argument");
    return o->default_x0(seed, perturb, x0);
}

// ------------------------------------------------------------------ box-constraint log barrier
// evalbarrier! (src/engine/primal_barrier.jl:112-133) with the box constraints of
// examples/constrained.jl:17-47 (fi = [x − ubs; lbs − x], dfi = [+e_d; −e_d]) around any device
// objective: the inner objective's trial kernels leave xp and g⁺ = ∇f0(xp); this BLAS-1 pass
// forms df = t·∇f0 + dψ in place (:130), ψ = −Σ log(−fi) after clamp!(fi, −Inf, 0) (:77-78), and —
// because g⁺ changed — every dot of the trial pack again (cg_utils.jl:20, optim.jl:107, getβ).
struct BarrierFinish {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 9;
    static constexpr int OCC = 2;
    struct In { double2 xp, gp, u, g, lo, hi; };
    const double2 *xp, *u, *g, *lo, *hi;
    double2 *gp;
    double t;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.xp = cgo_ld2(xp + q); r.gp = ld2rw(gp + q); r.u = cgo_ld2(u + q); r.g = cgo_ld2(g + q);
        r.lo = cgo_ld2(lo + q); r.hi = cgo_ld2(hi + q);
        return r;
    }
    __device__ __forceinline__ void one(double x, double g0, double uu, double gg, double lb, double ub, double &gn,
                                        double (&acc)[K]) const {
        double fu = x - ub, fl = lb - x;
        if (fu > 0.0) fu = 0.0;                      // clamp!(fi_evals, -Inf, 0): NaN stays NaN
        if (fl > 0.0) fl = 0.0;
        const double term = log(-fu) + log(-fl);
        double dpsi = 0.0 - 1.0 / fu;                // dψ[d] -= dfi[i][d]/fi[i], upper then lower (:80-85)
        dpsi = dpsi - (-1.0) / fl;
        gn = t * g0 + dpsi;                          // :130
        const double y = gn - gg;
        acc[CGO_P_PHI] = acc[CGO_P_PHI] + term;
        acc[CGO_P_DPHI] = acc[CGO_P_DPHI] + gn * uu;
        acc[CGO_P_GPGP] = acc[CGO_P_GPGP] + gn * gn;
        acc[CGO_P_YY] = acc[CGO_P_YY] + y * y;
        acc[CGO_P_UY] = acc[CGO_P_UY] + uu * y;
        acc[CGO_P_YGP] = acc[CGO_P_YGP] + y * gn;
        acc[CGO_P_GPG] = acc[CGO_P_GPG] + gn * gg;
        acc[CGO_P_UG] = acc[CGO_P_UG] + uu * gg;
        acc[CGO_P_UU] = acc[CGO_P_UU] + uu * uu;
    }
    __device__ __forceinline__ void apply(int64_t q, const In &in, double (&acc)[K], bool v2) const {
        double2 gn;
        one(in.xp.x, in.gp.x, in.u.x, in.g.x, in.lo.x, in.hi.x, gn.x, acc);
        if (v2) one(in.xp.y, in.gp.y, in.u.y, in.g.y, in.lo.y, in.hi.y, gn.y, acc);
        else gn.y = 0.0;
        cgo_st2(gp + q, gn);
    }
};
// any(fi_evals .>= 0) (primal_barrier.jl:189): number of coordinates on or outside the box
struct BoxInfeasible {
    static constexpr int TCLASS = CGO_T_OTHER;
    static constexpr int K = 1;
    static constexpr int OCC = 4;
    struct In { double2 x, lo, hi; };
    const double2 *x, *lo, *hi;
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ In load(int64_t q) const {
        In r;
        r.x = cgo_ld2(x + q); r.lo = cgo_ld2(lo + q); r.hi = cgo_ld2(hi + q);
        return r;
    }
    __device__ __forceinline__ void apply(int64_t, const In &in, double (&acc)[K], bool v2) const {
        if (in.x.x - in.hi.x >= 0.0 || in.lo.x - in.x.x >= 0.0) acc[0] = acc[0] + 1.0;
        if (v2 && (in.x.y - in.hi.y >= 0.0 || in.lo.y - in.x.y >= 0.0)) acc[0] = acc[0] + 1.0;
    }
};

struct BarrierObj : cgo_obj {
    cgo_obj *inner = nullptr;
    double *lo = nullptr, *hi = nullptr;
    double t = 1.0;
    ~BarrierObj() override {
        if (ctx && cgo_ctx_alive(ctx)) cudaSetDevice(ctx->device);
        cudaFree(lo); cudaFree(hi);
    }
    int eval_trial(cgo_state *st, double a, bool fused, double beta, double *out) override {
        double in[CGO_PACK_LEN];
        CGO_TRY(inner->eval_trial(st, a, fused, beta, in));      // xp, g⁺ = ∇f0(xp), f0, direction dots
        BarrierFinish op;
        op.xp = (const double2 *)st->xp; op.gp = (double2 *)st->gp; op.u = (const double2 *)st->u;
        op.g = (const double2 *)st->g; op.lo = (const double2 *)lo; op.hi = (const double2 *)hi; op.t = t;
        CGO_TRY(launch_blas1(ctx, op, st->n, cgo_red_args(ctx)));
        CGO_TRY(cgo_finish_pack(ctx, 9, out));
        out[CGO_P_PHI] = t * in[CGO_P_PHI] + (-out[CGO_P_PHI]);   // :132  t*f_x + ψ_x
        out[CGO_P_DIR_GU] = in[CGO_P_DIR_GU];
        out[CGO_P_DIR_UU] = in[CGO_P_DIR_UU];
        out[CGO_P_XPXP] = in[CGO_P_XPXP];
        return 0;
    }
    double bytes_per_eval() const override { return inner->bytes_per_eval() + 8.0 * 7.0 * (double)n_local; }
    void reduction_site(int32_t *V, int32_t *U) const override { *V = 2; *U = CGO_U_VEC; }
    int default_x0(uint64_t seed, double perturb, double *x0) override { return inner->default_x0(seed, perturb, x0); }
};

extern "C" int cgo_obj_box_barrier_create(cgo_ctx *ctx, cgo_obj *inner, const double *lbs, const double *ubs,
                                          double t, cgo_obj **out) {
    CGO_CHECK(ctx && inner && lbs && ubs && out, "NULL argument");
    CGO_CHECK(inner->ctx == ctx, "inner objective belongs to another ctx");
    CGO_CUDA(cudaSetDevice(ctx->device));
    BarrierObj *o = new BarrierObj();
    o->ctx = ctx; o->inner = inner; o->t = t;
    o->n_global = inner->n_global; o->n_local = inner->n_local; o->offset = inner->offset;
    o->halo = inner->halo; o->n_alloc = inner->n_alloc;
    const size_t len = (size_t)(o->n_local + 4);
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&o->lo, sizeof(double) * len));
        CGO_CUDA(cudaMalloc(&o->hi, sizeof(double) * len));
        CGO_CUDA(cudaMemsetAsync(o->lo, 0, sizeof(double) * len, ctx->stream));
        CGO_CUDA(cudaMemsetAsync(o->hi, 0, sizeof(double) * len, ctx->stream));
        CGO_CUDA(cudaMemcpyAsync(o->lo, lbs, sizeof(double) * (size_t)o->n_local, cudaMemcpyHostToDevice, ctx->stream));
        CGO_CUDA(cudaMemcpyAsync(o->hi, ubs, sizeof(double) * (size_t)o->n_local, cudaMemcpyHostToDevice, ctx->stream));
        CGO_CUDA(cudaStreamSynchronize(ctx->stream));
        return 0;
    };
    int rc = body();
    if (rc) { delete o; return rc; }
    *out = o;
    return 0;
}
extern "C" int cgo_obj_barrier_set_t(cgo_obj *obj, double t) {
    BarrierObj *o = dynamic_cast<BarrierObj *>(obj);
    CGO_CHECK(o != nullptr, "not a barrier objective");
    o->t = t;
    return 0;
}
extern "C" int cgo_obj_barrier_infeasible(cgo_obj *obj, const double *x_host, int64_t *count) {
    BarrierObj *o = dynamic_cast<BarrierObj *>(obj);
    CGO_CHECK(o && x_host && count, "not a barrier objective / NULL argument");
    cgo_ctx *c = o->ctx;
    CGO_CUDA(cudaSetDevice(c->device));
    double *dx = nullptr;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&dx, sizeof(double) * (size_t)(o->n_local + 4)));
        CGO_CUDA(cudaMemsetAsync(dx, 0, sizeof(double) * (size_t)(o->n_local + 4), c->stream));
        CGO_CUDA(cudaMemcpyAsync(dx, x_host, sizeof(double) * (size_t)o->n_local, cudaMemcpyHostToDevice, c->stream));
        BoxInfeasible op;
        op.x = (const double2 *)dx; op.lo = (const double2 *)o->lo; op.hi = (const double2 *)o->hi;
        CGO_TRY(launch_blas1(c, op, o->n_local, cgo_red_args(c)));
        double v[CGO_PACK_LEN];
        CGO_TRY(cgo_finish_pack(c, 1, v));
        *count = (int64_t)v[0];
        return 0;
    };
    int rc = body();
    cudaFree(dx);
    return rc;
}

// ------------------------------------------------------------------ solver state
static size_t vec_bytes(const cgo_state *st) { return sizeof(double) * (size_t)(st->n + 2 * st->halo + 4); }
static int alloc_vec(cgo_state *st, double **base, double **ptr) {
    void *p = nullptr;
    CGO_TRY(cgo_dev_alloc(st->ctx, vec_bytes(st), &p));
    *base = (double *)p;
    *ptr = *base + st->halo;
    return 0;
}

extern "C" int cgo_state_destroy(cgo_state *st) {
    if (!st) return 0;
    if (cgo_ctx_alive(st->ctx)) {
        cudaSetDevice(st->ctx->device);
        cudaStreamSynchronize(st->ctx->stream);
    } else {
        cudaDeviceSynchronize();
    }
    if (st->peer_x) {               // collective: the neighbours unmap before the owner frees
        for (int k = 0; k < 2; ++k) {
            if (st->xpeers[k].size() != (size_t)st->ctx->nranks) continue;
            double *mine = (double *)st->xpeers[k][(size_t)st->ctx->rank];
            for (int i = 0; i < 5; ++i) if (st->base[i] == mine) st->base[i] = nullptr;
            cgo_peer_free(st->ctx, mine, st->xpeers[k], true);
        }
    }
    for (int i = 0; i < 5; ++i) cgo_dev_free(st->ctx, st->base[i], vec_bytes(st));
    const size_t hist_bytes = sizeof(double) * (size_t)(st->n + 4);
    for (auto p : st->S) cgo_dev_free(st->ctx, p, hist_bytes);
    for (auto p : st->Y) cgo_dev_free(st->ctx, p, hist_bytes);
    cgo_dev_free(st->ctx, st->q, hist_bytes);
    cudaFree(st->xn);
    cudaFree(st->hv);
    delete st;
    return 0;
}

// x0: host pointer (x0_on_device = false: one H2D) or device pointer (one D2D)
static int state_create(cgo_ctx *ctx, cgo_obj *obj, const double *x0, bool x0_on_device, int32_t lbfgs_m,
                        cgo_state **out_state, double out[CGO_PACK_LEN]) {
    CGO_CHECK(ctx && obj && x0 && out_state && out, "cgo_state_create: NULL argument");
    CGO_CHECK(obj->ctx == ctx, "objective belongs to another ctx");
    CGO_CHECK(lbfgs_m >= 0 && lbfgs_m <= CGO_LBFGS_MAX_M, "lbfgs_m=%d out of [0,%d]", lbfgs_m, CGO_LBFGS_MAX_M);
    CGO_CHECK(obj->halo % 2 == 0, "halo must be even");      // keeps the local part 16-byte aligned
    CGO_CUDA(cudaSetDevice(ctx->device));
    cgo_state *st = new cgo_state();
    st->ctx = ctx; st->obj = obj; st->n = obj->n_local; st->halo = obj->halo;
    auto body = [&]() -> int {                     // (every failure below goes through cgo_state_destroy)
        double **ptrs[5] = {&st->x, &st->g, &st->u, &st->xp, &st->gp};
        st->peer_x = ctx->nranks > 1 && ctx->peer_ok && st->halo > 0;
        for (int i = 0; i < 5; ++i) {
            if (st->peer_x && (i == 0 || i == 3)) {      // x and xp: mapped by the ring neighbours
                void *p = nullptr;
                // same size on every rank: the ranks pool and reuse these blocks in lockstep
                const int64_t len = (obj->n_alloc > st->n ? obj->n_alloc : st->n) + 2 * st->halo + 4;
                CGO_TRY(cgo_peer_alloc(ctx, sizeof(double) * (size_t)len, &p, st->xpeers[i == 0 ? 0 : 1]));
                st->base[i] = (double *)p;
                *ptrs[i] = st->base[i] + st->halo;
            } else {
                CGO_TRY(alloc_vec(st, &st->base[i], ptrs[i]));
            }
        }
        st->xp_alloc = 1;
        st->m = lbfgs_m;
        if (lbfgs_m > 0) {
            // m + 1 slots: a pair is staged into the one slot no live pair occupies, so rejecting it touches nothing live
            const size_t hist_bytes = sizeof(double) * (size_t)(st->n + 4);
            for (int k = 0; k <= lbfgs_m; ++k) {
                void *s = nullptr, *y = nullptr;
                CGO_TRY(cgo_dev_alloc(ctx, hist_bytes, &s));
                st->S.push_back((double *)s);
                CGO_TRY(cgo_dev_alloc(ctx, hist_bytes, &y));
                st->Y.push_back((double *)y);
            }
            st->rho.assign(lbfgs_m + 1, 0.0);
            void *q = nullptr;
            CGO_TRY(cgo_dev_alloc(ctx, hist_bytes, &q));
            st->q = (double *)q;
        }
        // optim.jl:21 x = copy(x_initial); :25 f_x = fdf!(df_x, x): evaluate at x0 through the trial
        // kernels with u = 0, a = 0 (xp = x0 + 0*0 = x0 exactly), then adopt (xp, g⁺) as (x, g).
        CGO_CUDA(cudaMemcpyAsync(st->x, x0, sizeof(double) * (size_t)st->n,
                                 x0_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
        CGO_TRY(obj->eval_trial(st, 0.0, false, 0.0, out));
        return 0;
    };
    const int rc = body();
    if (rc) { cgo_state_destroy(st); return rc; }
    cgo_accept(st);
    *out_state = st;
    return 0;
}
extern "C" int cgo_state_create(cgo_ctx *ctx, cgo_obj *obj, const double *x0, int32_t lbfgs_m,
                                cgo_state **out_state, double out[CGO_PACK_LEN]) {
    return state_create(ctx, obj, x0, false, lbfgs_m, out_state, out);
}
extern "C" int cgo_state_create_from_state(cgo_ctx *ctx, cgo_obj *obj, cgo_state *src, int32_t which, int32_t lbfgs_m,
                                           cgo_state **out_state, double out[CGO_PACK_LEN]) {
    CGO_CHECK(src != nullptr, "cgo_state_create_from_state: NULL source state");
    CGO_CHECK(src->ctx == ctx && src->n == (obj ? obj->n_local : -1), "source state belongs to another ctx or has another dimension");
    double *v[5] = {src->x, src->g, src->u, src->xp, src->gp};
    CGO_CHECK(which >= 0 && which < 5, "which=%d out of range", which);
    return state_create(ctx, obj, v[which], true, lbfgs_m, out_state, out);
}

extern "C" int cgo_accept(cgo_state *st) {
    CGO_CHECK(st != nullptr, "NULL state");
    std::swap(st->x, st->xp);
    std::swap(st->g, st->gp);
    std::swap(st->base[0], st->base[3]);
    std::swap(st->base[1], st->base[4]);
    st->xp_alloc ^= 1;
    st->obj->on_accept(st);
    return 0;
}

extern "C" int cgo_eval_trial(cgo_state *st, double a, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    return st->obj->eval_trial(st, a, false, 0.0, out);
}
extern "C" int cgo_eval_trial_fused_dir(cgo_state *st, double beta, double a, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    return st->obj->eval_trial(st, a, true, beta, out);
}

extern "C" int cgo_update_dir(cgo_state *st, double beta, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    DirUpdate<false> op;
    op.g = (const double2 *)st->g; op.u = (double2 *)st->u; op.beta = beta;
    CGO_TRY(launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx)));
    return cgo_finish_pack(st->ctx, 2, out);
}
extern "C" int cgo_reset_direction(cgo_state *st, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    DirUpdate<true> op;
    op.g = (const double2 *)st->g; op.u = (double2 *)st->u; op.beta = 0.0;
    CGO_TRY(launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx)));
    return cgo_finish_pack(st->ctx, 2, out);
}
extern "C" int cgo_beta_literal(cgo_state *st, double R, double m, double *beta_out) {
    CGO_CHECK(st && beta_out, "NULL argument");
    BetaLiteral op;
    op.gp = (const double2 *)st->gp; op.g = (const double2 *)st->g; op.u = (const double2 *)st->u;
    op.R = R; op.m = m;
    CGO_TRY(launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx)));
    double tmp[CGO_PACK_LEN];
    CGO_TRY(cgo_finish_pack(st->ctx, 1, tmp));
    *beta_out = tmp[0];
    return 0;
}
extern "C" int cgo_norm_sq_u_plus_g(cgo_state *st, double *outv) {
    CGO_CHECK(st && outv, "NULL argument");
    NormUPlusG op;
    op.g = (const double2 *)st->g; op.u = (const double2 *)st->u;
    CGO_TRY(launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx)));
    double tmp[CGO_PACK_LEN];
    CGO_TRY(cgo_finish_pack(st->ctx, 1, tmp));
    *outv = tmp[0];
    return 0;
}

template <bool FUSED, int PUSH>
static int launch_axpy_dir(cgo_state *st, double a, double beta, const HaloPush *push) {
    // writes {g·u, u·u, xp·xp} to pack slots CGO_P_DIR_GU, CGO_P_DIR_UU, CGO_P_XPXP
    cgo_ctx *c = st->ctx;
    RedArgs red = cgo_red_args(c, CGO_P_DIR_GU);
    AxpyDir<FUSED, PUSH> op;
    op.x = (const double2 *)st->x; op.g = (const double2 *)st->g; op.u = (double2 *)st->u;
    op.xp = (double2 *)st->xp; op.a = a; op.beta = FUSED ? beta : 0.0;
    op.prev_right = op.next_left = nullptr; op.hq = 0; op.nq = st->n / 2;
    op.dst_all = nullptr; op.nranks = c->nranks;
    if (PUSH == 1) {
        op.prev_right = (double2 *)push->prev_right; op.next_left = (double2 *)push->next_left;
        op.hq = st->halo / 2;
        red.sig0 = push->sig_prev; red.sig1 = push->sig_next; red.sig_val = push->epoch;
    }
    if (PUSH == 2) {
        op.dst_all = push->dst_all;
        red.flags_all = c->d_flags_peer; red.sig_all_slot = CGO_F_XPALL; red.nranks = c->nranks; red.me = c->rank;
        red.sig_val = push->epoch;
    }
    return launch_blas1(c, op, st->n, red);
}
int cgo_blas1_axpy_dir(cgo_state *st, double a, bool fused, double beta, const HaloPush *push) {
    if (push && push->dst_all)
        return fused ? launch_axpy_dir<true, 2>(st, a, beta, push) : launch_axpy_dir<false, 2>(st, a, beta, push);
    if (push) return fused ? launch_axpy_dir<true, 1>(st, a, beta, push) : launch_axpy_dir<false, 1>(st, a, beta, push);
    return fused ? launch_axpy_dir<true, 0>(st, a, beta, nullptr) : launch_axpy_dir<false, 0>(st, a, beta, nullptr);
}

int cgo_blas1_sumsq(cgo_ctx *c, const double *a, int64_t n, int slot) {
    VecSumSq op;
    op.a = (const double2 *)a;
    return launch_blas1(c, op, n, cgo_red_args(c, slot));
}
int cgo_blas1_dots3(cgo_ctx *c, const double *a, const double *b, int64_t n, int slot) {
    Dots3 op;
    op.a = (const double2 *)a; op.b = (const double2 *)b;
    return launch_blas1(c, op, n, cgo_red_args(c, slot));
}
int cgo_blas1_logit(cgo_ctx *c, double *zc, const double *y, int64_t n, int slot, void *const *dst_all, unsigned long long epoch) {
    RedArgs red = cgo_red_args(c, slot);
    if (dst_all) {
        LogitLoss<true> op;
        op.zc = (double2 *)zc; op.y = (const double2 *)y; op.dst_all = dst_all; op.nranks = c->nranks;
        red.flags_all = c->d_flags_peer; red.sig_all_slot = CGO_F_GPART; red.nranks = c->nranks; red.me = c->rank;
        red.sig_val = epoch;
        return launch_blas1(c, op, n, red);
    }
    LogitLoss<false> op;
    op.zc = (double2 *)zc; op.y = (const double2 *)y; op.dst_all = nullptr; op.nranks = 1;
    return launch_blas1(c, op, n, red);
}
int cgo_blas1_grad_dots(cgo_state *st) {
    GradDots op;
    op.gp = (const double2 *)st->gp; op.g = (const double2 *)st->g; op.u = (const double2 *)st->u;
    return launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx, CGO_P_DPHI));
}

int cgo_blas1_grad_combine(cgo_state *st, const double *q, int nparts, int64_t stride, double invN, double lambda,
                           unsigned long long wait_epoch) {
    GradCombine op;
    op.q = (const double2 *)q; op.u = (const double2 *)st->u; op.g = (const double2 *)st->g;
    op.w = (const double2 *)st->xp; op.gp = (double2 *)st->gp;
    op.nparts = nparts; op.stride2 = stride / 2; op.invN = invN; op.lambda = lambda;
    RedArgs red = cgo_red_args(st->ctx, CGO_P_DPHI);
    if (wait_epoch) {
        red.wait_all = st->ctx->flags_local + CGO_F_GPART; red.wait_val = wait_epoch; red.nranks = st->ctx->nranks;
    }
    return launch_blas1(st->ctx, op, st->n, red);
}

// ------------------------------------------------------------------ solvesystem (solve_system.jl)
extern "C" int cgo_solvesys_begin(cgo_state *st) {
    CGO_CHECK(st != nullptr, "NULL state");
    cudaStream_t s = st->ctx->stream;
    if (!st->xn) CGO_CUDA(cudaMalloc(&st->xn, sizeof(double) * (size_t)(st->n + 4)));
    CGO_CUDA(cudaMemsetAsync(st->xn, 0, sizeof(double) * (size_t)(st->n + 4), s));
    CGO_CUDA(cudaMemcpyAsync(st->xn, st->x, sizeof(double) * (size_t)st->n, cudaMemcpyDeviceToDevice, s));   // :78 x_next = copy(x_initial)
    return 0;
}
extern "C" int cgo_solvesys_project(cgo_state *st, double m, int32_t fix_stale_iterate, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    CGO_CHECK(st->xn != nullptr, "cgo_solvesys_project before cgo_solvesys_begin");
    SolveSysProject op;
    op.base = (const double2 *)(fix_stale_iterate ? st->x : st->xn);
    op.gp = (const double2 *)st->gp; op.xn = (double2 *)st->xn; op.m = m;
    CGO_TRY(launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx, CGO_PACK_LEN - 1)));
    // f_x_next = fdf!(info.df_xp, x_next) (:179) through the trial kernels: xp = x_next + 0·u
    // (exact for finite u), g⁺ = g(x_next), and the whole dot pack against the OLD df_x and u,
    // which is what getβ (:201-206) reads
    double *x_saved = st->x;
    st->x = st->xn;
    int rc = st->obj->eval_trial(st, 0.0, false, 0.0, out);
    st->x = x_saved;
    return rc;
}
extern "C" int cgo_solvesys_accept(cgo_state *st, int32_t fix_stale_iterate) {
    CGO_CHECK(st != nullptr, "NULL state");
    // x, x_next = x_next, x (:198); df_x[:] = info.df_xp (:209); info.x[:] = x (:210).  xp holds a
    // copy of x_next (xp = x_next + 0·u), so the ordinary pointer swap adopts it; x_next then has
    // to hold the OLD x, which only the as-written variant reads again
    CGO_TRY(cgo_accept(st));
    if (!fix_stale_iterate)
        CGO_CUDA(cudaMemcpyAsync(st->xn, st->xp, sizeof(double) * (size_t)st->n, cudaMemcpyDeviceToDevice, st->ctx->stream));
    return 0;
}

// ------------------------------------------------------------------ L-BFGS
extern "C" int cgo_lbfgs_stage_pair(cgo_state *st, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    CGO_CHECK(st->m > 0, "state was created without an L-BFGS history (lbfgs_m = 0)");
    // the slot after the newest pair: the spare one (the ring has m + 1 slots and at most m pairs live)
    const int slot = (st->head + 1) % (st->m + 1);
    LbfgsStage op;
    op.xp = (const double2 *)st->xp; op.x = (const double2 *)st->x;
    op.gp = (const double2 *)st->gp; op.g = (const double2 *)st->g;
    op.S = (double2 *)st->S[slot]; op.Y = (double2 *)st->Y[slot];
    CGO_TRY(launch_blas1(st->ctx, op, st->n, cgo_red_args(st->ctx)));
    st->staged = slot;
    return cgo_finish_pack(st->ctx, 2, out);
}
extern "C" int cgo_lbfgs_commit_pair(cgo_state *st, int32_t commit, double rho, double gamma) {
    CGO_CHECK(st != nullptr, "NULL state");
    CGO_CHECK(st->staged >= 0, "cgo_lbfgs_commit_pair without a staged pair");
    if (commit) {        // the staged slot becomes the newest pair; at count == m the oldest one becomes the spare
        st->head = st->staged;
        if (st->count < st->m) st->count++;
        st->rho[st->staged] = rho;
        st->gamma = gamma;
    }                    // a rejected pair leaves the history as it was (N&W Alg. 7.5)
    st->staged = -1;
    return 0;
}

// publish the dot of the kernel that just ran into d_scal[slot] (all ranks, rank order)
static RedArgs red_to_slot(cgo_ctx *c, int slot) {
    RedArgs r = cgo_red_args(c);
    r.out = (c->nranks > 1) ? c->d_pack : c->d_scal + slot;
    return r;
}
static int publish_slot(cgo_ctx *c, int slot) {
    if (c->nranks > 1) CGO_TRY(cgo_combine_ranks(c, 1, c->d_scal + slot));
    return 0;
}

extern "C" int cgo_lbfgs_update_dir(cgo_state *st, double out[CGO_PACK_LEN]) {
    CGO_CHECK(st && out, "NULL argument");
    CGO_CHECK(st->m > 0, "state was created without an L-BFGS history (lbfgs_m = 0)");
    cgo_ctx *c = st->ctx;
    if (st->count == 0) return cgo_reset_direction(st, out);
    const int cnt = st->count, R = st->m + 1;
    auto slot_of = [&](int k) { return ((st->head - k) % R + R) % R; };   // k = 0 newest
    double2 *q = (double2 *)st->q;
    // loop 1 (newest → oldest): dots land in d_scal[k]
    for (int k = 0; k < cnt; ++k) {
        int s = slot_of(k);
        if (k == 0) {
            LbfgsStep<0> op{};
            op.q = q; op.A = (const double2 *)st->g; op.B = (const double2 *)st->S[s];
            CGO_TRY(launch_blas1(c, op, st->n, red_to_slot(c, k)));
        } else {
            int sp = slot_of(k - 1);
            LbfgsStep<1> op{};
            op.q = q; op.A = (const double2 *)st->Y[sp]; op.B = (const double2 *)st->S[s];
            op.dprev = c->d_scal + (k - 1); op.rho_prev = st->rho[sp];
            CGO_TRY(launch_blas1(c, op, st->n, red_to_slot(c, k)));
        }
        CGO_TRY(publish_slot(c, k));
    }
    // end of loop 1 + scaling + first dot of loop 2 (oldest pair): dots of loop 2 in d_scal[64+k]
    {
        int sp = slot_of(cnt - 1);
        LbfgsStep<2> op{};
        op.q = q; op.A = (const double2 *)st->Y[sp]; op.B = (const double2 *)st->Y[sp];
        op.dprev = c->d_scal + (cnt - 1); op.rho_prev = st->rho[sp]; op.gamma = st->gamma;
        CGO_TRY(launch_blas1(c, op, st->n, red_to_slot(c, 64 + cnt - 1)));
        CGO_TRY(publish_slot(c, 64 + cnt - 1));
    }
    // loop 2 (oldest → newest)
    for (int k = cnt - 2; k >= 0; --k) {
        int sp = slot_of(k + 1), s = slot_of(k);
        LbfgsStep<3> op{};
        op.q = q; op.A = (const double2 *)st->S[sp]; op.B = (const double2 *)st->Y[s];
        op.dprev = c->d_scal + 64 + (k + 1); op.alpha_dot = c->d_scal + (k + 1); op.rho_prev = st->rho[sp];
        CGO_TRY(launch_blas1(c, op, st->n, red_to_slot(c, 64 + k)));
        CGO_TRY(publish_slot(c, 64 + k));
    }
    {
        int sp = slot_of(0);
        LbfgsStep<4> op{};
        op.q = q; op.A = (const double2 *)st->S[sp]; op.B = (const double2 *)st->g; op.uout = (double2 *)st->u;
        op.dprev = c->d_scal + 64; op.alpha_dot = c->d_scal; op.rho_prev = st->rho[sp];
        CGO_TRY(launch_blas1(c, op, st->n, cgo_red_args(c)));
    }
    return cgo_finish_pack(c, 2, out);
}

// ------------------------------------------------------------------ downloads
extern "C" int cgo_download(cgo_state *st, double *x_host, double *g_host) {
    CGO_CHECK(st != nullptr, "NULL state");
    cudaStream_t s = st->ctx->stream;
    if (x_host) CGO_CUDA(cudaMemcpyAsync(x_host, st->x, sizeof(double) * (size_t)st->n, cudaMemcpyDeviceToHost, s));
    if (g_host) CGO_CUDA(cudaMemcpyAsync(g_host, st->g, sizeof(double) * (size_t)st->n, cudaMemcpyDeviceToHost, s));
    CGO_CUDA(cudaStreamSynchronize(s));
    return 0;
}
extern "C" int cgo_download_vector(cgo_state *st, int32_t which, double *host) {
    CGO_CHECK(st && host, "NULL argument");
    double *src[6] = {st->x, st->g, st->u, st->xp, st->gp, st->hv};
    CGO_CHECK(which >= 0 && which < 6 && src[which] != nullptr, "which=%d out of range (5 = hv needs cgo_hessvec_dir first)", which);
    CGO_CUDA(cudaMemcpyAsync(host, src[which], sizeof(double) * (size_t)st->n, cudaMemcpyDeviceToHost, st->ctx->stream));
    CGO_CUDA(cudaStreamSynchronize(st->ctx->stream));
    return 0;
}
