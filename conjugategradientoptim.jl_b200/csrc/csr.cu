// csr.cu — CSR objectives: sparse least squares ½‖Ax − b‖² and logistic regression.
//
// These are device-resident replacements of the user callback `fdf!(g, x) -> f` that the
// reference calls at src/engine/optim.jl:25 and src/cg_utils.jl:18 (the reference ships no
// large objective, SURVEY.md §0-3; the definitions are restated in oracle/cgo_oracle.c
// sparse_ls_fdf / logreg_fdf).  One trial  evalϕdϕ! (src/cg_utils.jl:3-22)  is three kernels:
//   K_a  xp = x + a u  [after u = −g + βu, cg_flavours.jl:10-12]           BLAS-1, blas1.cu
//   K_b  r  = A xp − b,  Σ r²                (logreg: margins, loss, c)     SpMV with A
//   K_c  g⁺ = Aᵀ r  + every dot of getβ / norm(df_xp) / dϕ                  SpMV with Aᵀ
// Aᵀ is an explicit CSR whose rows are sorted by source entry, so the gradient is a gather
// (no atomics on data) and reproduces the sequential scatter order of the oracle bit for bit.
// An objective runs every SpMV on one of two kernel families, chosen at creation (CsrObj::direct):
// the fused k_csr_rows, whose row epilogues reduce the dots, or — for matrices whose gathers do not
// coalesce — k_spmv_direct, which keeps no reduction, followed by BLAS-1 dot passes.
//
// k_csr_rows is a "CSR-stream" kernel: a CTA owns 256 consecutive rows at a time; their
// nonzeros are one contiguous range of val/col, which a producer warp streams into a circular
// shared-memory buffer with 1-D TMA bulk copies (cp.async.bulk + mbarrier, L2 evict-first) while
// the 256 row lanes gather the vector entries and add up their row's products in storage
// order.  Rows and tiles of any length work.
#include <cub/device/device_scan.cuh>
#include <cmath>
#include <utility>

#include "internal.cuh"
#include "reduce.cuh"


constexpr int CSR_PAD = 16;                 // slack entries behind every CSR array (see csr_alloc)

__device__ __forceinline__ double ld_stream_f64(const double *p) {
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ int32_t ld_stream_s32(const int32_t *p) {
    int32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_f64(double *p, double v) {
    asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

// ------------------------------------------------------------------ mbarrier / TMA (1-D bulk) PTX
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *b, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *b, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(b)), "r"(parity) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// global -> shared bulk copy (TMA engine), completion counted in bytes on `bar`; 16-byte
// aligned addresses and size
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}

// ------------------------------------------------------------------ the CSR row kernel
// Canonical reduction site: V = 1, U = 1 (item = row, lane t of a tile owns row t;
// include/cgoptim.h).  Warp-specialised: warp 8 is the producer (one lane drives the TMA
// engine), warps 0-7 are the 256 row lanes.  Everything that streams — matrix values, column
// indices, row pointers and the epilogue's per-row operands (b; u, g; w) — reaches shared memory
// only through bulk copies with an evict-first L2 policy; the lanes' only global loads are the
// gathers of the vector, issued with an evict-last policy so that the gathered window stays in
// L2 while the matrix streams through it.
//
// Shared-memory layout: a circular buffer of RING entries (values + column indices) that holds
// variable-length chunks back to back, and TS_ND chunk descriptors (full/empty mbarrier pair,
// the tile's row-pointer slice and operand slices).  A chunk is the entry range [p0 & ~3, p1)
// of one tile (tiles of Aᵀ vary in length), or a CHMAX piece of it when the tile is longer than
// half the ring.  The producer runs ahead as far as ring space and descriptors allow (about
// three tiles); it reclaims space in FIFO order as the lanes release chunks.
constexpr int TS_ND = 3;                    // chunk descriptors
constexpr int TS_THREADS = CGO_B + 32;
constexpr int TS_OCC = 2;
constexpr int TS_UN = 10;                   // gathers in flight per lane
constexpr int TS_SMEM_BUDGET = 115200;      // two CTAs per SM (228 KB - 2 x 1 KB reserved)
template <int NOPS>
struct TsLayout {
    static constexpr int BUDGET = TS_SMEM_BUDGET;
    static constexpr int RP_BYTES = (CGO_B + 2) * 8;
    static constexpr int OP_BYTES = CGO_B * 8;
    static constexpr int DESC_BYTES = RP_BYTES + NOPS * OP_BYTES;
    static constexpr int TAIL_BYTES = 2 * TS_ND * 8 + TS_ND * 4 + CGO_MAXK * CGO_NW * 8;
    static constexpr int RING = ((BUDGET - TS_ND * DESC_BYTES - TAIL_BYTES - 64) / 12) & ~3;
    static constexpr int CHMAX = (RING / 2) & ~3;
    // byte offsets (all multiples of 16)
    static constexpr int OFF_VAL = 0;
    static constexpr int OFF_COL = OFF_VAL + RING * 8;
    static constexpr int OFF_DESC = (OFF_COL + RING * 4 + 15) & ~15;
    static constexpr int OFF_BAR = OFF_DESC + TS_ND * DESC_BYTES;
    static constexpr int OFF_LEN = OFF_BAR + 2 * TS_ND * 8;
    static constexpr int OFF_RED = (OFF_LEN + TS_ND * 4 + 15) & ~15;
    static constexpr int BYTES = OFF_RED + CGO_MAXK * CGO_NW * 8;
    static_assert(BYTES <= BUDGET && RP_BYTES % 16 == 0 && DESC_BYTES % 16 == 0, "smem layout");
};

__device__ __forceinline__ bool ts_next_tile(int &v, int64_t &tile, int nact, int64_t ntiles, int G) {
    tile += G;
    if (tile < ntiles) return true;
    v += gridDim.x;
    if (v >= nact) return false;
    tile = v;
    return true;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ double ld_gather_f64(const double *p, uint64_t pol) {
    double r;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}
// predicated gather: a lane whose row has ended issues no request at all.  (A gather instruction
// costs one L1TEX wavefront per distinct 128-byte line; re-reading a dummy address on the idle
// lanes — the first version — spent half of the gather bandwidth of 5-entry rows on nothing.)
__device__ __forceinline__ double ld_gather_f64_if(const double *p, uint64_t pol, bool on) {
    double r = 0.0;
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.s32 q, %3, 0;\n"
        "@q ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;\n"
        "}\n" : "+d"(r) : "l"(p), "l"(pol), "r"((int)on));
    return r;
}

// ---------------- producer: one lane streams tiles into the ring, about three tiles ahead
template <class L, class Epi>
__device__ __forceinline__ void ts_produce(const CsrMat &A, const Epi &epi, const RedArgs &red,
                                           double *s_val, int32_t *s_col, unsigned char *s_desc, uint64_t *s_full,
                                           uint64_t *s_empty, uint32_t *s_len, int nact, int64_t ntiles) {
    constexpr int NOPS = Epi::NOPS;
    constexpr int RING = L::RING, CHMAX = L::CHMAX;
    const int64_t nrows = A.nrows;
    const uint64_t pol = l2_policy_evict_first();
    uint32_t c = 0, tail = 0;         // chunks issued / reclaimed
    uint32_t head = 0, nfree = RING;
    int v = blockIdx.x;
    int64_t tile = v;
    bool have = true;
    int nvalid_n = (int)(nrows - tile * CGO_B < CGO_B ? nrows - tile * CGO_B : CGO_B);
    int64_t p0n = __ldg(A.rowptr + tile * CGO_B), p1n = __ldg(A.rowptr + tile * CGO_B + nvalid_n);
    while (have) {
        const int64_t r0 = tile * CGO_B, p0 = p0n, p1 = p1n;
        const int nvalid = nvalid_n;
        have = ts_next_tile(v, tile, nact, ntiles, red.G);
        if (have) {                   // row pointers of the next tile: in flight during this one
            nvalid_n = (int)(nrows - tile * CGO_B < CGO_B ? nrows - tile * CGO_B : CGO_B);
            p0n = __ldg(A.rowptr + tile * CGO_B);
            p1n = __ldg(A.rowptr + tile * CGO_B + nvalid_n);
        }
        bool first = true;
        for (int64_t cs = p0 & ~(int64_t)3; first || cs < p1; cs += CHMAX) {
            const int64_t ce = cs + CHMAX < p1 ? cs + CHMAX : p1;
            const uint32_t cnt4 = p1 > p0 ? (uint32_t)((ce - cs + 3) & ~(int64_t)3) : 0u;
            // a free descriptor and cnt4 free ring entries: reclaim released chunks, oldest first
            while (tail + TS_ND <= c || nfree < cnt4) {
                mbar_wait(&s_empty[tail % TS_ND], (tail / TS_ND) & 1);
                nfree += s_len[tail % TS_ND];
                ++tail;
            }
            const int d = c % TS_ND;
            s_len[d] = cnt4;
            nfree -= cnt4;
            unsigned char *desc = s_desc + d * L::DESC_BYTES;
            const uint32_t rpb = first ? (uint32_t)((((nvalid + 1) * 8) + 15) & ~15) : 0u;
            const uint32_t opb = first ? (uint32_t)(((nvalid * 8) + 15) & ~15) : 0u;
            mbar_expect_tx(&s_full[d], cnt4 * 12u + rpb + NOPS * opb);
            if (first) {
                tma_load_1d(desc, A.rowptr + r0, rpb, &s_full[d], pol);
#pragma unroll
                for (int o = 0; o < NOPS; ++o)
                    tma_load_1d(desc + L::RP_BYTES + o * L::OP_BYTES, epi.operand(o) + r0, opb, &s_full[d], pol);
            }
            if (cnt4) {
                const uint32_t n1 = cnt4 < RING - head ? cnt4 : RING - head;   // up to the ring's end
                tma_load_1d(s_val + head, A.val + cs, n1 * 8u, &s_full[d], pol);
                tma_load_1d(s_col + head, A.col + cs, n1 * 4u, &s_full[d], pol);
                if (n1 < cnt4) {                                               // wrapped remainder
                    tma_load_1d(s_val, A.val + cs + n1, (cnt4 - n1) * 8u, &s_full[d], pol);
                    tma_load_1d(s_col, A.col + cs + n1, (cnt4 - n1) * 4u, &s_full[d], pol);
                }
                head += cnt4;
                if (head >= RING) head -= RING;
            }
            first = false;
            ++c;
        }
    }
}

template <class Epi>
__global__ void __launch_bounds__(TS_THREADS, TS_OCC)
k_csr_rows(CsrMat A, const double *__restrict__ xg, Epi epi, RedArgs red) {
    constexpr int K = Epi::K;
    constexpr int NOPS = Epi::NOPS;
    using L = TsLayout<NOPS>;
    constexpr int RING = L::RING, CHMAX = L::CHMAX;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *s_val = reinterpret_cast<double *>(smem_raw + L::OFF_VAL);
    int32_t *s_col = reinterpret_cast<int32_t *>(smem_raw + L::OFF_COL);
    unsigned char *s_desc = smem_raw + L::OFF_DESC;
    uint64_t *s_full = reinterpret_cast<uint64_t *>(smem_raw + L::OFF_BAR);
    uint64_t *s_empty = s_full + TS_ND;
    uint32_t *s_len = reinterpret_cast<uint32_t *>(smem_raw + L::OFF_LEN);   // producer's notes
    double *s_red = reinterpret_cast<double *>(smem_raw + L::OFF_RED);
    const int tid = threadIdx.x;
    const int64_t nrows = A.nrows;
    const int64_t ntiles = (nrows + CGO_B - 1) / CGO_B;
    const int nact = (int)(ntiles < (int64_t)red.G ? ntiles : (int64_t)red.G);
    if (tid == 0) {
        for (int s = 0; s < TS_ND; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], CGO_NW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (tid >= CGO_B) {                       // ---------------- producer warp
        if (tid == CGO_B && (int)blockIdx.x < nact)
            ts_produce<L, Epi>(A, epi, red, s_val, s_col, s_desc, s_full, s_empty, s_len, nact, ntiles);
        return;
    }

    // ---------------- 256 row lanes
    const BarLanes bar;
    cgo_wait_flags(red, bar);                 // sharded: the neighbours' halo pushes have landed
    const uint64_t gpol = l2_policy_evict_last();
    uint32_t c = 0, head = 0;                 // chunks consumed, ring offset of the next chunk
    for (int v = blockIdx.x; v < nact; v += gridDim.x) {
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.0;
        for (int64_t tile = v; tile < ntiles; tile += red.G) {
            const int64_t r0 = tile * CGO_B;
            const int nvalid = (int)(nrows - r0 < CGO_B ? nrows - r0 : CGO_B);
            const bool valid = tid < nvalid;
            typename Epi::Pre pre;
            int64_t rs = 0, re = 0, p0 = 0, p1 = 0, cs = 0;
            double sum = 0.0;
            bool first = true;
            do {
                const int d = c % TS_ND;
                mbar_wait(&s_full[d], (c / TS_ND) & 1);
                if (first) {
                    const unsigned char *desc = s_desc + d * L::DESC_BYTES;
                    const int64_t *rp = reinterpret_cast<const int64_t *>(desc);
                    if (valid) {
                        rs = rp[tid]; re = rp[tid + 1];
                        pre = epi.load(reinterpret_cast<const double *>(desc + L::RP_BYTES), tid);
                    }
                    p0 = rp[0];
                    p1 = rp[nvalid];
                    cs = p0 & ~(int64_t)3;
                    first = false;
                }
                const int64_t ce = cs + CHMAX < p1 ? cs + CHMAX : p1;
                const uint32_t cnt4 = p1 > p0 ? (uint32_t)((ce - cs + 3) & ~(int64_t)3) : 0u;
                const int lo = (int)((rs > cs ? rs : cs) - cs);
                const int hi = (int)((re < ce ? re : ce) - cs);
                for (int k0 = lo; k0 < hi; k0 += TS_UN) {
                    // branch-free batch: TS_UN gathers are issued back to back (entries past the
                    // row's end are predicated off and not added)
                    double vj[TS_UN], xj[TS_UN];
#pragma unroll
                    for (int j = 0; j < TS_UN; ++j) {
                        const int kk = k0 + j < hi ? k0 + j : hi - 1;
                        uint32_t idx = head + (uint32_t)kk;
                        if (idx >= RING) idx -= RING;
                        vj[j] = s_val[idx];
                        xj[j] = ld_gather_f64_if(xg + s_col[idx], gpol, k0 + j < hi);
                    }
#pragma unroll
                    for (int j = 0; j < TS_UN; ++j) {
                        const double t = sum + vj[j] * xj[j];
                        sum = k0 + j < hi ? t : sum;
                    }
                }
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&s_empty[d]);
                head += cnt4;
                if (head >= RING) head -= RING;
                ++c;
                cs += CHMAX;
            } while (cs < p1);
            if (valid) epi.row(r0 + tid, sum, pre, acc);
        }
        cgo_cta_combine<K, BarLanes>(acc, s_red, bar);
        cgo_publish<K>(red, v, acc);
    }
    cgo_grid_finish<K, BarLanes>(red, nact, s_red, bar);
}

template <class Epi>
static int launch_csr(cgo_ctx *c, const CsrMat &A, const double *xg, const Epi &epi, const RedArgs &red, int tclass) {
    const int64_t ntiles = (A.nrows + CGO_B - 1) / CGO_B;
    int64_t nact = ntiles < red.G ? ntiles : red.G;
    int64_t phys = (int64_t)c->sms * TS_OCC;
    int grid = (int)(nact < phys ? nact : phys);
    if (grid < 1) grid = 1;
    CGO_CHECK(!A.sliced, "internal: k_csr_rows on a matrix in the sliced layout");
    const size_t smem = TsLayout<Epi::NOPS>::BYTES;
    CGO_CUDA(cudaFuncSetAttribute(k_csr_rows<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cgo_timer_begin(c, tclass);
    k_csr_rows<Epi><<<grid, TS_THREADS, smem, c->stream>>>(A, xg, epi, red);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------ row epilogues
// operand(o): per-row input vectors of the epilogue; the producer stages the tile's slice of
// each in shared memory next to the row pointers (they must be 16-byte aligned and padded by
// one element).  load() picks lane t's values out of that slice; row() consumes them once the
// row sum is known.
struct EpiStore {                       // y = A x
    static constexpr int K = 1, NOPS = 0;
    struct Pre {};
    double *y;
    __device__ __forceinline__ const double *operand(int) const { return nullptr; }
    __device__ __forceinline__ Pre load(const double *, int) const { return Pre(); }
    __device__ __forceinline__ void row(int64_t i, double sum, const Pre &, double (&)[K]) const { y[i] = sum; }
};
// r = A xp − b ; Σ r².  PUSH: the first / last `halo` residuals also go straight into the ring
// neighbours' halos of r (peer memory), where their SpMVᵀ gathers them.
template <bool PUSH>
struct EpiResidualT {
    static constexpr int K = 1, NOPS = 1;
    struct Pre { double b; };
    const double *b;
    double *r;
    double *prev_right, *next_left;      // PUSH
    int64_t halo, nrows;                 // PUSH
    __device__ __forceinline__ const double *operand(int) const { return b; }
    __device__ __forceinline__ Pre load(const double *ops, int t) const { return Pre{ops[t]}; }
    __device__ __forceinline__ void row(int64_t i, double sum, const Pre &p, double (&acc)[K]) const {
        const double rr = sum - p.b;
        r[i] = rr;                      // re-read (gathered) by K_c: keep it cacheable
        if (PUSH) {
            if (i < halo) prev_right[i] = rr;
            if (i >= nrows - halo) next_left[i - (nrows - halo)] = rr;
        }
        acc[0] = acc[0] + rr * rr;
    }
};
// g⁺ = Aᵀ r [· 1/N + λ w], fused with norm(df_xp)² (optim.jl:107), dϕ = g⁺·u (cg_utils.jl:20) and
// the getβ dots (cg_flavours.jl:63-76, 96-105, 140-145, 164-167); fills pack slots 1..8.
template <bool LOGREG>
struct EpiGrad {
    static constexpr int K = 8, NOPS = LOGREG ? 3 : 2;
    struct Pre { double u, g, w; };
    double *gp;
    const double *g, *u, *w;
    double invN, lambda;
    __device__ __forceinline__ const double *operand(int o) const { return o == 0 ? u : (o == 1 ? g : w); }
    __device__ __forceinline__ Pre load(const double *ops, int t) const {
        Pre p;
        p.u = ops[t]; p.g = ops[CGO_B + t];
        p.w = LOGREG ? ops[2 * CGO_B + t] : 0.0;
        return p;
    }
    __device__ __forceinline__ void row(int64_t j, double sum, const Pre &p, double (&acc)[K]) const {
        double gn = sum;
        if (LOGREG) gn = sum * invN + lambda * p.w;
        st_stream_f64(gp + j, gn);
        const double uu = p.u, gg = p.g;
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
};
// logistic loss of sample i with margin z = a_i·w (oracle logreg_fdf):
//   t = −y z; e = exp(−|t|); ℓ = max(t,0) + log1p(e); σ = t ≥ 0 ? 1/(1+e) : e/(1+e); c = −y σ
struct EpiLogit {
    static constexpr int K = 1, NOPS = 1;
    struct Pre { double y; };
    const double *label;
    double *c;
    __device__ __forceinline__ const double *operand(int) const { return label; }
    __device__ __forceinline__ Pre load(const double *ops, int t) const { return Pre{ops[t]}; }
    __device__ __forceinline__ void row(int64_t i, double z, const Pre &p, double (&acc)[K]) const {
        const double y = p.y;
        const double t = -y * z;
        const double e = exp(-fabs(t));
        const double l = (t > 0.0 ? t : 0.0) + log1p(e);
        const double sg = t >= 0.0 ? 1.0 / (1.0 + e) : e / (1.0 + e);
        c[i] = -y * sg;
        acc[0] = acc[0] + l;
    }
};

// Hessian-vector product of least squares, ∇²f u = Aᵀ(A u): v = A u with Σ v² (= u·Hu), then
// hv = Aᵀ v with u·hv and hv·hv
struct EpiStoreSq {
    static constexpr int K = 1, NOPS = 0;
    struct Pre {};
    double *y;
    __device__ __forceinline__ const double *operand(int) const { return nullptr; }
    __device__ __forceinline__ Pre load(const double *, int) const { return Pre(); }
    __device__ __forceinline__ void row(int64_t i, double sum, const Pre &, double (&acc)[K]) const {
        y[i] = sum;
        acc[0] = acc[0] + sum * sum;
    }
};
struct EpiHv {
    static constexpr int K = 2, NOPS = 1;
    struct Pre { double u; };
    double *hv;
    const double *u;
    __device__ __forceinline__ const double *operand(int) const { return u; }
    __device__ __forceinline__ Pre load(const double *ops, int t) const { return Pre{ops[t]}; }
    __device__ __forceinline__ void row(int64_t j, double sum, const Pre &p, double (&acc)[K]) const {
        hv[j] = sum;
        acc[0] = acc[0] + p.u * sum;
        acc[1] = acc[1] + sum * sum;
    }
};

// quadratic-aware line search: v = A u with r·v, v·v and r·r (r = residual at x)
struct EpiQuadV {
    static constexpr int K = 3, NOPS = 1;
    struct Pre { double r; };
    double *v;
    const double *r;
    __device__ __forceinline__ const double *operand(int) const { return r; }
    __device__ __forceinline__ Pre load(const double *ops, int t) const { return Pre{ops[t]}; }
    __device__ __forceinline__ void row(int64_t i, double sum, const Pre &p, double (&acc)[K]) const {
        v[i] = sum;
        acc[0] = acc[0] + p.r * sum;
        acc[1] = acc[1] + sum * sum;
        acc[2] = acc[2] + p.r * p.r;
    }
};

// ------------------------------------------------------------------ the gather-bound SpMV kernel
// Matrices whose gathers do not coalesce — every lane of a warp-level gather touches its own 128-byte line: the
// per-row-random cfg-3 matrix (coh_log2 < 4), the column-block passes of logistic regression — are bound by
// L1TEX, one line per clock and SM: ≈ 245 G gathers/s on a B200 whatever the load path (scratch/gather_bench.cu:
// LDG, LDG with L2 hints, TEX, LDGSTS, TMA gather4 all measured).  What reaches that ceiling is many warps with
// a short instruction stream, each keeping a batch of gathers in flight: the prototype in gather_bench.cu gets
// 244 G gathers/s with 32 warps per SM, against ≈ 105 G/s for k_csr_rows, whose canonical reduction order caps
// the grid at G = 296 CTAs (16 warps per SM) and whose ring, barriers and epilogue leave those warps without a
// gather in flight half of the time.  So for these matrices the reductions leave the SpMV:
//   k_spmv_direct  y = A x [− b | /N + λw | + partial]: no reduction ⇒ no canonical order to respect ⇒ any
//                  grid, any schedule; 24-32 warps per SM, values and column indices read straight from HBM by
//                  coalesced loads (sliced layout: the k-th entries of a slice's 32 rows are consecutive), no
//                  shared memory, slices handed out dynamically — which also keeps all warps inside one band
//                  of the gathered vector, so it stays L2-resident (the static tile order of k_csr_rows lets its
//                  CTAs drift apart by more rows than the band is wide on a 2e8-row matrix: then every gather is
//                  a DRAM sector read, 86 GB of DRAM traffic against 30 GB algorithmic, 36 ms instead of 15);
//   k_blas1        the dots, in the BLAS-1 canonical order (V = 2, U = 4): Σ r² after K_b, the eight getβ dots
//                  after K_c — 16n more bytes per evaluation than the fused epilogues (+5 %).
// Each row's products are still added one by one in storage order: row sums are bit-identical to k_csr_rows'.
constexpr int DIR_GRAB = 4;                 // slices (of 32 rows) a warp takes from the queue at a time
struct DirArgs {
    unsigned long long *next;               // slice queue head (reset by the last CTA)
    unsigned int *ticket;
    // cross-GPU hand-off, as in RedArgs
    unsigned long long *sig0, *sig1;
    const unsigned long long *wait0, *wait1;
    unsigned long long sig_val, wait_val;
    void *const *flags_all;
    const unsigned long long *wait_all;
    int sig_all_slot, nranks, me;
};
__device__ __forceinline__ int32_t ld_stream_s32_if(const int32_t *p, bool on) {
    int32_t r = 0;
    asm volatile("{\n.reg .pred q;\nsetp.ne.s32 q, %2, 0;\n@q ld.global.nc.L1::no_allocate.s32 %0, [%1];\n}\n" : "+r"(r) : "l"(p), "r"((int)on));
    return r;
}
__device__ __forceinline__ double ld_stream_f64_if(const double *p, bool on) {
    double r = 0.0;
    asm volatile("{\n.reg .pred q;\nsetp.ne.s32 q, %2, 0;\n@q ld.global.nc.L1::no_allocate.f64 %0, [%1];\n}\n" : "+d"(r) : "l"(p), "r"((int)on));
    return r;
}

// one batch of UN levels of a slice: the lane's entries, gathered and added in order
template <int UN, bool UNIFORM>
__device__ __forceinline__ double dir_batch(const CsrMat &A, const double *__restrict__ xg, uint64_t gpol, int64_t sb,
                                            int64_t &off, int len, int k0, int lane, uint32_t lt, double sum) {
    int32_t cj[UN];
    double vj[UN], xj[UN];
#pragma unroll
    for (int j = 0; j < UN; ++j) {
        const bool on = len > k0 + j;
        int64_t idx;
        if (UNIFORM) { idx = sb + off + lane; off += 32; }
        else {
            const uint32_t m = __ballot_sync(0xffffffffu, on);
            idx = sb + off + __popc(m & lt);
            off += __popc(m);
        }
        cj[j] = ld_stream_s32_if(A.col + idx, on);
        vj[j] = ld_stream_f64_if(A.val + idx, on);
    }
#pragma unroll
    for (int j = 0; j < UN; ++j) xj[j] = ld_gather_f64_if(xg + cj[j], gpol, len > k0 + j);
#pragma unroll
    for (int j = 0; j < UN; ++j) {
        const double p = vj[j] * xj[j];
        if (len > k0 + j) sum = sum + p;
    }
    return sum;
}

template <class F, int UN, int OCC>
__global__ void __launch_bounds__(CGO_B, OCC)
k_spmv_direct(CsrMat A, const double *__restrict__ xg, F f, DirArgs da) {
    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const int64_t nrows = A.nrows, nslices = (nrows + 31) / 32;
    if (da.wait0 != nullptr || da.wait_all != nullptr) {        // sharded: the peers' pushes have landed
        if (tid == 0 && da.wait0 != nullptr) {
            cgo_spin_until(da.wait0, da.wait_val);
            if (da.wait1 != nullptr) cgo_spin_until(da.wait1, da.wait_val);
        }
        if (da.wait_all != nullptr && tid < da.nranks) cgo_spin_until(da.wait_all + tid, da.wait_val);
        __syncthreads();
    }
    const uint64_t gpol = l2_policy_evict_last();
    for (;;) {
        unsigned long long s0 = 0;
        if (lane == 0) s0 = atomicAdd(da.next, (unsigned long long)DIR_GRAB);
        s0 = __shfl_sync(0xffffffffu, s0, 0);
        if ((int64_t)s0 >= nslices) break;
#pragma unroll 1
        for (int g = 0; g < DIR_GRAB; ++g) {
            const int64_t s = (int64_t)s0 + g;
            if (s >= nslices) break;
            const int64_t row = s * 32 + lane;
            const bool valid = row < nrows;
            int64_t rp0 = 0, rp1 = 0;
            if (valid) { rp0 = __ldg(A.rowptr + row); rp1 = __ldg(A.rowptr + row + 1); }
            const int len = valid ? (int)(rp1 - rp0) : -1;
            const int64_t sb = __shfl_sync(0xffffffffu, rp0, 0);
            const int maxlen = __reduce_max_sync(0xffffffffu, len);
            const bool uniform = __all_sync(0xffffffffu, len == maxlen);
            double sum = valid ? f.init(row) : 0.0;
            int64_t off = 0;
            if (uniform) { for (int k0 = 0; k0 < maxlen; k0 += UN) sum = dir_batch<UN, true>(A, xg, gpol, sb, off, len, k0, lane, lt, sum); }
            else { for (int k0 = 0; k0 < maxlen; k0 += UN) sum = dir_batch<UN, false>(A, xg, gpol, sb, off, len, k0, lane, lt, sum); }
            if (valid) f.row(row, sum);
        }
    }
    // the last CTA re-arms the queue and hands the pushed halos to the peers
    __shared__ bool is_last;
    if (da.sig0 != nullptr || da.flags_all != nullptr) __threadfence_system();
    else __threadfence();
    __syncthreads();
    if (tid == 0) is_last = atomicAdd(da.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (is_last && tid == 0) {
        *da.ticket = 0u;
        *da.next = 0ULL;
        __threadfence_system();
        if (da.sig0 != nullptr) {
            cgo_st_release_sys(da.sig0, da.sig_val);
            if (da.sig1 != nullptr) cgo_st_release_sys(da.sig1, da.sig_val);
        }
        if (da.flags_all != nullptr)
            for (int r = 0; r < da.nranks; ++r)
                cgo_st_release_sys((unsigned long long *)da.flags_all[r] + da.sig_all_slot + da.me, da.sig_val);
    }
}

// row functors of k_spmv_direct: init(i) = what the row sum starts from, row(i, sum) = what to do with it
struct DirStore {                       // y = A x
    double *y;
    __device__ __forceinline__ double init(int64_t) const { return 0.0; }
    __device__ __forceinline__ void row(int64_t i, double sum) const { y[i] = sum; }
};
struct DirStoreInit {                   // column-block pass: y = partial + A_j x
    double *y;
    const double *partial;
    __device__ __forceinline__ double init(int64_t i) const { return ld_stream_f64(partial + i); }
    __device__ __forceinline__ void row(int64_t i, double sum) const { y[i] = sum; }
};
template <bool PUSH>
struct DirResidual {                    // r = A xp − b  (+ halo push, as EpiResidualT)
    const double *b;
    double *r;
    double *prev_right, *next_left;
    int64_t halo, nrows;
    __device__ __forceinline__ double init(int64_t) const { return 0.0; }
    __device__ __forceinline__ void row(int64_t i, double sum) const {
        const double rr = sum - ld_stream_f64(b + i);
        r[i] = rr;
        if (PUSH) {
            if (i < halo) prev_right[i] = rr;
            if (i >= nrows - halo) next_left[i - (nrows - halo)] = rr;
        }
    }
};
struct DirGradLS {                      // g⁺ = Aᵀ r
    double *gp;
    __device__ __forceinline__ double init(int64_t) const { return 0.0; }
    __device__ __forceinline__ void row(int64_t j, double sum) const { st_stream_f64(gp + j, sum); }
};

static DirArgs dir_args(cgo_ctx *c, const RedArgs *red = nullptr) {
    DirArgs d;
    d.next = c->d_progress + 4;
    d.ticket = c->d_ticket + 1;
    d.sig0 = d.sig1 = nullptr; d.wait0 = d.wait1 = nullptr; d.sig_val = d.wait_val = 0;
    d.flags_all = nullptr; d.wait_all = nullptr; d.sig_all_slot = -1; d.nranks = 1; d.me = 0;
    if (red) {
        d.sig0 = red->sig0; d.sig1 = red->sig1; d.wait0 = red->wait0; d.wait1 = red->wait1;
        d.sig_val = red->sig_val; d.wait_val = red->wait_val;
        d.flags_all = red->flags_all; d.wait_all = red->wait_all; d.sig_all_slot = red->sig_all_slot;
        d.nranks = red->nranks; d.me = red->me;
    }
    return d;
}
template <class F, int UN, int OCC>
static int launch_direct_k(cgo_ctx *c, const CsrMat &A, const double *xg, const F &f, const DirArgs &da, int tclass) {
    const int64_t nslices = (A.nrows + 31) / 32;
    int64_t want = (nslices + 8 * DIR_GRAB - 1) / (8 * DIR_GRAB), phys = (int64_t)c->sms * OCC;
    int grid = (int)(want < phys ? want : phys);
    if (grid < 1) grid = 1;
    cgo_timer_begin(c, tclass);
    k_spmv_direct<F, UN, OCC><<<grid, CGO_B, 0, c->stream>>>(A, xg, f, da);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    return 0;
}
template <class F>
static int launch_direct(cgo_ctx *c, const CsrMat &A, const double *xg, const F &f, const DirArgs &da, int tclass) {
    CGO_CHECK(A.sliced, "internal: k_spmv_direct needs the sliced layout");
    // gathers per batch × CTAs per SM, measured at n = 2e8, coh_log2 = 0 (K_b = ten entries in every row / K_c =
    // ragged rows of Aᵀ, ms; profiles/r2_exp_coh0_n2e8_k_spmv_direct_configs.txt): 10 × 4: 7.5–7.9 / 9.3–10.5;
    // 8 × 4: 8.0 / 9.1; 6 × 5: 7.7–8.1 / 9.1; 5 × 4: 7.7 / 9.3; 8 × 5 (spills): 8.4 / 9.5; 10 × 3: 7.9 / 10.5.
    // Ragged slices waste the tail of a wide batch, equal-length rows like the widest batch that does not spill.
    if (A.ragged) return launch_direct_k<F, 6, 5>(c, A, xg, f, da, tclass);
    return launch_direct_k<F, 10, 4>(c, A, xg, f, da, tclass);
}

// ------------------------------------------------------------------ the K-column SpMM (softmax regression)
// Y = A X with X (ncols × K) and Y (nrows × K) row-major: the SpMV of A ⊗ I_K on the flat vectors, whose row
// (i, k) holds row i's entries in storage order at columns col·K + k.  A group of GW = 2^gw_log2 lanes owns one
// row, lane k of the group one class (class tiles of 32 when K > 32).  The group's lanes read each entry's column
// index and value from the same address (one request per group, once per class tile) and gather x[col·K + k]:
// one gather instruction reads whole contiguous segments.  Each (row, class) sum is added entry by entry in
// storage order from f.init(i·K + k), so it is bit for bit the row sum k_spmv_direct makes of the expanded matrix,
// and column-block passes chain through DirStoreInit as they do there.  Plain row-major CSR (no sliced layout).
// Work units (32 / GW rows, one class tile) come from the slice queue of k_spmv_direct.
constexpr int MM_UN = 8;                    // entries per batch whose loads are in flight together
constexpr int MM_OCC = 4;
template <class F>
__global__ void __launch_bounds__(CGO_B, MM_OCC)
k_spmm_direct(CsrMat A, int K, int gw_log2, const double *__restrict__ xg, F f, DirArgs da) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int gw = 1 << gw_log2, rpw = 32 >> gw_log2;
    const int sub = lane >> gw_log2, kl = lane & (gw - 1);
    const int nct = (K + gw - 1) >> gw_log2;
    const int64_t nrows = A.nrows, nunits = (nrows + rpw - 1) / rpw * nct;
    const uint64_t gpol = l2_policy_evict_last();
    for (;;) {
        unsigned long long s0 = 0;
        if (lane == 0) s0 = atomicAdd(da.next, (unsigned long long)DIR_GRAB);
        s0 = __shfl_sync(0xffffffffu, s0, 0);
        if ((int64_t)s0 >= nunits) break;
#pragma unroll 1
        for (int g = 0; g < DIR_GRAB; ++g) {
            const int64_t s = (int64_t)s0 + g;
            if (s >= nunits) break;
            const int64_t rg = s / nct;
            const int k = (int)(s - rg * nct) * gw + kl;
            const int64_t row = rg * rpw + sub;
            const bool inrow = row < nrows, valid = inrow && k < K;
            int64_t rp0 = 0;
            int len = 0;
            if (inrow) { rp0 = __ldg(A.rowptr + row); len = (int)(__ldg(A.rowptr + row + 1) - rp0); }
            const int maxlen = __reduce_max_sync(0xffffffffu, len);
            const int64_t y = row * K + k;
            double sum = valid ? f.init(y) : 0.0;
            for (int k0 = 0; k0 < maxlen; k0 += MM_UN) {
                int32_t cj[MM_UN];
                double vj[MM_UN], xj[MM_UN];
#pragma unroll
                for (int j = 0; j < MM_UN; ++j) {
                    const bool on = len > k0 + j;
                    cj[j] = ld_stream_s32_if(A.col + rp0 + k0 + j, on);
                    vj[j] = ld_stream_f64_if(A.val + rp0 + k0 + j, on);
                }
#pragma unroll
                for (int j = 0; j < MM_UN; ++j) xj[j] = ld_gather_f64_if(xg + (int64_t)cj[j] * K + k, gpol, valid && len > k0 + j);
#pragma unroll
                for (int j = 0; j < MM_UN; ++j) {
                    const double p = vj[j] * xj[j];
                    if (len > k0 + j) sum = sum + p;
                }
            }
            if (valid) f.row(y, sum);
        }
    }
    // the last CTA re-arms the queue
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = atomicAdd(da.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (is_last && tid == 0) {
        *da.ticket = 0u;
        *da.next = 0ULL;
        __threadfence();
    }
}
template <class F>
static int launch_spmm(cgo_ctx *c, const CsrMat &A, int K, const double *xg, const F &f, int tclass) {
    CGO_CHECK(!A.sliced && K >= 1, "internal: k_spmm_direct needs a row-major matrix");
    int gw_log2 = 0;
    while ((1 << gw_log2) < K && gw_log2 < 5) ++gw_log2;
    const int64_t nct = (K + (1 << gw_log2) - 1) >> gw_log2;
    const int64_t nunits = (A.nrows + (32 >> gw_log2) - 1) / (32 >> gw_log2) * nct;
    int64_t want = (nunits + 8 * DIR_GRAB - 1) / (8 * DIR_GRAB), phys = (int64_t)c->sms * MM_OCC;
    int grid = (int)(want < phys ? want : phys);
    if (grid < 1) grid = 1;
    cgo_timer_begin(c, tclass);
    k_spmm_direct<F><<<grid, CGO_B, 0, c->stream>>>(A, K, gw_log2, xg, f, dir_args(c));
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------ counter-based hash
// (generator spec: oracle/cgo_oracle.c hash3 / u01; restated, identical arithmetic)
__host__ __device__ __forceinline__ uint64_t g_mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
__host__ __device__ __forceinline__ uint64_t g_hash3(uint64_t seed, uint64_t i, uint64_t k) {
    uint64_t h = g_mix64(seed + 0x9E3779B97F4A7C15ULL);
    h = g_mix64(h ^ (i + 0x9E3779B97F4A7C15ULL));
    h = g_mix64(h ^ (k + 0x632BE59BD9B4E019ULL));
    return h;
}
__host__ __device__ __forceinline__ double g_u01(uint64_t seed, uint64_t i, uint64_t k) {
    return (double)(g_hash3(seed, i, k) >> 11) * (1.0 / 9007199254740992.0);
}

// banded-random least-squares generator (spec text: oracle/cgo_oracle.c orc_obj_sparse_ls_synth)
struct LsSpec {
    int64_t n;          // global dimension
    int32_t K;          // entries per row
    int32_t coh;        // log2 of the number of consecutive rows sharing their offsets
    int64_t W, w;       // half band width, stratum width 2W/(K−1)
    uint64_t seed;
    // signed column offset and value of entry k of global row i
    __host__ __device__ __forceinline__ void entry(int64_t i, int k, int64_t &d, double &v) const {
        if (k == 0) { d = 0; v = 4.0 + g_u01(seed, (uint64_t)i, 0); return; }
        const int64_t lo = -W + (int64_t)(k - 1) * w;
        d = lo + (int64_t)(g_hash3(seed ^ 0xA5A5A5A5A5A5A5A5ULL, (uint64_t)(i >> coh), (uint64_t)k) % (uint64_t)w);
        if (d == 0) d = (lo + w > 1) ? 1 : -1;
        v = 0.3 * (2.0 * g_u01(seed, (uint64_t)i, (uint64_t)k) - 1.0);
    }
    __host__ __device__ __forceinline__ int64_t wrap(int64_t c) const {
        if (c < 0) c += n;
        if (c >= n) c -= n;
        return c;
    }
};
// logistic-regression generator (spec text: oracle/cgo_oracle.c orc_obj_logreg_synth)
struct LrSpec {
    int64_t N, d;
    int32_t K;
    int64_t w;          // stratum width d / K
    uint64_t seed;
    __host__ __device__ __forceinline__ void entry(int64_t i, int k, int64_t &c, double &v) const {
        c = (int64_t)k * w + (int64_t)(g_hash3(seed, (uint64_t)i, (uint64_t)k) % (uint64_t)w);
        v = 2.0 * g_u01(seed + 7, (uint64_t)i, (uint64_t)k) - 1.0;
    }
};

static inline int grid_for(int64_t items, int sms) {
    int64_t b = (items + 255) / 256;
    int64_t cap = (int64_t)sms * 32;
    return (int)(b < 1 ? 1 : (b < cap ? b : cap));
}
#define GRID_STRIDE(idx, total) \
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < (total); idx += (int64_t)gridDim.x * blockDim.x)

// rows [lo, lo + nloc) of A.  unwrapped: column index relative to lo, in [−W, nloc + W) (halo
// layout, multi-rank); else the wrapped global column (single rank).
__global__ void k_ls_fill_A(LsSpec s, int64_t lo, int64_t nloc, bool unwrapped, CsrMat A) {
    const int64_t total = nloc * s.K;
    GRID_STRIDE(p, total) {
        const int64_t il = p / s.K;
        const int k = (int)(p - il * s.K);
        int64_t d; double v;
        s.entry(lo + il, k, d, v);
        A.col[p] = (int32_t)(unwrapped ? il + d : s.wrap(lo + il + d));
        A.val[p] = v;
        if (k == 0) A.rowptr[il] = p;
        if (p == total - 1) A.rowptr[nloc] = total;
    }
}
// x_true over [lo − halo, lo + nloc + halo), wrapped
__global__ void k_ls_xtrue(LsSpec s, int64_t lo, int64_t nloc, int64_t halo, double *xt /* local origin */) {
    GRID_STRIDE(e, nloc + 2 * halo) {
        int64_t i = s.wrap(lo - halo + e);
        xt[e - halo] = 2.0 * g_u01(s.seed + 1, (uint64_t)i, 0) - 1.0;
    }
}
// samples [i0, i0 + nloc) of the generator; column = global feature index
__global__ void k_lr_fill_A(LrSpec s, int64_t i0, int64_t nloc, CsrMat A, double *label) {
    GRID_STRIDE(il, nloc) {
        const int64_t i = i0 + il;
        const int64_t p = il * s.K;
        A.rowptr[il] = p;
        double acc = 0.0;
        for (int k = 0; k < s.K; ++k) {
            int64_t c; double v;
            s.entry(i, k, c, v);
            A.col[p + k] = (int32_t)c;
            A.val[p + k] = v;
            const double wt = 2.0 * g_u01(s.seed + 2, (uint64_t)c, 0) - 1.0;
            acc += v * wt;
        }
        const double noise = 2.0 * g_u01(s.seed + 3, (uint64_t)i, 0) - 1.0;
        label[il] = (acc + 0.1 * noise >= 0.0) ? 1.0 : -1.0;
        if (il == nloc - 1) A.rowptr[nloc] = nloc * s.K;
    }
}

// ------------------------------------------------------------------ explicit transpose (setup)
// Entry sources enumerate (target row of Aᵀ, sort key) pairs; keys order the entries of one Aᵀ
// row exactly like the oracle's stable counting sort (ascending source entry).
struct CsrSrc {                 // a materialised CSR on this device
    const int32_t *col;
    int64_t total;
    __device__ __forceinline__ bool get(int64_t e, int64_t &trow, int64_t &key) const {
        trow = col[e]; key = e;
        return true;
    }
};
struct LsExtSrc {               // generator rows [lo − W, hi + W): entries landing in columns [lo, hi)
    LsSpec s;
    int64_t lo, hi, total;
    __device__ __forceinline__ bool get(int64_t e, int64_t &trow, int64_t &key) const {
        const int64_t ie = e / s.K;
        const int k = (int)(e - ie * s.K);
        const int64_t i = s.wrap(lo - s.W + ie);
        int64_t d; double v;
        s.entry(i, k, d, v);
        const int64_t c = s.wrap(i + d);
        if (c < lo || c >= hi) return false;
        trow = c - lo; key = i * s.K + k;
        return true;
    }
};
template <class Src>
__global__ void k_tr_count(Src src, unsigned long long *counts) {
    GRID_STRIDE(e, src.total) {
        int64_t trow, key;
        if (src.get(e, trow, key)) atomicAdd(counts + trow, 1ULL);
    }
}
template <class Src>
__global__ void k_tr_fill(Src src, unsigned long long *cursor, int64_t *perm) {
    GRID_STRIDE(e, src.total) {
        int64_t trow, key;
        if (src.get(e, trow, key)) perm[atomicAdd(cursor + trow, 1ULL)] = key;
    }
}
// each Aᵀ row's keys ascending (insertion sort for short rows, heapsort beyond)
__global__ void k_tr_sort(const int64_t *rowptrT, int64_t nT, int64_t *perm) {
    GRID_STRIDE(j, nT) {
        int64_t *a = perm + rowptrT[j];
        const int64_t L = rowptrT[j + 1] - rowptrT[j];
        if (L <= 48) {
            for (int64_t i = 1; i < L; ++i) {
                const int64_t key = a[i];
                int64_t q = i - 1;
                while (q >= 0 && a[q] > key) { a[q + 1] = a[q]; --q; }
                a[q + 1] = key;
            }
        } else {
            for (int64_t start = L / 2 - 1; start >= 0; --start) {       // heapify
                int64_t root = start;
                for (;;) {
                    int64_t ch = 2 * root + 1;
                    if (ch >= L) break;
                    if (ch + 1 < L && a[ch] < a[ch + 1]) ++ch;
                    if (a[root] >= a[ch]) break;
                    int64_t t = a[root]; a[root] = a[ch]; a[ch] = t;
                    root = ch;
                }
            }
            for (int64_t end = L - 1; end > 0; --end) {
                int64_t t = a[0]; a[0] = a[end]; a[end] = t;
                int64_t root = 0;
                for (;;) {
                    int64_t ch = 2 * root + 1;
                    if (ch >= end) break;
                    if (ch + 1 < end && a[ch] < a[ch + 1]) ++ch;
                    if (a[root] >= a[ch]) break;
                    int64_t t2 = a[root]; a[root] = a[ch]; a[ch] = t2;
                    root = ch;
                }
            }
        }
    }
}
struct CsrFin {                 // key = entry index of a materialised CSR
    const int64_t *rowptr;
    int64_t nrows;
    const double *val;
    __device__ __forceinline__ void get(int64_t key, int32_t &srow, double &v) const {
        int64_t lo = 0, hi = nrows;              // last row with rowptr[row] <= key
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (rowptr[mid] <= key) lo = mid; else hi = mid;
        }
        srow = (int32_t)lo; v = val[key];
    }
};
struct FixedKFin {              // materialised CSR with exactly K entries per row
    int32_t K;
    const double *val;
    __device__ __forceinline__ void get(int64_t key, int32_t &srow, double &v) const {
        srow = (int32_t)(key / K); v = val[key];
    }
};
struct LsExtFin {               // key = global entry index of the generator
    LsSpec s;
    int64_t lo;
    __device__ __forceinline__ void get(int64_t key, int32_t &srow, double &v) const {
        const int64_t i = key / s.K;
        const int k = (int)(key - i * s.K);
        int64_t d;
        s.entry(i, k, d, v);
        int64_t rel = i - lo;                    // unwrapped position relative to this shard
        if (rel < -s.W) rel += s.n;
        if (rel >= s.n - s.W) rel -= s.n;
        srow = (int32_t)rel;
    }
};
template <class Fin>
__global__ void k_tr_finalize(Fin fin, int64_t nnzT, const int64_t *perm, CsrMat AT) {
    GRID_STRIDE(q, nnzT) {
        int32_t srow; double v;
        fin.get(perm[q], srow, v);
        AT.col[q] = srow;
        AT.val[q] = v;
    }
}

static void csr_free(CsrMat &M) {
    cudaFree(M.rowptr); cudaFree(M.col); cudaFree(M.val);
    M = CsrMat();
}
static int csr_alloc(CsrMat &M, int64_t nrows, int64_t nnz) {
    M.nrows = nrows; M.nnz = nnz;
    // CSR_PAD: bulk copies are rounded up to 16 bytes and may read past the last entry
    CGO_CUDA(cudaMalloc(&M.rowptr, sizeof(int64_t) * (size_t)(nrows + 1 + CSR_PAD)));
    CGO_CUDA(cudaMalloc(&M.col, sizeof(int32_t) * (size_t)(nnz + CSR_PAD)));
    CGO_CUDA(cudaMalloc(&M.val, sizeof(double) * (size_t)(nnz + CSR_PAD)));
    return 0;
}

// ------------------------------------------------------------------ sliced layout (setup)
// Re-order the entries of every 32-row slice level-major (CsrMat::sliced; k_csr_rows ts_issue).  Row pointers
// stay CSR row pointers: a slice still owns the range [rowptr[32s], rowptr[32s+32)), only the order inside it
// changes, and each row's own entries keep their relative order.
// one warp per slice; inverse = back to row-major; *n_ragged (optional) += slices whose rows differ in length
__global__ void k_slice_permute(CsrMat M, const int32_t *col_in, const double *val_in, int32_t *col_out, double *val_out,
                                bool inverse, unsigned long long *n_ragged = nullptr) {
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const int64_t nslices = (M.nrows + 31) / 32;
    const int64_t wstride = (int64_t)gridDim.x * (blockDim.x / 32);
    for (int64_t s = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); s < nslices; s += wstride) {
        const int64_t row = s * 32 + lane;
        int64_t rs = 0, len = 0;
        if (row < M.nrows) { rs = M.rowptr[row]; len = M.rowptr[row + 1] - rs; }
        const int64_t sb = M.rowptr[s * 32];
        if (n_ragged != nullptr) {
            const int64_t len0 = __shfl_sync(0xffffffffu, len, 0);
            const bool same = __all_sync(0xffffffffu, row >= M.nrows || len == len0);
            if (!same && lane == 0) atomicAdd(n_ragged, 1ULL);
        }
        int64_t off = 0;
        for (int64_t k = 0;; ++k) {
            const uint32_t m = __ballot_sync(0xffffffffu, len > k);
            if (m == 0) break;
            if (len > k) {
                const int64_t lvl = sb + off + __popc(m & lt), rm = rs + k;
                const int64_t src = inverse ? lvl : rm, dst = inverse ? rm : lvl;
                col_out[dst] = col_in[src];
                val_out[dst] = val_in[src];
            }
            off += __popc(m);
        }
    }
}
// a 1-in-64 sample of the 32-row slices of a row-major matrix: stats[0] += warp-level gathers (the k-th entries
// of a slice's rows), stats[1] += distinct 128-byte lines of the gathered vector they touch
__global__ void k_gather_lines(CsrMat M, unsigned long long *stats) {
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const int64_t nslices = (M.nrows + 31) / 32;
    const int64_t wstride = (int64_t)gridDim.x * (blockDim.x / 32);
    for (int64_t s = ((int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5)) * 64; s < nslices; s += wstride * 64) {
        const int64_t row = s * 32 + lane;
        int64_t rs = 0, len = 0;
        if (row < M.nrows) { rs = M.rowptr[row]; len = M.rowptr[row + 1] - rs; }
        unsigned int nlev = 0, nlines = 0;
        for (int64_t k = 0;; ++k) {
            const uint32_t m = __ballot_sync(0xffffffffu, len > k);
            if (m == 0) break;
            if (len > k) {
                const uint32_t same = __match_any_sync(m, M.col[rs + k] >> 4);
                if ((same & lt) == 0) ++nlines;          // first lane of its line
            }
            ++nlev;
        }
        nlines = __reduce_add_sync(0xffffffffu, nlines);
        if (lane == 0) { atomicAdd(stats, (unsigned long long)nlev); atomicAdd(stats + 1, (unsigned long long)nlines); }
    }
}
// distinct 128-byte lines of the gathered vector one warp-level gather touches (row-major matrix, sampled)
static int csr_gather_lines(cgo_ctx *c, const CsrMat &M, float *lines) {
    unsigned long long *d_stats = c->d_progress + 2, h_stats[2] = {0, 0};
    *lines = 1.0f;
    if (M.nnz == 0) return 0;
    CGO_CUDA(cudaMemsetAsync(d_stats, 0, sizeof(h_stats), c->stream));
    k_gather_lines<<<grid_for((M.nrows + 31) / 32 * 32, c->sms), 256, 0, c->stream>>>(M, d_stats);
    CGO_CUDA(cudaGetLastError());
    CGO_CUDA(cudaMemcpyAsync(h_stats, d_stats, sizeof(h_stats), cudaMemcpyDeviceToHost, c->stream));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    if (h_stats[0]) *lines = (float)((double)h_stats[1] / (double)h_stats[0]);
    return 0;
}
static int csr_make_sliced(cgo_ctx *c, CsrMat &M) {
    if (M.sliced || M.nnz == 0 || !M.col || !M.val) return 0;
    int32_t *col2 = nullptr; double *val2 = nullptr;
    unsigned long long n_ragged = 0;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&col2, sizeof(int32_t) * (size_t)(M.nnz + CSR_PAD)));
        CGO_CUDA(cudaMalloc(&val2, sizeof(double) * (size_t)(M.nnz + CSR_PAD)));
        CGO_CUDA(cudaMemsetAsync(col2 + M.nnz, 0, sizeof(int32_t) * CSR_PAD, c->stream));
        CGO_CUDA(cudaMemsetAsync(val2 + M.nnz, 0, sizeof(double) * CSR_PAD, c->stream));
        unsigned long long *d_ragged = c->d_progress + 1;
        CGO_CUDA(cudaMemsetAsync(d_ragged, 0, sizeof(unsigned long long), c->stream));
        k_slice_permute<<<grid_for((M.nrows + 31) / 32 * 32, c->sms), 256, 0, c->stream>>>(M, M.col, M.val, col2, val2, false,
                                                                                          d_ragged);
        CGO_CUDA(cudaGetLastError());
        CGO_CUDA(cudaMemcpyAsync(&n_ragged, d_ragged, sizeof(n_ragged), cudaMemcpyDeviceToHost, c->stream));
        CGO_CUDA(cudaStreamSynchronize(c->stream));
        return 0;
    };
    int rc = body();
    if (rc) { cudaFree(col2); cudaFree(val2); return rc; }
    cudaFree(M.col); cudaFree(M.val);
    M.col = col2; M.val = val2;
    M.sliced = 1;
    M.ragged = 16 * n_ragged > (unsigned long long)((M.nrows + 31) / 32);   // more than 1 slice in 16
    return 0;
}

template <class Src, class Fin>
static int build_transpose(cgo_ctx *c, const Src &src, const Fin &fin, int64_t nT, CsrMat &AT) {
    cudaStream_t s = c->stream;
    unsigned long long *counts = nullptr, *cursor = nullptr;
    int64_t *perm = nullptr;
    void *tmp = nullptr;
    int rc = 0;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&counts, sizeof(unsigned long long) * (size_t)(nT + 1)));
        CGO_CUDA(cudaMemsetAsync(counts, 0, sizeof(unsigned long long) * (size_t)(nT + 1), s));
        if (src.total > 0) k_tr_count<<<grid_for(src.total, c->sms), 256, 0, s>>>(src, counts);
        CGO_CUDA(cudaGetLastError());
        AT.nrows = nT;
        CGO_CUDA(cudaMalloc(&AT.rowptr, sizeof(int64_t) * (size_t)(nT + 1 + CSR_PAD)));
        size_t tmp_bytes = 0;
        CGO_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (const int64_t *)counts, AT.rowptr, nT + 1, s));
        CGO_CUDA(cudaMalloc(&tmp, tmp_bytes > 0 ? tmp_bytes : 1));
        CGO_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, (const int64_t *)counts, AT.rowptr, nT + 1, s));
        int64_t nnzT = 0;
        CGO_CUDA(cudaMemcpyAsync(&nnzT, AT.rowptr + nT, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        CGO_CUDA(cudaStreamSynchronize(s));
        AT.nnz = nnzT;
        cudaFree(counts); counts = nullptr;
        cudaFree(tmp); tmp = nullptr;
        CGO_CUDA(cudaMalloc(&cursor, sizeof(unsigned long long) * (size_t)(nT + 1)));
        CGO_CUDA(cudaMemcpyAsync(cursor, AT.rowptr, sizeof(int64_t) * (size_t)(nT + 1), cudaMemcpyDeviceToDevice, s));
        CGO_CUDA(cudaMalloc(&perm, sizeof(int64_t) * (size_t)(nnzT > 0 ? nnzT : 1)));
        if (src.total > 0) k_tr_fill<<<grid_for(src.total, c->sms), 256, 0, s>>>(src, cursor, perm);
        CGO_CUDA(cudaGetLastError());
        if (nT > 0) k_tr_sort<<<grid_for(nT, c->sms), 256, 0, s>>>(AT.rowptr, nT, perm);
        CGO_CUDA(cudaGetLastError());
        CGO_CUDA(cudaMalloc(&AT.col, sizeof(int32_t) * (size_t)(nnzT + CSR_PAD)));
        CGO_CUDA(cudaMalloc(&AT.val, sizeof(double) * (size_t)(nnzT + CSR_PAD)));
        if (nnzT > 0) k_tr_finalize<<<grid_for(nnzT, c->sms), 256, 0, s>>>(fin, nnzT, perm, AT);
        CGO_CUDA(cudaGetLastError());
        CGO_CUDA(cudaStreamSynchronize(s));
        return 0;
    };
    rc = body();
    cudaFree(counts); cudaFree(cursor); cudaFree(perm); cudaFree(tmp);
    return rc;
}

// ------------------------------------------------------------------ column blocking (setup)
// A gather that ranges over more than about half of the 126 MB L2 (measured cliff: 48 MB still
// hits, 60 MB starts missing) turns every 8-byte gather into a 32-byte DRAM sector read.  For
// such matrices the columns are cut into nb blocks of at most ctx->gather_block_bytes and the
// matrix is stored block-major: blk[j] holds the entries of every row whose column lies in block
// j (rows' columns must ascend, which both logistic-regression matrices do by construction).  One
// k_spmv_direct pass per block keeps its window of the gathered vector L2-resident; passes chain the
// row sums (DirStoreInit), so the arithmetic order is unchanged.
struct CsrBlocked {
    std::vector<CsrMat> blk;
    void free_all() { for (auto &m : blk) csr_free(m); blk.clear(); }
};
__global__ void k_blk_check_sorted(CsrMat A, int *bad) {
    GRID_STRIDE(i, A.nrows) {
        for (int64_t p = A.rowptr[i] + 1; p < A.rowptr[i + 1]; ++p)
            if (A.col[p] < A.col[p - 1]) { *bad = 1; break; }
    }
}
// entries of row i with c0 <= col < c1: first[i] = their start in A, cnt[i] = how many
__global__ void k_blk_count(CsrMat A, int32_t c0, int32_t c1, int64_t *first, int64_t *cnt) {
    GRID_STRIDE(i, A.nrows + 1) {
        if (i == A.nrows) { cnt[i] = 0; continue; }
        const int64_t rs = A.rowptr[i], re = A.rowptr[i + 1];
        int64_t lo = rs, hi = re;                // lower_bound(c0)
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (A.col[mid] < c0) lo = mid + 1; else hi = mid; }
        const int64_t b0 = lo;
        hi = re;                                 // lower_bound(c1)
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (A.col[mid] < c1) lo = mid + 1; else hi = mid; }
        first[i] = b0;
        cnt[i] = lo - b0;
    }
}
__global__ void k_blk_copy(CsrMat A, const int64_t *first, CsrMat B) {
    GRID_STRIDE(i, A.nrows) {
        const int64_t d0 = B.rowptr[i], n = B.rowptr[i + 1] - d0, s0 = first[i];
        for (int64_t e = 0; e < n; ++e) { B.col[d0 + e] = A.col[s0 + e]; B.val[d0 + e] = A.val[s0 + e]; }
    }
}
// `width`: doubles gathered per column (1 for an SpMV, K for the K-column SpMM)
static int build_blocked(cgo_ctx *c, const CsrMat &A, int64_t ncols, int64_t width, CsrBlocked &out) {
    out.free_all();
    const int64_t cap = (int64_t)(c->gather_block_bytes / (sizeof(double) * (size_t)width));
    if (cap <= 0 || ncols <= cap || A.nnz == 0) return 0;
    const int64_t nb = (ncols + cap - 1) / cap;
    const int64_t bc = (((ncols + nb - 1) / nb) + 1) & ~(int64_t)1;
    cudaStream_t s = c->stream;
    int *bad = nullptr;
    int64_t *first = nullptr, *cnt = nullptr;
    void *tmp = nullptr;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&bad, sizeof(int)));
        CGO_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), s));
        k_blk_check_sorted<<<grid_for(A.nrows, c->sms), 256, 0, s>>>(A, bad);
        int hbad = 0;
        CGO_CUDA(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, s));
        CGO_CUDA(cudaStreamSynchronize(s));
        if (hbad) return 0;                      // columns not ascending: stay single-pass
        CGO_CUDA(cudaMalloc(&first, sizeof(int64_t) * (size_t)(A.nrows + 1)));
        CGO_CUDA(cudaMalloc(&cnt, sizeof(int64_t) * (size_t)(A.nrows + 1)));
        size_t tmp_bytes = 0;
        CGO_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, cnt, cnt, A.nrows + 1, s));
        CGO_CUDA(cudaMalloc(&tmp, tmp_bytes > 0 ? tmp_bytes : 1));
        out.blk.resize((size_t)nb);
        for (int64_t j = 0; j < nb; ++j) {
            CsrMat &B = out.blk[(size_t)j];
            const int64_t c0 = j * bc, c1 = (j + 1) * bc < ncols ? (j + 1) * bc : ncols;
            k_blk_count<<<grid_for(A.nrows + 1, c->sms), 256, 0, s>>>(A, (int32_t)c0, (int32_t)c1, first, cnt);
            CGO_CUDA(cudaGetLastError());
            B.nrows = A.nrows;
            CGO_CUDA(cudaMalloc(&B.rowptr, sizeof(int64_t) * (size_t)(A.nrows + 1 + CSR_PAD)));
            CGO_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, cnt, B.rowptr, A.nrows + 1, s));
            int64_t nnzb = 0;
            CGO_CUDA(cudaMemcpyAsync(&nnzb, B.rowptr + A.nrows, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            CGO_CUDA(cudaStreamSynchronize(s));
            B.nnz = nnzb;
            CGO_CUDA(cudaMalloc(&B.col, sizeof(int32_t) * (size_t)(nnzb + CSR_PAD)));
            CGO_CUDA(cudaMalloc(&B.val, sizeof(double) * (size_t)(nnzb + CSR_PAD)));
            k_blk_copy<<<grid_for(A.nrows, c->sms), 256, 0, s>>>(A, first, B);
            CGO_CUDA(cudaGetLastError());
        }
        CGO_CUDA(cudaStreamSynchronize(s));
        return 0;
    };
    int rc = body();
    cudaFree(bad); cudaFree(first); cudaFree(cnt); cudaFree(tmp);
    if (rc) out.free_all();
    return rc;
}
// one k_spmv_direct pass per column block (sliced blocks): every pass just stores the running row sums, the
// epilogue and its reductions are a BLAS-1 kernel of the caller's.  `wait`: flag hand-off that guards the gathered
// vector (first pass)
static int spmv_direct_passes(cgo_ctx *c, const CsrMat &M, const CsrBlocked &B, const double *xg, double *out,
                              const RedArgs *wait, int tclass) {
    if (B.blk.empty()) return launch_direct(c, M, xg, DirStore{out}, dir_args(c, wait), tclass);
    for (size_t j = 0; j < B.blk.size(); ++j) {
        if (j == 0) CGO_TRY(launch_direct(c, B.blk[j], xg, DirStore{out}, dir_args(c, wait), tclass));
        else CGO_TRY(launch_direct(c, B.blk[j], xg, DirStoreInit{out, out}, dir_args(c), tclass));
    }
    return 0;
}
// the same for the K-column SpMM (row-major blocks)
static int spmm_passes(cgo_ctx *c, const CsrMat &M, const CsrBlocked &B, int K, const double *xg, double *out, int tclass) {
    if (B.blk.empty()) return launch_spmm(c, M, K, xg, DirStore{out}, tclass);
    for (size_t j = 0; j < B.blk.size(); ++j) {
        if (j == 0) CGO_TRY(launch_spmm(c, B.blk[j], K, xg, DirStore{out}, tclass));
        else CGO_TRY(launch_spmm(c, B.blk[j], K, xg, DirStoreInit{out, out}, tclass));
    }
    return 0;
}

// ------------------------------------------------------------------ long rows (logistic regression from a host CSR)
// A row with more than CGO_LONG_ROW entries would chain its products on one lane of k_spmv_direct: the ones column
// of an intercept is a row of Aᵀ with N entries.  Such rows are taken out of the matrix the row kernels see (they
// are empty in its sliced copy and in every column block), stored once, unblocked, and summed in the canonical order
// of include/cgoptim.h with V = 1, U = 4.  A work unit is one (long row, virtual CTA) pair with data; k_long_rows
// spreads the units over the whole grid, and each adds its lanes' products and combines its 256 lanes into one
// partial.  k_long_finish, one CTA per long row, combines the row's partials and stores the row sum where the row
// kernel stores the others.
constexpr int LONG_U = 4;                    // items per lane and tile
constexpr int LONG_TILE = CGO_B * LONG_U;
constexpr int LONG_TB = 2;                   // tiles of one unit whose loads are in flight together
struct LongRows {
    int64_t n = 0;                           // long rows
    CsrMat M;                                // the long rows, row-major, entries in storage order
    int64_t *row = nullptr;                  // their indices in the whole matrix (device)
    std::vector<int64_t> h_row, h_rowptr;    // host copies of `row` and M.rowptr
    int G = 0;                               // the G the work units are laid out for
    int width = 1;                           // sums per long row (K for the K-column SpMM)
    // an intercept's unit row (add_unit_row): the last of the n rows, not stored in M, with ulen entries 1.0
    int64_t ulen = 0;
    int64_t nunits = 0;
    int2 *unit = nullptr;                    // (long row, virtual CTA) of every unit
    int64_t *ubase = nullptr;                // first unit of every long row, n + 1
    double *partial = nullptr;               // `width` per unit
    void free_all() {
        csr_free(M);
        cudaFree(row); cudaFree(unit); cudaFree(ubase); cudaFree(partial);
        *this = LongRows();
    }
};

// UNIT: the last long row may be the unit row of an intercept (row index >= L.nrows): a virtual row of Aᵀ whose
// entries are 1.0 at columns 0 … ulen − 1, synthesised instead of stored
template <bool UNIT>
__device__ __forceinline__ void long_rows_body(const CsrMat &L, const int2 *__restrict__ unit, int64_t nunits, int G,
                                               int64_t ulen, const double *__restrict__ xg, double *__restrict__ partial) {
    __shared__ double s_red[CGO_NW];
    const int t = threadIdx.x;
    const uint64_t gpol = l2_policy_evict_last();
    for (int64_t u = blockIdx.x; u < nunits; u += gridDim.x) {
        const int2 w = unit[u];
        const bool urow = UNIT && w.x >= L.nrows;
        const int64_t p0 = urow ? 0 : L.rowptr[w.x], len = urow ? ulen : L.rowptr[w.x + 1] - p0;
        const int64_t ntiles = (len + LONG_TILE - 1) / LONG_TILE;
        double acc[1] = {0.0};
#pragma unroll 1
        for (int64_t tile = w.y; tile < ntiles; tile += (int64_t)LONG_TB * G) {
            // the lane's items of tiles tile, tile + G, …: index order, values and indices coalesced across the lanes
            constexpr int NI = LONG_TB * LONG_U;
            int32_t cj[NI];
            double vj[NI], xj[NI];
            bool on[NI];
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                const int64_t k = (tile + (int64_t)(j / LONG_U) * G) * LONG_TILE + (j % LONG_U) * CGO_B + t;
                on[j] = k < len;
                if (urow) {
                    cj[j] = (int32_t)k;
                    vj[j] = 1.0;
                } else {
                    cj[j] = ld_stream_s32_if(L.col + p0 + k, on[j]);
                    vj[j] = ld_stream_f64_if(L.val + p0 + k, on[j]);
                }
            }
#pragma unroll
            for (int j = 0; j < NI; ++j) xj[j] = ld_gather_f64_if(xg + cj[j], gpol, on[j]);
#pragma unroll
            for (int j = 0; j < NI; ++j) {
                const double p = vj[j] * xj[j];
                if (on[j]) acc[0] = acc[0] + p;
            }
        }
        cgo_cta_combine<1>(acc, s_red);
        if (t == 0) partial[u] = acc[0];
    }
}
__global__ void __launch_bounds__(CGO_B) k_long_rows(CsrMat L, const int2 *__restrict__ unit, int64_t nunits, int G,
                                                     const double *__restrict__ xg, double *__restrict__ partial) {
    long_rows_body<false>(L, unit, nunits, G, 0, xg, partial);
}
__global__ void __launch_bounds__(CGO_B) k_long_rows_unit(CsrMat L, const int2 *__restrict__ unit, int64_t nunits, int G,
                                                          int64_t ulen, const double *__restrict__ xg,
                                                          double *__restrict__ partial) {
    long_rows_body<true>(L, unit, nunits, G, ulen, xg, partial);
}
// one CTA per long row: lane t adds the row's partials t, t + 256, …, then the CTA combine
__global__ void __launch_bounds__(CGO_B) k_long_finish(const int64_t *__restrict__ ubase, const int64_t *__restrict__ row,
                                                       const double *__restrict__ partial, double *out) {
    __shared__ double s_red[CGO_NW];
    const int64_t b = ubase[blockIdx.x], nact = ubase[blockIdx.x + 1] - b;
    double acc[1] = {0.0};
    for (int64_t c = threadIdx.x; c < nact; c += CGO_B) acc[0] = acc[0] + partial[b + c];
    cgo_cta_combine<1>(acc, s_red);
    if (threadIdx.x == 0) out[row[blockIdx.x]] = acc[0];
}

// lay the work units out for the ctx's G (at the first evaluation, and again when G changes)
static int long_units(cgo_ctx *c, LongRows &L) {
    if (L.G == c->G) return 0;
    std::vector<int2> unit;
    std::vector<int64_t> ubase((size_t)L.n + 1, 0);
    for (int64_t r = 0; r < L.n; ++r) {
        const int64_t ntiles = (L.h_rowptr[(size_t)r + 1] - L.h_rowptr[(size_t)r] + LONG_TILE - 1) / LONG_TILE;
        const int64_t nact = ntiles < c->G ? ntiles : c->G;
        for (int64_t v = 0; v < nact; ++v) unit.push_back(make_int2((int)r, (int)v));
        ubase[(size_t)r + 1] = (int64_t)unit.size();
    }
    cudaFree(L.unit); cudaFree(L.partial);
    L.unit = nullptr; L.partial = nullptr; L.G = 0;
    L.nunits = (int64_t)unit.size();
    CGO_CUDA(cudaMalloc(&L.unit, sizeof(int2) * unit.size()));
    CGO_CUDA(cudaMalloc(&L.partial, sizeof(double) * unit.size() * (size_t)L.width));
    CGO_CUDA(cudaMemcpyAsync(L.unit, unit.data(), sizeof(int2) * unit.size(), cudaMemcpyHostToDevice, c->stream));
    CGO_CUDA(cudaMemcpyAsync(L.ubase, ubase.data(), sizeof(int64_t) * ubase.size(), cudaMemcpyHostToDevice, c->stream));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    L.G = c->G;
    return 0;
}
// out[row] = the sum of every long row, after the row kernels' last pass over the same output
static int long_rows_sum(cgo_ctx *c, LongRows &L, const double *xg, double *out, int tclass) {
    if (L.n == 0) return 0;
    CGO_TRY(long_units(c, L));
    const int64_t phys = (int64_t)c->sms * 8;
    const int grid = (int)(L.nunits < phys ? L.nunits : phys);
    cgo_timer_begin(c, tclass);
    if (L.ulen > 0) k_long_rows_unit<<<grid, CGO_B, 0, c->stream>>>(L.M, L.unit, L.nunits, L.G, L.ulen, xg, L.partial);
    else k_long_rows<<<grid, CGO_B, 0, c->stream>>>(L.M, L.unit, L.nunits, L.G, xg, L.partial);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    cgo_timer_begin(c, tclass);
    k_long_finish<<<(unsigned)L.n, CGO_B, 0, c->stream>>>(L.ubase, L.row, L.partial, out);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    return 0;
}

// The long rows of the K-column SpMM: for every class k the items of a long row are val_p · x[col_p·K + k], summed
// exactly as k_long_rows + k_long_finish sum that row of A ⊗ I_K.  The (long row, virtual CTA) units are those of
// the SpMV; k_long_rows_k spreads (unit, tile of LONG_KT classes) over the grid, so each lane reads its entries once
// per class tile and keeps LONG_KT accumulators, and the CTA combine reduces each of them as it reduces one.
// Partials are stored unit-major, K per unit; k_long_finish_k runs one CTA per (long row, class).
constexpr int LONG_KT = 8;
template <bool UNIT>
__device__ __forceinline__ void long_rows_k_body(const CsrMat &L, const int2 *__restrict__ unit, int64_t nunits, int G,
                                                 int K, int64_t ulen, const double *__restrict__ xg,
                                                 double *__restrict__ partial) {
    __shared__ double s_red[LONG_KT * CGO_NW];
    const int t = threadIdx.x;
    const uint64_t gpol = l2_policy_evict_last();
    const int nct = (K + LONG_KT - 1) / LONG_KT;
    for (int64_t wi = blockIdx.x; wi < nunits * nct; wi += gridDim.x) {
        const int64_t u = wi / nct;
        const int k0 = (int)(wi - u * nct) * LONG_KT;
        const int2 w = unit[u];
        const bool urow = UNIT && w.x >= L.nrows;
        const int64_t p0 = urow ? 0 : L.rowptr[w.x], len = urow ? ulen : L.rowptr[w.x + 1] - p0;
        const int64_t ntiles = (len + LONG_TILE - 1) / LONG_TILE;
        double acc[LONG_KT];
#pragma unroll
        for (int kk = 0; kk < LONG_KT; ++kk) acc[kk] = 0.0;
#pragma unroll 1
        for (int64_t tile = w.y; tile < ntiles; tile += G) {
            int32_t cj[LONG_U];
            double vj[LONG_U];
            bool on[LONG_U];
#pragma unroll
            for (int j = 0; j < LONG_U; ++j) {
                const int64_t k = tile * LONG_TILE + j * CGO_B + t;
                on[j] = k < len;
                if (urow) {
                    cj[j] = (int32_t)k;
                    vj[j] = 1.0;
                } else {
                    cj[j] = ld_stream_s32_if(L.col + p0 + k, on[j]);
                    vj[j] = ld_stream_f64_if(L.val + p0 + k, on[j]);
                }
            }
            double xj[LONG_U][LONG_KT];
#pragma unroll
            for (int j = 0; j < LONG_U; ++j)
#pragma unroll
                for (int kk = 0; kk < LONG_KT; ++kk)
                    xj[j][kk] = ld_gather_f64_if(xg + (int64_t)cj[j] * K + k0 + kk, gpol, on[j] && k0 + kk < K);
#pragma unroll
            for (int j = 0; j < LONG_U; ++j)
#pragma unroll
                for (int kk = 0; kk < LONG_KT; ++kk) {
                    const double p = vj[j] * xj[j][kk];
                    if (on[j]) acc[kk] = acc[kk] + p;
                }
        }
        cgo_cta_combine<LONG_KT>(acc, s_red);
        if (t == 0) {
#pragma unroll
            for (int kk = 0; kk < LONG_KT; ++kk)
                if (k0 + kk < K) partial[u * K + k0 + kk] = acc[kk];
        }
    }
}
__global__ void __launch_bounds__(CGO_B) k_long_rows_k(CsrMat L, const int2 *__restrict__ unit, int64_t nunits, int G, int K,
                                                       const double *__restrict__ xg, double *__restrict__ partial) {
    long_rows_k_body<false>(L, unit, nunits, G, K, 0, xg, partial);
}
__global__ void __launch_bounds__(CGO_B) k_long_rows_k_unit(CsrMat L, const int2 *__restrict__ unit, int64_t nunits, int G,
                                                            int K, int64_t ulen, const double *__restrict__ xg,
                                                            double *__restrict__ partial) {
    long_rows_k_body<true>(L, unit, nunits, G, K, ulen, xg, partial);
}
__global__ void __launch_bounds__(CGO_B) k_long_finish_k(const int64_t *__restrict__ ubase, const int64_t *__restrict__ row, int K,
                                                         const double *__restrict__ partial, double *out) {
    __shared__ double s_red[CGO_NW];
    const int k = (int)blockIdx.y;
    const int64_t b = ubase[blockIdx.x], nact = ubase[blockIdx.x + 1] - b;
    double acc[1] = {0.0};
    for (int64_t c = threadIdx.x; c < nact; c += CGO_B) acc[0] = acc[0] + partial[(b + c) * K + k];
    cgo_cta_combine<1>(acc, s_red);
    if (threadIdx.x == 0) out[row[blockIdx.x] * K + k] = acc[0];
}
static int long_rows_sum_k(cgo_ctx *c, LongRows &L, const double *xg, double *out, int tclass) {
    if (L.n == 0) return 0;
    CGO_TRY(long_units(c, L));
    const int K = L.width;
    const int64_t items = L.nunits * ((K + LONG_KT - 1) / LONG_KT), phys = (int64_t)c->sms * 8;
    const int grid = (int)(items < phys ? items : phys);
    cgo_timer_begin(c, tclass);
    if (L.ulen > 0) k_long_rows_k_unit<<<grid, CGO_B, 0, c->stream>>>(L.M, L.unit, L.nunits, L.G, K, L.ulen, xg, L.partial);
    else k_long_rows_k<<<grid, CGO_B, 0, c->stream>>>(L.M, L.unit, L.nunits, L.G, K, xg, L.partial);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    cgo_timer_begin(c, tclass);
    k_long_finish_k<<<dim3((unsigned)L.n, (unsigned)K), CGO_B, 0, c->stream>>>(L.ubase, L.row, K, L.partial, out);
    cgo_timer_end(c);
    c->launches++;
    CGO_CUDA(cudaGetLastError());
    return 0;
}

// set-up: the rows of A longer than CGO_LONG_ROW move to L; A keeps them as empty rows (count + scan + copy)
__global__ void k_strip_count(CsrMat A, int64_t *cnt) {
    GRID_STRIDE(i, A.nrows + 1) {
        const int64_t len = i < A.nrows ? A.rowptr[i + 1] - A.rowptr[i] : 0;
        cnt[i] = len > CGO_LONG_ROW ? 0 : len;
    }
}
__global__ void k_long_copy(CsrMat A, const int64_t *row, CsrMat L) {
    for (int64_t r = blockIdx.x; r < L.nrows; r += gridDim.x) {
        const int64_t s0 = A.rowptr[row[r]], d0 = L.rowptr[r], n = L.rowptr[r + 1] - d0;
        for (int64_t e = threadIdx.x; e < n; e += blockDim.x) { L.col[d0 + e] = A.col[s0 + e]; L.val[d0 + e] = A.val[s0 + e]; }
    }
}
static int split_long_rows(cgo_ctx *c, CsrMat &A, LongRows &L) {
    cudaStream_t s = c->stream;
    std::vector<int64_t> rp((size_t)A.nrows + 1);
    CGO_CUDA(cudaMemcpyAsync(rp.data(), A.rowptr, sizeof(int64_t) * rp.size(), cudaMemcpyDeviceToHost, s));
    CGO_CUDA(cudaStreamSynchronize(s));
    L.h_rowptr.assign(1, 0);
    for (int64_t i = 0; i < A.nrows; ++i) {
        const int64_t len = rp[(size_t)i + 1] - rp[(size_t)i];
        if (len <= CGO_LONG_ROW) continue;
        L.h_row.push_back(i);
        L.h_rowptr.push_back(L.h_rowptr.back() + len);
    }
    L.n = (int64_t)L.h_row.size();
    if (L.n == 0) return 0;
    CsrMat S;
    int64_t *cnt = nullptr;
    void *tmp = nullptr;
    auto body = [&]() -> int {
        CGO_TRY(csr_alloc(L.M, L.n, L.h_rowptr.back()));
        CGO_CUDA(cudaMalloc(&L.row, sizeof(int64_t) * (size_t)L.n));
        CGO_CUDA(cudaMalloc(&L.ubase, sizeof(int64_t) * (size_t)(L.n + 1)));
        CGO_CUDA(cudaMemcpyAsync(L.M.rowptr, L.h_rowptr.data(), sizeof(int64_t) * (size_t)(L.n + 1), cudaMemcpyHostToDevice, s));
        CGO_CUDA(cudaMemcpyAsync(L.row, L.h_row.data(), sizeof(int64_t) * (size_t)L.n, cudaMemcpyHostToDevice, s));
        k_long_copy<<<(unsigned)(L.n < (int64_t)c->sms * 4 ? L.n : (int64_t)c->sms * 4), 256, 0, s>>>(A, L.row, L.M);
        CGO_CUDA(cudaGetLastError());
        CGO_CUDA(cudaMalloc(&cnt, sizeof(int64_t) * (size_t)(A.nrows + 1)));
        k_strip_count<<<grid_for(A.nrows + 1, c->sms), 256, 0, s>>>(A, cnt);
        CGO_CUDA(cudaGetLastError());
        S.nrows = A.nrows;
        CGO_CUDA(cudaMalloc(&S.rowptr, sizeof(int64_t) * (size_t)(A.nrows + 1 + CSR_PAD)));
        size_t tmp_bytes = 0;
        CGO_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, cnt, S.rowptr, A.nrows + 1, s));
        CGO_CUDA(cudaMalloc(&tmp, tmp_bytes > 0 ? tmp_bytes : 1));
        CGO_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, cnt, S.rowptr, A.nrows + 1, s));
        CGO_CUDA(cudaMemcpyAsync(&S.nnz, S.rowptr + A.nrows, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        CGO_CUDA(cudaStreamSynchronize(s));
        CGO_CUDA(cudaMalloc(&S.col, sizeof(int32_t) * (size_t)(S.nnz + CSR_PAD)));
        CGO_CUDA(cudaMalloc(&S.val, sizeof(double) * (size_t)(S.nnz + CSR_PAD)));
        k_blk_copy<<<grid_for(A.nrows, c->sms), 256, 0, s>>>(A, A.rowptr, S);
        CGO_CUDA(cudaGetLastError());
        CGO_CUDA(cudaStreamSynchronize(s));
        return 0;
    };
    const int rc = body();
    cudaFree(cnt); cudaFree(tmp);
    if (rc) { csr_free(S); return rc; }
    csr_free(A);
    A = S;
    return 0;
}
// an intercept: its gradient is the sum of a row of Aᵀ that is not stored, 1.0 at every sample.  It joins L as one
// more long row, stored at index `row` of the output, so the intercept adds work units, not launches
static int add_unit_row(cgo_ctx *c, LongRows &L, int64_t row, int64_t len) {
    L.h_row.push_back(row);
    L.h_rowptr.push_back(L.h_rowptr.back() + len);
    L.n = (int64_t)L.h_row.size();
    L.ulen = len;
    cudaFree(L.row); cudaFree(L.ubase);
    L.row = nullptr; L.ubase = nullptr;
    CGO_CUDA(cudaMalloc(&L.row, sizeof(int64_t) * (size_t)L.n));
    CGO_CUDA(cudaMalloc(&L.ubase, sizeof(int64_t) * (size_t)(L.n + 1)));
    CGO_CUDA(cudaMemcpyAsync(L.row, L.h_row.data(), sizeof(int64_t) * (size_t)L.n, cudaMemcpyHostToDevice, c->stream));
    CGO_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------ the objective
struct CsrObj : cgo_obj {
    bool logreg = false;
    // classes of the softmax objective (logreg also true): the state vector is W (d × K, feature-major), Z = A W and
    // C = P − Y live in `r` (N × K, row-major), and every product with A or Aᵀ is the K-column SpMM.  1 otherwise
    int32_t nclass = 1;
    // the SpMV kernel family of every evaluation, fixed at creation.  false: the fused k_csr_rows, whose epilogues
    // reduce the dots (reduction site V = 1, U = 1).  true: k_spmv_direct on the sliced layout, the dots are
    // BLAS-1 passes (V = 2, U = CGO_U_VEC).  Least squares: A.sliced after set-up; logistic regression: also when
    // column-blocked or sharded.
    bool direct = false;
    CsrMat A, AT;
    CsrBlocked Ab, ATb;                // column-blocked copies (logreg on k_spmv_direct, large gather ranges)
    LongRows LA, LAT;                  // rows taken out of A / AT (logreg from a host CSR on k_spmv_direct)
    bool have_unblocked = true;        // A / AT arrays still allocated (test hooks need them)
    int64_t nrows = 0;                 // local rows of A (residuals / samples)
    double *b = nullptr;               // rhs (LS) or labels (logreg), nrows
    double *r_base = nullptr, *r = nullptr;   // residual / c vector with halo
    double *qv = nullptr;                     // v = A u of the quadratic-aware line search (nrows)
    // whose residual `r` holds: every trial leaves r(xp) of its state; cgo_accept makes that r(x); the
    // Hessian-vector product and trials of OTHER states on the same objective overwrite it
    const cgo_state *r_state = nullptr;
    bool r_at_xp = false, r_at_x = false;
    int quad_steps = 0;                       // accepted steps since r was last formed as A x − b
    std::vector<void *> rpeers;               // peer mappings of r_base (sharded LS with peer memory)
    bool r_is_peer = false;
    double lambda = 0.0;
    int64_t nsamples = 0;
    // logistic and softmax regression: S, the sum of the sample weights (nsamples without weights); the weights
    // (nullptr: unit weights, nsamples + CSR_PAD); fit_intercept: the last nclass coordinates of the state are the
    // intercept, which λ does not penalise (k_spmv_direct / the SpMM only)
    double wsum = 0.0;
    double *wt = nullptr;
    bool icpt = false;
    bool glm() const { return wt != nullptr || icpt; }
    int64_t npen() const { return icpt ? n_local - nclass : n_local; }
    // sharded logistic regression (nranks > 1): samples AND features are sharded.  A holds this rank's samples ×
    // all features and gathers the all-gathered trial point; AT holds this rank's FEATURES × all samples (built
    // straight from the generator) and gathers the all-gathered c, so every row of Aᵀc is added over all samples in
    // the single-GPU order.  The state vectors are feature shards [flo[rank], flo[rank+1]).
    bool lr_sharded = false;
    std::vector<int64_t> flo, slo;     // feature / sample shard boundaries, nranks + 1
    double *xp_full = nullptr;         // all-gathered trial point, n_global
    double *c_full = nullptr;          // all-gathered c = −y σ, nsamples
    // peer-memory variant: xp_full and c_full are mapped by every rank
    bool lr_peer = false;
    std::vector<void *> xpf_peers, cf_peers;
    void **d_xpf_dst = nullptr;        // rank r's xp_full + flo[me]
    void **d_cf_dst = nullptr;         // rank r's c_full + slo[me]
    ~CsrObj() override {
        if (ctx && cgo_ctx_alive(ctx)) cudaSetDevice(ctx->device);
        csr_free(A); csr_free(AT);
        Ab.free_all(); ATb.free_all();
        LA.free_all(); LAT.free_all();
        if (r_is_peer) { cgo_peer_free(ctx, r_base, rpeers, true); r_base = nullptr; }
        if (lr_peer) {
            cgo_peer_free(ctx, xp_full, xpf_peers, true); xp_full = nullptr;
            cgo_peer_free(ctx, c_full, cf_peers, true); c_full = nullptr;
        }
        cudaFree(d_xpf_dst); cudaFree(d_cf_dst);
        cudaFree(b); cudaFree(wt); cudaFree(r_base); cudaFree(qv);
        cudaFree(xp_full); cudaFree(c_full);
    }
    int alloc_r() {
        size_t bytes = sizeof(double) * (size_t)(nrows * nclass + 2 * halo + 4);
        if (ctx->nranks > 1 && ctx->peer_ok && halo > 0) {
            bytes = sizeof(double) * (size_t)((n_alloc > nrows ? n_alloc : nrows) + 2 * halo + 4);   // rank-independent
            void *p = nullptr;
            r_is_peer = true;
            CGO_TRY(cgo_peer_alloc(ctx, bytes, &p, rpeers));
            r_base = (double *)p;
        } else {
            CGO_CUDA(cudaMalloc(&r_base, bytes));
            CGO_CUDA(cudaMemsetAsync(r_base, 0, bytes, ctx->stream));
        }
        r = r_base + halo;
        return 0;
    }
    // local length of rank q's shard (the vector shards and the row shards coincide for LS)
    int64_t shard_len_of(int q) const {
        int64_t lo, hi;
        cgo_shard_range(n_global, ctx->nranks, q, 2, &lo, &hi);
        return hi - lo;
    }
    // fill v[−halo, 0) and v[nloc, nloc + halo) from the ring neighbours
    int exchange(double *v, int64_t nloc) {
        if (halo == 0) return 0;
        return cgo_sendrecv_ring(ctx, v, v + nloc, v + nloc - halo, v - halo, halo);
    }
    void reduction_site(int32_t *V, int32_t *U) const override {
        if (direct) { *V = 2; *U = CGO_U_VEC; } else { *V = 1; *U = 1; }
    }

    // ---- least squares: one trial = K_a, K_b (residual), K_c (gradient), on either kernel family
    // sharded least squares over peer memory: K_a and K_b push their boundary elements into the ring neighbours'
    // halos and hand off with flags; there is no separate exchange step
    struct PeerLinks {
        HaloPush xp;                            // K_a: xp's boundary elements, flags CGO_F_XP_FROM_*
        double *r_prev_right, *r_next_left;     // K_b: where r's boundary elements go
        RedArgs kb, kc;                         // K_b: waits for xp's halos, signals r's; K_c: waits for r's
    };
    PeerLinks peer_links(cgo_state *st) {
        const int R = ctx->nranks, me = ctx->rank, prev = (me + R - 1) % R, next = (me + 1) % R;
        const unsigned long long e = ++ctx->epoch;
        unsigned long long *fprev = (unsigned long long *)ctx->flags_peer[(size_t)prev];
        unsigned long long *fnext = (unsigned long long *)ctx->flags_peer[(size_t)next];
        const int64_t nprev = shard_len_of(prev);
        PeerLinks pl;
        pl.xp.prev_right = (double *)st->xpeers[st->xp_alloc][(size_t)prev] + halo + nprev;   // prev's xp + its n
        pl.xp.next_left = (double *)st->xpeers[st->xp_alloc][(size_t)next];                    // next's xp − halo
        pl.xp.sig_prev = fprev + CGO_F_XP_FROM_NEXT;                                           // I am prev's next
        pl.xp.sig_next = fnext + CGO_F_XP_FROM_PREV;
        pl.xp.epoch = e;
        pl.r_prev_right = (double *)rpeers[(size_t)prev] + halo + nprev;
        pl.r_next_left = (double *)rpeers[(size_t)next];
        pl.kb = cgo_red_args(ctx, CGO_P_PHI);
        pl.kb.wait0 = ctx->flags_local + CGO_F_XP_FROM_PREV; pl.kb.wait1 = ctx->flags_local + CGO_F_XP_FROM_NEXT;
        pl.kb.wait_val = e;
        pl.kb.sig0 = fprev + CGO_F_R_FROM_NEXT; pl.kb.sig1 = fnext + CGO_F_R_FROM_PREV; pl.kb.sig_val = e;
        pl.kc = cgo_red_args(ctx, CGO_P_DPHI);
        pl.kc.wait0 = ctx->flags_local + CGO_F_R_FROM_PREV; pl.kc.wait1 = ctx->flags_local + CGO_F_R_FROM_NEXT;
        pl.kc.wait_val = e;
        return pl;
    }
    // K_b: r = A x − b, and Σ r² into pack slot CGO_P_PHI when `sumsq` (without it, k_csr_rows still reduces, into
    // the scratch slot; k_spmv_direct runs no BLAS-1 pass).  pl: also push r's boundary elements to the neighbours
    int residual(const double *x, bool sumsq, const PeerLinks *pl) {
        if (direct) {
            if (pl) {
                DirResidual<true> f{b, r, pl->r_prev_right, pl->r_next_left, halo, nrows};
                CGO_TRY(launch_direct(ctx, A, x, f, dir_args(ctx, &pl->kb), CGO_T_SPMV));
            } else {
                CGO_TRY(launch_direct(ctx, A, x, DirResidual<false>{b, r, nullptr, nullptr, 0, nrows}, dir_args(ctx), CGO_T_SPMV));
            }
            return sumsq ? cgo_blas1_sumsq(ctx, r, nrows, CGO_P_PHI) : 0;
        }
        if (pl) {
            EpiResidualT<true> e{b, r, pl->r_prev_right, pl->r_next_left, halo, nrows};
            return launch_csr(ctx, A, x, e, pl->kb, CGO_T_SPMV);
        }
        EpiResidualT<false> e{b, r, nullptr, nullptr, 0, nrows};
        return launch_csr(ctx, A, x, e, cgo_red_args(ctx, sumsq ? CGO_P_PHI : CGO_PACK_LEN - 1), CGO_T_SPMV);
    }
    // K_c: g⁺ = Aᵀ r with dϕ, ‖g⁺‖² and the getβ dots into pack slots CGO_P_DPHI…  pl: wait for r's halos
    int gradient(cgo_state *st, const PeerLinks *pl) {
        if (direct) {
            CGO_TRY(launch_direct(ctx, AT, r, DirGradLS{st->gp}, pl ? dir_args(ctx, &pl->kc) : dir_args(ctx), CGO_T_SPMVT));
            return cgo_blas1_grad_dots(st);
        }
        EpiGrad<false> e{st->gp, st->g, st->u, nullptr, 0.0, 0.0};
        return launch_csr(ctx, AT, r, e, pl ? pl->kc : cgo_red_args(ctx, CGO_P_DPHI), CGO_T_SPMVT);
    }
    int finish_ls(double *out) {
        CGO_TRY(cgo_finish_pack(ctx, 12, out));
        out[CGO_P_PHI] = 0.5 * out[CGO_P_PHI];
        return 0;
    }
    int eval_trial_ls(cgo_state *st, double a, bool fused, double beta, double *out) {
        const bool peer = r_is_peer && st->peer_x;
        PeerLinks links;
        const PeerLinks *pl = nullptr;
        if (peer) { links = peer_links(st); pl = &links; }
        CGO_TRY(cgo_blas1_axpy_dir(st, a, fused, beta, pl ? &pl->xp : nullptr));      // K_a (+ halo push)
        if (!peer) CGO_TRY(exchange(st->xp, st->n));
        CGO_TRY(residual(st->xp, true, pl));                                           // K_b (+ halo push)
        if (!peer) CGO_TRY(exchange(r, nrows));
        CGO_TRY(gradient(st, pl));                                                     // K_c
        return finish_ls(out);
    }
    // ∇²f u = Aᵀ(A u) along the current direction (north_star's Hessian-vector product; the reference
    // engine never calls one, src/engine/optim.jl:83-145).  `r` is scratch here.
    int hessvec_dir(cgo_state *st, double *out) override {
        CGO_CHECK(!logreg, "the Hessian-vector product is implemented for least squares");
        r_state = nullptr; r_at_x = r_at_xp = false;                                      // r is scratch here
        CGO_TRY(cgo_sendrecv_ring(ctx, st->u, st->u + st->n, st->u + st->n - halo, st->u - halo, halo));
        if (direct) {
            CGO_TRY(launch_direct(ctx, A, st->u, DirStore{r}, dir_args(ctx), CGO_T_SPMV));
            CGO_TRY(cgo_blas1_sumsq(ctx, r, nrows, 0));                                   // u·Hu = ‖Au‖²
            CGO_TRY(exchange(r, nrows));
            CGO_TRY(launch_direct(ctx, AT, r, DirStore{st->hv}, dir_args(ctx), CGO_T_SPMVT));
            CGO_TRY(cgo_blas1_dots3(ctx, st->u, st->hv, st->n, 1));                       // u·hv, hv·hv
            return cgo_finish_pack(ctx, 3, out);
        }
        EpiStoreSq e1{r};
        CGO_TRY(launch_csr(ctx, A, st->u, e1, cgo_red_args(ctx, 0), CGO_T_SPMV));
        CGO_TRY(exchange(r, nrows));
        EpiHv e2{st->hv, st->u};
        CGO_TRY(launch_csr(ctx, AT, r, e2, cgo_red_args(ctx, 1), CGO_T_SPMVT));
        return cgo_finish_pack(ctx, 3, out);
    }
    // SURVEY.md §8f N1.  `r` must hold the residual at x: true after state creation and after every
    // accepted step whose last trial was the accepted one (strong-Wolfe / Wolfe searches).
    int quad_begin(cgo_state *st, double *out) override {
        CGO_CHECK(!logreg, "the quadratic-aware line search is for least squares");
        if (!qv) {
            CGO_CUDA(cudaMalloc(&qv, sizeof(double) * (size_t)(nrows + CSR_PAD)));
            CGO_CUDA(cudaMemsetAsync(qv, 0, sizeof(double) * (size_t)(nrows + CSR_PAD), ctx->stream));
        }
        // r must be the residual at THIS state's x.  It is after a trial of this state was accepted; it is not after
        // a Hessian-vector product, after another state used the objective, or — the recursive update r += a v
        // drifts by ≈ ε‖r₀‖ per step — after 64 accepted steps: then r = A x − b is formed again
        if (!(r_state == st && r_at_x) || quad_steps >= 64) {
            CGO_TRY(cgo_sendrecv_ring(ctx, st->x, st->x + st->n, st->x + st->n - halo, st->x - halo, halo));
            CGO_TRY(residual(st->x, false, nullptr));
            r_state = st; r_at_x = true; r_at_xp = false; quad_steps = 0;
        }
        CGO_TRY(cgo_sendrecv_ring(ctx, st->u, st->u + st->n, st->u + st->n - halo, st->u - halo, halo));
        if (direct) {
            CGO_TRY(launch_direct(ctx, A, st->u, DirStore{qv}, dir_args(ctx), CGO_T_SPMV));
            CGO_TRY(cgo_blas1_dots3(ctx, r, qv, nrows, 0));                               // r·v, v·v, r·r
            return cgo_finish_pack(ctx, 3, out);
        }
        EpiQuadV e1{qv, r};
        CGO_TRY(launch_csr(ctx, A, st->u, e1, cgo_red_args(ctx, 0), CGO_T_SPMV));
        return cgo_finish_pack(ctx, 3, out);
    }
    int quad_accept(cgo_state *st, double a, double *out) override {
        CGO_CHECK(!logreg && qv != nullptr, "cgo_quad_accept before cgo_quad_begin");
        CGO_CHECK(r_state == st && r_at_x, "cgo_quad_accept: the residual of this state was overwritten since cgo_quad_begin");
        r_at_x = false; r_at_xp = true; ++quad_steps;                                     // r becomes r(xp) below
        CGO_TRY(cgo_blas1_axpy_dir(st, a, false, 0.0));                                   // xp = x + a u
        CGO_TRY(cgo_blas1_residual_axpy(ctx, r, qv, a, nrows, CGO_P_PHI));                // r += a v, Σ r²
        CGO_TRY(exchange(r, nrows));
        CGO_TRY(gradient(st, nullptr));                                                   // K_c
        return finish_ls(out);
    }

    // ---- logistic regression
    // k_spmv_direct.  One rank: K_a | passes of A → margins | logit + loss (BLAS-1) | passes of Aᵀ | /N + λw + dots
    // (BLAS-1).  R ranks: K_a also stores its shard of xp into every rank's all-gathered copy; the logit kernel stores
    // its shard of c into every rank's all-gathered c; flags hand the data to the consuming passes (without peer
    // memory: two NCCL all-gathers).
    int eval_trial_lr_direct(cgo_state *st, double a, bool fused, double beta, double *out) {
        const int R = ctx->nranks;
        RedArgs wx, wc;                           // flag waits of the first K_b / K_c pass
        const RedArgs *pwx = nullptr, *pwc = nullptr;
        unsigned long long e = 0;
        if (R > 1 && lr_peer) {
            e = ++ctx->epoch;
            HaloPush hp;
            hp.dst_all = d_xpf_dst; hp.epoch = e;
            CGO_TRY(cgo_blas1_axpy_dir(st, a, fused, beta, &hp));                     // K_a + all-gather of xp
            wx.wait_all = ctx->flags_local + CGO_F_XPALL; wx.wait_val = e; wx.nranks = R; pwx = &wx;
            wc.wait_all = ctx->flags_local + CGO_F_CALL; wc.wait_val = e; wc.nranks = R; pwc = &wc;
        } else {
            CGO_TRY(trial_axpy(st, a, fused, beta));                                   // K_a
            if (R > 1) CGO_TRY(cgo_allgatherv_f64(ctx, st->xp, xp_full, flo.data()));
        }
        const double *w_all = R > 1 ? xp_full : st->xp;
        CGO_TRY(spmv_direct_passes(ctx, A, Ab, w_all, r, pwx, CGO_T_SPMV));            // K_b: margins of my samples
        CGO_TRY(long_rows_sum(ctx, LA, w_all, r, CGO_T_SPMV));                           // … of the long rows
        if (glm()) CGO_TRY(cgo_blas1_logit_glm(ctx, r, b, wt, icpt ? st->xp + npen() : nullptr, nrows, CGO_P_PHI));   // c, Σ s ℓ
        else CGO_TRY(cgo_blas1_logit(ctx, r, b, nrows, CGO_P_PHI, (R > 1 && lr_peer) ? d_cf_dst : nullptr, e));   // c, Σ loss [+ all-gather of c]
        if (R > 1 && !lr_peer) CGO_TRY(cgo_allgatherv_f64(ctx, r, c_full, slo.data()));
        const double *c_all = R > 1 ? c_full : r;
        CGO_TRY(spmv_direct_passes(ctx, AT, ATb, c_all, st->gp, pwc, CGO_T_SPMVT));    // K_c: Aᵀc over my features
        CGO_TRY(long_rows_sum(ctx, LAT, c_all, st->gp, CGO_T_SPMVT));                    // … and over the long rows [and Σ c]
        CGO_TRY(grad_combine(st));                                                      // /S + λw, dots
        return finish_lr(out);
    }
    // the fused k_csr_rows, one pass of each matrix (single rank)
    int eval_trial_lr_fused(cgo_state *st, double a, bool fused, double beta, double *out) {
        CGO_TRY(cgo_blas1_axpy_dir(st, a, fused, beta));                                             // K_a
        EpiLogit e1{b, r};
        CGO_TRY(launch_csr(ctx, A, st->xp, e1, cgo_red_args(ctx, CGO_P_PHI), CGO_T_SPMV));            // K_b
        EpiGrad<true> e2{st->gp, st->g, st->u, st->xp, 1.0 / (double)nsamples, lambda};
        CGO_TRY(launch_csr(ctx, AT, r, e2, cgo_red_args(ctx, CGO_P_DPHI), CGO_T_SPMVT));              // K_c
        return finish_lr(out);
    }
    // softmax regression, single rank: K_a | SpMM passes of A → Z | softmax + loss (BLAS-1) | SpMM passes of Aᵀ |
    // /N + λW + dots (BLAS-1)
    int eval_trial_softmax(cgo_state *st, double a, bool fused, double beta, double *out) {
        CGO_TRY(trial_axpy(st, a, fused, beta));                                           // K_a
        CGO_TRY(spmm_passes(ctx, A, Ab, nclass, st->xp, r, CGO_T_SPMV));                    // K_b: Z = A W
        CGO_TRY(long_rows_sum_k(ctx, LA, st->xp, r, CGO_T_SPMV));                           // … of the long rows
        if (glm()) CGO_TRY(cgo_blas1_softmax_glm(ctx, r, b, wt, icpt ? st->xp + npen() : nullptr, nrows, nclass, CGO_P_PHI));
        else CGO_TRY(cgo_blas1_softmax(ctx, r, b, nrows, nclass, CGO_P_PHI));              // C = P − Y, Σ loss
        CGO_TRY(spmm_passes(ctx, AT, ATb, nclass, r, st->gp, CGO_T_SPMVT));                 // K_c: Aᵀ C
        CGO_TRY(long_rows_sum_k(ctx, LAT, r, st->gp, CGO_T_SPMVT));                         // … and over the long rows [and Σ C]
        CGO_TRY(grad_combine(st));                                                          // /S + λW, dots
        return finish_lr(out);
    }
    // K_a; with an intercept P, the penalised part of xp·xp, replaces xp·xp in slot CGO_P_XPXP
    int trial_axpy(cgo_state *st, double a, bool fused, double beta) {
        return icpt ? cgo_blas1_axpy_dir_pen(st, a, fused, beta, npen()) : cgo_blas1_axpy_dir(st, a, fused, beta);
    }
    int grad_combine(cgo_state *st) {
        return icpt ? cgo_blas1_grad_combine_pen(st, 1.0 / wsum, lambda, npen()) : cgo_blas1_grad_combine(st, 1.0 / wsum, lambda);
    }
    int finish_lr(double *out) {
        CGO_TRY(cgo_finish_pack(ctx, 12, out));
        out[CGO_P_PHI] = out[CGO_P_PHI] / wsum + (0.5 * lambda) * out[CGO_P_XPXP];
        return 0;
    }

    void on_accept(cgo_state *st) override {
        r_at_x = (r_state == st) && r_at_xp;
        r_at_xp = false;
        if (r_state != st) r_state = nullptr;
    }
    int eval_trial(cgo_state *st, double a, bool fused, double beta, double *out) override {
        r_state = st; r_at_xp = true; r_at_x = false; quad_steps = 0;        // r = A xp − b (least squares) / c (logreg)
        if (!logreg) return eval_trial_ls(st, a, fused, beta, out);
        if (nclass > 1) return eval_trial_softmax(st, a, fused, beta, out);
        return direct ? eval_trial_lr_direct(st, a, fused, beta, out) : eval_trial_lr_fused(st, a, fused, beta, out);
    }
    // SURVEY.md §8(d): A and Aᵀ streamed once (8 B value + 4 B index per entry + row pointers)
    // plus the vector passes R x,u W xp | gather xp, R b, W r | gather r, W g⁺, R u (,g)
    double bytes_per_eval() const override {
        // weights: the loss op reads s (8N); intercept: its unit row reads c (8N, 8NK), and no matrix bytes
        const double glm_bytes = 8.0 * ((wt ? (double)nrows : 0.0) + (icpt ? (double)nrows * (double)nclass : 0.0));
        if (nclass > 1)         // K_a 24n | A_r + W Z | softmax R Z, y W C | Aᵀ_r + W g⁺ | R g⁺, u, g, w W g⁺  (n = d K)
            return 12.0 * (double)(A.nnz + AT.nnz + LA.M.nnz + LAT.M.nnz) + 8.0 * (double)(A.nrows + 1 + AT.nrows + 1) +
                   8.0 * (3.0 * (double)nrows * (double)nclass + (double)nrows + 11.0 * (double)n_local) + glm_bytes;
        if (logreg && direct)   // K_a 24d_loc | A_r + gather + W z | logit R z, y W c | Aᵀ_f + gather + W q | R q, u, g, w W g⁺
            return 12.0 * (double)(A.nnz + AT.nnz + LA.M.nnz + LAT.M.nnz) + 8.0 * (double)(A.nrows + 1 + AT.nrows + 1) +
                   8.0 * (5.0 * (double)nrows + (ctx->nranks > 1 ? (double)n_global + (double)nsamples : 0.0) + 11.0 * (double)n_local) +
                   glm_bytes;
        // (k_spmv_direct: the dots are separate BLAS-1 passes, R r | R g⁺, g, u instead of the staged u, g)
        return 12.0 * (double)(A.nnz + AT.nnz) + 8.0 * (double)(A.nrows + 1 + AT.nrows + 1) +
               8.0 * (3.0 * (double)nrows + 6.0 * (double)n_local) + (direct ? 8.0 * ((double)nrows + (double)n_local) : 0.0);
    }
    int default_x0(uint64_t, double, double *x0) override {
        for (int64_t i = 0; i < n_local; ++i) x0[i] = 0.0;
        return 0;
    }
};

static int check_i32(int64_t v, const char *what) {
    CGO_CHECK(v < 2147483647LL, "%s = %lld does not fit the int32 column index", what, (long long)v);
    return 0;
}

// a host CSR's arrays (both host-CSR constructors): argument errors name the offending row or entry
static int check_host_csr(int64_t nrows, int64_t ncols, const int64_t *rowptr, const int32_t *col, const double *val) {
    const int64_t nnz = rowptr[nrows];
    CGO_CHECK(nnz == 0 || (col && val), "NULL col/val");
    for (int64_t i = 0; i < nrows; ++i) CGO_CHECK(rowptr[i] <= rowptr[i + 1], "rowptr not monotone at row %lld", (long long)i);
    for (int64_t p = 0; p < nnz; ++p) CGO_CHECK(col[p] >= 0 && col[p] < ncols, "column index out of range at entry %lld", (long long)p);
    return 0;
}

extern "C" int cgo_obj_sparse_ls_create_synthetic(cgo_ctx *ctx, int64_t n, int32_t K, int64_t W,
                                                  uint64_t seed, int32_t coh_log2, cgo_obj **out) {
    CGO_CHECK(ctx && out, "NULL argument");
    const int64_t S = K - 1;
    CGO_CHECK(K >= 1 && n >= 2 && n % 2 == 0, "sparse_ls: need nnz_per_row >= 1 and an even n >= 2");
    CGO_CHECK(S == 0 || (W >= S && n > 2 * W), "sparse_ls: need W >= nnz_per_row-1 and n > 2W (n=%lld, W=%lld)", (long long)n, (long long)W);
    CGO_CHECK(coh_log2 >= 0 && coh_log2 < 31, "sparse_ls: coh_log2 out of range");
    CGO_CUDA(cudaSetDevice(ctx->device));
    int64_t lo, hi, n_alloc = 0;
    CGO_TRY(cgo_shard_range(n, ctx->nranks, ctx->rank, 2, &lo, &hi));
    for (int q = 0; q < ctx->nranks; ++q) {
        int64_t a, b;
        CGO_TRY(cgo_shard_range(n, ctx->nranks, q, 2, &a, &b));
        if (b - a > n_alloc) n_alloc = b - a;
    }
    const bool multi = ctx->nranks > 1;
    if (multi) {
        CGO_CHECK(hi - lo >= W && hi - lo + 2 * W <= n, "sparse_ls: shard of %lld rows needs W <= rows and rows + 2W <= n (W=%lld, n=%lld)",
                  (long long)(hi - lo), (long long)W, (long long)n);
        CGO_CHECK(W % 2 == 0, "sparse_ls: W must be even with more than one rank");
    }
    CsrObj *o = new CsrObj();          // (nothing below returns without deleting it)
    o->ctx = ctx; o->n_global = n;
    o->offset = lo; o->n_local = hi - lo; o->nrows = hi - lo; o->n_alloc = n_alloc;
    o->halo = multi ? W : 0;
    LsSpec sp;
    sp.n = n; sp.K = K; sp.coh = coh_log2; sp.W = W; sp.w = S > 0 ? (2 * W) / S : 0; sp.seed = seed;
    const int64_t nloc = o->n_local, nnz = nloc * K;
    double *xt_base = nullptr;
    auto body = [&]() -> int {
        CGO_TRY(check_i32(nloc + 2 * o->halo, "local dimension + halo"));
        CGO_TRY(csr_alloc(o->A, nloc, nnz));
        k_ls_fill_A<<<grid_for(nnz, ctx->sms), 256, 0, ctx->stream>>>(sp, lo, nloc, multi, o->A);
        CGO_CUDA(cudaGetLastError());
        // b = A x_true
        CGO_CUDA(cudaMalloc(&xt_base, sizeof(double) * (size_t)(nloc + 2 * o->halo)));
        k_ls_xtrue<<<grid_for(nloc + 2 * o->halo, ctx->sms), 256, 0, ctx->stream>>>(sp, lo, nloc, o->halo, xt_base + o->halo);
        CGO_CUDA(cudaGetLastError());
        CGO_CUDA(cudaMalloc(&o->b, sizeof(double) * (size_t)(nloc + CSR_PAD)));
        EpiStore es{o->b};
        CGO_TRY(launch_csr(ctx, o->A, xt_base + o->halo, es, cgo_red_args(ctx, CGO_PACK_LEN - 1), CGO_T_OTHER));
        CGO_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaFree(xt_base); xt_base = nullptr;
        CGO_TRY(o->alloc_r());
        if (multi) {
            LsExtSrc src{sp, lo, hi, (nloc + 2 * W) * K};
            LsExtFin fin{sp, lo};
            CGO_TRY(build_transpose(ctx, src, fin, nloc, o->AT));
        } else {
            CsrSrc src{o->A.col, nnz};
            FixedKFin fin{K, o->A.val};
            CGO_TRY(build_transpose(ctx, src, fin, nloc, o->AT));
        }
        // offsets redrawn at least every 8 rows: no two lanes of a warp-level gather share a line ⇒ gather-bound
        // (the rule is part of the canonical order: include/cgoptim.h; CGO_CSR_MODE = 1 / 2 forces never / always)
        if (ctx->csr_mode == 2 || (ctx->csr_mode == 0 && coh_log2 < 4 && K > 1)) {
            CGO_TRY(csr_make_sliced(ctx, o->A));
            CGO_TRY(csr_make_sliced(ctx, o->AT));
        }
        o->direct = o->A.sliced != 0;          // (not sliced without entries)
        return 0;
    };
    int rc = body();
    cudaFree(xt_base);
    if (rc) { delete o; return rc; }
    *out = o;
    return 0;
}

extern "C" int cgo_obj_sparse_ls_create_csr(cgo_ctx *ctx, int64_t nrows, int64_t ncols, const int64_t *rowptr,
                                            const int32_t *col, const double *val, const double *b,
                                            cgo_obj **out) {
    CGO_CHECK(ctx && rowptr && b && out, "NULL argument");
    CGO_CHECK(ctx->nranks == 1, "cgo_obj_sparse_ls_create_csr is single-GPU");
    CGO_CHECK(nrows >= 1 && ncols >= 1, "empty matrix");
    CGO_TRY(check_host_csr(nrows, ncols, rowptr, col, val));
    const int64_t nnz = rowptr[nrows];
    CGO_CUDA(cudaSetDevice(ctx->device));
    CsrObj *o = new CsrObj();
    o->ctx = ctx; o->n_global = ncols; o->n_local = ncols; o->offset = 0; o->nrows = nrows; o->halo = 0;
    auto body = [&]() -> int {
        CGO_TRY(check_i32(nrows > ncols ? nrows : ncols, "matrix dimension"));
        CGO_TRY(csr_alloc(o->A, nrows, nnz));
        cudaStream_t s = ctx->stream;
        CGO_CUDA(cudaMemcpyAsync(o->A.rowptr, rowptr, sizeof(int64_t) * (size_t)(nrows + 1), cudaMemcpyHostToDevice, s));
        if (nnz) {
            CGO_CUDA(cudaMemcpyAsync(o->A.col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, s));
            CGO_CUDA(cudaMemcpyAsync(o->A.val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, s));
        }
        CGO_CUDA(cudaMalloc(&o->b, sizeof(double) * (size_t)(nrows + CSR_PAD)));
        CGO_CUDA(cudaMemcpyAsync(o->b, b, sizeof(double) * (size_t)nrows, cudaMemcpyHostToDevice, s));
        CGO_TRY(o->alloc_r());
        CsrSrc src{o->A.col, nnz};
        CsrFin fin{o->A.rowptr, nrows, o->A.val};
        CGO_TRY(build_transpose(ctx, src, fin, ncols, o->AT));
        float la = 1.f, lt = 1.f;
        CGO_TRY(csr_gather_lines(ctx, o->A, &la));
        CGO_TRY(csr_gather_lines(ctx, o->AT, &lt));
        if (ctx->csr_mode == 2 || (ctx->csr_mode == 0 && la > 4.0f && lt > 4.0f && nrows >= 4096)) {
            CGO_TRY(csr_make_sliced(ctx, o->A));
            CGO_TRY(csr_make_sliced(ctx, o->AT));
        }
        o->direct = o->A.sliced != 0;          // (not sliced without entries)
        return 0;
    };
    int rc = body();
    if (rc) { delete o; return rc; }
    *out = o;
    return 0;
}

// rows [flo, fhi) of Aᵀ over ALL samples, straight from the generator (sharded logistic regression): feature c
// lies in stratum c / w, so only the entries k of the strata that overlap the shard have to be looked at
struct LrFeatSrc {
    LrSpec s;
    int64_t flo, fhi, total;        // total = N * nk candidates
    int32_t k0, nk;
    __device__ __forceinline__ bool get(int64_t e, int64_t &trow, int64_t &key) const {
        const int64_t i = e / nk;
        const int k = k0 + (int)(e - i * nk);
        int64_t c; double v;
        s.entry(i, k, c, v);
        if (c < flo || c >= fhi) return false;
        trow = c - flo; key = i * s.K + k;
        return true;
    }
};
struct LrFeatFin {                  // key = global entry index of the generator; column = global sample index
    LrSpec s;
    __device__ __forceinline__ void get(int64_t key, int32_t &srow, double &v) const {
        const int64_t i = key / s.K;
        int64_t c;
        s.entry(i, (int)(key - i * s.K), c, v);
        srow = (int32_t)i;
    }
};

// column blocks, kernel family and layout of a logistic regression's A (samples × all features) and Aᵀ (both
// constructors).  `long_rows`: rows were taken out of A or Aᵀ (split_long_rows), which only k_spmv_direct adds back;
// also set for weights or an intercept, which only the k_spmv_direct trial applies.
static int lr_layout(cgo_ctx *ctx, CsrObj *o, bool long_rows) {
    const int R = ctx->nranks;
    // K_b gathers over all d features, K_c over all N samples.  Column blocks are k_spmv_direct passes: the
    // forced k_csr_rows (CGO_CSR_MODE=1) runs single-pass whatever the gather range
    if (ctx->csr_mode != 1) {
        CGO_TRY(build_blocked(ctx, o->A, o->n_global - (o->icpt ? 1 : 0), 1, o->Ab));
        CGO_TRY(build_blocked(ctx, o->AT, o->nsamples, 1, o->ATb));
    }
    const bool blocked = !o->Ab.blk.empty() || !o->ATb.blk.empty();
    if (blocked && o->A.nnz > (int64_t)200000000 / R) {
        // production sizes: drop the single-pass copies (only the CSR test hooks read them)
        if (!o->Ab.blk.empty()) { cudaFree(o->A.col); cudaFree(o->A.val); o->A.col = nullptr; o->A.val = nullptr; }
        if (!o->ATb.blk.empty()) { cudaFree(o->AT.col); cudaFree(o->AT.val); o->AT.col = nullptr; o->AT.val = nullptr; }
        o->have_unblocked = false;
    }
    // uniformly random columns: gather-bound (k_spmv_direct + BLAS-1 epilogues) whenever the gathers are what
    // costs — column-blocked sizes, and always when sharded
    o->direct = ctx->csr_mode != 1 && (R > 1 || blocked || ctx->csr_mode == 2 || long_rows);
    if (o->direct) {
        if (o->Ab.blk.empty()) CGO_TRY(csr_make_sliced(ctx, o->A));
        if (o->ATb.blk.empty()) CGO_TRY(csr_make_sliced(ctx, o->AT));
        for (auto &m : o->Ab.blk) CGO_TRY(csr_make_sliced(ctx, m));
        for (auto &m : o->ATb.blk) CGO_TRY(csr_make_sliced(ctx, m));
        // a matrix left without entries (every row long) has nothing to reorder: its empty rows are stored as zeros
        if (o->A.nnz == 0) o->A.sliced = 1;
        if (o->AT.nnz == 0) o->AT.sliced = 1;
    }
    return 0;
}

extern "C" int cgo_obj_logreg_create_synthetic(cgo_ctx *ctx, int64_t N, int64_t d, int32_t K, uint64_t seed,
                                               double lambda, cgo_obj **out) {
    CGO_CHECK(ctx && out, "NULL argument");
    CGO_CHECK(K >= 1 && N >= 1 && d >= K, "logreg: need nnz_per_row >= 1, nsamples >= 1, nfeat >= nnz_per_row");
    const int R = ctx->nranks, me = ctx->rank;
    CGO_CHECK(R == 1 || (N >= 2 * R && d >= 2 * R), "logreg: %d ranks need nsamples >= %d and nfeat >= %d", R, 2 * R, 2 * R);
    CGO_CHECK(R == 1 || ctx->csr_mode != 1, "logreg: the sharded objective runs on k_spmv_direct (CGO_CSR_MODE=1 forbids it)");
    CGO_CUDA(cudaSetDevice(ctx->device));
    CsrObj *o = new CsrObj();
    o->ctx = ctx; o->logreg = true; o->lambda = lambda; o->nsamples = N; o->wsum = (double)N;
    o->n_global = d; o->halo = 0;
    LrSpec sp;
    sp.N = N; sp.d = d; sp.K = K; sp.w = d / K; sp.seed = seed;
    auto body = [&]() -> int {
        // samples (rows of A) and features (state vectors, rows of Aᵀ) are both sharded contiguously
        o->flo.assign(R + 1, 0); o->slo.assign(R + 1, 0);
        for (int r = 0; r < R; ++r) {
            int64_t lo, hi;
            CGO_TRY(cgo_shard_range(d, R, r, 2, &lo, &hi));
            o->flo[r] = lo; o->flo[r + 1] = hi;
            CGO_TRY(cgo_shard_range(N, R, r, 2, &lo, &hi));
            o->slo[r] = lo; o->slo[r + 1] = hi;
        }
        const int64_t slo = o->slo[me], nloc = o->slo[me + 1] - o->slo[me];
        o->offset = o->flo[me]; o->n_local = o->flo[me + 1] - o->flo[me];
        o->nrows = nloc;
        o->lr_sharded = R > 1;
        CGO_TRY(check_i32(N > d ? N : d, "matrix dimension"));
        CGO_TRY(csr_alloc(o->A, nloc, nloc * K));
        CGO_CUDA(cudaMalloc(&o->b, sizeof(double) * (size_t)(nloc + CSR_PAD)));
        CGO_CUDA(cudaMemsetAsync(o->b, 0, sizeof(double) * (size_t)(nloc + CSR_PAD), ctx->stream));
        k_lr_fill_A<<<grid_for(nloc, ctx->sms), 256, 0, ctx->stream>>>(sp, slo, nloc, o->A, o->b);
        CGO_CUDA(cudaGetLastError());
        CGO_TRY(o->alloc_r());
        if (R == 1) {
            CsrSrc src{o->A.col, nloc * K};
            FixedKFin fin{K, o->A.val};
            CGO_TRY(build_transpose(ctx, src, fin, d, o->AT));
        } else {
            const int64_t flo = o->flo[me], fhi = o->flo[me + 1];
            int64_t k0 = flo / sp.w, k1 = (fhi - 1) / sp.w;
            if (k0 > K - 1) k0 = K - 1;
            if (k1 > K - 1) k1 = K - 1;
            LrFeatSrc src{sp, flo, fhi, N * (k1 - k0 + 1), (int32_t)k0, (int32_t)(k1 - k0 + 1)};
            LrFeatFin fin{sp};
            CGO_TRY(build_transpose(ctx, src, fin, fhi - flo, o->AT));
        }
        CGO_TRY(lr_layout(ctx, o, false));
        if (o->lr_sharded) {
            const size_t xb = sizeof(double) * (size_t)(d + CSR_PAD), cb = sizeof(double) * (size_t)(N + CSR_PAD);
            if (ctx->peer_ok) {
                void *p = nullptr;
                o->lr_peer = true;
                CGO_TRY(cgo_peer_alloc(ctx, xb, &p, o->xpf_peers));
                o->xp_full = (double *)p;
                CGO_TRY(cgo_peer_alloc(ctx, cb, &p, o->cf_peers));
                o->c_full = (double *)p;
                std::vector<void *> xd((size_t)R), cd((size_t)R);
                for (int r = 0; r < R; ++r) {
                    xd[(size_t)r] = (double *)o->xpf_peers[(size_t)r] + o->flo[(size_t)me];
                    cd[(size_t)r] = (double *)o->cf_peers[(size_t)r] + o->slo[(size_t)me];
                }
                CGO_CUDA(cudaMalloc(&o->d_xpf_dst, sizeof(void *) * (size_t)R));
                CGO_CUDA(cudaMalloc(&o->d_cf_dst, sizeof(void *) * (size_t)R));
                CGO_CUDA(cudaMemcpy(o->d_xpf_dst, xd.data(), sizeof(void *) * (size_t)R, cudaMemcpyHostToDevice));
                CGO_CUDA(cudaMemcpy(o->d_cf_dst, cd.data(), sizeof(void *) * (size_t)R, cudaMemcpyHostToDevice));
            } else {
                CGO_CUDA(cudaMalloc(&o->xp_full, xb));
                CGO_CUDA(cudaMalloc(&o->c_full, cb));
                CGO_CUDA(cudaMemsetAsync(o->xp_full, 0, xb, ctx->stream));
                CGO_CUDA(cudaMemsetAsync(o->c_full, 0, cb, ctx->stream));
            }
            CGO_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        return 0;
    };
    int rc = body();
    if (rc) { delete o; return rc; }
    *out = o;
    return 0;
}

// the correctly rounded sum of x[0 … n) (Shewchuk's exact partials, rounded as Python's math.fsum rounds them)
static double exact_sum(const double *x, int64_t n) {
    std::vector<double> part;
    for (int64_t k = 0; k < n; ++k) {
        double v = x[k];
        size_t i = 0;
        for (double y : part) {
            if (std::fabs(v) < std::fabs(y)) std::swap(v, y);
            const double hi = v + y, lo = y - (hi - v);
            if (lo != 0.0) part[i++] = lo;
            v = hi;
        }
        part.resize(i);
        part.push_back(v);
    }
    size_t m = part.size();
    if (m == 0) return 0.0;
    double hi = part[--m], lo = 0.0;
    while (m > 0) {
        const double v = hi, y = part[--m];
        hi = v + y;
        lo = y - (hi - v);
        if (lo != 0.0) break;
    }
    if (m > 0 && ((lo < 0.0 && part[m - 1] < 0.0) || (lo > 0.0 && part[m - 1] > 0.0))) {
        const double y = lo * 2.0, v = hi + y;
        if (y == v - hi) hi = v;
    }
    return hi;
}

// weights and intercept of the logistic and softmax objectives: argument errors name the offending sample or value.
// S = Σ s_i, correctly rounded (N without weights)
static int check_glm(cgo_ctx *ctx, const char *who, int64_t N, int64_t d, const double *w, int32_t fit_intercept, double *S) {
    CGO_CHECK(fit_intercept == 0 || fit_intercept == 1, "%s: fit_intercept = %d must be 0 or 1", who, (int)fit_intercept);
    *S = (double)N;
    if (!w && !fit_intercept) return 0;
    CGO_CHECK(ctx->csr_mode != 1, "%s: weights and the intercept run on k_spmv_direct (CGO_CSR_MODE=1 forbids them)", who);
    if (fit_intercept) CGO_TRY(check_i32(d + 1, "nfeat + 1 (the intercept's feature)"));
    if (!w) return 0;
    for (int64_t i = 0; i < N; ++i)
        CGO_CHECK(std::isfinite(w[i]) && w[i] >= 0.0, "%s: sample_weight %g of sample %lld must be finite and >= 0", who, w[i],
                  (long long)i);
    *S = exact_sum(w, N);
    CGO_CHECK(std::isfinite(*S) && *S > 0.0, "%s: the sample weights add up to %g; their sum must be finite and > 0", who, *S);
    return 0;
}
// weights on the device, padded for the double2 loads of the loss ops
static int upload_weights(cgo_ctx *ctx, CsrObj *o, const double *w, int64_t N) {
    if (!w) return 0;
    CGO_CUDA(cudaMalloc(&o->wt, sizeof(double) * (size_t)(N + CSR_PAD)));
    CGO_CUDA(cudaMemsetAsync(o->wt, 0, sizeof(double) * (size_t)(N + CSR_PAD), ctx->stream));
    CGO_CUDA(cudaMemcpyAsync(o->wt, w, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

extern "C" int cgo_obj_logreg_create_csr_ex(cgo_ctx *ctx, int64_t N, int64_t d, const int64_t *rowptr, const int32_t *col,
                                            const double *val, const double *y, const double *sample_weight,
                                            int32_t fit_intercept, double lambda, cgo_obj **out) {
    CGO_CHECK(ctx && rowptr && y && out, "NULL argument");
    CGO_CHECK(ctx->nranks == 1, "cgo_obj_logreg_create_csr is single-GPU");
    CGO_CHECK(N >= 1 && d >= 1, "logreg: need nsamples >= 1 and nfeat >= 1 (nsamples=%lld, nfeat=%lld)", (long long)N, (long long)d);
    CGO_TRY(check_i32(N, "nsamples"));
    CGO_TRY(check_i32(d, "nfeat"));
    CGO_CHECK(rowptr[0] == 0, "rowptr[0] = %lld: row pointers are 0-based", (long long)rowptr[0]);
    CGO_TRY(check_host_csr(N, d, rowptr, col, val));
    for (int64_t i = 0; i < N; ++i) CGO_CHECK(y[i] == 1.0 || y[i] == -1.0, "label %g of sample %lld is not +1 or -1", y[i], (long long)i);
    CGO_CHECK(std::isfinite(lambda) && lambda >= 0.0, "logreg: lambda = %g must be finite and >= 0", lambda);
    double S;
    CGO_TRY(check_glm(ctx, "logreg", N, d, sample_weight, fit_intercept, &S));
    CGO_CUDA(cudaSetDevice(ctx->device));
    const int64_t nnz = rowptr[N], n = d + fit_intercept;
    CsrObj *o = new CsrObj();
    o->ctx = ctx; o->logreg = true; o->lambda = lambda; o->nsamples = N; o->wsum = S; o->icpt = fit_intercept == 1;
    o->n_global = n; o->n_local = n; o->offset = 0; o->nrows = N; o->halo = 0;
    auto body = [&]() -> int {
        cudaStream_t s = ctx->stream;
        CGO_TRY(csr_alloc(o->A, N, nnz));
        CGO_CUDA(cudaMemcpyAsync(o->A.rowptr, rowptr, sizeof(int64_t) * (size_t)(N + 1), cudaMemcpyHostToDevice, s));
        if (nnz) {
            CGO_CUDA(cudaMemcpyAsync(o->A.col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, s));
            CGO_CUDA(cudaMemcpyAsync(o->A.val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, s));
        }
        CGO_CUDA(cudaMalloc(&o->b, sizeof(double) * (size_t)(N + CSR_PAD)));
        CGO_CUDA(cudaMemsetAsync(o->b, 0, sizeof(double) * (size_t)(N + CSR_PAD), s));
        CGO_CUDA(cudaMemcpyAsync(o->b, y, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, s));
        CGO_TRY(upload_weights(ctx, o, sample_weight, N));
        CGO_TRY(o->alloc_r());
        CsrSrc src{o->A.col, nnz};
        CsrFin fin{o->A.rowptr, N, o->A.val};
        CGO_TRY(build_transpose(ctx, src, fin, d, o->AT));
        if (ctx->csr_mode != 1) {            // k_csr_rows keeps every row (sequential sums)
            CGO_TRY(split_long_rows(ctx, o->A, o->LA));
            CGO_TRY(split_long_rows(ctx, o->AT, o->LAT));
        }
        if (o->icpt) CGO_TRY(add_unit_row(ctx, o->LAT, d, N));
        return lr_layout(ctx, o, o->LA.n > 0 || o->LAT.n > 0 || o->glm());
    };
    int rc = body();
    if (rc) { delete o; return rc; }
    *out = o;
    return 0;
}
extern "C" int cgo_obj_logreg_create_csr(cgo_ctx *ctx, int64_t N, int64_t d, const int64_t *rowptr, const int32_t *col,
                                         const double *val, const double *y, double lambda, cgo_obj **out) {
    return cgo_obj_logreg_create_csr_ex(ctx, N, d, rowptr, col, val, y, nullptr, 0, lambda, out);
}

extern "C" int cgo_obj_softmax_create_csr_ex(cgo_ctx *ctx, int64_t N, int64_t d, int32_t K, const int64_t *rowptr,
                                             const int32_t *col, const double *val, const int32_t *labels,
                                             const double *sample_weight, int32_t fit_intercept, double lambda,
                                             cgo_obj **out) {
    CGO_CHECK(ctx && rowptr && labels && out, "NULL argument");
    CGO_CHECK(ctx->nranks == 1, "cgo_obj_softmax_create_csr is single-GPU");
    CGO_CHECK(ctx->csr_mode != 1, "softmax: the objective runs on the K-column SpMM (CGO_CSR_MODE=1 forbids it)");
    CGO_CHECK(N >= 1 && d >= 1, "softmax: need nsamples >= 1 and nfeat >= 1 (nsamples=%lld, nfeat=%lld)", (long long)N, (long long)d);
    CGO_CHECK(K >= 2 && K <= 256, "softmax: nclasses = %d must be in [2, 256]", (int)K);
    CGO_TRY(check_i32(N, "nsamples"));
    CGO_TRY(check_i32(d, "nfeat"));
    CGO_CHECK(rowptr[0] == 0, "rowptr[0] = %lld: row pointers are 0-based", (long long)rowptr[0]);
    CGO_TRY(check_host_csr(N, d, rowptr, col, val));
    for (int64_t i = 0; i < N; ++i)
        CGO_CHECK(labels[i] >= 0 && labels[i] < K, "label %d of sample %lld is not in [0, %d)", (int)labels[i], (long long)i, (int)K);
    CGO_CHECK(std::isfinite(lambda) && lambda >= 0.0, "softmax: lambda = %g must be finite and >= 0", lambda);
    double S;
    CGO_TRY(check_glm(ctx, "softmax", N, d, sample_weight, fit_intercept, &S));
    CGO_CUDA(cudaSetDevice(ctx->device));
    const int64_t nnz = rowptr[N], n = (d + fit_intercept) * K;
    CsrObj *o = new CsrObj();
    o->ctx = ctx; o->logreg = true; o->nclass = K; o->lambda = lambda; o->nsamples = N; o->wsum = S;
    o->icpt = fit_intercept == 1;
    o->n_global = n; o->n_local = n; o->offset = 0; o->nrows = N; o->halo = 0;
    o->LA.width = o->LAT.width = K;
    auto body = [&]() -> int {
        cudaStream_t s = ctx->stream;
        CGO_TRY(csr_alloc(o->A, N, nnz));
        CGO_CUDA(cudaMemcpyAsync(o->A.rowptr, rowptr, sizeof(int64_t) * (size_t)(N + 1), cudaMemcpyHostToDevice, s));
        if (nnz) {
            CGO_CUDA(cudaMemcpyAsync(o->A.col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, s));
            CGO_CUDA(cudaMemcpyAsync(o->A.val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, s));
        }
        // labels as doubles (exact below 2^53), read in pairs by the softmax kernel
        std::vector<double> yd((size_t)N);
        for (int64_t i = 0; i < N; ++i) yd[(size_t)i] = (double)labels[i];
        CGO_CUDA(cudaMalloc(&o->b, sizeof(double) * (size_t)(N + CSR_PAD)));
        CGO_CUDA(cudaMemsetAsync(o->b, 0, sizeof(double) * (size_t)(N + CSR_PAD), s));
        CGO_CUDA(cudaMemcpyAsync(o->b, yd.data(), sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, s));
        CGO_TRY(upload_weights(ctx, o, sample_weight, N));
        CGO_TRY(o->alloc_r());
        CsrSrc src{o->A.col, nnz};
        CsrFin fin{o->A.rowptr, N, o->A.val};
        CGO_TRY(build_transpose(ctx, src, fin, d, o->AT));
        CGO_TRY(split_long_rows(ctx, o->A, o->LA));
        CGO_TRY(split_long_rows(ctx, o->AT, o->LAT));
        if (o->icpt) CGO_TRY(add_unit_row(ctx, o->LAT, d, N));
        // K_b gathers d·K doubles, K_c N·K: column blocks of gather_block_bytes / 8K features / samples
        CGO_TRY(build_blocked(ctx, o->A, d, K, o->Ab));
        CGO_TRY(build_blocked(ctx, o->AT, N, K, o->ATb));
        if ((!o->Ab.blk.empty() || !o->ATb.blk.empty()) && o->A.nnz > (int64_t)200000000) {
            // production sizes: drop the single-pass copies (only the CSR download reads them)
            if (!o->Ab.blk.empty()) { cudaFree(o->A.col); cudaFree(o->A.val); o->A.col = nullptr; o->A.val = nullptr; }
            if (!o->ATb.blk.empty()) { cudaFree(o->AT.col); cudaFree(o->AT.val); o->AT.col = nullptr; o->AT.val = nullptr; }
            o->have_unblocked = false;
        }
        CGO_CUDA(cudaStreamSynchronize(s));
        o->direct = true;                     // dots in BLAS-1 passes: reduction site (2, 4)
        return 0;
    };
    int rc = body();
    if (rc) { delete o; return rc; }
    *out = o;
    return 0;
}
extern "C" int cgo_obj_softmax_create_csr(cgo_ctx *ctx, int64_t N, int64_t d, int32_t K, const int64_t *rowptr,
                                          const int32_t *col, const double *val, const int32_t *labels, double lambda,
                                          cgo_obj **out) {
    return cgo_obj_softmax_create_csr_ex(ctx, N, d, K, rowptr, col, val, labels, nullptr, 0, lambda, out);
}

// ------------------------------------------------------------------ test hooks
static CsrObj *as_csr(cgo_obj *o) { return dynamic_cast<CsrObj *>(o); }

extern "C" int cgo_obj_csr_blocks(cgo_obj *obj, int transposed, int32_t *nblocks) {
    CsrObj *o = as_csr(obj);
    CGO_CHECK(o && nblocks, "not a CSR objective / NULL argument");
    const CsrBlocked &B = transposed ? o->ATb : o->Ab;
    *nblocks = B.blk.empty() ? 1 : (int32_t)B.blk.size();
    return 0;
}
extern "C" int cgo_obj_csr_nnz(cgo_obj *obj, int transposed, int64_t *nrows, int64_t *nnz) {
    CsrObj *o = as_csr(obj);
    CGO_CHECK(o != nullptr, "not a CSR objective");
    const CsrMat &M = transposed ? o->AT : o->A;
    if (nrows) *nrows = M.nrows;
    if (nnz) *nnz = M.nnz + (transposed ? o->LAT : o->LA).M.nnz;
    return 0;
}
// M row-major on the host (any of the three may be NULL)
static int csr_download_mat(cgo_ctx *c, const CsrMat &M, int64_t *rowptr, int32_t *col, double *val) {
    cudaStream_t s = c->stream;
    if (rowptr) CGO_CUDA(cudaMemcpyAsync(rowptr, M.rowptr, sizeof(int64_t) * (size_t)(M.nrows + 1), cudaMemcpyDeviceToHost, s));
    int32_t *ctmp = nullptr; double *vtmp = nullptr;          // row-major copies of a sliced matrix
    auto body = [&]() -> int {
        const int32_t *csrc = M.col; const double *vsrc = M.val;
        if (M.sliced && M.nnz && (col || val)) {
            CGO_CUDA(cudaMalloc(&ctmp, sizeof(int32_t) * (size_t)M.nnz));
            CGO_CUDA(cudaMalloc(&vtmp, sizeof(double) * (size_t)M.nnz));
            k_slice_permute<<<grid_for((M.nrows + 31) / 32 * 32, c->sms), 256, 0, s>>>(M, M.col, M.val, ctmp, vtmp, true);
            CGO_CUDA(cudaGetLastError());
            csrc = ctmp; vsrc = vtmp;
        }
        if (col && M.nnz) CGO_CUDA(cudaMemcpyAsync(col, csrc, sizeof(int32_t) * (size_t)M.nnz, cudaMemcpyDeviceToHost, s));
        if (val && M.nnz) CGO_CUDA(cudaMemcpyAsync(val, vsrc, sizeof(double) * (size_t)M.nnz, cudaMemcpyDeviceToHost, s));
        CGO_CUDA(cudaStreamSynchronize(s));
        return 0;
    };
    int rc = body();
    cudaFree(ctmp); cudaFree(vtmp);
    return rc;
}
// the whole matrix: M with the long rows of L put back in their places
static int csr_download_whole(cgo_ctx *c, const CsrMat &M, const LongRows &L, int64_t *rowptr, int32_t *col, double *val) {
    if (L.n == 0) return csr_download_mat(c, M, rowptr, col, val);
    std::vector<int64_t> rp((size_t)M.nrows + 1);
    std::vector<int32_t> ci((size_t)M.nnz), lc((size_t)L.M.nnz);
    std::vector<double> va((size_t)M.nnz), lv((size_t)L.M.nnz);
    CGO_TRY(csr_download_mat(c, M, rp.data(), ci.data(), va.data()));
    CGO_TRY(csr_download_mat(c, L.M, nullptr, lc.data(), lv.data()));
    int64_t q = 0, r = 0;
    for (int64_t i = 0; i < M.nrows; ++i) {
        if (rowptr) rowptr[i] = q;
        int64_t p0 = rp[(size_t)i], p1 = rp[(size_t)i + 1];
        const int32_t *cs = ci.data(); const double *vs = va.data();
        if (r < L.n && L.h_row[(size_t)r] == i) {
            p0 = L.h_rowptr[(size_t)r]; p1 = L.h_rowptr[(size_t)r + 1];
            cs = lc.data(); vs = lv.data();
            ++r;
        }
        for (int64_t p = p0; p < p1; ++p, ++q) {
            if (col) col[q] = cs[p];
            if (val) val[q] = vs[p];
        }
    }
    if (rowptr) rowptr[M.nrows] = q;
    return 0;
}
extern "C" int cgo_obj_csr_download(cgo_obj *obj, int transposed, int64_t *rowptr, int32_t *col, double *val, double *b) {
    CsrObj *o = as_csr(obj);
    CGO_CHECK(o != nullptr, "not a CSR objective");
    CGO_CHECK(o->have_unblocked, "the single-pass CSR copy was dropped at this size (column-blocked storage only)");
    CGO_CUDA(cudaSetDevice(o->ctx->device));
    CGO_TRY(csr_download_whole(o->ctx, transposed ? o->AT : o->A, transposed ? o->LAT : o->LA, rowptr, col, val));
    if (b) {
        CGO_CUDA(cudaMemcpyAsync(b, o->b, sizeof(double) * (size_t)o->nrows, cudaMemcpyDeviceToHost, o->ctx->stream));
        CGO_CUDA(cudaStreamSynchronize(o->ctx->stream));
    }
    return 0;
}
// softmax objective: Z = A W (d·K → N·K) or Aᵀ C (N·K → d·K), through the trial's passes (column blocks included)
static int spmm_hook(CsrObj *o, int transposed, const double *x_host, double *y_host) {
    cgo_ctx *c = o->ctx;
    CGO_CUDA(cudaSetDevice(c->device));
    // transposed: all n entries of the state, Aᵀ C followed by the intercept's sums
    const int64_t K = o->nclass, nin = (transposed ? o->A.nrows : o->AT.nrows) * K, nout = transposed ? o->n_local : o->A.nrows * K;
    const int tclass = transposed ? CGO_T_SPMVT : CGO_T_SPMV;
    double *dx = nullptr, *dy = nullptr;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&dx, sizeof(double) * (size_t)nin));
        CGO_CUDA(cudaMalloc(&dy, sizeof(double) * (size_t)nout));
        CGO_CUDA(cudaMemcpyAsync(dx, x_host, sizeof(double) * (size_t)nin, cudaMemcpyHostToDevice, c->stream));
        CGO_TRY(spmm_passes(c, transposed ? o->AT : o->A, transposed ? o->ATb : o->Ab, o->nclass, dx, dy, tclass));
        CGO_TRY(long_rows_sum_k(c, transposed ? o->LAT : o->LA, dx, dy, tclass));
        CGO_CUDA(cudaMemcpyAsync(y_host, dy, sizeof(double) * (size_t)nout, cudaMemcpyDeviceToHost, c->stream));
        CGO_CUDA(cudaStreamSynchronize(c->stream));
        return 0;
    };
    int rc = body();
    cudaFree(dx); cudaFree(dy);
    return rc;
}
// y = A x (transposed: Aᵀ x) through the production kernel; single GPU (no halo)
extern "C" int cgo_obj_spmv(cgo_obj *obj, int transposed, const double *x_host, double *y_host) {
    CsrObj *o = as_csr(obj);
    CGO_CHECK(o && x_host && y_host, "not a CSR objective / NULL argument");
    CGO_CHECK(o->halo == 0 && !o->lr_sharded, "cgo_obj_spmv is a single-GPU test hook");
    if (o->nclass > 1) return spmm_hook(o, transposed, x_host, y_host);
    CGO_CHECK(o->have_unblocked, "the single-pass CSR copy was dropped at this size (column-blocked storage only)");
    cgo_ctx *c = o->ctx;
    CGO_CUDA(cudaSetDevice(c->device));
    const CsrMat &M = transposed ? o->AT : o->A;
    const int64_t nin = transposed ? o->A.nrows : o->AT.nrows, nout = transposed ? o->n_local : M.nrows;   // Aᵀ x [, Σ x]
    double *dx = nullptr, *dy = nullptr;
    auto body = [&]() -> int {
        CGO_CUDA(cudaMalloc(&dx, sizeof(double) * (size_t)nin));
        CGO_CUDA(cudaMalloc(&dy, sizeof(double) * (size_t)nout));
        CGO_CUDA(cudaMemcpyAsync(dx, x_host, sizeof(double) * (size_t)nin, cudaMemcpyHostToDevice, c->stream));
        if (M.sliced) {
            CGO_TRY(launch_direct(c, M, dx, DirStore{dy}, dir_args(c), transposed ? CGO_T_SPMVT : CGO_T_SPMV));
        } else {
            EpiStore es{dy};
            CGO_TRY(launch_csr(c, M, dx, es, cgo_red_args(c, CGO_PACK_LEN - 1), transposed ? CGO_T_SPMVT : CGO_T_SPMV));
        }
        CGO_TRY(long_rows_sum(c, transposed ? o->LAT : o->LA, dx, dy, transposed ? CGO_T_SPMVT : CGO_T_SPMV));
        CGO_CUDA(cudaMemcpyAsync(y_host, dy, sizeof(double) * (size_t)nout, cudaMemcpyDeviceToHost, c->stream));
        CGO_CUDA(cudaStreamSynchronize(c->stream));
        return 0;
    };
    int rc = body();
    cudaFree(dx); cudaFree(dy);
    return rc;
}
