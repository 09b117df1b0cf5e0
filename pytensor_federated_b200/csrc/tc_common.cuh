// tcgen05 / TMEM / TMA / mbarrier PTX wrappers and UMMA descriptor builders shared by the
// tensor-core GLM kernels (glm_tc.cu: bf16, glm_fp8.cu: block-scaled fp8).  sm_100a only.
#pragma once
#include <cstdlib>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "fed_comm.cuh"

namespace tc {

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// CTA-wide "the mbarrier pipeline stalled" flag.  A wait that exceeds 4 s raises it instead of trapping (a
// trap poisons the whole CUDA context: engine, torch and all); once it is up every wait returns at once, so the
// roles run off the end of their loops, the CTA reports B200FED_ERR_PIPELINE through fed::epilogue and the host
// raises an ordinary exception with the context intact.  Results of such a launch are garbage by definition.
__device__ __forceinline__ volatile int* pipeline_fault() {
    __shared__ int fault;
    return &fault;
}
// Bounded wait: a pipeline bug must surface as an error status, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const unsigned long long t0 = fed::globaltimer();
    volatile int* fault = pipeline_fault();
    while (!mbar_try_wait(bar, parity)) {
        if (*fault) return;
        if (fed::globaltimer() - t0 > 4000000000ull) {
            *fault = 1;
            return;
        }
    }
}
// One lane of a fully active warp (the role loops stay warp-uniform; only the issue is predicated, so the
// compiler keeps descriptors and addresses in uniform registers instead of a per-instruction waterfall).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_out, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_out)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, float (&v)[4]) {
    uint32_t a, b, c, d;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(a), "=r"(b), "=r"(c), "=r"(d)
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    v[0] = __uint_as_float(a); v[1] = __uint_as_float(b); v[2] = __uint_as_float(c); v[3] = __uint_as_float(d);
}
// N consecutive fp32 columns of this warp's 32 TMEM lanes in ONE round trip: every tcgen05.ld of the request is
// issued before the single tcgen05.wait::ld (issue + wait live in one asm statement, so the compiler cannot
// touch the destination registers in between).  N in {4, 8, 16, 24, 32}.
template <int N>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[N]) {
    static_assert(N == 4 || N == 8 || N == 16 || N == 24 || N == 32, "supported widths");
    uint32_t r[N];
    if constexpr (N == 4) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n\ttcgen05.wait::ld.sync.aligned;"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
    } else if constexpr (N == 8) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n\ttcgen05.wait::ld.sync.aligned;"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
    } else if constexpr (N == 16) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\ttcgen05.wait::ld.sync.aligned;"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr) : "memory");
    } else if constexpr (N == 24) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%24];\n\t"
                     "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%16, %17, %18, %19, %20, %21, %22, %23}, [%25];\n\ttcgen05.wait::ld.sync.aligned;"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]) : "r"(taddr), "r"(taddr + 16) : "memory");
    } else {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\ttcgen05.wait::ld.sync.aligned;"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]) : "r"(taddr) : "memory");
    }
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, float (&v)[16]) { tmem_ld_cols<16>(taddr, v); }

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor (sm_100): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout type [61,64) (0 = none/interleave, 2 = 128B swizzle).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(layout & 7) << 61;
    return d;
}
// Instruction descriptor for kind::f16 with bf16 operands and fp32 accumulation.
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4)      // D format: f32
           | (1u << 7)    // A format: bf16
           | (1u << 10)   // B format: bf16
           | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// Programmatic dependent launch for back-to-back evaluations (B200FED_NO_PDL=1 disables it for A/B runs).
inline bool use_pdl() {
    static const bool on = [] {
        const char* v = getenv("B200FED_NO_PDL");
        return !(v && *v && *v != '0');
    }();
    return on;
}

// Index + phase bit of an n-deep circular buffer, advanced without division (the single-thread
// TMA / MMA issue loops are latency chains: a 64-bit `it % n`, `it / n` pair costs ~100 instructions).
struct Ring {
    int idx = 0;
    uint32_t phase = 0;
    __host__ __device__ __forceinline__ void advance(int n) {
        if (++idx == n) {
            idx = 0;
            phase ^= 1u;
        }
    }
};

__device__ __forceinline__ void link_loglik(int family, float y, float eta, float& ll, float& r) {
    if (family == 0) {
        const float e = __expf(-fabsf(eta));
        const float sp = fmaxf(eta, 0.f) + __logf(1.f + e);
        const float inv = __fdividef(1.f, 1.f + e);
        const float p = eta >= 0.f ? inv : e * inv;
        ll = y * eta - sp;
        r = y - p;
    } else if (family == 1) {
        const float mu = __expf(eta);
        ll = y * eta - mu;
        r = y - mu;
    } else {
        const float d = y - eta;
        ll = -0.5f * d * d - 0.918938533204672742f;
        r = d;
    }
}

// ------------------------------------------------------------------ families with fitted parameters phi
// Family codes 3 = normal (sigma), 4 = student_t (sigma, nu), 5 = negative_binomial (alpha, NB2: var = mu + mu^2 / alpha).
// They are fully normalised.  Everything that depends on phi alone is computed ONCE per chain (phi_chain, fp64):
// fp32 helpers for the per-row maths, and the per-row constants c of the log-likelihood and of d/dphi, which the
// kernel adds in fp64 as (valid rows of a chunk) x c instead of summing them row by row.
struct PhiChain {
    double c_ll, c_d0, c_d1;   // per-row constants of LL, dLL/dphi0, dLL/dphi1
    float p[4];                // fp32 helpers of the per-row maths (family-specific, see phi_chain)
};

// Digamma for x > 0: recurrence up to x >= 10, then the asymptotic series (error < 1e-13 there).
template <typename T>
__host__ __device__ inline T digamma(T x) {
    T acc = 0;
    while (x < T(10)) {
        acc -= T(1) / x;
        x += T(1);
    }
    const T inv = T(1) / x, inv2 = inv * inv;
    const T series = inv2 * (T(1) / 12 - inv2 * (T(1) / 120 - inv2 * (T(1) / 252 - inv2 * (T(1) / 240 - inv2 * (T(1) / 132)))));
    return acc + log(x) - T(0.5) * inv - series;
}

__device__ inline PhiChain phi_chain(int family, const float* phi) {
    PhiChain c{0.0, 0.0, 0.0, {0.f, 0.f, 0.f, 0.f}};
    const double s = phi[0];
    if (family == 3) {
        c.p[0] = (float)(1.0 / s);
        c.c_ll = -log(s) - 0.918938533204672742;
        c.c_d0 = -1.0 / s;
    } else if (family == 4) {
        const double nu = phi[1];
        c.p[0] = (float)(1.0 / s);
        c.p[1] = phi[1];
        c.p[2] = (float)(1.0 / nu);
        c.p[3] = (float)(nu + 1.0);
        c.c_ll = lgamma(0.5 * (nu + 1.0)) - lgamma(0.5 * nu) - 0.5 * log(nu * 3.14159265358979323846) - log(s);
        c.c_d0 = -1.0 / s;
        c.c_d1 = 0.5 * (digamma(0.5 * (nu + 1.0)) - digamma(0.5 * nu) - 1.0 / nu);
    } else if (family == 5) {
        c.p[0] = phi[0];
        c.p[1] = (float)(1.0 / s);
        c.p[2] = (float)log(s);
    }
    return c;
}

// Counts below this use the exact short sums  lgamma(y+a) - lgamma(a) - lgamma(y+1) = sum_{j<y} log((a+j)/(j+1))  and
// psi(y+a) - psi(a) = sum_{j<y} 1/(a+j)  in fp32; larger counts take lgamma / digamma in fp64 (the fp32 difference of
// two lgammas near 1e3..1e4 cancels catastrophically: lgammaf(1000) ~ 5905 has an ulp of ~5e-4).
constexpr int kNbShortSum = 16;

__device__ __forceinline__ void nb_count_terms(float y, float a, float& lg, float& dg) {
    const int n = (int)y;
    if (n < kNbShortSum) {
        float lsum = 0.f, dsum = 0.f, prod = 1.f;
        for (int j = 0; j < n; ++j) {
            const float aj = a + (float)j;
            prod *= __fdividef(aj, (float)(j + 1));
            dsum += __fdividef(1.f, aj);
            if (j & 1) {   // pairs of ratios: no fp32 overflow for a up to ~1e19
                lsum += __logf(prod);
                prod = 1.f;
            }
        }
        lg = lsum + __logf(prod);
        dg = dsum;
    } else {
        const double yd = y, ad = a;
        lg = (float)(lgamma(yd + ad) - lgamma(ad) - lgamma(yd + 1.0));
        dg = (float)(digamma(yd + ad) - digamma(ad));
    }
}

// Per row: the phi-free part of LL, r = dLL/deta and the row parts of dLL/dphi (the per-chain constants of
// PhiChain are added per chunk).  p = PhiChain::p of the chain.
__device__ __forceinline__ void link_loglik_phi(int family, float y, float eta, const float* p, float& ll, float& r,
                                                float& d0, float& d1) {
    if (family == 3) {                               // p = (1/sigma)
        const float z = (y - eta) * p[0];
        ll = -0.5f * z * z;
        r = z * p[0];
        d0 = z * z * p[0];
        d1 = 0.f;
    } else if (family == 4) {                        // p = (1/sigma, nu, 1/nu, nu + 1)
        const float z = (y - eta) * p[0];
        const float z2 = z * z;
        const float l1p = log1pf(z2 * p[2]);
        const float w = __fdividef(p[3], p[1] + z2);  // (nu + 1) / (nu + z^2)
        ll = -0.5f * p[3] * l1p;
        r = w * z * p[0];
        d0 = w * z2 * p[0];
        d1 = 0.5f * (w * z2 * p[2] - l1p);
    } else {                                         // p = (alpha, 1/alpha, log alpha)
        const float mu = expf(eta);
        const float l1 = log1pf(mu * p[1]);          // log((alpha + mu) / alpha)
        const float inv = __fdividef(1.f, p[0] + mu);
        float lg, dg;
        nb_count_terms(y, p[0], lg, dg);
        ll = lg - p[0] * l1 + y * (eta - p[2] - l1);
        r = p[0] * (y - mu) * inv;
        d0 = dg - l1 + (mu - y) * inv;
        d1 = 0.f;
    }
}


}  // namespace tc
