// Shared device/host helpers for libuem_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <math.h>

#include "../../include/uem_b200.h"

#define UEM_MAX_C UEM_MAX_CLASSES
#define UEM_SMS 148  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

int uem_fail(const char* fmt, ...);
// tuning knobs set through uem_set_option (0 = the kernel's own choice); see uem_api.cu
extern int g_uem_refine_ctas_per_sm;   // cap on resident CTAs per SM of the fused refine kernel (co-residency with the next batch's streaming kernels)
extern int g_uem_region_ctas_per_sm;   // same for the region-max kernel
extern int g_uem_l2_stream;            // 1: maps a step reads or writes exactly once carry an L2 evict_first hint, so that they do not push
                                       // out what the next kernel of the chain re-reads (soft labels + ids: region max -> refine;
                                       // refined labels: refine -> selection)
extern int g_uem_l2_keep;              // hint of the refined map between the refine kernel and the selection: 0 = default priority, 2 = evict_last
extern int g_uem_l2_region;            // hint of the region-max kernel's reads of soft / ids on the fused chain: 0 | 1 evict_first | 2 evict_last
                                       // (default 1: the refine kernel is not faster on L2-hot inputs, the selection is, so the
                                       // refined map is the one thing worth the capacity; profiles/r02_l2_hints.txt)
extern int g_uem_l2_last_use;          // 1: the refine kernel's reads of soft / ids (their last use in the chain) are evict_first
extern int g_uem_proto_ctas_per_sm;    // same for the prototype-sum kernel (so that a Pearson CTA fits beside it)
void uem_note_launches(int n);  // bookkeeping for uem_kernel_launches()
void uem_take_profile_events(void** start, void** stop);

#define UEM_REQUIRE(cond, ...)                                    \
    do {                                                          \
        if (!(cond)) return uem_fail(__VA_ARGS__);                \
    } while (0)

// n = number of kernels the enclosing function has just launched
#define UEM_CHECK_LAUNCH_N(n)                                                               \
    do {                                                                                    \
        cudaError_t e__ = cudaGetLastError();                                               \
        if (e__ != cudaSuccess) return uem_fail("%s: %s", __func__, cudaGetErrorString(e__)); \
        uem_note_launches(n);                                                               \
    } while (0)
#define UEM_CHECK_LAUNCH() UEM_CHECK_LAUNCH_N(1)

#define UEM_CUDA(call)                                                                      \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) return uem_fail("%s: %s", #call, cudaGetErrorString(e__)); \
    } while (0)

// compile-time class count dispatch: kernels keep the per-pixel class vector in registers
#define UEM_DISPATCH_C(c, ...)                                                        \
    switch (c) {                                                                      \
        case 1: { constexpr int C = 1; __VA_ARGS__; } break;                          \
        case 2: { constexpr int C = 2; __VA_ARGS__; } break;                          \
        case 3: { constexpr int C = 3; __VA_ARGS__; } break;                          \
        case 4: { constexpr int C = 4; __VA_ARGS__; } break;                          \
        case 5: { constexpr int C = 5; __VA_ARGS__; } break;                          \
        case 6: { constexpr int C = 6; __VA_ARGS__; } break;                          \
        case 7: { constexpr int C = 7; __VA_ARGS__; } break;                          \
        case 8: { constexpr int C = 8; __VA_ARGS__; } break;                          \
        default: return uem_fail("%s: class count %d outside [1,%d]", __func__, (int)(c), UEM_MAX_C); \
    }

static inline bool uem_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline int uem_div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------
// 128-bit streaming loads/stores (read-only path, no L1 allocation: every map is touched once
// per kernel; L2 residency is left to the default policy so the next phase can hit)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_f4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float ldg_f1(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void ldg_i64x2(const int64_t* p, int64_t& a, int64_t& b) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.s64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p));
}
__device__ __forceinline__ int64_t ldg_i64(const int64_t* p) {
    int64_t r;
    asm volatile("ld.global.nc.L1::no_allocate.s64 %0, [%1];" : "=l"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_f4(float* p, float4 v) {
    asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void stg_i64x2(int64_t* p, int64_t a, int64_t b) {
    asm volatile("st.global.v2.s64 [%0], {%1,%2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
// ---- the same with an L2 eviction-priority hint (createpolicy handle in a register; kind 0 = evict_normal = no hint)
__device__ __forceinline__ uint64_t l2_policy(int kind) {
    uint64_t pol;
    if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    else if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ float4 ldg_f4(const float* p, uint64_t pol) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ldg_f1(const float* p, uint64_t pol) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ void ldg_i64x2(const int64_t* p, int64_t& a, int64_t& b, uint64_t pol) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.s64 {%0,%1}, [%2], %3;" : "=l"(a), "=l"(b) : "l"(p), "l"(pol));
}
__device__ __forceinline__ int64_t ldg_i64(const int64_t* p, uint64_t pol) {
    int64_t r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s64 %0, [%1], %2;" : "=l"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ void stg_f4(float* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_f1(float* p, float v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_i64x2(int64_t* p, int64_t a, int64_t b, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v2.s64 [%0], {%1,%2}, %3;" ::"l"(p), "l"(a), "l"(b), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_i64(int64_t* p, int64_t a, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.s64 [%0], %1, %2;" ::"l"(p), "l"(a), "l"(pol) : "memory");
}
// L2-coherent (skips L1) scalar load: used by test-then-atomic on tables other CTAs update
__device__ __forceinline__ unsigned ld_cg_u32(const unsigned* p) {
    unsigned r;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(r) : "l"(p) : "memory");
    return r;
}

// cp.async (LDGSTS): global -> shared without staging registers
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem, uint64_t pol) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(sa), "l"(gmem), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// VEC pixels per thread (4 = 128-bit path, 1 = scalar fallback for unaligned / ragged rows)
template <int VEC> struct PixVec;
template <> struct PixVec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float* p) { float4 t = ldg_f4(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    __device__ __forceinline__ void load(const float* p, uint64_t pol) { float4 t = ldg_f4(p, pol); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
    __device__ __forceinline__ void store(float* p) const { stg_f4(p, make_float4(v[0], v[1], v[2], v[3])); }
    __device__ __forceinline__ void store(float* p, uint64_t pol) const { stg_f4(p, make_float4(v[0], v[1], v[2], v[3]), pol); }
};
template <> struct PixVec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float* p) { v[0] = ldg_f1(p); }
    __device__ __forceinline__ void load(const float* p, uint64_t pol) { v[0] = ldg_f1(p, pol); }
    __device__ __forceinline__ void store(float* p) const { p[0] = v[0]; }
    __device__ __forceinline__ void store(float* p, uint64_t pol) const { stg_f1(p, v[0], pol); }
};
template <int VEC> __device__ __forceinline__ void load_ids(const int64_t* p, int64_t (&id)[VEC]);
template <> __device__ __forceinline__ void load_ids<4>(const int64_t* p, int64_t (&id)[4]) {
    ldg_i64x2(p, id[0], id[1]);
    ldg_i64x2(p + 2, id[2], id[3]);
}
template <> __device__ __forceinline__ void load_ids<1>(const int64_t* p, int64_t (&id)[1]) { id[0] = ldg_i64(p); }
template <int VEC> __device__ __forceinline__ void load_ids(const int64_t* p, int64_t (&id)[VEC], uint64_t pol);
template <> __device__ __forceinline__ void load_ids<4>(const int64_t* p, int64_t (&id)[4], uint64_t pol) {
    ldg_i64x2(p, id[0], id[1], pol);
    ldg_i64x2(p + 2, id[2], id[3], pol);
}
template <> __device__ __forceinline__ void load_ids<1>(const int64_t* p, int64_t (&id)[1], uint64_t pol) { id[0] = ldg_i64(p, pol); }
template <int VEC> __device__ __forceinline__ void store_ids(int64_t* p, const int64_t (&id)[VEC], uint64_t pol);
template <> __device__ __forceinline__ void store_ids<4>(int64_t* p, const int64_t (&id)[4], uint64_t pol) {
    stg_i64x2(p, id[0], id[1], pol);
    stg_i64x2(p + 2, id[2], id[3], pol);
}
template <> __device__ __forceinline__ void store_ids<1>(int64_t* p, const int64_t (&id)[1], uint64_t pol) { stg_i64(p, id[0], pol); }
template <int VEC> __device__ __forceinline__ void store_ids(int64_t* p, const int64_t (&id)[VEC]);
template <> __device__ __forceinline__ void store_ids<4>(int64_t* p, const int64_t (&id)[4]) {
    stg_i64x2(p, id[0], id[1]);
    stg_i64x2(p + 2, id[2], id[3]);
}
template <> __device__ __forceinline__ void store_ids<1>(int64_t* p, const int64_t (&id)[1]) { p[0] = id[0]; }

// ------------------------------------------------------------------------------------------
// order-preserving float <-> uint32 encoding for atomicMax/atomicMin on arbitrary floats;
// 0 never encodes a real float > -NaN, so a zeroed table means "untouched"
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned f32_to_ordered(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_f32(unsigned e) {
    unsigned u = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
    return __uint_as_float(u);
}

// ------------------------------------------------------------------------------------------
// warp / block reductions
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// torch.max semantics: NaN is sticky
__device__ __forceinline__ float nanmax(float a, float b) { return (a != a) ? a : ((b != b) ? b : fmaxf(a, b)); }
__device__ __forceinline__ float warp_nanmax(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = nanmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------------------
// bilinear (align_corners=True) source coordinates, PyTorch upsample_bilinear2d arithmetic:
// scale = fp32(in-1)/fp32(out-1) (0 if out==1), src = scale*dst, i0=(int)src, i1=i0+(i0<in-1)
// ------------------------------------------------------------------------------------------
struct Lerp {
    int i0, i1;
    float l0, l1;
};
__device__ __forceinline__ Lerp make_lerp(int dst, int in_size, float scale) {
    Lerp r;
    float src = scale * (float)dst;
    r.i0 = min((int)src, in_size - 1);
    r.i1 = r.i0 + ((r.i0 < in_size - 1) ? 1 : 0);
    r.l1 = src - (float)r.i0;
    r.l0 = 1.0f - r.l1;
    return r;
}
static inline float uem_align_corners_scale(int in_size, int out_size) {
    return out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.0f;
}

// single-MUFU approximations (2 ulp): reciprocal and 2^x
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// e_c = exp(z_c - max z) (one MUFU each; results below 2^-126 flush to 0, irrelevant for a softmax numerator),
// returns S = sum e_c
template <int C> __device__ __forceinline__ float exp_shifted(float (&z)[C]) {
    float mx = z[0];
#pragma unroll
    for (int i = 1; i < C; ++i) mx = fmaxf(mx, z[i]);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < C; ++i) {
        z[i] = ex2_approx((z[i] - mx) * 1.4426950408889634f);
        s += z[i];
    }
    return s;
}

// softmax over a register vector: y = exp(x - max) / sum, matches torch.softmax to ~2 ulp
template <int C> __device__ __forceinline__ void softmax_regs(float (&x)[C]) {
    float mx = x[0];
#pragma unroll
    for (int i = 1; i < C; ++i) mx = fmaxf(mx, x[i]);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < C; ++i) {
        x[i] = __expf(x[i] - mx);
        s += x[i];
    }
    float inv = 1.0f / s;
#pragma unroll
    for (int i = 0; i < C; ++i) x[i] *= inv;
}
// x / (max_c x + 1e-7)  (alignment.py:222,235,253)
template <int C> __device__ __forceinline__ void peak_norm_regs(float (&x)[C]) {
    float mx = x[0];
#pragma unroll
    for (int i = 1; i < C; ++i) mx = fmaxf(mx, x[i]);
    float inv = 1.0f / (mx + 1e-7f);
#pragma unroll
    for (int i = 0; i < C; ++i) x[i] *= inv;
}

// UVEMLoss.get_weight (balance.py:396-423), operation by operation (no FMA contraction)
__device__ __forceinline__ float uvem_weight_dev(float u, float m, float t, float inv_gamma, float cl, float cr) {
    // only the branch that the final where() selects is evaluated; NaN fails every comparison and lands on the
    // right branch with the substitute value 0, exactly like the reference
    const bool left = (u <= m);
    const bool enabled = left ? (m > 0.f) : (m < t);
    const float sub = left ? ((u >= 0.f) ? u : 1.0f) : ((u > m && u <= t) ? u : 0.0f);
    const float d = __fsub_rn(sub, m);
    float x = __fadd_rn(__fmul_rn(left ? cl : cr, __fmul_rn(d, d)), 1.0f);
    x = fminf(fmaxf(x, 0.f), 1.f);
    // x^(1/gamma) = 2^(lg2(x)/gamma): lg2.approx is 2^-22 absolute on [0.5,2] and 2 ulp elsewhere, 1/gamma <= 1
    // keeps the result within ~1e-6 relative of the reference's pow; x = 0 -> 0, x = 1 -> 1 exactly
    float w = __powf(x, inv_gamma);
    if (!enabled) w = left ? 1.0f : 0.0f;
    return (u >= t) ? 0.f : w;
}

// entropy sum_c -p log p (balance.py:372) = -ln2 * sum_c p*lg2(p): one MUFU.LG2 + one FFMA per class.
// lg2.approx is 2 ulp for p < 0.5 but only 2^-22 ABSOLUTE on [0.5, 2), which would dominate the small term of a
// confident pixel; the (at most one) class with p >= 1 - 2^-6 therefore gets log(p) = log1p(-d), d = 1 - p, from its
// series (-d - d^2/2 - d^3/3 - d^4/4, truncation < 2e-8 relative), everything branch-free.  Below that bound the other
// classes carry enough entropy for the absolute error to stay under 1e-5 relative.  p == 0 yields NaN (0 * -inf)
// exactly like the reference.
template <int C>
__device__ __forceinline__ float entropy_px(const float (&p)[C]) {
    float t = 0.f, vmax = p[0];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
        const float v = p[ci];
        vmax = fmaxf(vmax, v);
        float l;
        asm("lg2.approx.f32 %0, %1;" : "=f"(l) : "f"(v));
        t = fmaf(v, l, t);
    }
    float u = t * -0.69314718055994531f;
    // swap the approximate term of the dominant class for the series when it is within 2^-6 of 1
    const float d = 1.0f - vmax;
    float lm;
    asm("lg2.approx.f32 %0, %1;" : "=f"(lm) : "f"(vmax));
    const float approx_term = (vmax * lm) * -0.69314718055994531f;
    const float series = -d * fmaf(d, fmaf(d, fmaf(d, 0.25f, 0.33333334f), 0.5f), 1.0f);   // log(1 - d)
    const float exact_term = -vmax * series;
    return (d < 0.015625f) ? (u - approx_term) + exact_term : u;
}
