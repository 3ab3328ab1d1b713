// a6: Aligner.label_refine as ONE full-resolution kernel, plus the fused refine->select chain.
// Reference: uemda/gast/alignment.py:194-293 (~60 eager kernels, ~58 full-res map passes):
//   prototype view  :215-223  1/pearson (low-res) -> bilinear up -> softmax(T=1) -> /max
//   prediction view :225-236  logits (low-res) -> bilinear up -> softmax(/temp) [mean of 2 heads] -> /max
//   superpixel view :238-258  region max of soft (torch_scatter 'max') -> gather -> softmax(/temp) -> /max,
//                             applied multiplicatively outside the batch-global "ignored" id (:241-243,:255)
//   final           :291-292  soft' = w*soft / (sum_c w*soft + 1e-7)
// Compulsory traffic per pixel: read soft (4c) + sup (8), write refined (4c); everything else (three
// low-res maps, the per-region weight table) is L2/L1 resident.
//
// Two kernels, chosen from the configuration by launch_refine:
//   * refine_col_kernel -- the default configuration (all three views, two heads, W % 4 == 0): a lane owns one or two
//     image COLUMNS and walks down a range of rows, so the horizontal half of the bilinear interpolation is hoisted out
//     of the row loop (one packed FFMA per class pair and row); rows arrive by per-warp cp.async three rows ahead; no
//     barrier in the row loop.  See the comment above the kernel and DESIGN.md section 3 for the measurements that led
//     here (a row-major 4-pixels-per-thread TMA kernel with a 3-tap table, 37 us, was the previous default).
//   * refine_kernel -- any view subset / one head / ragged or unaligned rows: persistent CTAs of 128 threads over image
//     rows, a thread = 4 (or 1) consecutive pixels, low-res maps interpolated vertically once per row into shared memory.
// Shared by both: softmax followed by "/ (max + 1e-7)" collapses algebraically (max_c softmax = 1/S, hence
// w_c = e_c * (1 - 1e-7*S) to O(1e-13)): no division, exp is one MUFU (ex2.approx.ftz); the superpixel view depends only
// on (image, region): softmax(/temp)/max of the region maxima is precomputed per region (by the region-max kernel's tail
// on the fused chain), the pixel kernels gather 2 x LDG.128; per-(image,class) maxima for pseudo_selection
// (pseudo_generation.py:76) fall out as a (b, c+2) stats table raised with atomicMax.
#include "uem_tma.cuh"
#include "uem_xchg_dev.cuh"
#include <string.h>

int uem_region_table_f32(const float* src, int64_t sb, int64_t sn, int64_t sc, const int64_t* index, int b, int64_t N,
                         int c, int64_t R, int op, const int64_t* hot_ptr, int64_t hot_val, int skip_hot, unsigned* table,
                         unsigned* cnt, int* status, cudaStream_t st);
int uem_i64_max_accumulate(const int64_t* x, int64_t n, int64_t* out_max, cudaStream_t st);
int uem_region_max_f32(const float* src, int64_t sb, int64_t sc, const int64_t* index, int b, int64_t N, int c, int64_t R,
                       unsigned* table, int64_t* maxid_out, int* status, float* tail_sw, int* tail_done, float temp,
                       unsigned* zero_words, int n_zero, const RegionXchg* xchg, cudaStream_t st);
int uem_select_entropy_stats_impl(const float* mask, const uint32_t* class_stats, int b, int c, int64_t hw, float cutoff_top,
                                  float cutoff_low, int64_t ignore_label, int64_t* out, const float* uvem, float* entropy,
                                  float* weight, int64_t* zero_after, int pdl, cudaStream_t st);

#define UEM_FFMA2(a, b, c) __ffma2_rn(a, b, c)
#define UEM_FMUL2(a, b) __fmul2_rn(a, b)
#define UEM_FADD2(a, b) __fadd2_rn(a, b)

namespace {

constexpr int kRefineThreads = 128;

template <int C> struct Lay {
    static constexpr int CP = (C + 3) & ~3;   // class slots per map, padded for LDS.128 / LDG.128
    static constexpr int STRIDE = 3 * CP;     // floats per low-res column: [simi | pred1 | pred2]
    static constexpr int PC = (C + 1) / 2;    // class pairs for packed fp32x2 math
};

__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
}

struct RefineParams {
    int views;
    const float* maps[3];   // slot 0 simi, 1 pred1, 2 pred2 (low-res (b,C,h,w)); null = unused
    float map_scale[3];     // folded into the staged rows (1/temp for the logits when temp is a power of two)
    int n_pred;             // prediction heads (0..2)
    int b, h, w, H, W;
    float sy, sx;
    float temp;
    int div_temp;           // temp is not a power of two: the staged logits are divided (one rounding) instead
    const int64_t* sup;
    const float* sw;        // (b,R+1,CP) per-region superpixel-view weights
    int64_t R;
    const int64_t* ignored_id;
    const float* soft;
    float* out;
    unsigned* stats;        // (b, C+2) ordered-u32: per-class max of `out`, -(min of out), bad flag; atomically raised
    int l2_in, l2_out;      // L2 eviction-priority hints (l2_policy kinds) of the soft / id reads and of the stores of `out`
};

// softmax numerators over PC class pairs, inputs in the log2 domain (taps pre-scaled by log2 e): e_c = 2^(z_c - max z);
// returns their sum
template <int PC> __device__ __forceinline__ float exp2_shifted2(float2 (&z)[PC]) {
    float mx = fmaxf(z[0].x, z[0].y);
#pragma unroll
    for (int j = 1; j < PC; ++j) mx = fmaxf(mx, fmaxf(z[j].x, z[j].y));
    const float2 nmx = make_float2(-mx, -mx);
    float2 acc;
#pragma unroll
    for (int j = 0; j < PC; ++j) {
        const float2 d = UEM_FADD2(z[j], nmx);
        z[j] = make_float2(ex2_approx(d.x), ex2_approx(d.y));
        acc = j ? UEM_FADD2(acc, z[j]) : z[j];
    }
    return acc.x + acc.y;
}

template <int C> __device__ __forceinline__ void load_tap(const float* col, float (&t)[Lay<C>::CP]) {
#pragma unroll
    for (int q = 0; q < Lay<C>::CP / 4; ++q) {
        const float4 v = *reinterpret_cast<const float4*>(col + 4 * q);
        t[4 * q] = v.x; t[4 * q + 1] = v.y; t[4 * q + 2] = v.z; t[4 * q + 3] = v.w;
    }
}

// vertical lerp of the low-res rows feeding output row y into row[(w+2)][STRIDE]:
// warp -> (map, class slot), lane -> low-res column: coalesced loads, no integer division by runtime values.
// Two replicated columns at the right edge (column a+2 of the 3-tap form always exists); padded class slots hold
// -1e30 so they exponentiate to exactly 0 and never win a max.
template <int C>
__device__ __forceinline__ void stage_row(float* row, const RefineParams& p, int bi, int y) {
    constexpr int CP = Lay<C>::CP, STRIDE = Lay<C>::STRIDE;
    const Lerp ly = make_lerp(y, p.h, p.sy);
    const int nwarps = blockDim.x >> 5, wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int hw_low = p.h * p.w;
    for (int mc = wid; mc < 3 * CP; mc += nwarps) {
        const int m = mc / CP, ci = mc - m * CP;
        if (p.maps[m] == nullptr) continue;
        if (ci >= C) {
            for (int x = lane; x < p.w + 2; x += 32) row[x * STRIDE + m * CP + ci] = -1e30f;
            continue;
        }
        const float* plane = p.maps[m] + ((int64_t)bi * C + ci) * hw_low;
        const float* r0 = plane + ly.i0 * p.w;
        const float* r1 = plane + ly.i1 * p.w;
        const float sc = p.map_scale[m];
        const bool dv = p.div_temp && m > 0;
        for (int x = lane; x < p.w + 2; x += 32) {
            const int xs = min(x, p.w - 1);
            const float v = ly.l0 * __ldg(r0 + xs) + ly.l1 * __ldg(r1 + xs);
            row[x * STRIDE + m * CP + ci] = dv ? __fdiv_rn(v, p.temp) : v * sc;
        }
    }
}

// block-reduce the running statistics of image bi and raise its stats row (one atomic per class per CTA)
template <int C>
__device__ __forceinline__ void flush_stats(unsigned* stats, int bi, float (&cmax)[C], float& cmin, bool& bad, float (*red)[C + 2]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
        const float v = warp_max(cmax[ci]);
        if (lane == 0) red[warp][ci] = v;
    }
    const float mn = warp_min(cmin);
    const int anybad = __any_sync(0xffffffffu, bad);
    if (lane == 0) { red[warp][C] = mn; red[warp][C + 1] = anybad ? 1.f : 0.f; }
    __syncthreads();
    if (threadIdx.x <= C + 1) {
        const int nw = blockDim.x >> 5;
        float v = red[0][threadIdx.x];
        for (int i = 1; i < nw; ++i) v = (threadIdx.x == C) ? fminf(v, red[i][threadIdx.x]) : fmaxf(v, red[i][threadIdx.x]);
        unsigned* s = stats + (int64_t)bi * (C + 2);
        if (threadIdx.x < C) atomicMax(s + threadIdx.x, f32_to_ordered(v));
        else if (threadIdx.x == C) atomicMax(s + C, f32_to_ordered(-v));
        else if (v != 0.f) atomicOr(s + C + 1, 1u);
    }
    __syncthreads();
#pragma unroll
    for (int ci = 0; ci < C; ++ci) cmax[ci] = -INFINITY;
    cmin = INFINITY;
    bad = false;
}

// Generic form: any view subset / one head / scalar path / any scale (2-tap scalar math, runtime view flags).
// The default configuration (all views, two heads, W % 4 == 0) runs refine_col_kernel below.
template <int C, int VEC>
__global__ void __launch_bounds__(kRefineThreads) refine_kernel(const RefineParams p) {
    constexpr int CP = Lay<C>::CP, STRIDE = Lay<C>::STRIDE;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* row = reinterpret_cast<float*>(smem_raw);                                        // [w+2][STRIDE]
    float* soft_s = row + (size_t)(p.w + 2) * STRIDE;                                       // [C][threads][VEC]
    int64_t* ids_s = reinterpret_cast<int64_t*>(soft_s + (size_t)C * kRefineThreads * VEC); // [threads][VEC]
    __shared__ float red[kRefineThreads / 32][C + 2];

    const int64_t HW = (int64_t)p.H * p.W;
    const bool vP = p.views & UEM_VIEW_PROTO, vL = p.views & UEM_VIEW_PRED, vS = p.views & UEM_VIEW_SUP;
    const int64_t ignored_id = vS ? *p.ignored_id : -1;
    const bool have_maps = vP || vL;

    float cmax[C];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) cmax[ci] = -INFINITY;
    float cmin = INFINITY;
    bool bad = false;

    // persistent: CTA i owns the contiguous rows [R0, R1) of the flattened (image, row) space
    const int64_t total_rows = (int64_t)p.b * p.H;
    const int64_t R0 = total_rows * blockIdx.x / gridDim.x, R1 = total_rows * (blockIdx.x + 1) / gridDim.x;
    const int groups = p.W / VEC;
    int cur_b = -1;
    for (int64_t rr = R0; rr < R1; ++rr) {
        const int bi = (int)(rr / p.H), y = (int)(rr - (int64_t)bi * p.H);
        if (bi != cur_b) {
            if (cur_b >= 0 && p.stats) flush_stats<C>(p.stats, cur_b, cmax, cmin, bad, red);
            cur_b = bi;
        }
        const float* softb = p.soft + (int64_t)bi * C * HW;
        float* outb = p.out + (int64_t)bi * C * HW;
        const float* swb = p.sw + (int64_t)bi * (p.R + 1) * CP;  // row R of every image: the all-ones sentinel
        for (int g0 = 0; g0 < groups; g0 += kRefineThreads) {
            const int g = g0 + threadIdx.x;
            const bool active = g < groups;
            const int x0 = g * VEC;
            const int64_t px = (int64_t)y * p.W + x0;
            // ---- async: soft tile (+ ids) global -> shared, consumed by this same thread at the end
            if (active) {
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    float* dst = soft_s + ((size_t)ci * kRefineThreads + threadIdx.x) * VEC;
                    if constexpr (VEC == 4) cp_async_16(dst, softb + (int64_t)ci * HW + px);
                    else cp_async_4(dst, softb + (int64_t)ci * HW + px);
                }
                if (vS) {
                    int64_t* dst = ids_s + (size_t)threadIdx.x * VEC;
                    const int64_t* src = p.sup + (int64_t)bi * HW + px;
                    if constexpr (VEC == 4) { cp_async_16(dst, src); cp_async_16(dst + 2, src + 2); }
                    else cp_async_8(dst, src);
                }
            }
            cp_async_commit_group();
            if (have_maps && g0 == 0) {
                __syncthreads();  // previous row's readers are done
                stage_row<C>(row, p, bi, y);
                __syncthreads();
            }
            if (!active) { cp_async_wait_group<0>(); continue; }

            float wgt[C][VEC];
            {
                bool have = false;
                if (vP) {  // prototype view: softmax(T=1) of the up-sampled 1/distance, peak-normalised
#pragma unroll
                    for (int i = 0; i < VEC; ++i) {
                        const Lerp lx = make_lerp(x0 + i, p.w, p.sx);
                        float t0[CP], t1[CP], z[C];
                        load_tap<C>(row + lx.i0 * STRIDE, t0);
                        load_tap<C>(row + lx.i1 * STRIDE, t1);
#pragma unroll
                        for (int ci = 0; ci < C; ++ci) z[ci] = lx.l0 * t0[ci] + lx.l1 * t1[ci];
                        const float S = exp_shifted<C>(z);
                        const float rs = fmaf(-1e-7f, S, 1.0f);
#pragma unroll
                        for (int ci = 0; ci < C; ++ci) wgt[ci][i] = z[ci] * rs;
                    }
                    have = true;
                }
                if (vL) {  // prediction view: softmax(logits/temp), mean of the heads, peak-normalised
#pragma unroll
                    for (int i = 0; i < VEC; ++i) {
                        const Lerp lx = make_lerp(x0 + i, p.w, p.sx);
                        float t0[CP], t1[CP], z[C], acc[C];
                        load_tap<C>(row + lx.i0 * STRIDE + CP, t0);
                        load_tap<C>(row + lx.i1 * STRIDE + CP, t1);
#pragma unroll
                        for (int ci = 0; ci < C; ++ci) z[ci] = lx.l0 * t0[ci] + lx.l1 * t1[ci];
                        const float S1 = exp_shifted<C>(z);
                        if (p.n_pred == 2) {
                            float z2[C];
                            load_tap<C>(row + lx.i0 * STRIDE + 2 * CP, t0);
                            load_tap<C>(row + lx.i1 * STRIDE + 2 * CP, t1);
#pragma unroll
                            for (int ci = 0; ci < C; ++ci) z2[ci] = lx.l0 * t0[ci] + lx.l1 * t1[ci];
                            const float S2 = exp_shifted<C>(z2);
                            const float h1 = 0.5f * rcp_approx(S1), h2 = 0.5f * rcp_approx(S2);
                            float mx = 0.f;
#pragma unroll
                            for (int ci = 0; ci < C; ++ci) { acc[ci] = fmaf(z[ci], h1, z2[ci] * h2); mx = fmaxf(mx, acc[ci]); }
                            const float inv = rcp_approx(mx + 1e-7f);
#pragma unroll
                            for (int ci = 0; ci < C; ++ci) acc[ci] *= inv;
                        } else {
                            const float rs = fmaf(-1e-7f, S1, 1.0f);
#pragma unroll
                            for (int ci = 0; ci < C; ++ci) acc[ci] = z[ci] * rs;
                        }
#pragma unroll
                        for (int ci = 0; ci < C; ++ci) wgt[ci][i] = have ? wgt[ci][i] + acc[ci] : acc[ci];
                    }
                    have = true;
                }
                cp_async_wait_group<0>();
                if (vS) {  // superpixel view: per-region weights, multiplicative outside the ignored id
#pragma unroll
                    for (int i = 0; i < VEC; ++i) {
                        const int64_t rid = ids_s[(size_t)threadIdx.x * VEC + i];
                        if (rid != ignored_id && (uint64_t)rid < (uint64_t)p.R) {
                            float sw[CP];
#pragma unroll
                            for (int q = 0; q < CP / 4; ++q) {
                                const float4 v = __ldg(reinterpret_cast<const float4*>(swb + rid * CP) + q);
                                sw[4 * q] = v.x; sw[4 * q + 1] = v.y; sw[4 * q + 2] = v.z; sw[4 * q + 3] = v.w;
                            }
#pragma unroll
                            for (int ci = 0; ci < C; ++ci) wgt[ci][i] = have ? wgt[ci][i] * sw[ci] : sw[ci];
                        } else if (!have) {
#pragma unroll
                            for (int ci = 0; ci < C; ++ci) wgt[ci][i] = 1.0f;
                        }
                    }
                }
            }
            // ---- soft' = w*soft / (sum + 1e-7)   (alignment.py:291-292, :324-325)
#pragma unroll
            for (int ci = 0; ci < C; ++ci) {
                const float* sp = soft_s + ((size_t)ci * kRefineThreads + threadIdx.x) * VEC;
                if constexpr (VEC == 4) {
                    const float4 v = *reinterpret_cast<const float4*>(sp);
                    wgt[ci][0] *= v.x; wgt[ci][1] *= v.y; wgt[ci][2] *= v.z; wgt[ci][3] *= v.w;
                } else {
                    wgt[ci][0] *= sp[0];
                }
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                float s = 0.f;
#pragma unroll
                for (int ci = 0; ci < C; ++ci) s += wgt[ci][i];
                const float inv = rcp_approx(s + 1e-7f);
                bad |= !(s < INFINITY);
                float lo = INFINITY;
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const float o = wgt[ci][i] * inv;
                    wgt[ci][i] = o;
                    cmax[ci] = fmaxf(cmax[ci], o);
                    lo = fminf(lo, o);
                }
                cmin = fminf(cmin, lo);
            }
#pragma unroll
            for (int ci = 0; ci < C; ++ci) {
                PixVec<VEC> t;
#pragma unroll
                for (int i = 0; i < VEC; ++i) t.v[i] = wgt[ci][i];
                t.store(outb + (int64_t)ci * HW + px);
            }
        }
    }
    if (cur_b >= 0 && p.stats) flush_stats<C>(p.stats, cur_b, cmax, cmin, bad, red);
}

// ------------------------------------------------------------------------------------------------
// Column-walk kernel (default configuration: all three views, two heads, W % 4 == 0).
// A thread owns ONE image column of a strip of NT columns and walks down a contiguous range of rows, so everything
// that depends on the column only is hoisted out of the row loop:
//   * the horizontal half of the bilinear interpolation is done once per low-res row pair (every ~H/h output rows):
//     A_c = lerp_x(map[i0]), B_c = lerp_x(map[i1]) for the 3C (map, class) planes, kept in registers as
//     A' = kappa*A and D' = kappa*(B - A) (kappa = log2 e [/temp]); per output row the interpolated, pre-scaled
//     logit is ONE packed FFMA per class pair: z' = A' + t_y * D', and the softmax exponent is a bare EX2;
//   * no tap row in shared memory, no per-row vertical interpolation pass, and NO barrier of any kind in the row
//     loop: every thread copies its own 4C+8 bytes of a row (C soft planes + the superpixel id) global -> shared
//     with cp.async (LDGSTS, 128 contiguous bytes per warp and plane), NS-1 rows ahead, and reads back only what it
//     copied itself, so cp.async.wait_group is the only synchronisation (a first version that fed NT-column strips
//     with 512-byte cp.async.bulk copies was bound by the per-copy cost of the TMA unit: 66 us);
//   * the global stores are 32-bit per lane, contiguous over the warp (full 128-byte lines), class maps stay planar.
// 1 pixel per thread keeps the state at 6*PC registers + temporaries, so 5 CTAs of 128 threads are resident per SM.
// ------------------------------------------------------------------------------------------------
// region-weight gather: keep the table rows in L1 (neighbouring pixels and rows hit the same 32 bytes)
__device__ __forceinline__ float4 ldg_f4_l1(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::evict_last.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

#ifndef UEM_REFINE_COL_MINB
#define UEM_REFINE_COL_MINB 4   // 128 registers: no spills for C <= 8 (5 resident CTAs spill and run 30% slower at C = 7)
#endif

// VX = image columns per lane (1 or 2).  With VX = 2 a lane owns two adjacent columns: the per-row bookkeeping (loop,
// prefetch cursor, row coordinate, store addressing) is shared by two pixels, their two dependent chains interleave,
// shared-memory reads and global stores become 64-bit; the price is twice the column state (12*PC registers).
#ifndef UEM_REFINE_COL_MINB_VX2
#define UEM_REFINE_COL_MINB_VX2 3
#endif
#ifdef UEM_REFINE_TIMING
// development (tools/refine_timing.py): per-CTA %globaltimer stamps {entry, ignored id loaded, first setup done, first row
// landed, first row done, last row done, statistics flushed}
__device__ unsigned long long g_refine_t[1024][8];
#define UEM_T(i) do { if (threadIdx.x == 0 && blockIdx.x < 1024) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); g_refine_t[blockIdx.x][i] = t_; } } while (0)
#else
#define UEM_T(i) do { } while (0)
#endif
template <int C, int NT, int NS, int VX>
__global__ void __launch_bounds__(NT, ((VX == 2 ? UEM_REFINE_COL_MINB_VX2 : UEM_REFINE_COL_MINB) * 128) / NT)
refine_col_kernel(const RefineParams p, const int ncols_max) {
    UEM_T(0);
#ifdef UEM_REFINE_TIMING
    if (threadIdx.x == 0 && blockIdx.x < 1024) { unsigned sm_; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_)); g_refine_t[blockIdx.x][7] = sm_; }
#endif
    constexpr int CP = Lay<C>::CP, PC = Lay<C>::PC, NW = NT / 32, WC = 32 * VX;
    constexpr int TS = 3 * CP;                                   // floats per (row, low-res column) of the warp's tap scratch
    constexpr uint32_t kPlane = (uint32_t)WC * 4u;               // bytes of one soft plane of a warp row
    constexpr uint32_t kWarpStage = (uint32_t)WC * (4u * C + 8u);   // bytes of one row of a warp's WC columns
    constexpr int CPP = WC / 4;                                  // 16-byte chunks per soft plane
    constexpr int NCHUNK = CPP * C + WC / 2;                     // + the ids (2 per chunk)
    constexpr int NCP = (NCHUNK + 31) / 32;                      // cp.async per lane and row
    extern __shared__ __align__(128) unsigned char smem_col[];
    const int W = p.W, H = p.H, w = p.w, h = p.h;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int64_t HW = (int64_t)H * W;
    const int hw_low = h * w;
    const int nstrips = (W + NT * VX - 1) / (NT * VX);
    // shared memory: [warp][stage][C planes x WC floats | WC ids]  then  [warp][2 rows][ncols_max][TS] tap scratch
    unsigned char* const wstage = smem_col + (size_t)wid * NS * kWarpStage;
    float* const taps = reinterpret_cast<float*>(smem_col + (size_t)NW * NS * kWarpStage) + (size_t)wid * 2 * ncols_max * TS;

    // flattened (image, strip, row) space, row fastest; this CTA owns [U0, U1)
    const int64_t total = (int64_t)p.b * nstrips * H;
    const int64_t U0 = total * blockIdx.x / gridDim.x, U1 = total * (blockIdx.x + 1) / gridDim.x;
    const int n = (int)(U1 - U0);
    if (n <= 0) return;
    const int bs0 = (int)(U0 / H), y0 = (int)(U0 - (int64_t)bs0 * H);

    // ---- prefetch side.  A row of the warp's WC columns is NCHUNK 16-byte chunks (chunk k sits at byte 16k of the
    // stage: the planes are contiguous, ids follow); lane l copies chunks l, l+32, ... with cp.async.cg 16.
    // The source pointer of each chunk advances by one image row per unit; recomputed when the strip changes.
    // L2 hints only in the two-column build (c <= 6): the one-column build sits at its register limit, and the batches it
    // serves at c >= 7 (LoveDA) are larger than L2 anyway
    constexpr bool HINT = (VX == 2);
    const uint64_t pol_in = HINT ? l2_policy(p.l2_in) : 0ull;   // last reader of soft / ids on the fused chain: evict_first
    const uint64_t pol_out = HINT ? l2_policy(p.l2_out) : 0ull;
    const uint32_t wstage_u32 = smem_u32(wstage) + (uint32_t)lane * 16u;
    const uint32_t rd_base = smem_u32(wstage) + (uint32_t)lane * (4u * VX);
    int ibs = bs0, iy = y0, ibs_cur = -1;
    const char* csrc[NCP];
    uint32_t cstride[NCP];
    bool cvalid[NCP];
#pragma unroll
    for (int q = 0; q < NCP; ++q) { csrc[q] = nullptr; cstride[q] = 0; cvalid[q] = false; }
    auto prefetch = [&](int stage) {
        if (ibs != ibs_cur) {
            const int bi = ibs / nstrips, s = ibs - bi * nstrips;
            const int xw = s * NT * VX + wid * WC;
#pragma unroll
            for (int q = 0; q < NCP; ++q) {
                const int k = lane + 32 * q;
                if (k < CPP * C) {
                    const int ci = k / CPP, x = xw + (k - ci * CPP) * 4;
                    cvalid[q] = x < W;
                    csrc[q] = reinterpret_cast<const char*>(p.soft + ((int64_t)bi * C + ci) * HW + (int64_t)iy * W + (cvalid[q] ? x : 0));
                    cstride[q] = (uint32_t)W * 4u;
                } else {
                    const int x = xw + (k - CPP * C) * 2;
                    cvalid[q] = (k < NCHUNK) && x < W;
                    csrc[q] = reinterpret_cast<const char*>(p.sup + (int64_t)bi * HW + (int64_t)iy * W + (cvalid[q] ? x : 0));
                    cstride[q] = (uint32_t)W * 8u;
                }
            }
            ibs_cur = ibs;
        }
        const uint32_t d = wstage_u32 + (uint32_t)stage * kWarpStage;
#pragma unroll
        for (int q = 0; q < NCP; ++q) {
            if constexpr (HINT) {
                if (cvalid[q]) asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(d + 512u * q), "l"(csrc[q]), "l"(pol_in) : "memory");
            } else {
                if (cvalid[q]) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 512u * q), "l"(csrc[q]) : "memory");
            }
            csrc[q] += cstride[q];
        }
        if (++iy == H) { iy = 0; ++ibs; }
    };
#pragma unroll
    for (int s = 0; s < NS - 1; ++s) {   // inputs only: safe before the dependency wait
        if (s < n) prefetch(s);
        cp_async_commit_group();
    }
    // programmatic dependent launch: the similarity map, the region weights and the ignored id come from the
    // preceding kernels; everything above touched this kernel's inputs and its own shared memory only
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int64_t ignored_id = *p.ignored_id;
    const uint32_t ign_lo = ((uint64_t)ignored_id >> 32) == 0 ? (uint32_t)ignored_id : 0xffffffffu;
    const uint32_t Ru = (uint32_t)p.R;
#ifdef UEM_REFINE_TIMING
    if (ign_lo == 0x12345678u) return;   // force the load to complete before the stamp
#endif
    UEM_T(1);

    // column state: pre-scaled row-pair interpolants of the three maps (pairs of classes; padded slot -> e = 0)
    float2 A[VX][3][PC], D[VX][3][PC];
    int cur_bs = -1, cur_i0 = -1, cur_b = -1;
    int a0[VX], a1[VX], abase = 0, ncols = 1;
    float l0x[VX], l1x[VX];
#pragma unroll
    for (int v = 0; v < VX; ++v) { a0[v] = a1[v] = 0; l0x[v] = l1x[v] = 0.f; }
    bool active = false;
    const float* ob = nullptr;      // out + (bi*C)*HW
    uint32_t x = 0;                 // first of the lane's VX columns
    const float4* swb = nullptr;

    float cmax[C];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) cmax[ci] = -INFINITY;
    float cmin = INFINITY, nanacc = 0.f;

    auto flush = [&](int bi) {      // per warp: shuffle-reduce, one atomic per statistic
        float mn = warp_min(cmin);
        const int anybad = __any_sync(0xffffffffu, nanacc != nanacc);
        float mine = 0.f;
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            const float v = warp_max(cmax[ci]);
            if (lane == ci) mine = v;
            cmax[ci] = -INFINITY;
        }
        unsigned* srow = p.stats + (int64_t)bi * (C + 2);
        if (lane < C) { if (mine > -INFINITY) atomicMax(srow + lane, f32_to_ordered(mine)); }
        else if (lane == C) { if (mn < INFINITY) atomicMax(srow + C, f32_to_ordered(-mn)); }
        else if (lane == C + 1) { if (anybad) atomicOr(srow + C + 1, 1u); }
        cmin = INFINITY;
        nanacc = 0.f;
    };

    int bs = bs0, y = y0;
    int stage = 0, pstage = NS - 1;
    for (int it = 0; it < n; ++it) {
        __syncwarp();                            // every lane is done with the stage row it-1 has just left
        if (it + NS - 1 < n) prefetch(pstage);   // row it+NS-1 goes there
        cp_async_commit_group();
        if (bs != cur_bs) {        // new (image, strip): column geometry
            const int bi = bs / nstrips, s = bs - bi * nstrips;
            if (bi != cur_b) {
                if (cur_b >= 0 && p.stats) flush(cur_b);
                cur_b = bi;
            }
            const int xw = s * NT * VX + wid * WC;
            x = (uint32_t)(xw + lane * VX);
            active = (int)x < W;     // W % 4 == 0 and x % VX == 0: the lane's columns are all inside or all outside
#pragma unroll
            for (int v = 0; v < VX; ++v) {
                const Lerp lx = make_lerp(active ? (int)x + v : W - 1, w, p.sx);
                a0[v] = lx.i0; a1[v] = lx.i1; l0x[v] = lx.l0; l1x[v] = lx.l1;
            }
            abase = make_lerp(min(xw, W - 1), w, p.sx).i0;                      // warp-uniform: first low-res column
            ncols = make_lerp(min(xw + WC - 1, W - 1), w, p.sx).i1 - abase + 1;   // <= ncols_max
            ob = p.out + (int64_t)bi * C * HW;
            swb = reinterpret_cast<const float4*>(p.sw + (int64_t)bi * (p.R + 1) * CP);
            cur_bs = bs;
            cur_i0 = -1;
        }
        const Lerp ly = make_lerp(y, h, p.sy);
        if (ly.i0 != cur_i0) {
            // new low-res row pair.  The warp's WC columns span `ncols` low-res columns: their 2 x ncols x 3C values are
            // fetched once per warp (lane -> (map, class)), pre-scaled by log2 e [/temp], and every lane then reads the
            // four corners of each of its columns as 128-bit shared-memory loads and interpolates horizontally, once.
            cur_i0 = ly.i0;
            __syncwarp();
            if (lane < 3 * C) {
                const int m = lane / C, ci = lane - m * C;
                const float* plane = p.maps[m] + ((int64_t)cur_b * C + ci) * hw_low + abase;
                const float sc = p.map_scale[m];
                float* dst = taps + m * CP + ci;
                const float* r0 = plane + ly.i0 * w;
                const float* r1 = plane + ly.i1 * w;
                for (int j0 = 0; j0 < ncols; j0 += 4) {   // 8 loads in flight: one L2 round trip per 4 columns
                    float u0[4], u1[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int j = min(j0 + u, ncols - 1);
                        u0[u] = __ldg(r0 + j);
                        u1[u] = __ldg(r1 + j);
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        if (j0 + u < ncols) {
                            dst[(j0 + u) * TS] = u0[u] * sc;
                            dst[(ncols_max + j0 + u) * TS] = u1[u] * sc;
                        }
                }
            }
            __syncwarp();
#pragma unroll
            for (int v = 0; v < VX; ++v) {
                const float* t00 = taps + (a0[v] - abase) * TS;
                const float* t01 = taps + (a1[v] - abase) * TS;
                const float2 l0 = make_float2(l0x[v], l0x[v]), l1 = make_float2(l1x[v], l1x[v]);
#pragma unroll
                for (int m = 0; m < 3; ++m) {
                    float v00[CP], v01[CP], v10[CP], v11[CP];
                    load_tap<C>(t00 + m * CP, v00);
                    load_tap<C>(t01 + m * CP, v01);
                    load_tap<C>(t00 + ncols_max * TS + m * CP, v10);
                    load_tap<C>(t01 + ncols_max * TS + m * CP, v11);
#pragma unroll
                    for (int j = 0; j < PC; ++j) {
                        const bool pad = 2 * j + 1 >= C;   // odd class count: the last pair's second slot is padding
                        const float2 p00 = make_float2(v00[2 * j], pad ? 0.f : v00[2 * j + 1]);
                        const float2 p01 = make_float2(v01[2 * j], pad ? 0.f : v01[2 * j + 1]);
                        const float2 p10 = make_float2(v10[2 * j], pad ? 0.f : v10[2 * j + 1]);
                        const float2 p11 = make_float2(v11[2 * j], pad ? 0.f : v11[2 * j + 1]);
                        float2 ta = UEM_FFMA2(l1, p01, UEM_FMUL2(l0, p00));
                        const float2 tb = UEM_FFMA2(l1, p11, UEM_FMUL2(l0, p10));
                        float2 td = UEM_FADD2(tb, make_float2(-ta.x, -ta.y));
                        if (pad) { ta.y = -1e30f; td.y = 0.f; }   // EX2 gives exactly 0, never wins a max
                        A[v][m][j] = ta;
                        D[v][m][j] = td;
                    }
                }
            }
        }
        if (it == 0) UEM_T(2);
        cp_async_wait_group<NS - 1>();   // this lane's chunks of row `it` have landed ...
        __syncwarp();                    // ... and so have the other lanes' (the row is read across lanes)
        if (it == 0) UEM_T(3);
        if (active) {
            const uint32_t rd = rd_base + (uint32_t)stage * kWarpStage;   // this lane's first float of plane 0
            int64_t rid[VX];
            if constexpr (VX == 2)
                asm volatile("ld.shared.v2.b64 {%0,%1}, [%2];" : "=l"(rid[0]), "=l"(rid[1]) : "r"(rd + (uint32_t)lane * 8u + (uint32_t)C * kPlane));
            else
                asm volatile("ld.shared.b64 %0, [%1];" : "=l"(rid[0]) : "r"(rd + (uint32_t)lane * 4u + (uint32_t)C * kPlane));
            // superpixel view first (its gather is the only long-latency access of the row): multiplicative outside the
            // ignored id; the ignored id and any id outside [0,R) are redirected to the all-ones sentinel row R
            float4 swv[VX][CP / 4];
#pragma unroll
            for (int v = 0; v < VX; ++v) {
                const uint32_t lo = (uint32_t)rid[v], hi = (uint32_t)((uint64_t)rid[v] >> 32);
                const bool in_region = (hi == 0u) & (lo < Ru) & (lo != ign_lo);
                const uint32_t r = in_region ? lo : Ru;
                const float4* wp = swb + r * (uint32_t)(CP / 4);
#pragma unroll
                for (int q = 0; q < CP / 4; ++q) swv[v][q] = ldg_f4_l1(wp + q);
            }
            float sv[C][VX];
#pragma unroll
            for (int ci = 0; ci < C; ++ci) {
                if constexpr (VX == 2)
                    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(sv[ci][0]), "=f"(sv[ci][1]) : "r"(rd + (uint32_t)ci * kPlane));
                else
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(sv[ci][0]) : "r"(rd + (uint32_t)ci * kPlane));
            }
            const float2 t2 = make_float2(ly.l1, ly.l1);
            float o[C][VX];
#pragma unroll
            for (int v = 0; v < VX; ++v) {
                float2 wgt2[PC];
                {   // prototype view: softmax(T=1) of the up-sampled 1/distance, / (max + 1e-7) == e_c * (1 - 1e-7 S)
                    float2 z[PC];
#pragma unroll
                    for (int j = 0; j < PC; ++j) z[j] = UEM_FFMA2(t2, D[v][0][j], A[v][0][j]);
                    const float S = exp2_shifted2<PC>(z);
                    const float rs = fmaf(-1e-7f, S, 1.0f);
                    const float2 rs2 = make_float2(rs, rs);
#pragma unroll
                    for (int j = 0; j < PC; ++j) wgt2[j] = UEM_FMUL2(z[j], rs2);
                }
                {   // prediction view: mean of the two heads' softmax(logits/temp), / (max + 1e-7); the 0.5 of the mean is
                    // folded into the epsilon (q/(max q + 2e-7) == (q/2)/(max q/2 + 1e-7), exact power-of-two scaling)
                    float2 z[PC], z2[PC];
#pragma unroll
                    for (int j = 0; j < PC; ++j) {
                        z[j] = UEM_FFMA2(t2, D[v][1][j], A[v][1][j]);
                        z2[j] = UEM_FFMA2(t2, D[v][2][j], A[v][2][j]);
                    }
                    const float S1 = exp2_shifted2<PC>(z);
                    const float S2 = exp2_shifted2<PC>(z2);
                    // q_c = e1_c/S1 + e2_c/S2, scaled through by S1*S2 (in [1, C^2]): no reciprocal of the two sums
                    const float2 h1v = make_float2(S2, S2), h2v = make_float2(S1, S1);
                    float mx = 0.f;
#pragma unroll
                    for (int j = 0; j < PC; ++j) {
                        z[j] = UEM_FFMA2(z[j], h1v, UEM_FMUL2(z2[j], h2v));
                        mx = fmaxf(mx, fmaxf(z[j].x, z[j].y));
                    }
                    const float inv = rcp_approx(fmaf(2e-7f, S1 * S2, mx));
                    const float2 inv2 = make_float2(inv, inv);
#pragma unroll
                    for (int j = 0; j < PC; ++j) wgt2[j] = UEM_FFMA2(z[j], inv2, wgt2[j]);
                }
#pragma unroll
                for (int q = 0; q < CP / 4; ++q) {
                    wgt2[2 * q] = UEM_FMUL2(wgt2[2 * q], make_float2(swv[v][q].x, swv[v][q].y));
                    if (2 * q + 1 < PC) wgt2[2 * q + 1] = UEM_FMUL2(wgt2[2 * q + 1], make_float2(swv[v][q].z, swv[v][q].w));
                }
                // soft' = w*soft / (sum + 1e-7)   (alignment.py:291-292, :324-325)
#pragma unroll
                for (int ci = 0; ci < C; ++ci) o[ci][v] = ((ci & 1) ? wgt2[ci >> 1].y : wgt2[ci >> 1].x) * sv[ci][v];
                float ps[PC];   // pairwise tree: depth log2(C) instead of a chain of C dependent adds
#pragma unroll
                for (int j = 0; j < PC; ++j) ps[j] = (2 * j + 1 < C) ? o[2 * j][v] + o[2 * j + 1][v] : o[2 * j][v];
#pragma unroll
                for (int st2 = 1; st2 < PC; st2 *= 2)
#pragma unroll
                    for (int j = 0; j + st2 < PC; j += 2 * st2) ps[j] += ps[j + st2];
                const float s = ps[0];
                const float inv = rcp_approx(s + 1e-7f);
                nanacc = fmaf(s, 0.f, nanacc);   // s*0 accumulates to NaN iff a row sum was inf/NaN
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const float ov = o[ci][v] * inv;
                    o[ci][v] = ov;
                    cmax[ci] = fmaxf(cmax[ci], ov);
                    cmin = fminf(cmin, ov);
                }
            }
            const uint32_t idx = (uint32_t)y * (uint32_t)W + x;   // < 2^31: one plane of one image
#pragma unroll
            for (int ci = 0; ci < C; ++ci) {
                float* dst = const_cast<float*>(ob + (int64_t)ci * HW) + idx;
                if constexpr (VX == 2)
                    asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1,%2}, %3;" ::"l"(dst), "f"(o[ci][0]), "f"(o[ci][1]), "l"(pol_out) : "memory");
                else *dst = o[ci][0];
            }
        }
        if (it == 0) UEM_T(4);
        if (++y == H) { y = 0; ++bs; }
        pstage = stage;
        if (++stage == NS) stage = 0;
    }
    UEM_T(5);
    if (p.stats) flush(cur_b);
    UEM_T(6);
}

// superpixel-view weight of every (image, region): softmax(region_max/temp) / (max + 1e-7)  (alignment.py:252-253)
// table: (b,R,C) ordered-u32 (encoded != 0) or fp32 region maxima -> sw (b,R+1,CP); row R (the sentinel the ignored
// id and out-of-range ids are redirected to) is all ones.  On the fused chain the region-max kernel does this itself.
template <int C>
__global__ void __launch_bounds__(256) region_weight_kernel(const void* __restrict__ table, int encoded, int b, int64_t R,
                                                            const int64_t* __restrict__ ignored_ptr, float temp, float inv_temp,
                                                            int div_temp, float* __restrict__ sw) {
    constexpr int CP = Lay<C>::CP;
    const int64_t rows = (int64_t)b * (R + 1);
    (void)ignored_ptr;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t bi = i / (R + 1), rl = i - bi * (R + 1);
        float4* dst = reinterpret_cast<float4*>(sw + i * CP);
        if (rl == R) {
#pragma unroll
            for (int q = 0; q < CP / 4; ++q) dst[q] = make_float4(1.f, 1.f, 1.f, 1.f);
            continue;
        }
        const int64_t r = bi * R + rl;
        float z[C];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            float v;
            if (encoded) { const unsigned e = reinterpret_cast<const unsigned*>(table)[r * C + ci]; v = e ? ordered_to_f32(e) : 0.f; }
            else v = reinterpret_cast<const float*>(table)[r * C + ci];
            z[ci] = div_temp ? __fdiv_rn(v, temp) : v * inv_temp;
        }
        const float S = exp_shifted<C>(z);
        const float rs = fmaf(-1e-7f, S, 1.0f);
        float o[CP];
#pragma unroll
        for (int ci = 0; ci < CP; ++ci) o[ci] = ci < C ? z[ci < C ? ci : 0] * rs : 0.f;
#pragma unroll
        for (int q = 0; q < CP / 4; ++q) dst[q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    }
}

// a13: weight of each pixel's own hard-label class under the prototype view (alignment.py:295-309)
template <int C>
__global__ void __launch_bounds__(256) proto_weight_4pixel_kernel(const float* __restrict__ simi, int h, int w, int H, int W, float sy,
                                                                  float sx, const int64_t* __restrict__ hard, int64_t ignore_label,
                                                                  float eps, float* __restrict__ out) {
    extern __shared__ float prow[];
    const int y = blockIdx.x, bi = blockIdx.y;
    const Lerp ly = make_lerp(y, h, sy);
    for (int i = threadIdx.x; i < C * w; i += blockDim.x) {
        const int x = i % w, ci = i / w;
        const float* plane = simi + ((int64_t)bi * C + ci) * h * w;
        prow[i] = ly.l0 * __ldg(plane + (int64_t)ly.i0 * w + x) + ly.l1 * __ldg(plane + (int64_t)ly.i1 * w + x);
    }
    __syncthreads();
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        const Lerp lx = make_lerp(x, w, sx);
        float z[C];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) z[ci] = lx.l0 * prow[ci * w + lx.i0] + lx.l1 * prow[ci * w + lx.i1];
        softmax_regs<C>(z);
        float mx = z[0];
#pragma unroll
        for (int ci = 1; ci < C; ++ci) mx = fmaxf(mx, z[ci]);
        const float inv = 1.0f / (mx + eps);
        const int64_t l = hard[((int64_t)bi * H + y) * W + x];
        float o = 0.f;
#pragma unroll
        for (int ci = 0; ci < C; ++ci) o = (l == ci && l != ignore_label) ? z[ci] * inv : o;
        out[((int64_t)bi * H + y) * W + x] = o;
    }
}

static inline int64_t align16(int64_t x) { return (x + 15) & ~(int64_t)15; }
static inline int cp_of(int c) { return (c + 3) & ~3; }

static int sm_count() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = UEM_SMS;
    }
    return n;
}

template <typename K>
static int launch_persistent(K kernel, const RefineParams& p, int threads, size_t smem, cudaStream_t st) {
    if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    UEM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) per_sm = 1;
    const int64_t total_rows = (int64_t)p.b * p.H;
    const int grid = (int)min(total_rows, (int64_t)sm_count() * per_sm);
    kernel<<<grid, threads, smem, st>>>(p);
    return 0;
}

// column-walk kernel: strips of 128 columns, 4 rows in flight per CTA
#ifndef UEM_REFINE_COL_NS
#define UEM_REFINE_COL_NS 4
#endif
#ifndef UEM_REFINE_COL_NT
#define UEM_REFINE_COL_NT 128
#endif
#ifndef UEM_REFINE_COL_VX
#define UEM_REFINE_COL_VX 2
#endif
template <int C>
static int launch_refine_col(RefineParams p, cudaStream_t st, bool pdl, bool* done) {
    // two columns per lane while their state fits 168 registers (c <= 6); 7 and 8 classes would spill: one column
    constexpr int NT = UEM_REFINE_COL_NT, NS = UEM_REFINE_COL_NS, VX = (C <= 6) ? UEM_REFINE_COL_VX : 1;
    *done = false;
    constexpr float kL2E = 1.4426950408889634f;
    p.map_scale[0] = kL2E;
    p.map_scale[1] = p.map_scale[2] = (float)(1.4426950408889634 / (double)p.temp);
    // low-res columns one warp's 32*VX image columns can span (+1 for the right neighbour)
    int ncols_max = (int)((32 * VX - 1) * p.sx) + 3;
    if (ncols_max > p.w) ncols_max = p.w;
    const size_t smem = (size_t)NS * NT * VX * (4 * C + 8) + (size_t)(NT / 32) * 2 * ncols_max * 3 * cp_of(C) * 4;
    if (smem > 100 * 1024 || (int64_t)p.H * p.W >= ((int64_t)1 << 31)) return 0;   // generic kernels take it
    auto kernel = refine_col_kernel<C, NT, NS, VX>;
    if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    UEM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NT, smem));
    if (per_sm < 1) per_sm = 1;
    if (g_uem_refine_ctas_per_sm > 0 && per_sm > g_uem_refine_ctas_per_sm) per_sm = g_uem_refine_ctas_per_sm;
    const int nstrips = (p.W + NT * VX - 1) / (NT * VX);
    const int64_t total = (int64_t)p.b * nstrips * p.H;
    const int grid = (int)min(total, (int64_t)sm_count() * per_sm);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(NT, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    UEM_CUDA(cudaLaunchKernelEx(&cfg, kernel, p, ncols_max));
    *done = true;
    return 0;
}

// sw_ws: b*(R+1)*CP floats of scratch for the per-region weights (superpixel view only)
static int launch_refine(int views, const float* simi, const float* pred1, const float* pred2, int h, int w, const int64_t* sup,
                         const void* table, int table_encoded, int64_t R, const int64_t* ignored_id, const float* soft, int b,
                         int c, int H, int W, float temp, float* out, unsigned* stats, float* sw_ws, cudaStream_t st,
                         bool weights_ready = false, bool pdl = false) {
    // weights_ready: sw_ws already holds the per-region weights (fused tail of the region-max kernel); pdl: that kernel
    // directly precedes this launch in the stream, so the column-walk kernel may overlap its prologue with it
    UEM_REQUIRE(soft && out && b > 0 && H > 0 && W > 0, "uem_label_refine_f32: bad arguments");
    UEM_REQUIRE(views > 0 && views < 8, "uem_label_refine_f32: views must be a non-empty mask of UEM_VIEW_*");
    UEM_REQUIRE(temp > 0.f, "uem_label_refine_f32: temp must be > 0");  // alignment.py:313
    UEM_REQUIRE(R < ((int64_t)1 << 30), "uem_label_refine_f32: region capacity %lld too large", (long long)R);
    RefineParams p{};
    p.views = views;
    int ex;
    const bool pow2 = (frexpf(temp, &ex) == 0.5f);
    for (int m = 0; m < 3; ++m) p.map_scale[m] = 1.0f;
    if (views & UEM_VIEW_PROTO) { UEM_REQUIRE(simi, "uem_label_refine_f32: prototype view needs simi"); p.maps[0] = simi; }
    if (views & UEM_VIEW_PRED) {
        UEM_REQUIRE(pred1, "uem_label_refine_f32: prediction view needs pred1");
        p.maps[1] = pred1;
        p.n_pred = 1;
        if (pred2) { p.maps[2] = pred2; p.n_pred = 2; }
        if (pow2) p.map_scale[1] = p.map_scale[2] = 1.0f / temp;  // exact: scaling by 2^k commutes with rounding
    }
    const bool maps = views & (UEM_VIEW_PROTO | UEM_VIEW_PRED);
    if (views & UEM_VIEW_SUP)
        UEM_REQUIRE(sup && table && ignored_id && R > 0 && sw_ws, "uem_label_refine_f32: superpixel view needs sup, region table, ignored id, ws");
    if (maps) UEM_REQUIRE(h > 0 && w > 0, "uem_label_refine_f32: bad low-res size");
    if (!maps) { w = 0; h = 0; }
    p.b = b; p.h = h; p.w = w; p.H = H; p.W = W;
    p.sy = uem_align_corners_scale(h, H);
    p.sx = uem_align_corners_scale(w, W);
    p.temp = temp;
    p.div_temp = pow2 ? 0 : 1;
    p.sup = sup; p.sw = sw_ws; p.R = R; p.ignored_id = ignored_id;
    p.soft = soft; p.out = out; p.stats = stats;
    p.l2_in = (weights_ready && g_uem_l2_last_use) ? 1 : 0;   // on the fused chain this is the last read of soft / ids
    p.l2_out = g_uem_l2_keep;                                  // the selection reads `out` next
    const bool vec = (W % 4 == 0) && uem_aligned16(soft) && uem_aligned16(out) && (!sup || uem_aligned16(sup));
    // column-walk kernel: any up-sampling ratio, any low-res width
    const bool colwalk = vec && views == (UEM_VIEW_PROTO | UEM_VIEW_PRED | UEM_VIEW_SUP) && p.n_pred == 2;
    void *ev0 = nullptr, *ev1 = nullptr;
    int launched = 1, rc = 0;
    UEM_DISPATCH_C(c, {
        if ((views & UEM_VIEW_SUP) && !weights_ready) {
            const int64_t rows = (int64_t)b * (R + 1);
            region_weight_kernel<C><<<(int)min((int64_t)UEM_SMS * 4, (rows + 255) / 256), 256, 0, st>>>(
                table, table_encoded, b, R, ignored_id, temp, 1.0f / temp, p.div_temp, sw_ws);
            launched = 2;
        }
        uem_take_profile_events(&ev0, &ev1);
        if (ev0) UEM_CUDA(cudaEventRecord((cudaEvent_t)ev0, st));
        bool done = false;
        if (colwalk) rc = launch_refine_col<C>(p, st, pdl && weights_ready && !ev0, &done);
        if (!done && rc == 0) {
            const int vecw = vec ? 4 : 1;
            const size_t smem = (size_t)(w + 2) * Lay<C>::STRIDE * 4 + (size_t)C * kRefineThreads * vecw * 4 + (size_t)kRefineThreads * vecw * 8;
            UEM_REQUIRE(smem <= 200 * 1024, "uem_label_refine_f32: low-res width %d too large", w);
            if (vec) rc = launch_persistent(refine_kernel<C, 4>, p, kRefineThreads, smem, st);
            else rc = launch_persistent(refine_kernel<C, 1>, p, kRefineThreads, smem, st);
        }
    });
    if (rc) return rc;
    if (ev1) UEM_CUDA(cudaEventRecord((cudaEvent_t)ev1, st));
    UEM_CHECK_LAUNCH_N(launched);
    return 0;
}

}  // namespace

#ifdef UEM_REFINE_TIMING
extern "C" __attribute__((visibility("default"))) int uem_debug_refine_timing(unsigned long long* host_out /* [1024][8] */) {
    UEM_CUDA(cudaDeviceSynchronize());
    UEM_CUDA(cudaMemcpyFromSymbol(host_out, g_refine_t, sizeof(unsigned long long) * 1024 * 8));
    return 0;
}
#endif

extern "C" int uem_set_option(const char* name, int value) {
    UEM_REQUIRE(name, "uem_set_option: NULL name");
    if (strcmp(name, "refine_ctas_per_sm") == 0) { g_uem_refine_ctas_per_sm = value; return 0; }
    if (strcmp(name, "region_ctas_per_sm") == 0) { g_uem_region_ctas_per_sm = value; return 0; }
    if (strcmp(name, "proto_ctas_per_sm") == 0) { g_uem_proto_ctas_per_sm = value; return 0; }
    if (strcmp(name, "l2_stream") == 0) { g_uem_l2_stream = value ? 1 : 0; return 0; }
    if (strcmp(name, "l2_keep") == 0) { g_uem_l2_keep = value == 2 ? 2 : 0; return 0; }
    if (strcmp(name, "l2_region") == 0) { g_uem_l2_region = (value >= 0 && value <= 2) ? value : 0; return 0; }
    if (strcmp(name, "l2_last_use") == 0) { g_uem_l2_last_use = value ? 1 : 0; return 0; }
    return uem_fail("uem_set_option: unknown option '%s'", name);
}

extern "C" int64_t uem_class_stats_bytes(int b, int c) { return align16((int64_t)b * (c + 2) * 4); }

extern "C" int64_t uem_label_refine_ws_bytes(int b, int c, int64_t R, int W) {
    return align16((int64_t)b * ((R > 0 ? R : 0) + 1) * cp_of(c) * 4) + align16((int64_t)(W / 4 + 1) * 64);
}

extern "C" int uem_label_refine_f32(int views, const float* simi, const float* pred1, const float* pred2, int h, int w,
                                    const int64_t* sup, const float* region_max, int64_t R, const int64_t* ignored_id,
                                    const float* soft, int b, int c, int H, int W, float temp, float* out,
                                    uint32_t* class_stats, void* ws, void* stream) {
    return launch_refine(views, simi, pred1, pred2, h, w, sup, region_max, 0, R, ignored_id, soft, b, c, H, W, temp, out,
                         class_stats, (float*)ws, (cudaStream_t)stream);
}

extern "C" int uem_proto_weight_4pixel_f32(const float* simi, int h, int w, const int64_t* hard, int b, int c, int H, int W,
                                           int64_t ignore_label, float eps, float* out, void* stream) {
    UEM_REQUIRE(simi && hard && out && b > 0 && h > 0 && w > 0 && H > 0 && W > 0, "uem_proto_weight_4pixel_f32: bad arguments");
    const float sy = uem_align_corners_scale(h, H), sx = uem_align_corners_scale(w, W);
    UEM_DISPATCH_C(c, {
        size_t smem = (size_t)C * w * sizeof(float);
        UEM_REQUIRE(smem <= 48 * 1024, "uem_proto_weight_4pixel_f32: low-res width %d too large", w);
        dim3 grid(H, b);
        proto_weight_4pixel_kernel<C><<<grid, 256, smem, (cudaStream_t)stream>>>(simi, h, w, H, W, sy, sx, hard, ignore_label, eps, out);
    });
    UEM_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Fused chain: label_refine (all requested views) -> pseudo_selection (+ entropy / UVEM weight of the
// refined map), one C call, no host sync.  tools/train_ssl_uem.py:209-214, balance.py:372-396.
// ws layout (all 16-byte aligned):
//   [0]      status   int32[4]   bit1: label out of range, bit2: superpixel id outside [0,R)
//   [16]     --- self-cleaned block: zero on entry, zero again on exit; position depends on (b, c, R) only ---
//            maxid    int64[2]     [0] = batch max superpixel id (alignment.py:241), ids are >= 0
//            done     i32[b]       per-image arrival counters of the region-max kernel
//            stats    u32[b*(c+2)] class stats of the refined map (ordered-encoded, atomically raised)
//            region   u32[b*R*c]   ordered-encoded region maxima
//            --- plain scratch ---
//            simi     f32[b*c*h*w]
//            pearson ws (uem_pearson_ws_bytes)
//            sw       f32[b*(R+1)*CP] per-region superpixel-view weights (+ column tables)
// ------------------------------------------------------------------------------------------------
struct MineLayout {
    int64_t simi, pearson, sw, zero_begin, zero_end, maxid, done, stats, region, end;
};
static MineLayout mine_layout(int b, int c, int W, int h, int w, int k, int64_t R) {
    // The self-cleaned block comes first and depends on (b, c, R) only, so calls with different view subsets /
    // feature shapes on the same workspace agree on where it lives.
    MineLayout L;
    int64_t n = 16;
    L.zero_begin = n;
    L.maxid = n; n += 16;
    L.done = n; n += align16((int64_t)b * 4);
    L.stats = n; n += uem_class_stats_bytes(b, c);
    L.region = n; n += align16((int64_t)b * R * c * 4);
    L.zero_end = n;
    L.simi = n; n += align16((int64_t)b * c * h * w * 4);
    L.pearson = n; n += align16(uem_pearson_nchw_ws_bytes(b, (int64_t)h * w, c, k));
    L.sw = n; n += uem_label_refine_ws_bytes(b, c, R, W);
    L.end = n;
    return L;
}

extern "C" int64_t uem_mine_ws_bytes(int b, int c, int H, int W, int h, int w, int k, int64_t R) {
    (void)H;
    return mine_layout(b, c, W, h, w, k, R).end;
}
extern "C" int64_t uem_mine_ws_stats_offset(int b, int c, int H, int W, int h, int w, int k, int64_t R) {
    (void)H;
    return mine_layout(b, c, W, h, w, k, R).stats;
}
extern "C" int64_t uem_mine_ws_maxid_offset(int b, int c, int H, int W, int h, int w, int k, int64_t R) {
    (void)H;
    return mine_layout(b, c, W, h, w, k, R).maxid;
}

static bool mine_selfclean(int views, int c, int64_t R) {
    return (views & UEM_VIEW_SUP) && R > 0 && R * ((int64_t)cp_of(c) * 4 + 1) + 64 <= 200 * 1024;
}

// Region half of the fused chain on its own (multi-GPU form, SURVEY section 8e): region maxima of soft -> per-region
// superpixel-view weights, and the rank-LOCAL max superpixel id at byte offset uem_mine_ws_maxid_offset(...) of ws.
// The batch-global id (all-gather / all-reduce MAX across ranks, alignment.py:241) is only needed by the refine kernel,
// so this half can run one step ahead of the exchange; uem_mine_refine_select_f32 with UEM_VIEW_REGIONS_READY then skips
// it.  Same workspace, same self-cleaning protocol (the selection kernel zeroes the max-id slot again).  xchg: the id
// part of the step's multi-GPU send carried by the region-max kernel's last CTA, or nullptr.
static int mine_region_phase(const int64_t* sup, int64_t R, const float* soft, int b, int c, int H, int W, int h, int w, int k,
                             float temp, void* ws, const RegionXchg* xchg, void* stream) {
    UEM_REQUIRE(ws && soft && sup && b > 0 && H > 0 && W > 0, "uem_mine_region_phase_f32: bad arguments");
    UEM_REQUIRE(mine_selfclean(UEM_VIEW_SUP, c, R), "uem_mine_region_phase_f32: region capacity %lld does not fit the shared-memory table",
                (long long)R);
    char* base = (char*)ws;
    const MineLayout L = mine_layout(b, c, W, h, w, k, R);
    const int64_t HW = (int64_t)H * W;
    return uem_region_max_f32(soft, (int64_t)c * HW, HW, sup, b, HW, c, R, (unsigned*)(base + L.region), (int64_t*)(base + L.maxid),
                              (int*)base, (float*)(base + L.sw), (int*)(base + L.done), temp, (unsigned*)(base + L.stats), b * (c + 2),
                              xchg, (cudaStream_t)stream);
}

extern "C" int uem_mine_region_phase_f32(const int64_t* sup, int64_t R, const float* soft, int b, int c, int H, int W, int h,
                                         int w, int k, float temp, void* ws, void* stream) {
    return mine_region_phase(sup, R, soft, b, c, H, W, h, w, k, temp, ws, nullptr, stream);
}

// Same, and the LAST CTA of the region-max kernel also carries the id part of the step's multi-GPU send (uem_exchange.cu):
// this rank's max id goes into slot `slot` of every rank and, with global_id_out, the batch-global id (alignment.py:241) is
// left there once every rank's id of this step has arrived -- uem_xchg_send_f32(parts = 2) without a launch of its own.
extern "C" int uem_mine_region_phase_xchg_f32(const int64_t* sup, int64_t R, const float* soft, int b, int c, int H, int W, int h,
                                              int w, int k, float temp, void* ws, const void* const* peer_regions, int rank, int world,
                                              int depth, int slot, int64_t* global_id_out, void* stream) {
    UEM_REQUIRE(c > 0 && k > 0, "uem_mine_region_phase_xchg_f32: bad arguments");
    RegionXchg x{};
    if (int rc = fill_peers(&x.peers, peer_regions, rank, world, depth, slot, "uem_mine_region_phase_xchg_f32")) return rc;
    x.rank = rank; x.world = world; x.slot = slot; x.c = c; x.k = k;
    x.global_id_out = (long long*)global_id_out;
    return mine_region_phase(sup, R, soft, b, c, H, W, h, w, k, temp, ws, &x, stream);
}

extern "C" int uem_mine_proto_phase_f32(const float* feat, int k, const float* protos, int b, int c, int H, int W, int h, int w,
                                        int64_t R, float eps, void* ws, void* stream) {
    UEM_REQUIRE(ws && feat && protos && b > 0 && k > 0 && h > 0 && w > 0, "uem_mine_proto_phase_f32: bad arguments");
    (void)H;
    char* base = (char*)ws;
    const MineLayout L = mine_layout(b, c, W, h, w, k, R);
    return uem_pearson_dist_nchw_f32(feat, b, k, (int64_t)h * w, protos, c, eps, 1, (float*)(base + L.simi), base + L.pearson, stream);
}

// Side stream of the fused chain: the feature-map pass (Pearson similarity) and the soft/superpixel pass (region
// maxima) are independent until the refine kernel, so they are forked onto two streams and joined with events
// (capturable: inside a CUDA graph they become two parallel branches).  One set per host thread and device.
namespace {
struct SideStream {
    int device = -1;
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
int side_stream(SideStream** out) {
    static thread_local SideStream side[16];
    int dev = 0;
    UEM_CUDA(cudaGetDevice(&dev));
    UEM_REQUIRE(dev >= 0 && dev < 16, "uem_mine_refine_select_f32: device index %d out of range", dev);
    SideStream& s = side[dev];
    if (s.device != dev) {
        int least = 0, greatest = 0;
        UEM_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        UEM_CUDA(cudaStreamCreateWithPriority(&s.stream, cudaStreamNonBlocking, greatest));  // part of the critical chain
        UEM_CUDA(cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming));
        UEM_CUDA(cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming));
        s.device = dev;
    }
    *out = &s;
    return 0;
}
}  // namespace

extern "C" int uem_mine_refine_select_f32(int views, const float* feat, int k, const float* protos, const float* pred1,
                                          const float* pred2, int h, int w, const int64_t* sup, int64_t R,
                                          const int64_t* ignored_id, const float* soft, int b, int c, int H, int W, float temp,
                                          float eps, float cutoff_top, float cutoff_low, int64_t ignore_label, float* refined,
                                          int64_t* hard, const float* uvem /* NULL or host {m,t,1/gamma,coef_left,coef_right} */,
                                          float* entropy, float* weight, void* ws, void* stream) {
    UEM_REQUIRE(ws && soft && refined, "uem_mine_refine_select_f32: bad arguments");
    const bool regions_ready = (views & UEM_VIEW_REGIONS_READY) != 0;   // uem_mine_region_phase_f32 already ran on this ws
    const bool simi_ready = (views & UEM_VIEW_SIMI_READY) != 0;         // uem_mine_proto_phase_f32 already ran on this ws
    views &= ~(UEM_VIEW_REGIONS_READY | UEM_VIEW_SIMI_READY);
    cudaStream_t st = (cudaStream_t)stream;
    char* base = (char*)ws;
    const MineLayout L = mine_layout(b, c, W, h, w, k, R);
    int* status = (int*)base;
    float* simi = (float*)(base + L.simi);
    void* pws = base + L.pearson;
    float* sw = (float*)(base + L.sw);
    int64_t* maxid = (int64_t*)(base + L.maxid);
    unsigned* stats = (unsigned*)(base + L.stats);
    unsigned* table = (unsigned*)(base + L.region);
    const int64_t HW = (int64_t)H * W;
    int rc;
    // Self-cleaning fast path (superpixel view, region table fits shared memory): ws is zero on entry (zero-initialised
    // by the allocator, then kept clean by every call) -- the region-max kernel clears the class statistics, its tail
    // zeroes the table rows and arrival counters again, the selection kernel zeroes the max-id slot -- so no memset
    // node sits on the critical path.  Every other configuration zeroes the region before and after the call.
    const bool selfclean = mine_selfclean(views, c, R);
    UEM_REQUIRE(!regions_ready || (selfclean && ignored_id), "uem_mine_refine_select_f32: UEM_VIEW_REGIONS_READY needs the superpixel view, "
                "a region capacity that fits shared memory and the batch-global ignored id");
    if (!selfclean) UEM_CUDA(cudaMemsetAsync(base + L.zero_begin, 0, (size_t)(L.zero_end - L.zero_begin), st));
    // fork: the feature pass runs on the side stream while the region-max pass (below) runs on the caller's stream
    SideStream* side = nullptr;
    UEM_REQUIRE(!simi_ready || (views & UEM_VIEW_PROTO), "uem_mine_refine_select_f32: UEM_VIEW_SIMI_READY needs the prototype view");
    const bool fork = (views & UEM_VIEW_PROTO) && (views & UEM_VIEW_SUP) && !simi_ready;
    if ((views & UEM_VIEW_PROTO) && !simi_ready) {
        UEM_REQUIRE(feat && protos, "uem_mine_refine_select_f32: prototype view needs feat and prototypes");
        void* pst = stream;
        if (fork) {
            if ((rc = side_stream(&side))) return rc;
            UEM_CUDA(cudaEventRecord(side->fork, st));
            UEM_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
            pst = (void*)side->stream;
        }
        if ((rc = uem_pearson_dist_nchw_f32(feat, b, k, (int64_t)h * w, protos, c, eps, 1, simi, pws, pst))) return rc;
        if (fork) UEM_CUDA(cudaEventRecord(side->join, side->stream));
    }
    bool own_maxid = false;
    if (regions_ready) {
        own_maxid = true;   // the slot holds the rank-local id: the selection kernel zeroes it again
    } else if (views & UEM_VIEW_SUP) {
        UEM_REQUIRE(sup && R > 0, "uem_mine_refine_select_f32: superpixel view needs sup and a region capacity R");
        own_maxid = (ignored_id == nullptr);
        // region maxima of soft, NCHW viewed as (b,N,c): class stride HW; the batch max id (alignment.py:241) comes out
        // of the same pass when the caller did not supply it
        if (selfclean) {
            if ((rc = uem_region_max_f32(soft, (int64_t)c * HW, HW, sup, b, HW, c, R, table, own_maxid ? maxid : nullptr, status, sw,
                                         (int*)(base + L.done), temp, stats, b * (c + 2), nullptr, st)))
                return rc;
            if (own_maxid) ignored_id = maxid;
        } else {
            if (own_maxid) {
                if ((rc = uem_i64_max_accumulate(sup, (int64_t)b * HW, maxid, st))) return rc;
                ignored_id = maxid;
            }
            if ((rc = uem_region_table_f32(soft, (int64_t)c * HW, 1, HW, sup, b, HW, c, R, UEM_REDUCE_MAX, ignored_id, -1, 1, table,
                                           nullptr, status, st)))
                return rc;
        }
    }
    // join before the refine kernel reads simi; an event wait is a full dependency, so the programmatic overlap with
    // the region-max kernel is only requested when nothing else sits between the two launches
    if (fork) UEM_CUDA(cudaStreamWaitEvent(st, side->join, 0));
    if ((rc = launch_refine(views, simi, pred1, pred2, h, w, sup, table, 1, R, ignored_id, soft, b, c, H, W, temp, refined,
                            stats, sw, st, selfclean, selfclean && !regions_ready)))
        return rc;
    const bool select = hard || entropy || weight;
    if (select) {
        UEM_REQUIRE(hard, "uem_mine_refine_select_f32: entropy/weight outputs come with the selection (hard must be given)");
        UEM_REQUIRE(!(weight && !uvem), "uem_mine_refine_select_f32: weight output needs the uvem parameter block");
        if ((rc = uem_select_entropy_stats_impl(refined, stats, b, c, HW, cutoff_top, cutoff_low, ignore_label, hard, uvem, entropy,
                                                weight, (selfclean && own_maxid) ? maxid : nullptr, 1, st)))
            return rc;
    }
    if (selfclean && own_maxid && !select) UEM_CUDA(cudaMemsetAsync(maxid, 0, 16, st));
    if (!selfclean) {
        // leave the block clean -- except the class statistics: the drop-in pairing label_refine -> pseudo_selection reads
        // them after this call returns (mining.refine_select); every path clears them at entry (the memset above here,
        // the region-max kernel on the self-cleaning path), so they need not be zero on exit
        UEM_CUDA(cudaMemsetAsync(base + L.zero_begin, 0, (size_t)(L.stats - L.zero_begin), st));
        UEM_CUDA(cudaMemsetAsync(base + L.region, 0, (size_t)(L.zero_end - L.region), st));
    }
    return 0;
}
