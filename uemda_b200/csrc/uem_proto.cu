// a8: DownscaleLabel; a10-a12: masked class-prototype accumulation, soft-weighted accumulation, EMA.
// Reference: uemda/gast/alignment.py:484-509 (DownscaleLabel.forward), :328-355
// (_compute_local_prototypes), :107-126 (update_avg/init_avg), :92-105 (update_prototype_bytarget),
// :463-466 (_ema), :468-481 (_index2onehot).
//
// The reference builds one-hot tensors ((b,c+1,H,W) f32, (n,c) int64) and an (n,c,k) broadcast product
// (403 MB at config 2).  Here: DownscaleLabel is one pass over the int64 label map with per-thread
// register bins; the prototype sums read the NCHW feature map exactly once (TMA tiles and one-hot
// class planes when hw % 4 == 0, otherwise one warp per (image, channel rows) with the class ids staged
// as bytes in shared memory) into per-image partials, which every consumer folds over the batch in
// image order with the helpers of uem_proto_stats.cuh, so results are bit-reproducible run to run.
#include "uem_proto_stats.cuh"
#include "uem_tma.cuh"

#ifndef UEM_PROTO_RW
#define UEM_PROTO_RW 4   // channel rows per consumer warp of the TMA accumulate kernel (item = 8*RW channels of one image)
#endif

namespace {

// ------------------------------------------------------------------------------- DownscaleLabel
// one CTA per (output row, image): s input rows x W columns
template <int C>
__global__ void __launch_bounds__(512) downscale_kernel(const int64_t* __restrict__ label, int H, int W, int s, int h, int w,
                                                        int64_t ignore_label, float min_ratio, int vec,
                                                        int64_t* __restrict__ out, int32_t* __restrict__ status) {
    extern __shared__ unsigned bins[];  // [w][C+1]
    const int oy = blockIdx.x, bi = blockIdx.y;
    // blockDim = (column pairs, kRowGroups): the s input rows of a block row are spread over threadIdx.y so that all
    // of a thread's 128-bit loads are independent and issued together
    const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
    for (int i = tid; i < w * (C + 1); i += nthr) bins[i] = 0;
    __syncthreads();
    const int64_t* base = label + ((int64_t)bi * H + (int64_t)oy * s) * W;
    // trailing columns that do not fill a block are dropped (alignment.py:500); gridDim.z CTAs share one output row
    const int cells_per = (w + gridDim.z - 1) / gridDim.z;
    const int cxs = blockIdx.z * cells_per, cxe = min(w, cxs + cells_per);
    const int xs = cxs * s, xe = cxe * s;
    const int step = vec ? 2 : 1;
    int bad = 0;
    for (int x0 = xs + threadIdx.x * step; x0 < xe; x0 += blockDim.x * step) {
        unsigned cnt0[C + 1], cnt1[C + 1];
#pragma unroll
        for (int ci = 0; ci <= C; ++ci) { cnt0[ci] = 0; cnt1[ci] = 0; }
        const bool two = vec && (x0 + 1 < xe);
#pragma unroll 4
        for (int r = threadIdx.y; r < s; r += blockDim.y) {
            int64_t a, b2 = ignore_label;
            if (vec) ldg_i64x2(base + (int64_t)r * W + x0, a, b2);
            else a = ldg_i64(base + (int64_t)r * W + x0);
            int la = (a == ignore_label) ? C : (int)a;
            int lb = (b2 == ignore_label) ? C : (int)b2;
            bad |= (a != ignore_label && (a < 0 || a >= C)) || (b2 != ignore_label && (b2 < 0 || b2 >= C));
#pragma unroll
            for (int ci = 0; ci <= C; ++ci) { cnt0[ci] += (la == ci); cnt1[ci] += (lb == ci); }
        }
        const int c0 = x0 / s, c1 = (x0 + 1) / s;
        if (two && c1 == c0) {
#pragma unroll
            for (int ci = 0; ci <= C; ++ci) { unsigned v = cnt0[ci] + cnt1[ci]; if (v) atomicAdd(&bins[c0 * (C + 1) + ci], v); }
        } else {
#pragma unroll
            for (int ci = 0; ci <= C; ++ci) {
                if (cnt0[ci]) atomicAdd(&bins[c0 * (C + 1) + ci], cnt0[ci]);
                if (two && cnt1[ci]) atomicAdd(&bins[c1 * (C + 1) + ci], cnt1[ci]);
            }
        }
    }
    if (bad && status) atomicOr(status, 1);
    __syncthreads();
    const float area = (float)(s * s);
    for (int cx = cxs + tid; cx < cxe; cx += nthr) {
        const unsigned* bn = bins + cx * (C + 1);
        unsigned best = bn[0];
        int arg = 0;
#pragma unroll
        for (int ci = 1; ci <= C; ++ci)
            if (bn[ci] > best) { best = bn[ci]; arg = ci; }  // first index wins ties (torch.max)
        const float ratio = __fdiv_rn((float)best, area);   // avg_pool2d of the one-hot: count / (s*s)
        int64_t o = (arg == C || ratio < min_ratio) ? ignore_label : (int64_t)arg;
        out[((int64_t)bi * h + oy) * w + cx] = o;
    }
}

// Power-of-two scale factors (the reference hard-wires 16): s/2 consecutive lanes own one output cell, each lane
// streams its two columns over the s rows with independent 128-bit loads (BR in flight), and counts classes in packed
// 16-bit fields (two 64-bit registers hold bins 0..7, bin 8 separately), so a label costs a shift and an add instead
// of C+1 compares.  The lanes of a cell fold their counters with xor-shuffles; lane 0 takes the first-index argmax.
// BR = rows per batch of independent loads: 16 (128 registers, 2 CTAs/SM: lowest latency when the whole grid is resident
// at once) or 8 (3 CTAs/SM overlap their load and count phases: higher throughput on grids of several waves)
template <int C, int BR>
__device__ __forceinline__ void downscale_pow2_body(const int64_t* __restrict__ label, int H, int W, int s, int h, int w,
                                                    int64_t cells, int64_t ignore_label, float min_ratio,
                                                    int64_t* __restrict__ out, int32_t* __restrict__ status, int l2_in) {
    const uint64_t pol = l2_policy(l2_in);   // the full-resolution labels are read once
    const int tpc = s >> 1;  // lanes per cell (1..32)
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t cell = gid / tpc;
    const int sub = (int)(gid - cell * tpc);
    const bool live = cell < cells;
    unsigned long long lo = 0ull, hi = 0ull;
    unsigned b8 = 0u;
    int bad = 0;
    int ox = 0, oy = 0, bi = 0;
    if (live) {
        ox = (int)(cell % w);
        const int64_t t = cell / w;
        oy = (int)(t % h);
        bi = (int)(t / h);
        const int64_t* base = label + ((int64_t)bi * H + (int64_t)oy * s) * W + (int64_t)ox * s + sub * 2;
        auto add = [&](int64_t v) {
            const bool ign = (v == ignore_label);
            const bool oob = !ign && (v < 0 || v >= C);
            bad |= oob;
            const int bin = ign ? C : (int)v;  // ignore -> bin C (alignment.py:497)
            if (!oob) {
                const unsigned long long one = 1ull << ((bin & 3) * 16);
                if (bin < 4) lo += one;
                else if (bin < 8) hi += one;
                else ++b8;
            }
        };
        for (int r0 = 0; r0 < s; r0 += BR) {
            int64_t a[BR], c2[BR];
#pragma unroll
            for (int r = 0; r < BR; ++r)
                if (r0 + r < s) ldg_i64x2(base + (int64_t)(r0 + r) * W, a[r], c2[r], pol);
#pragma unroll
            for (int r = 0; r < BR; ++r)
                if (r0 + r < s) { add(a[r]); add(c2[r]); }
        }
    }
    for (int o = tpc >> 1; o > 0; o >>= 1) {
        lo += __shfl_xor_sync(0xffffffffu, lo, o);
        hi += __shfl_xor_sync(0xffffffffu, hi, o);
        b8 += __shfl_xor_sync(0xffffffffu, b8, o);
    }
    if (bad && status) atomicOr(status, 1);
    if (live && sub == 0) {
        unsigned best = (unsigned)(lo & 0xffffu);
        int arg = 0;
#pragma unroll
        for (int ci = 1; ci <= C; ++ci) {
            const unsigned v = ci < 4 ? (unsigned)((lo >> (16 * ci)) & 0xffffu) : (ci < 8 ? (unsigned)((hi >> (16 * (ci - 4))) & 0xffffu) : b8);
            if (v > best) { best = v; arg = ci; }  // first index wins ties (torch.max)
        }
        const float ratio = __fdiv_rn((float)best, (float)(s * s));  // avg_pool2d of the one-hot: count / (s*s)
        out[((int64_t)bi * h + oy) * w + ox] = (arg == C || ratio < min_ratio) ? ignore_label : (int64_t)arg;
    }
}

template <int C>
__global__ void __launch_bounds__(256) downscale_pow2_kernel(const int64_t* __restrict__ label, int H, int W, int s, int h, int w,
                                                             int64_t cells, int64_t ignore_label, float min_ratio,
                                                             int64_t* __restrict__ out, int32_t* __restrict__ status, int l2_in) {
    downscale_pow2_body<C, 16>(label, H, W, s, h, w, cells, ignore_label, min_ratio, out, status, l2_in);
}
template <int C>
__global__ void __launch_bounds__(256, 3) downscale_pow2_stream_kernel(const int64_t* __restrict__ label, int H, int W, int s, int h,
                                                                       int w, int64_t cells, int64_t ignore_label, float min_ratio,
                                                                       int64_t* __restrict__ out, int32_t* __restrict__ status, int l2_in) {
    downscale_pow2_body<C, 8>(label, H, W, s, h, w, cells, ignore_label, min_ratio, out, status, l2_in);
}

// ------------------------------------------------------------------------------- prototype sums
constexpr int kAccThreads = 256;  // 8 warps
constexpr int kChPerWarp = 4;     // channel rows per warp -> 32 channels per CTA

// stage the class ids of image bi as bytes (255 = ignore / out of range)
__device__ __forceinline__ void stage_labels(unsigned char* lab, const int64_t* __restrict__ label, int64_t hw, int c,
                                             int64_t ignore_label) {
    for (int64_t i = threadIdx.x; i < hw; i += blockDim.x) {
        int64_t v = label[i];
        lab[i] = (v >= 0 && v < c && v != ignore_label) ? (unsigned char)v : (unsigned char)255;
    }
}

// partial[(bi*C + ci)*k + kk] = sum over pixels of image bi with label ci of feat[bi,kk,:]
template <int C, int VEC>
__global__ void __launch_bounds__(kAccThreads) proto_accum_kernel(const float* __restrict__ feat, int k, int64_t hw,
                                                                  const int64_t* __restrict__ label, int64_t ignore_label,
                                                                  float* __restrict__ partial, int* __restrict__ cnt_partial) {
    extern __shared__ unsigned char lab[];
    const int bi = blockIdx.y;
    stage_labels(lab, label + (int64_t)bi * hw, hw, C, ignore_label);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (blockIdx.x == 0) {  // class counts of this image, once
        for (int ci = warp; ci < C; ci += kAccThreads / 32) {
            int n = 0;
            for (int64_t i = lane; i < hw; i += 32) n += (lab[i] == ci);
            n = __reduce_add_sync(0xffffffffu, n);
            if (lane == 0) cnt_partial[bi * C + ci] = n;
        }
    }
    // each warp streams kChPerWarp consecutive channel rows at once: kChPerWarp independent 128-bit loads in flight
    // per thread and step, the byte label of a pixel is read once for all of them
    const int kk0 = (blockIdx.x * (kAccThreads / 32) + warp) * kChPerWarp;
    if (kk0 >= k) return;
    const float* f = feat + ((int64_t)bi * k + kk0) * hw;
    float acc[kChPerWarp][C];
#pragma unroll
    for (int q = 0; q < kChPerWarp; ++q)
#pragma unroll
        for (int ci = 0; ci < C; ++ci) acc[q][ci] = 0.f;
    const int64_t groups = hw / VEC;
#pragma unroll 2
    for (int64_t g = lane; g < groups; g += 32) {
        PixVec<VEC> v[kChPerWarp];
#pragma unroll
        for (int q = 0; q < kChPerWarp; ++q)
            if (kk0 + q < k) v[q].load(f + (int64_t)q * hw + g * VEC);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int l = lab[g * VEC + i];
#pragma unroll
            for (int q = 0; q < kChPerWarp; ++q)
#pragma unroll
                for (int ci = 0; ci < C; ++ci) acc[q][ci] += (l == ci) ? v[q].v[i] : 0.f;
        }
    }
#pragma unroll
    for (int q = 0; q < kChPerWarp; ++q) {
        if (kk0 + q >= k) break;
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            float x = warp_sum(acc[q][ci]);
            if (lane == 0) partial[((int64_t)bi * C + ci) * k + kk0 + q] = x;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// TMA form of the masked class sums (hw % 4 == 0): persistent CTAs loop over (image, block of 8*RW channels) items
// and stream each item's [8*RW channels x 128 pixels] tiles (cp.async.bulk.tensor) through an mbarrier ring.
// The producer warp also turns the int64 labels of the tile's 128 pixels into C one-hot fp32 planes (published with
// the same full-barrier arrival as the tile), so the 8 consumer warps only do LDS.128 + packed FFMA2:
//     acc2[row][class] += (mask.x,mask.y)*(v.x,v.y) ; += (mask.z,mask.w)*(v.z,v.w)
// Per-image partial sums are folded afterwards in image order (deterministic).
// ------------------------------------------------------------------------------------------------
constexpr int kTilePx = 128;
constexpr int kTmaConsumers = 256;
constexpr int kTmaThreads = kTmaConsumers + 32;

template <int C, int RW>
struct ProtoTma {
    static constexpr int ROWS = 8 * RW;                      // channels per item / tile
    static constexpr int STAGES = 64 / ROWS * 2 > 8 ? 8 : 64 / ROWS * 2;  // ~64 KB of tiles in flight
    static constexpr int TILE_BYTES = ROWS * kTilePx * 4;
    static constexpr int MASK_BYTES = C * kTilePx * 4;
    static constexpr size_t SMEM = (size_t)STAGES * (TILE_BYTES + MASK_BYTES) + 2 * STAGES * 8;
};

template <int C, int RW>
__global__ void __launch_bounds__(kTmaThreads) proto_accum_tma_kernel(const __grid_constant__ CUtensorMap tmap, int k, int hw, int b,
                                                                      const int64_t* __restrict__ label, int64_t ignore_label,
                                                                      float* __restrict__ partial, int* __restrict__ cnt_partial,
                                                                      int l2_feat) {
    using P = ProtoTma<C, RW>;
    extern __shared__ __align__(128) unsigned char smem_q[];
    float* tiles = reinterpret_cast<float*>(smem_q);                                              // [STAGES][ROWS][128]
    float* masks = reinterpret_cast<float*>(smem_q + (size_t)P::STAGES * P::TILE_BYTES);          // [STAGES][C][128]
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_q + (size_t)P::STAGES * (P::TILE_BYTES + P::MASK_BYTES));
    uint64_t* empty = full + P::STAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb = (k + P::ROWS - 1) / P::ROWS, ntiles = (hw + kTilePx - 1) / kTilePx;
    const int total = b * nkb;

    if (threadIdx.x == 0) {
        for (int s = 0; s < P::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kTmaConsumers / 32); }
        mbar_fence_init();
    }
    __syncthreads();

    uint32_t T = 0;  // tiles handled so far by this CTA (ring position), same sequence on both sides
    if (warp == kTmaConsumers / 32) {
        if (lane == 0) tma_prefetch_desc(&tmap);
        const uint64_t pol = l2_policy(l2_feat);   // the feature map is read once
        // the labels of the NEXT tile are fetched while the current one waits for its ring slot, so the label round trip
        // never sits between two TMA issues
        auto fetch_labels = [&](int item, int t, int64_t (&l)[4]) {
            l[0] = l[1] = l[2] = l[3] = ignore_label;
            if (item < total) {
                const int bi = item / nkb;
                const int px = t * kTilePx + lane * 4;
                if (px < hw) load_ids<4>(label + (int64_t)bi * hw + px, l);  // hw % 4 == 0
            }
        };
        int64_t l[4];
        fetch_labels(blockIdx.x, 0, l);
        for (int item = blockIdx.x; item < total; item += gridDim.x) {
            const int bi = item / nkb, kb = item - bi * nkb;
            int cnt[C];
#pragma unroll
            for (int ci = 0; ci < C; ++ci) cnt[ci] = 0;
            for (int t = 0; t < ntiles; ++t, ++T) {
                const uint32_t s = T % P::STAGES, r = T / P::STAGES;
                int64_t ln[4];
                if (t + 1 < ntiles) fetch_labels(item, t + 1, ln);
                else fetch_labels(item + gridDim.x, 0, ln);
                if (r > 0) mbar_wait(&empty[s], (r - 1) & 1u);
                float* mk = masks + (size_t)s * C * kTilePx + lane * 4;
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    float4 m;
                    m.x = (l[0] == ci && l[0] != ignore_label) ? 1.f : 0.f;
                    m.y = (l[1] == ci && l[1] != ignore_label) ? 1.f : 0.f;
                    m.z = (l[2] == ci && l[2] != ignore_label) ? 1.f : 0.f;
                    m.w = (l[3] == ci && l[3] != ignore_label) ? 1.f : 0.f;
                    *reinterpret_cast<float4*>(mk + ci * kTilePx) = m;
                    cnt[ci] += (int)(m.x + m.y + m.z + m.w);
                }
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive_expect_tx(&full[s], P::TILE_BYTES);
                    tma_load_3d(tiles + (size_t)s * P::ROWS * kTilePx, &tmap, t * kTilePx, kb * P::ROWS, bi, &full[s], pol);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) l[i] = ln[i];
            }
            if (kb == 0) {  // class counts of this image, once
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const int n = __reduce_add_sync(0xffffffffu, cnt[ci]);
                    if (lane == 0) cnt_partial[bi * C + ci] = n;
                }
            }
        }
    } else {
        for (int item = blockIdx.x; item < total; item += gridDim.x) {
            const int bi = item / nkb, kb = item - bi * nkb;
            float2 acc2[RW][C];
#pragma unroll
            for (int q = 0; q < RW; ++q)
#pragma unroll
                for (int ci = 0; ci < C; ++ci) acc2[q][ci] = make_float2(0.f, 0.f);
            for (int t = 0; t < ntiles; ++t, ++T) {
                const uint32_t s = T % P::STAGES;
                mbar_wait(&full[s], (T / P::STAGES) & 1u);
                const float* tile = tiles + (size_t)s * P::ROWS * kTilePx + (size_t)(warp * RW) * kTilePx + lane * 4;
                const float* mk = masks + (size_t)s * C * kTilePx + lane * 4;
                float4 v[RW];
#pragma unroll
                for (int q = 0; q < RW; ++q) v[q] = *reinterpret_cast<const float4*>(tile + q * kTilePx);
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const float4 m = *reinterpret_cast<const float4*>(mk + ci * kTilePx);
                    const float2 m01 = make_float2(m.x, m.y), m23 = make_float2(m.z, m.w);
#pragma unroll
                    for (int q = 0; q < RW; ++q) {
                        acc2[q][ci] = __ffma2_rn(m01, make_float2(v[q].x, v[q].y), acc2[q][ci]);
                        acc2[q][ci] = __ffma2_rn(m23, make_float2(v[q].z, v[q].w), acc2[q][ci]);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
            }
#pragma unroll
            for (int q = 0; q < RW; ++q) {
                const int kk = kb * P::ROWS + warp * RW + q;
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const float x = warp_sum(acc2[q][ci].x + acc2[q][ci].y);
                    if (lane == 0 && kk < k) partial[((int64_t)bi * C + ci) * k + kk] = x;
                }
            }
        }
    }
}

// soft weights: bilinear (align_corners=True) down-sampling of soft (b,C,H,W) to (h,w) (alignment.py:102)
__global__ void __launch_bounds__(256) soft_down_kernel(const float* __restrict__ soft, int planes, int H, int W, int h, int w,
                                                        float sy, float sx, float* __restrict__ down) {
    const int64_t total = (int64_t)planes * h * w;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
        const int x = (int)(i % w);
        const int y = (int)((i / w) % h);
        const int64_t pl = i / ((int64_t)w * h);
        const Lerp ly = make_lerp(y, H, sy), lx = make_lerp(x, W, sx);
        const float* p = soft + pl * H * W;
        const float top = lx.l0 * p[(int64_t)ly.i0 * W + lx.i0] + lx.l1 * p[(int64_t)ly.i0 * W + lx.i1];
        const float bot = lx.l0 * p[(int64_t)ly.i1 * W + lx.i0] + lx.l1 * p[(int64_t)ly.i1 * W + lx.i1];
        down[i] = ly.l0 * top + ly.l1 * bot;
    }
}

// partial[(bi*C + ci)*k + kk] = sum_px feat[bi,kk,px] * down[bi,ci,px]
template <int C, int VEC>
__global__ void __launch_bounds__(kAccThreads) proto_accum_soft_kernel(const float* __restrict__ feat, int k, int64_t hw,
                                                                       const float* __restrict__ down, float* __restrict__ partial) {
    const int bi = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kk = blockIdx.x * (kAccThreads / 32) + warp;
    if (kk >= k) return;
    const float* f = feat + ((int64_t)bi * k + kk) * hw;
    const float* wd = down + (int64_t)bi * C * hw;
    float acc[C];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) acc[ci] = 0.f;
    const int64_t groups = hw / VEC;
    for (int64_t g = lane; g < groups; g += 32) {
        PixVec<VEC> v;
        v.load(f + g * VEC);
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[ci] = fmaf(v.v[i], __ldg(wd + (int64_t)ci * hw + g * VEC + i), acc[ci]);
        }
    }
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
        float x = warp_sum(acc[ci]);
        if (lane == 0) partial[((int64_t)bi * C + ci) * k + kk] = x;
    }
}

// fold the per-image partials (sums; counts when both are given)
__global__ void __launch_bounds__(256) proto_fold_kernel(const float* __restrict__ partial, const int* __restrict__ cnt_partial,
                                                         int b, int ck, int c, float* __restrict__ sums, int64_t* __restrict__ counts) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < ck) sums[i] = fold_images(partial, b, ck, i);
    if (counts && cnt_partial && i < c) counts[i] = fold_image_counts(cnt_partial, b, c, i);
}

__global__ void __launch_bounds__(256) proto_finalize_kernel(const float* __restrict__ sums, const int64_t* __restrict__ counts,
                                                             const float* __restrict__ proto_old, int c, int k, float eps,
                                                             float one_minus_decay, float decay, int64_t mean_n,
                                                             float* __restrict__ local_out, float* __restrict__ proto_new) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= c * k) return;
    const float old = proto_old[i];
    const float local = counts ? proto_local(sums[i], counts[i / k], old, eps)
                               : sums[i] / (float)mean_n;   // torch.mean over n pixels, alignment.py:104
    if (local_out) local_out[i] = local;
    if (proto_new) proto_new[i] = proto_ema_of(local, old, one_minus_decay, decay);
}

// fold of the per-image partials + local mean + keep-old rule + EMA in ONE launch: the single-GPU step needs neither the
// folded sums nor a separate fold kernel
__global__ void __launch_bounds__(256) proto_fold_finalize_kernel(const float* __restrict__ partial, const int* __restrict__ cnt_partial,
                                                                  int b, int c, int k, const float* __restrict__ proto_old, float eps,
                                                                  float one_minus_decay, float decay, float* __restrict__ proto_new) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= c * k) return;
    proto_new[i] = proto_ema(fold_images(partial, b, (int64_t)c * k, i), fold_image_counts(cnt_partial, b, c, i / k), proto_old[i], eps,
                             one_minus_decay, decay);
}

}  // namespace

extern "C" int uem_downscale_label_i64(const int64_t* label, int b, int H, int W, int scale, int n_classes, int64_t ignore_label,
                                       float min_ratio, int64_t* out, int32_t* status, void* stream) {
    UEM_REQUIRE(label && out && b > 0 && H > 0 && W > 0, "uem_downscale_label_i64: bad arguments");
    UEM_REQUIRE(scale > 1, "uem_downscale_label_i64: scale_factor must be > 1");  // alignment.py:488
    const int h = H / scale, w = W / scale;
    if (h == 0 || w == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int vec = (W % 2 == 0) && uem_aligned16(label) && (scale % 2 == 0);
    if (vec && (scale & (scale - 1)) == 0 && scale <= 64) {  // power of two: packed-counter kernel
        const int64_t cells = (int64_t)b * h * w;
        const int64_t threads = cells * (scale / 2);
        UEM_DISPATCH_C(n_classes, {
            const int nblk = uem_div_up(threads, 256);
            if (nblk <= 2 * UEM_SMS)
                downscale_pow2_kernel<C><<<nblk, 256, 0, st>>>(label, H, W, scale, h, w, cells, ignore_label, min_ratio, out, status, g_uem_l2_stream ? 1 : 0);
            else
                downscale_pow2_stream_kernel<C><<<nblk, 256, 0, st>>>(label, H, W, scale, h, w, cells, ignore_label, min_ratio, out, status, g_uem_l2_stream ? 1 : 0);
        });
        UEM_CHECK_LAUNCH();
        return 0;
    }
    // enough CTAs for ~4 waves: split every output row into column segments of whole cells
    int nseg = (int)min((int64_t)w, max((int64_t)1, (int64_t)(4 * UEM_SMS + (int64_t)h * b - 1) / ((int64_t)h * b)));
    nseg = min(nseg, 64);
    const int seg_cells = (w + nseg - 1) / nseg;
    const int cols = vec ? (seg_cells * scale + 1) / 2 : seg_cells * scale;
    const int threads = min(128, max(32, ((cols + 31) / 32) * 32));
    const int row_groups = scale >= 8 ? 4 : (scale >= 4 ? 2 : 1);
    UEM_DISPATCH_C(n_classes, {
        size_t smem = (size_t)w * (C + 1) * sizeof(unsigned);
        UEM_REQUIRE(smem <= 48 * 1024, "uem_downscale_label_i64: output width %d too large", w);
        dim3 grid(h, b, nseg);
        downscale_kernel<C><<<grid, dim3(threads, row_groups), smem, st>>>(label, H, W, scale, h, w, ignore_label, min_ratio, vec, out, status);
    });
    UEM_CHECK_LAUNCH();
    return 0;
}

// ws layout: [partial b*c*k f32][cnt_partial b*c i32]; the soft variant appends [down b*c*h*w f32]
extern "C" int64_t uem_proto_accum_ws_bytes(int b, int c, int k) {
    return (((int64_t)b * c * k + (int64_t)b * c + 4) * 4 + 15) & ~(int64_t)15;
}
extern "C" int64_t uem_proto_accum_soft_ws_bytes(int b, int c, int k, int h, int w) {
    return uem_proto_accum_ws_bytes(b, c, k) + (int64_t)b * c * h * w * 4;
}

extern "C" int uem_proto_accum_nchw_f32(const float* feat, int b, int k, int64_t hw, const int64_t* label, int c,
                                        int64_t ignore_label, float* sums, int64_t* counts, void* ws, void* stream) {
    UEM_REQUIRE(feat && label && ws && b > 0 && k > 0 && hw > 0 && (!sums == !counts), "uem_proto_accum_nchw_f32: bad arguments");
    UEM_REQUIRE(hw <= 200 * 1024, "uem_proto_accum_nchw_f32: %lld feature pixels per image exceed the shared-memory label stage", (long long)hw);
    cudaStream_t st = (cudaStream_t)stream;
    float* partial = (float*)ws;
    int* cnt_partial = (int*)proto_partials(ws, b, c, k).counts;
    // the TMA form reads the labels in 16-byte loads (load_ids<4>): both maps must be 16-byte aligned
    const bool vec = (hw % 4 == 0) && uem_aligned16(feat) && uem_aligned16(label);
    UEM_DISPATCH_C(c, {
        if (vec) {   // TMA form (hw fits int: at most 200K pixels)
            using P = ProtoTma<C, UEM_PROTO_RW>;
            CUtensorMap tmap;
            UEM_REQUIRE(uem_make_tmap_3d_f32(&tmap, feat, (uint64_t)hw, (uint64_t)k, (uint64_t)b, (uint64_t)hw, (uint64_t)k * hw, kTilePx,
                                             P::ROWS) == 0,
                        "uem_proto_accum_nchw_f32: cuTensorMapEncodeTiled failed");
            UEM_CUDA(cudaFuncSetAttribute(proto_accum_tma_kernel<C, UEM_PROTO_RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P::SMEM));
            int per_sm = 0;
            UEM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, proto_accum_tma_kernel<C, UEM_PROTO_RW>, kTmaThreads, P::SMEM));
            if (per_sm < 1) per_sm = 1;
            if (g_uem_proto_ctas_per_sm > 0 && per_sm > g_uem_proto_ctas_per_sm) per_sm = g_uem_proto_ctas_per_sm;
            const int total = b * uem_div_up(k, P::ROWS);
            const int nblk = min(total, UEM_SMS * per_sm);
            proto_accum_tma_kernel<C, UEM_PROTO_RW><<<nblk, kTmaThreads, P::SMEM, st>>>(tmap, k, (int)hw, b, label, ignore_label, partial,
                                                                                         cnt_partial, g_uem_l2_stream ? 1 : 0);
        } else {
            const dim3 grid(uem_div_up(k, (kAccThreads / 32) * kChPerWarp), b);
            const size_t smem = (size_t)((hw + 15) / 16) * 16;
            if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(proto_accum_kernel<C, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            proto_accum_kernel<C, 1><<<grid, kAccThreads, smem, st>>>(feat, k, hw, label, ignore_label, partial, cnt_partial);
        }
    });
    if (sums) proto_fold_kernel<<<uem_div_up((int64_t)c * k, 256), 256, 0, st>>>(partial, cnt_partial, b, c * k, c, sums, counts);
    UEM_CHECK_LAUNCH_N(sums ? 2 : 1);
    return 0;
}

extern "C" int uem_proto_fold_finalize_ema_f32(const void* ws, int b, int c, int k, const float* proto_old, float eps,
                                               float one_minus_decay, float decay, float* proto_new, void* stream) {
    UEM_REQUIRE(ws && proto_old && proto_new && b > 0 && c > 0 && k > 0, "uem_proto_fold_finalize_ema_f32: bad arguments");
    const ProtoPartials P = proto_partials(ws, b, c, k);
    proto_fold_finalize_kernel<<<uem_div_up((int64_t)c * k, 256), 256, 0, (cudaStream_t)stream>>>(P.sums, P.counts, b, c, k, proto_old, eps,
                                                                                                one_minus_decay, decay, proto_new);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_proto_accum_soft_f32(const float* feat, int b, int k, int h, int w, const float* soft, int c, int H, int W,
                                        float* sums, void* ws, void* stream) {
    UEM_REQUIRE(feat && soft && sums && ws && b > 0 && k > 0 && h > 0 && w > 0, "uem_proto_accum_soft_f32: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t hw = (int64_t)h * w;
    float* partial = (float*)ws;
    float* down = (float*)((char*)ws + uem_proto_accum_ws_bytes(b, c, k));
    const float sy = uem_align_corners_scale(H, h), sx = uem_align_corners_scale(W, w);
    const int64_t total = (int64_t)b * c * hw;
    soft_down_kernel<<<(int)min((int64_t)UEM_SMS * 8, (total + 255) / 256), 256, 0, st>>>(soft, b * c, H, W, h, w, sy, sx, down);
    const bool vec = (hw % 4 == 0) && uem_aligned16(feat);
    UEM_DISPATCH_C(c, {
        dim3 grid(uem_div_up(k, kAccThreads / 32), b);
        if (vec) proto_accum_soft_kernel<C, 4><<<grid, kAccThreads, 0, st>>>(feat, k, hw, down, partial);
        else proto_accum_soft_kernel<C, 1><<<grid, kAccThreads, 0, st>>>(feat, k, hw, down, partial);
    });
    proto_fold_kernel<<<uem_div_up((int64_t)c * k, 256), 256, 0, st>>>(partial, nullptr, b, c * k, c, sums, nullptr);
    UEM_CHECK_LAUNCH_N(3);
    return 0;
}

extern "C" int uem_proto_finalize_ema_f32(const float* sums, const int64_t* counts, int64_t mean_n, const float* proto_old, int c,
                                          int k, float eps, float one_minus_decay, float decay, float* local_out,
                                          float* proto_new, void* stream) {
    UEM_REQUIRE(sums && proto_old && c > 0 && k > 0 && (local_out || proto_new), "uem_proto_finalize_ema_f32: bad arguments");
    UEM_REQUIRE(counts || mean_n > 0, "uem_proto_finalize_ema_f32: need counts or mean_n");
    proto_finalize_kernel<<<uem_div_up((int64_t)c * k, 256), 256, 0, (cudaStream_t)stream>>>(
        sums, counts, proto_old, c, k, eps, one_minus_decay, decay, mean_n, local_out, proto_new);
    UEM_CHECK_LAUNCH();
    return 0;
}


// ------------------------------------------------------------------------------------------------
// Multi-GPU exchange helpers (SURVEY section 8e): the rank-local statistics of a step travel as ONE fp64 vector
// [c*k prototype sums | c counts | max superpixel id]; every part is exact in fp64.  One launch packs it, one launch
// folds the all-gathered (world, n) matrix in RANK ORDER (so every rank gets bit-identical sums) back into fp32 sums,
// int64 counts and the batch-global max id (alignment.py:241, :347-353).  They replace ~13 tiny elementwise launches
// that sat on the critical path of every sharded step.
// ------------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) pack_local_kernel(const float* __restrict__ sums, const int64_t* __restrict__ counts,
                                                         const int64_t* __restrict__ max_id, int ck, int c, double* __restrict__ out) {
    const int n = ck + c + 1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = i < ck ? (double)sums[i] : (i < ck + c ? (double)counts[i - ck] : (double)max_id[0]);
}
__global__ void __launch_bounds__(256) fold_gathered_kernel(const double* __restrict__ gathered, int world, int ck, int c,
                                                            float* __restrict__ sums, int64_t* __restrict__ counts,
                                                            int64_t* __restrict__ max_id) {
    const int n = ck + c + 1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        double tot = gathered[i];
        if (i < ck + c) {
            for (int r = 1; r < world; ++r) tot += gathered[(int64_t)r * n + i];   // rank order: identical on every rank
            if (i < ck) sums[i] = (float)tot;
            else counts[i - ck] = llrint(tot);
        } else {
            for (int r = 1; r < world; ++r) tot = fmax(tot, gathered[(int64_t)r * n + i]);
            max_id[0] = llrint(tot);
        }
    }
}
}  // namespace

namespace {
// per-image partials of proto_accumulate folded and packed in the same launch
__global__ void __launch_bounds__(256) pack_partials_kernel(const float* __restrict__ partial, const int* __restrict__ cnt_partial,
                                                            const int64_t* __restrict__ max_id, int b, int ck, int c,
                                                            double* __restrict__ out) {
    const int n = ck + c + 1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = i < ck ? (double)fold_images(partial, b, ck, i)
                        : (i < ck + c ? (double)fold_image_counts(cnt_partial, b, c, i - ck) : (double)max_id[0]);
}
}  // namespace

// ws: the per-image partials uem_proto_accum_nchw_f32 leaves when called with sums == NULL
extern "C" int uem_pack_local_partials_f64(const void* ws, int b, int c, int k, const int64_t* max_id, double* out, void* stream) {
    UEM_REQUIRE(ws && max_id && out && b > 0 && c > 0 && k > 0, "uem_pack_local_partials_f64: bad arguments");
    const ProtoPartials P = proto_partials(ws, b, c, k);
    const int n = c * k + c + 1;
    pack_partials_kernel<<<min(uem_div_up(n, 256), UEM_SMS), 256, 0, (cudaStream_t)stream>>>(P.sums, P.counts, max_id, b, c * k, c, out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_pack_local_f64(const float* sums, const int64_t* counts, const int64_t* max_id, int c, int k, double* out,
                                  void* stream) {
    UEM_REQUIRE(sums && counts && max_id && out && c > 0 && k > 0, "uem_pack_local_f64: bad arguments");
    const int n = c * k + c + 1;
    pack_local_kernel<<<min(uem_div_up(n, 256), UEM_SMS), 256, 0, (cudaStream_t)stream>>>(sums, counts, max_id, c * k, c, out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_fold_gathered_f64(const double* gathered, int world, int c, int k, float* sums, int64_t* counts,
                                     int64_t* max_id, void* stream) {
    UEM_REQUIRE(gathered && sums && counts && max_id && world > 0 && c > 0 && k > 0, "uem_fold_gathered_f64: bad arguments");
    const int n = c * k + c + 1;
    fold_gathered_kernel<<<min(uem_div_up(n, 256), UEM_SMS), 256, 0, (cudaStream_t)stream>>>(gathered, world, c * k, c, sums, counts,
                                                                                            max_id);
    UEM_CHECK_LAUNCH();
    return 0;
}
