// a9: Pearson distance between every feature vector and every class prototype.
// Reference: Aligner._pearson_dist, uemda/gast/alignment.py:424-451:
//   d[i,j] = ( -cov(f_i,p_j) / ((k-1+eps) * (std(f_i)*std(p_j) + eps)) + 1 ) * 0.5, unbiased std.
// The reference transposes NCHW features to (n,k) (alignment.py:213) and materialises an (n,c,k)
// product (:438-440, 403 MB at config 2).  Here the NCHW map is read exactly once, in place:
// threads run along the pixel dimension (128-bit loads, 128 B per class-of-8-lanes), the k dimension is
// split over 32 slices per CTA, and each thread keeps 2+m running sums per pixel:
//   S1 = sum g, S2 = sum g^2, Cj = sum g * pc_j      with g = f - pivot
// The pivot is the pixel's mean over 8 channels spread over k (channels i*(k/8)): an estimate of the per-pixel mean
// that is within sigma/sqrt(8) of it, so the one-pass variance S2 - S1^2/k loses ~1.1x (a 4-sigma channel-0 value used
// as the pivot would lose 17x) and |g| stays at the scale of the centred feature.  Measured against fp64 at k = 2048 on
// the near-prototype set (feat = proto + 0.05 noise, dist ~ 5e-4): 2.4e-7 absolute on dist, the reference's own fp32
// centre-then-dot form is at 1.7e-7 (tests/test_gpu_parity.py::test_pearson_benchmarked_shapes).
// where pc_j is the centred prototype (sum_k pc_j ~ 0, so centring f is unnecessary for the covariance;
// the residual mean(g)*sum(pc_j) is subtracted anyway).  HBM-bound on feat: 4k B per feature pixel.
#include "uem_common.cuh"
#include "uem_tma.cuh"

namespace {

constexpr int kPearsonThreads = 256;
constexpr int kPxLanes = 4;    // lanes along pixels; each handles VEC pixels (64 B of a channel row per warp quarter)
constexpr int kSlices = kPearsonThreads / kPxLanes;  // k-slices per CTA (64): 512 CTAs of 16 pixels at config 2
constexpr int kDepth = 8;      // cp.async ring depth per thread
constexpr int kPcStride = 8;   // transposed centred prototypes: pcT[kk][8] -> two LDG.128 fetch all classes of a channel

// centre the prototypes once: pc (m,k), stats[j] = {std_j (unbiased), sum_k pc_j}
__global__ void __launch_bounds__(256) proto_center_kernel(const float* __restrict__ protos, int k, int transposed,
                                                           float* __restrict__ pc, float* __restrict__ stats,
                                                           int* __restrict__ zero_ints, int n_zero) {
    const int j = blockIdx.x;
    if (j == 0)  // arrival counters of the k-split fold (uninitialised caller workspace)
        for (int i = threadIdx.x; i < n_zero; i += 256) zero_ints[i] = 0;
    const float* p = protos + (int64_t)j * k;
    __shared__ float red[8];
    __shared__ float bc;
    float s = 0.f;
    for (int i = threadIdx.x; i < k; i += 256) s += p[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { float t = 0.f; for (int i = 0; i < 8; ++i) t += red[i]; bc = t / (float)k; }
    __syncthreads();
    const float mean = bc;
    float s2 = 0.f, s1 = 0.f;
    for (int i = threadIdx.x; i < k; i += 256) {
        float d = p[i] - mean;
        if (transposed) {
            pc[(int64_t)i * kPcStride + j] = d;
            if (j == 0)  // unused class slots of the (k,8) table stay 0
                for (int u = gridDim.x; u < kPcStride; ++u) pc[(int64_t)i * kPcStride + u] = 0.f;
        } else {
            pc[(int64_t)j * k + i] = d;
        }
        s2 += d * d;
        s1 += d;
    }
    s2 = warp_sum(s2);
    s1 = warp_sum(s1);
    __syncthreads();
    __shared__ float red1[8];
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = s2; red1[threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float t2 = 0.f, t1 = 0.f;
        for (int i = 0; i < 8; ++i) { t2 += red[i]; t1 += red1[i]; }
        stats[2 * j] = sqrtf(t2 / (float)(k - 1));
        stats[2 * j + 1] = t1;
    }
}

__device__ __forceinline__ float pearson_finish(float S1, float S2, float Cj, float std_p, float sum_pc, int k, float eps,
                                                int reciprocal) {
    const float kf = (float)k;
    const float mean_g = S1 / kf;
    float var = (S2 - S1 * mean_g) / (float)(k - 1);
    var = fmaxf(var, 0.f);
    const float std_f = sqrtf(var);
    const float cov = (Cj - mean_g * sum_pc) / ((float)(k - 1) + eps);
    const float den = std_f * std_p + eps;
    const float d = (-1.0f * cov / den + 1.0f) * 0.5f;
    return reciprocal ? 1.0f / d : d;
}

// feat (b,k,hw) planar -> out (b,M,hw) planar
template <int M, int VEC>
__global__ void __launch_bounds__(kPearsonThreads, 4) pearson_nchw_kernel(const float* __restrict__ feat, int k, int64_t hw,
                                                                       const float* __restrict__ pc, const float* __restrict__ stats,
                                                                       float eps, int reciprocal, float* __restrict__ out) {
    constexpr int NA = 2 + M;
    constexpr int TILE = kPxLanes * VEC;
    const int bi = blockIdx.y;
    const int pl = threadIdx.x % kPxLanes, ks = threadIdx.x / kPxLanes;
    const int64_t px0 = (int64_t)blockIdx.x * TILE + pl * VEC;
    const bool active = px0 < hw;  // hw % VEC == 0 on the vector path
    const float* f = feat + (int64_t)bi * k * hw + px0;

    float acc[NA][VEC];
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[a][i] = 0.f;

    if (active) {
        PixVec<VEC> piv;   // mean over 8 spread channels: the shift that keeps the one-pass variance stable
        {
            const int kstep = k >> 3;
#pragma unroll
            for (int i = 0; i < VEC; ++i) piv.v[i] = 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                PixVec<VEC> q;
                q.load(f + (int64_t)(u * kstep) * hw);
#pragma unroll
                for (int i = 0; i < VEC; ++i) piv.v[i] += q.v[i];
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) piv.v[i] *= 0.125f;
        }
        auto consume = [&](const PixVec<VEC>& v, int kk) {
            float pcv[kPcStride];
            const float4 a = __ldg(reinterpret_cast<const float4*>(pc + (int64_t)kk * kPcStride));
            pcv[0] = a.x; pcv[1] = a.y; pcv[2] = a.z; pcv[3] = a.w;
            if (M > 4) {
                const float4 c4 = __ldg(reinterpret_cast<const float4*>(pc + (int64_t)kk * kPcStride) + 1);
                pcv[4] = c4.x; pcv[5] = c4.y; pcv[6] = c4.z; pcv[7] = c4.w;
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                const float g = v.v[i] - piv.v[i];
                acc[0][i] += g;
                acc[1][i] = fmaf(g, g, acc[1][i]);
#pragma unroll
                for (int j = 0; j < M; ++j) acc[2 + j][i] = fmaf(g, pcv[j], acc[2 + j][i]);
            }
        };
        if constexpr (VEC == 4) {
            // register-free software pipeline: every thread keeps kDepth 16-byte cp.async copies in flight in its own
            // shared-memory ring slots (128 B per thread, ~16 MB chip-wide: enough to cover HBM latency)
            __shared__ float4 ring[kDepth][kPearsonThreads];
            const int n_it = (k - ks + kSlices - 1) / kSlices;
#pragma unroll
            for (int d = 0; d < kDepth; ++d) {
                if (d < n_it) cp_async_16(&ring[d][threadIdx.x], f + (int64_t)(ks + d * kSlices) * hw);
                cp_async_commit_group();
            }
            for (int it = 0; it < n_it; ++it) {
                cp_async_wait_group<kDepth - 1>();
                const float4 q = ring[it % kDepth][threadIdx.x];
                if (it + kDepth < n_it) cp_async_16(&ring[it % kDepth][threadIdx.x], f + (int64_t)(ks + (it + kDepth) * kSlices) * hw);
                cp_async_commit_group();
                PixVec<VEC> v;
                v.v[0] = q.x; v.v[1] = q.y; v.v[2] = q.z; v.v[3] = q.w;
                consume(v, ks + it * kSlices);
            }
            cp_async_wait_group<0>();
        } else {
#pragma unroll 4
            for (int kk = ks; kk < k; kk += kSlices) {
                PixVec<VEC> v;
                v.load(f + (int64_t)kk * hw);
                consume(v, kk);
            }
        }
    }
    // fold the 8 slices that share a warp (lanes l, l+4, ..., l+28 hold the same pixels)
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            float x = acc[a][i];
            x += __shfl_xor_sync(0xffffffffu, x, 4);
            x += __shfl_xor_sync(0xffffffffu, x, 8);
            x += __shfl_xor_sync(0xffffffffu, x, 16);
            acc[a][i] = x;
        }
    __shared__ float red[kPearsonThreads / 32][TILE][NA + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane < kPxLanes) {
#pragma unroll
        for (int i = 0; i < VEC; ++i)
#pragma unroll
            for (int a = 0; a < NA; ++a) red[warp][lane * VEC + i][a] = acc[a][i];
    }
    __syncthreads();
    if (threadIdx.x < TILE) {
        const int64_t px = (int64_t)blockIdx.x * TILE + threadIdx.x;
        if (px < hw) {
            float s[NA];
#pragma unroll
            for (int a = 0; a < NA; ++a) {
                float t = 0.f;
#pragma unroll
                for (int wv = 0; wv < kPearsonThreads / 32; ++wv) t += red[wv][threadIdx.x][a];
                s[a] = t;
            }
#pragma unroll
            for (int j = 0; j < M; ++j)
                out[((int64_t)bi * M + j) * hw + px] =
                    pearson_finish(s[0], s[1], s[2 + j], stats[2 * j], stats[2 * j + 1], k, eps, reciprocal);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// TMA form (hw % 4 == 0): the NCHW map is streamed as [kKT channels x kPT pixels] tiles (cp.async.bulk.tensor,
// 16 KB each) through a kStages-deep mbarrier ring filled by a dedicated producer warp; 8 consumer warps keep the
// 2+M running sums of their 4 pixels in registers (packed FFMA2 over pixel pairs, the centred prototype as the
// scalar operand).  The k dimension is split over KS CTAs per pixel tile; their partial sums meet in an L2-resident
// scratch array and the last CTA to arrive adds them in split order (deterministic) and finishes the distance.
// ------------------------------------------------------------------------------------------------
constexpr int kPT = 128;      // pixels per tile (512 B rows)
constexpr int kKT = 32;       // channels per tile
constexpr int kStages = 4;    // tiles in flight per CTA (64 KB)
constexpr int kConsumers = 256;
constexpr int kTmaThreads = kConsumers + 32;

template <int M>
__global__ void __launch_bounds__(kTmaThreads) pearson_tma_kernel(const __grid_constant__ CUtensorMap tmap, const float* __restrict__ feat,
                                                                  int k, int hw, int kper, int KS, const float* __restrict__ pc,
                                                                  const float* __restrict__ stats, float eps, int reciprocal,
                                                                  float* __restrict__ gpart, int* __restrict__ arrivals,
                                                                  float* __restrict__ out, int l2_feat) {
    constexpr int NA = 2 + M;
    extern __shared__ __align__(128) unsigned char smem_p[];
    float* tiles = reinterpret_cast<float*>(smem_p);                                   // [kStages][kKT][kPT]
    float* pcs = tiles + (size_t)kStages * kKT * kPT;                                  // [kStages][kKT][kPcStride] centred prototypes
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_p + (size_t)kStages * (kKT * kPT + kKT * kPcStride) * 4);
    uint64_t* empty = full + kStages;
    float* part = reinterpret_cast<float*>(empty + kStages);                           // [NA][kPT] CTA partial
    __shared__ int s_last;
    const int ks = blockIdx.x % KS;
    const int ptile = blockIdx.x / KS, bi = blockIdx.y;
    const int px0 = ptile * kPT;
    const int kbeg = ks * kper, kend = min(k, kbeg + kper);
    const int ntiles = kend > kbeg ? (kend - kbeg + kKT - 1) / kKT : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumers / 32); }
        mbar_fence_init();
        tma_prefetch_desc(&tmap);
    }
    __syncthreads();

    if (warp == kConsumers / 32) {
        // ---- producer warp: one lane streams the tiles of this CTA's channel range
        if (lane == 0) {
            const uint64_t pol = l2_policy(l2_feat);   // the feature map is read once: evict_first keeps it from displacing the label maps
            for (int t = 0; t < ntiles; ++t) {
                const int s = t % kStages, r = t / kStages;
                if (r > 0) mbar_wait(&empty[s], (uint32_t)(r - 1) & 1u);
                const int kk0 = kbeg + t * kKT;
                const uint32_t pc_bytes = (uint32_t)min(kKT, k - kk0) * kPcStride * 4u;  // the tile's rows of the (k,8) table
                mbar_arrive_expect_tx(&full[s], kKT * kPT * 4 + pc_bytes);
                tma_load_3d(tiles + (size_t)s * kKT * kPT, &tmap, px0, kk0, bi, &full[s], pol);
                tma_load_1d(pcs + (size_t)s * kKT * kPcStride, pc + (int64_t)kk0 * kPcStride, pc_bytes, &full[s]);
            }
        }
        __syncwarp();
    } else {
        // ---- consumers: warp -> channels warp, warp+8, .. of the tile; lane -> 4 consecutive pixels
        const int px = px0 + lane * 4;
        const bool inb = px < hw;  // hw % 4 == 0
        float2 piv01 = make_float2(0.f, 0.f), piv23 = make_float2(0.f, 0.f);
        if (inb) {  // mean over 8 spread channels of these pixels: the shift that keeps the one-pass variance stable
            // (same channels, same order for every k split: the splits' partial sums share one pivot bit for bit)
            const float* f0 = feat + (int64_t)bi * k * hw + px;
            const int64_t kstep = (int64_t)(k >> 3) * hw;
            float4 q[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) q[u] = ldg_f4(f0 + u * kstep);
            float4 pv = q[0];
#pragma unroll
            for (int u = 1; u < 8; ++u) { pv.x += q[u].x; pv.y += q[u].y; pv.z += q[u].z; pv.w += q[u].w; }
            piv01 = make_float2(-0.125f * pv.x, -0.125f * pv.y);
            piv23 = make_float2(-0.125f * pv.z, -0.125f * pv.w);
        }
        float2 acc[NA][2];
#pragma unroll
        for (int a = 0; a < NA; ++a) { acc[a][0] = make_float2(0.f, 0.f); acc[a][1] = make_float2(0.f, 0.f); }
        for (int t = 0; t < ntiles; ++t) {
            const int s = t % kStages;
            mbar_wait(&full[s], (uint32_t)(t / kStages) & 1u);
            const float* tile = tiles + (size_t)s * kKT * kPT + lane * 4;
            const float* pct = pcs + (size_t)s * kKT * kPcStride;
            const int kk0 = kbeg + t * kKT;
#pragma unroll
            for (int j = 0; j < kKT / 8; ++j) {
                const int row = warp + 8 * j, kk = kk0 + row;
                if (kk < kend) {
                    const float4 v = *reinterpret_cast<const float4*>(tile + row * kPT);
                    const float4 p0 = *reinterpret_cast<const float4*>(pct + row * kPcStride);  // broadcast LDS.128
                    float pcv[kPcStride];
                    pcv[0] = p0.x; pcv[1] = p0.y; pcv[2] = p0.z; pcv[3] = p0.w;
                    if (M > 4) {
                        const float4 p1 = *reinterpret_cast<const float4*>(pct + row * kPcStride + 4);
                        pcv[4] = p1.x; pcv[5] = p1.y; pcv[6] = p1.z; pcv[7] = p1.w;
                    }
                    const float2 g01 = __fadd2_rn(make_float2(v.x, v.y), piv01), g23 = __fadd2_rn(make_float2(v.z, v.w), piv23);
                    acc[0][0] = __fadd2_rn(acc[0][0], g01);
                    acc[0][1] = __fadd2_rn(acc[0][1], g23);
                    acc[1][0] = __ffma2_rn(g01, g01, acc[1][0]);
                    acc[1][1] = __ffma2_rn(g23, g23, acc[1][1]);
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        const float2 pm = make_float2(pcv[m], pcv[m]);
                        acc[2 + m][0] = __ffma2_rn(g01, pm, acc[2 + m][0]);
                        acc[2 + m][1] = __ffma2_rn(g23, pm, acc[2 + m][1]);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
        }
        // ---- fold the 8 warps (channel sub-slices) of this CTA: red[warp][NA][pixel] in the drained tile ring
        asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");  // every consumer is past its last tile read
        float* red = tiles;
#pragma unroll
        for (int a = 0; a < NA; ++a)
            *reinterpret_cast<float4*>(red + ((size_t)warp * NA + a) * kPT + lane * 4) =
                make_float4(acc[a][0].x, acc[a][0].y, acc[a][1].x, acc[a][1].y);
        asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");
        if (threadIdx.x < kPT) {
#pragma unroll
            for (int a = 0; a < NA; ++a) {
                float sum = 0.f;
#pragma unroll
                for (int wv = 0; wv < kConsumers / 32; ++wv) sum += red[((size_t)wv * NA + a) * kPT + threadIdx.x];
                part[a * kPT + threadIdx.x] = sum;
            }
        }
    }
    // ---- fold the k splits: every CTA parks its partial sums in global memory (L2), the last one to arrive for this
    // (image, pixel tile) adds them in split order (deterministic) and finishes the distance.  (A thread-block cluster
    // with a DSMEM fold measured slower: the cluster barrier holds every CTA until the slowest of the group is done.)
    __syncthreads();
    float* mine = gpart + ((size_t)(blockIdx.y * (gridDim.x / KS) + ptile) * KS) * NA * kPT;
    if (KS > 1) {
        if (threadIdx.x < kPT) {
#pragma unroll
            for (int a = 0; a < NA; ++a) mine[((size_t)ks * NA + a) * kPT + threadIdx.x] = part[a * kPT + threadIdx.x];
        }
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = (atomicAdd(arrivals + blockIdx.y * (gridDim.x / KS) + ptile, 1) == KS - 1);
        __syncthreads();
        if (!s_last) return;
        __threadfence();
    }
    if (threadIdx.x < kPT) {
        const int px = px0 + threadIdx.x;
        float sacc[NA];
        if (KS > 1) {
#pragma unroll
            for (int a = 0; a < NA; ++a) sacc[a] = 0.f;
            for (int r = 0; r < KS; ++r) {
#pragma unroll
                for (int a = 0; a < NA; ++a) sacc[a] += __ldcg(mine + ((size_t)r * NA + a) * kPT + threadIdx.x);
            }
        } else {
#pragma unroll
            for (int a = 0; a < NA; ++a) sacc[a] = part[a * kPT + threadIdx.x];
        }
        if (px < hw) {
#pragma unroll
            for (int j = 0; j < M; ++j)
                out[((int64_t)bi * M + j) * hw + px] =
                    pearson_finish(sacc[0], sacc[1], sacc[2 + j], stats[2 * j], stats[2 * j + 1], k, eps, reciprocal);
        }
    }
    if (KS > 1 && threadIdx.x == 0) arrivals[blockIdx.y * (gridDim.x / KS) + ptile] = 0;  // clean for the next call
}

// generic row-major (n,k) x (m,k): one warp per feat1 row, classes in chunks of 8
__global__ void __launch_bounds__(256) pearson_rows_kernel(const float* __restrict__ f1, int64_t n, int k, const float* __restrict__ pc,
                                                           const float* __restrict__ stats, int m, float eps, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n) return;
    const float* f = f1 + row * k;
    float piv = 0.f;   // mean over 8 spread elements (see the header comment)
#pragma unroll
    for (int u = 0; u < 8; ++u) piv += f[u * (k >> 3)];
    piv *= 0.125f;
    for (int j0 = 0; j0 < m; j0 += 8) {
        const int mj = min(8, m - j0);
        float S1 = 0.f, S2 = 0.f, Cj[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) Cj[j] = 0.f;
        for (int kk = lane; kk < k; kk += 32) {
            const float g = f[kk] - piv;
            S1 += g;
            S2 = fmaf(g, g, S2);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < mj) Cj[j] = fmaf(g, __ldg(pc + (int64_t)(j0 + j) * k + kk), Cj[j]);
        }
        S1 = warp_sum(S1);
        S2 = warp_sum(S2);
#pragma unroll
        for (int j = 0; j < 8; ++j) Cj[j] = warp_sum(Cj[j]);
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < mj)
                    out[row * m + j0 + j] = pearson_finish(S1, S2, Cj[j], stats[2 * (j0 + j)], stats[2 * (j0 + j) + 1], k, eps, 0);
        }
    }
}

}  // namespace

// ws layout: [pc max(m,8)*k f32 (row-major (m,k), or transposed (k,8) for the NCHW kernel)][stats 2*m f32]
extern "C" int64_t uem_pearson_ws_bytes(int m, int k) {
    const int64_t rows = m > kPcStride ? m : kPcStride;
    return (rows * k + 2 * (int64_t)m + 4) * sizeof(float);
}

// k split of the TMA kernel: at most ~2 CTAs per SM (all resident at once), each with at least 4 tiles of its own
static int pearson_ksplit(int b, int64_t hw, int k) {
    const int ptiles = uem_div_up(hw, kPT);
    int KS = 1;
    while (KS < 8 && (int64_t)ptiles * b * KS * 2 <= 2 * UEM_SMS && k / (KS * 2) >= 4 * kKT) KS *= 2;
    return KS;
}

// NCHW entry: [pc k*8 f32][stats 2*m f32 (+pad)][arrival counters b*ptiles i32][k-split partial sums]
extern "C" int64_t uem_pearson_nchw_ws_bytes(int b, int64_t hw, int m, int k) {
    const int64_t ptiles = (hw + kPT - 1) / kPT;
    const int KS = pearson_ksplit(b, hw, k);
    int64_t n = ((int64_t)kPcStride * k + 2 * (int64_t)m + 4) * 4;
    n = (n + 15) & ~(int64_t)15;
    n += ((int64_t)b * ptiles * 4 + 15) & ~(int64_t)15;
    n += (KS > 1) ? (int64_t)b * ptiles * KS * (2 + m) * kPT * 4 : 0;
    return n;
}

extern "C" int uem_pearson_dist_nchw_f32(const float* feat, int b, int k, int64_t hw, const float* protos, int m, float eps,
                                         int reciprocal, float* out, void* ws, void* stream) {
    UEM_REQUIRE(feat && protos && out && ws && b > 0 && k > 0 && hw > 0, "uem_pearson_dist_nchw_f32: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    float* pc = (float*)ws;
    float* stats = pc + (int64_t)kPcStride * k;
    const int64_t ptiles64 = (hw + kPT - 1) / kPT;
    int* arrivals = (int*)((char*)ws + ((((int64_t)kPcStride * k + 2 * (int64_t)m + 4) * 4 + 15) & ~(int64_t)15));
    float* gpart = (float*)((char*)arrivals + (((int64_t)b * ptiles64 * 4 + 15) & ~(int64_t)15));
    const bool vec = (hw % 4 == 0) && uem_aligned16(feat);
    const bool tma = vec && hw < (1 << 30) && k >= kKT;
    UEM_DISPATCH_C(m, {
        proto_center_kernel<<<C, 256, 0, st>>>(protos, k, 1, pc, stats, arrivals, tma ? (int)(b * ptiles64) : 0);
        if (tma) {
            CUtensorMap tmap;
            UEM_REQUIRE(uem_make_tmap_3d_f32(&tmap, feat, (uint64_t)hw, (uint64_t)k, (uint64_t)b, (uint64_t)hw, (uint64_t)k * hw, kPT,
                                             kKT) == 0,
                        "uem_pearson_dist_nchw_f32: cuTensorMapEncodeTiled failed");
            const int ptiles = uem_div_up(hw, kPT);
            const int KS = pearson_ksplit(b, hw, k);
            const int kper = ((k + KS - 1) / KS + kKT - 1) / kKT * kKT;
            const size_t smem = (size_t)kStages * (kKT * kPT + kKT * kPcStride) * 4 + 2 * kStages * 8 + (size_t)kPT * (2 + C) * 4;
            UEM_CUDA(cudaFuncSetAttribute(pearson_tma_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            pearson_tma_kernel<C><<<dim3(ptiles * KS, b), kTmaThreads, smem, st>>>(tmap, feat, k, (int)hw, kper, KS, pc, stats, eps, reciprocal,
                                                                                   gpart, arrivals, out, g_uem_l2_stream ? 1 : 0);
        } else if (vec) {
            dim3 grid(uem_div_up(hw, kPxLanes * 4), b);
            pearson_nchw_kernel<C, 4><<<grid, kPearsonThreads, 0, st>>>(feat, k, hw, pc, stats, eps, reciprocal, out);
        } else {
            dim3 grid(uem_div_up(hw, kPxLanes), b);
            pearson_nchw_kernel<C, 1><<<grid, kPearsonThreads, 0, st>>>(feat, k, hw, pc, stats, eps, reciprocal, out);
        }
    });
    UEM_CHECK_LAUNCH_N(2);
    return 0;
}

extern "C" int uem_pearson_dist_rows_f32(const float* feat1, int64_t n, int k, const float* feat2, int m, float eps, float* out,
                                         void* ws, void* stream) {
    UEM_REQUIRE(feat1 && feat2 && out && ws && n > 0 && k > 0 && m > 0, "uem_pearson_dist_rows_f32: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    float* pc = (float*)ws;
    float* stats = pc + (int64_t)(m > kPcStride ? m : kPcStride) * k;
    proto_center_kernel<<<m, 256, 0, st>>>(feat2, k, 0, pc, stats, nullptr, 0);
    pearson_rows_kernel<<<uem_div_up(n, 8), 256, 0, st>>>(feat1, n, k, pc, stats, m, eps, out);
    UEM_CHECK_LAUNCH_N(2);
    return 0;
}
