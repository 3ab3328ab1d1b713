// Next row (SURVEY 8f-2): PrototypeContrastiveLoss, forward and backward, fused.
// Reference: uemda/loss.py:10-47, called at tools/train_align_uem.py:176-177:
//     feat (b,k,h,w) -> rows (N,k); drop ignore-label pixels; f^ = f / max(||f||, 1e-12), P^ likewise;
//     logits = f^ P^T / T;  loss = mean_valid CrossEntropy(logits, label)
// The reference permutes the NCHW feature map into an (N,k) copy, normalises it (another copy), multiplies by the
// (k,c) prototype matrix and lets autograd replay all of it backwards.  Here the map is read in place, twice:
//   forward   one TMA-tiled pass over feat (same ring as the Pearson kernel): per pixel sum f^2 and the c dot products
//             with the normalised prototypes; the finishing threads turn them into logits, the CE term and the
//             per-pixel backward coefficients a_j = G_j / (n T), beta = sum_j a_j (f.P^_j) / n^2, G = (softmax - onehot)/Nv;
//   backward  one TMA-tiled pass: grad[k,px] = g_out * (sum_j a_j[px] P^_j[k] - beta[px] f[k,px]), written with 128-bit
//             stores (d/df of f/||f|| is (I - f^ f^T)/||f||).
// Both passes are HBM-bound (4k B read per feature pixel; the backward also writes 4k B): CUDA cores, N = c <= 8.
#include "uem_common.cuh"
#include "uem_tma.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace {

constexpr int kPT = 128;      // pixels per tile
constexpr int kKT = 32;       // channels per tile
constexpr int kStages = 4;
constexpr int kConsumers = 256;
constexpr int kThreads = kConsumers + 32;
constexpr int kPS = 8;        // stride of the transposed normalised prototype table ph[k][8]

// blocks 0..m-1: ph[kk][j] = P[j][kk] / max(||P_j||, 1e-12) (F.normalize); block m: number of non-ignored labels
__global__ void __launch_bounds__(256) pcl_prep_kernel(const float* __restrict__ protos, int m, int k, const int64_t* __restrict__ labels,
                                                       int64_t n, int64_t ignore_label, float* __restrict__ ph,
                                                       long long* __restrict__ nvalid) {
    __shared__ float red[8];
    __shared__ long long redl[8];
    const int j = blockIdx.x;
    if (j == m) {
        long long cnt = 0;
        for (int64_t i = threadIdx.x; i < n; i += 256) cnt += (labels[i] != ignore_label);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if ((threadIdx.x & 31) == 0) redl[threadIdx.x >> 5] = cnt;
        __syncthreads();
        if (threadIdx.x == 0) {
            long long t = 0;
            for (int i = 0; i < 8; ++i) t += redl[i];
            nvalid[0] = t;
        }
        return;
    }
    const float* p = protos + (int64_t)j * k;
    float s2 = 0.f;
    for (int i = threadIdx.x; i < k; i += 256) s2 = fmaf(p[i], p[i], s2);
    s2 = warp_sum(s2);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s2;
    __syncthreads();
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    const float inv = 1.0f / fmaxf(sqrtf(t), 1e-12f);
    for (int i = threadIdx.x; i < k; i += 256) {
        ph[(int64_t)i * kPS + j] = p[i] * inv;
        if (j == 0)
            for (int u = m; u < kPS; ++u) ph[(int64_t)i * kPS + u] = 0.f;
    }
}

struct Ring {
    float* tiles;
    float* tabs;
    uint64_t* full;
    uint64_t* empty;
};
__device__ __forceinline__ Ring ring_carve(unsigned char* smem) {
    Ring r;
    r.tiles = reinterpret_cast<float*>(smem);
    r.tabs = r.tiles + (size_t)kStages * kKT * kPT;
    r.full = reinterpret_cast<uint64_t*>(smem + (size_t)kStages * (kKT * kPT + kKT * kPS) * 4);
    r.empty = r.full + kStages;
    return r;
}
constexpr size_t kTileRingBytes = (size_t)kStages * (kKT * kPT + kKT * kPS) * 4 + 2 * kStages * 8;

// producer lane: feature tiles [kKT x kPT] + the matching rows of the (k,8) prototype table, one barrier per stage
__device__ __forceinline__ void ring_produce(const Ring& r, const CUtensorMap* tmap, const float* ph, int k, int px0, int kbeg, int ntiles,
                                             int bi) {
    tma_prefetch_desc(tmap);
    for (int t = 0; t < ntiles; ++t) {
        const int s = t % kStages, rr = t / kStages;
        if (rr > 0) mbar_wait(&r.empty[s], (uint32_t)(rr - 1) & 1u);
        const int kk0 = kbeg + t * kKT;
        const uint32_t tab_bytes = (uint32_t)min(kKT, k - kk0) * kPS * 4u;
        mbar_arrive_expect_tx(&r.full[s], kKT * kPT * 4 + tab_bytes);
        tma_load_3d(r.tiles + (size_t)s * kKT * kPT, tmap, px0, kk0, bi, &r.full[s]);
        tma_load_1d(r.tabs + (size_t)s * kKT * kPS, ph + (int64_t)kk0 * kPS, tab_bytes, &r.full[s]);
    }
}

template <int M>
__global__ void __launch_bounds__(kThreads) pcl_forward_tma_kernel(const __grid_constant__ CUtensorMap tmap, int k, int hw, int kper,
                                                                   const float* __restrict__ ph, const int64_t* __restrict__ labels,
                                                                   int64_t ignore_label, float inv_temp,
                                                                   const long long* __restrict__ nvalid, float* __restrict__ coef,
                                                                   float* __restrict__ loss_terms, int* __restrict__ status) {
    constexpr int NA = 1 + M;
    extern __shared__ __align__(128) unsigned char smem_f[];
    const Ring r = ring_carve(smem_f);
    float* part = reinterpret_cast<float*>(smem_f + kTileRingBytes);  // [NA][kPT] CTA partial (cluster-visible)
    cg::cluster_group cluster = cg::this_cluster();
    const int ks = (int)cluster.block_rank(), KS = (int)cluster.num_blocks();
    const int ptile = blockIdx.x / KS, bi = blockIdx.y;
    const int px0 = ptile * kPT;
    const int kbeg = ks * kper, kend = min(k, kbeg + kper);
    const int ntiles = kend > kbeg ? (kend - kbeg + kKT - 1) / kKT : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&r.full[s], 1); mbar_init(&r.empty[s], kConsumers / 32); }
        mbar_fence_init();
    }
    __syncthreads();
    if (warp == kConsumers / 32) {
        if (lane == 0) ring_produce(r, &tmap, ph, k, px0, kbeg, ntiles, bi);
        __syncwarp();
    } else {
        float2 acc[NA][2];
#pragma unroll
        for (int a = 0; a < NA; ++a) { acc[a][0] = make_float2(0.f, 0.f); acc[a][1] = make_float2(0.f, 0.f); }
        for (int t = 0; t < ntiles; ++t) {
            const int s = t % kStages;
            mbar_wait(&r.full[s], (uint32_t)(t / kStages) & 1u);
            const float* tile = r.tiles + (size_t)s * kKT * kPT + lane * 4;
            const float* tab = r.tabs + (size_t)s * kKT * kPS;
            const int kk0 = kbeg + t * kKT;
#pragma unroll
            for (int j = 0; j < kKT / 8; ++j) {
                const int row = warp + 8 * j;
                if (kk0 + row < kend) {
                    const float4 v = *reinterpret_cast<const float4*>(tile + row * kPT);
                    const float4 p0 = *reinterpret_cast<const float4*>(tab + row * kPS);
                    float pv[kPS];
                    pv[0] = p0.x; pv[1] = p0.y; pv[2] = p0.z; pv[3] = p0.w;
                    if (M > 4) {
                        const float4 p1 = *reinterpret_cast<const float4*>(tab + row * kPS + 4);
                        pv[4] = p1.x; pv[5] = p1.y; pv[6] = p1.z; pv[7] = p1.w;
                    }
                    const float2 f01 = make_float2(v.x, v.y), f23 = make_float2(v.z, v.w);
                    acc[0][0] = __ffma2_rn(f01, f01, acc[0][0]);
                    acc[0][1] = __ffma2_rn(f23, f23, acc[0][1]);
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        const float2 pm = make_float2(pv[m], pv[m]);
                        acc[1 + m][0] = __ffma2_rn(f01, pm, acc[1 + m][0]);
                        acc[1 + m][1] = __ffma2_rn(f23, pm, acc[1 + m][1]);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&r.empty[s]);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");
        float* red = r.tiles;  // [warp][NA][kPT] in the drained ring
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
    cluster.sync();
    if (ks == 0 && threadIdx.x < kPT) {
        const int px = px0 + threadIdx.x;
        float sacc[NA];
#pragma unroll
        for (int a = 0; a < NA; ++a) sacc[a] = part[a * kPT + threadIdx.x];
        for (int rk = 1; rk < KS; ++rk) {
            const float* rp = cluster.map_shared_rank(part, rk);
#pragma unroll
            for (int a = 0; a < NA; ++a) sacc[a] += rp[a * kPT + threadIdx.x];
        }
        if (px < hw) {
            const int64_t l = labels[(int64_t)bi * hw + px];
            const bool valid = (l != ignore_label) && l >= 0 && l < M;
            if (l != ignore_label && !valid && status) atomicOr(status, 1);  // CrossEntropyLoss would raise
            const float n = fmaxf(sqrtf(sacc[0]), 1e-12f);
            const float inv_n = 1.0f / n;
            float z[M];
            float mx = -INFINITY;
#pragma unroll
            for (int j = 0; j < M; ++j) { z[j] = sacc[1 + j] * inv_n * inv_temp; mx = fmaxf(mx, z[j]); }
            float se = 0.f, e[M];
#pragma unroll
            for (int j = 0; j < M; ++j) { e[j] = expf(z[j] - mx); se += e[j]; }
            float zl = 0.f;
#pragma unroll
            for (int j = 0; j < M; ++j) zl = (l == j) ? z[j] : zl;
            loss_terms[(int64_t)bi * hw + px] = valid ? (logf(se) + mx) - zl : 0.f;
            const float inv_nv = 1.0f / (float)nvalid[0];
            const float scale = valid ? inv_nv * inv_temp * inv_n : 0.f;
            float beta = 0.f;
#pragma unroll
            for (int j = 0; j < M; ++j) {
                const float a = ((e[j] / se) - ((l == j) ? 1.f : 0.f)) * scale;
                coef[((int64_t)bi * (M + 1) + j) * hw + px] = a;
                beta = fmaf(a, sacc[1 + j], beta);
            }
            coef[((int64_t)bi * (M + 1) + M) * hw + px] = beta * inv_n * inv_n;
        }
    }
    cluster.sync();
}

// loss = sum(terms) / Nv in a fixed order (one block): deterministic, NaN when there is no valid pixel like the reference
__global__ void __launch_bounds__(1024) pcl_loss_kernel(const float* __restrict__ terms, int64_t n, const long long* __restrict__ nvalid,
                                                        float* __restrict__ loss) {
    __shared__ float red[32];
    float s = 0.f;
    for (int64_t i = threadIdx.x; i < n; i += 1024) s += terms[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < 32; ++i) t += red[i];
        loss[0] = t / (float)nvalid[0];
    }
}

template <int M>
__global__ void __launch_bounds__(kThreads) pcl_backward_tma_kernel(const __grid_constant__ CUtensorMap tmap, int k, int hw, int kper,
                                                                    const float* __restrict__ ph, const float* __restrict__ coef,
                                                                    const float* __restrict__ gout, float* __restrict__ grad) {
    extern __shared__ __align__(128) unsigned char smem_b[];
    const Ring r = ring_carve(smem_b);
    const int ksplit = gridDim.z;
    const int ptile = blockIdx.x, bi = blockIdx.y, ks = blockIdx.z;
    (void)ksplit;
    const int px0 = ptile * kPT;
    const int kbeg = ks * kper, kend = min(k, kbeg + kper);
    const int ntiles = kend > kbeg ? (kend - kbeg + kKT - 1) / kKT : 0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&r.full[s], 1); mbar_init(&r.empty[s], kConsumers / 32); }
        mbar_fence_init();
    }
    __syncthreads();
    if (warp == kConsumers / 32) {
        if (lane == 0) ring_produce(r, &tmap, ph, k, px0, kbeg, ntiles, bi);
        return;
    }
    const int px = px0 + lane * 4;
    const bool inb = px < hw;  // hw % 4 == 0
    const float g = gout ? gout[0] : 1.0f;
    float2 a01[M], a23[M], b01 = make_float2(0.f, 0.f), b23 = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < M; ++j) { a01[j] = make_float2(0.f, 0.f); a23[j] = make_float2(0.f, 0.f); }
    if (inb) {
#pragma unroll
        for (int j = 0; j < M; ++j) {
            const float4 a = ldg_f4(coef + ((int64_t)bi * (M + 1) + j) * hw + px);
            a01[j] = make_float2(a.x * g, a.y * g);
            a23[j] = make_float2(a.z * g, a.w * g);
        }
        const float4 bt = ldg_f4(coef + ((int64_t)bi * (M + 1) + M) * hw + px);
        b01 = make_float2(-bt.x * g, -bt.y * g);
        b23 = make_float2(-bt.z * g, -bt.w * g);
    }
    float* gb = grad + (int64_t)bi * k * hw + px;
    for (int t = 0; t < ntiles; ++t) {
        const int s = t % kStages;
        mbar_wait(&r.full[s], (uint32_t)(t / kStages) & 1u);
        const float* tile = r.tiles + (size_t)s * kKT * kPT + lane * 4;
        const float* tab = r.tabs + (size_t)s * kKT * kPS;
        const int kk0 = kbeg + t * kKT;
#pragma unroll
        for (int j = 0; j < kKT / 8; ++j) {
            const int row = warp + 8 * j, kk = kk0 + row;
            if (kk < kend) {
                const float4 v = *reinterpret_cast<const float4*>(tile + row * kPT);
                const float4 p0 = *reinterpret_cast<const float4*>(tab + row * kPS);
                float pv[kPS];
                pv[0] = p0.x; pv[1] = p0.y; pv[2] = p0.z; pv[3] = p0.w;
                if (M > 4) {
                    const float4 p1 = *reinterpret_cast<const float4*>(tab + row * kPS + 4);
                    pv[4] = p1.x; pv[5] = p1.y; pv[6] = p1.z; pv[7] = p1.w;
                }
                float2 o01 = __fmul2_rn(b01, make_float2(v.x, v.y)), o23 = __fmul2_rn(b23, make_float2(v.z, v.w));
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    const float2 pm = make_float2(pv[m], pv[m]);
                    o01 = __ffma2_rn(a01[m], pm, o01);
                    o23 = __ffma2_rn(a23[m], pm, o23);
                }
                if (inb) stg_f4(gb + (int64_t)kk * hw, make_float4(o01.x, o01.y, o23.x, o23.y));
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&r.empty[s]);
    }
}

}  // namespace

// ws: [ph k*8 f32][nvalid i64 (+pad)][loss_terms b*hw f32][status i32 (+pad)]
extern "C" int64_t uem_pcl_ws_bytes(int b, int k, int64_t hw) {
    return ((int64_t)k * kPS * 4 + 16 + (((int64_t)b * hw * 4 + 15) & ~(int64_t)15) + 16);
}

static int pcl_tmap(CUtensorMap* tmap, const float* feat, int b, int k, int64_t hw) {
    return uem_make_tmap_3d_f32(tmap, feat, (uint64_t)hw, (uint64_t)k, (uint64_t)b, (uint64_t)hw, (uint64_t)k * hw, kPT, kKT);
}

extern "C" int uem_pcl_forward_f32(const float* feat, int b, int k, int64_t hw, const float* protos, int c, const int64_t* labels,
                                   int64_t ignore_label, float temperature, float* loss, float* coef, void* ws, void* stream) {
    UEM_REQUIRE(feat && protos && labels && loss && coef && ws && b > 0 && k >= kKT && hw > 0 && temperature > 0.f,
                "uem_pcl_forward_f32: bad arguments");
    UEM_REQUIRE(hw % 4 == 0 && uem_aligned16(feat) && hw < (1 << 30), "uem_pcl_forward_f32: feature rows must be 16-byte aligned (h*w %% 4 == 0)");
    cudaStream_t st = (cudaStream_t)stream;
    float* ph = (float*)ws;
    long long* nvalid = (long long*)(ph + (int64_t)k * kPS);
    float* terms = (float*)((char*)nvalid + 16);
    int* status = (int*)((char*)terms + (((int64_t)b * hw * 4 + 15) & ~(int64_t)15));
    UEM_CUDA(cudaMemsetAsync(status, 0, 16, st));
    CUtensorMap tmap;
    UEM_REQUIRE(pcl_tmap(&tmap, feat, b, k, hw) == 0, "uem_pcl_forward_f32: cuTensorMapEncodeTiled failed");
    const int ptiles = uem_div_up(hw, kPT);
    int KS = 1;
    while (KS < 8 && (int64_t)ptiles * b * KS * 2 <= 2 * UEM_SMS && k / (KS * 2) >= 4 * kKT) KS *= 2;
    const int kper = ((k + KS - 1) / KS + kKT - 1) / kKT * kKT;
    UEM_DISPATCH_C(c, {
        pcl_prep_kernel<<<C + 1, 256, 0, st>>>(protos, C, k, labels, (int64_t)b * hw, ignore_label, ph, nvalid);
        const size_t smem = kTileRingBytes + (size_t)kPT * (1 + C) * 4;
        UEM_CUDA(cudaFuncSetAttribute(pcl_forward_tma_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(ptiles * KS, b, 1);
        cfg.blockDim = dim3(kThreads, 1, 1);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = KS;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        UEM_CUDA(cudaLaunchKernelEx(&cfg, pcl_forward_tma_kernel<C>, tmap, k, (int)hw, kper, (const float*)ph, labels, ignore_label,
                                    1.0f / temperature, (const long long*)nvalid, coef, terms, status));
    });
    pcl_loss_kernel<<<1, 1024, 0, st>>>(terms, (int64_t)b * hw, nvalid, loss);
    UEM_CHECK_LAUNCH_N(3);
    return 0;
}

extern "C" int uem_pcl_backward_f32(const float* feat, int b, int k, int64_t hw, int c, const float* coef, const float* grad_out,
                                    float* grad_feat, const void* ws, void* stream) {
    UEM_REQUIRE(feat && coef && grad_feat && ws && b > 0 && k >= kKT && hw > 0, "uem_pcl_backward_f32: bad arguments");
    UEM_REQUIRE(hw % 4 == 0 && uem_aligned16(feat) && uem_aligned16(grad_feat) && uem_aligned16(coef) && hw < (1 << 30),
                "uem_pcl_backward_f32: feature rows must be 16-byte aligned (h*w %% 4 == 0)");
    cudaStream_t st = (cudaStream_t)stream;
    const float* ph = (const float*)ws;
    CUtensorMap tmap;
    UEM_REQUIRE(pcl_tmap(&tmap, feat, b, k, hw) == 0, "uem_pcl_backward_f32: cuTensorMapEncodeTiled failed");
    const int ptiles = uem_div_up(hw, kPT);
    int KS = 1;
    while (KS < 16 && (int64_t)ptiles * b * KS < 3 * UEM_SMS && k / (KS * 2) >= 4 * kKT) KS *= 2;
    const int kper = ((k + KS - 1) / KS + kKT - 1) / kKT * kKT;
    UEM_DISPATCH_C(c, {
        UEM_CUDA(cudaFuncSetAttribute(pcl_backward_tma_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileRingBytes));
        pcl_backward_tma_kernel<C><<<dim3(ptiles, b, KS), kThreads, kTileRingBytes, st>>>(tmap, k, (int)hw, kper, ph, coef, grad_out, grad_feat);
    });
    UEM_CHECK_LAUNCH();
    return 0;
}
