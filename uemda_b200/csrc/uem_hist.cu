// a14/a15: per-class label histogram, class-weight lookup, generic fp32 histogram.
// Reference: ClassBalance._local_freq / _one_hot / get_class_weight_4pixel, uemda/gast/balance.py:27-67
// (the reference materialises an (n,c) int64 one-hot: 96 MiB at config 2); torch.histc at
// balance.py:193,261 and the entropy-range statistics of pseudo_generation.py:167-207.
//
// HBM-bound single pass over int64 labels (8 B/px): per-thread register bins -> warp REDUX ->
// shared-memory privatised histogram -> one global atomic per bin per CTA.
#include "uem_common.cuh"

namespace {

constexpr int kThreads = 256;

template <int C>
__global__ void __launch_bounds__(kThreads) class_hist_kernel(const int64_t* __restrict__ label, int64_t n, int vec,
                                                              int64_t ignore_label, unsigned long long* __restrict__ hist) {
    unsigned bins[C + 1];
#pragma unroll
    for (int ci = 0; ci <= C; ++ci) bins[ci] = 0;
    const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x, nth = (int64_t)gridDim.x * kThreads;
    auto add = [&](int64_t v) {
        bins[C] += (v != ignore_label);  // local_cnt, balance.py:49
#pragma unroll
        for (int ci = 0; ci < C; ++ci) bins[ci] += (v == ci) && (v != ignore_label);
    };
    if (vec) {
        for (int64_t i = tid; i < n / 2; i += nth) {
            int64_t a, b2;
            ldg_i64x2(label + 2 * i, a, b2);
            add(a);
            add(b2);
        }
        if (tid == 0 && (n & 1)) add(label[n - 1]);
    } else {
        for (int64_t i = tid; i < n; i += nth) add(label[i]);
    }
    __shared__ unsigned sh[C + 1];
    if (threadIdx.x <= C) sh[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int ci = 0; ci <= C; ++ci) {
        unsigned x = __reduce_add_sync(0xffffffffu, bins[ci]);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(&sh[ci], x);
    }
    __syncthreads();
    if (threadIdx.x <= C && sh[threadIdx.x]) atomicAdd(hist + threadIdx.x, (unsigned long long)sh[threadIdx.x]);
}

__global__ void __launch_bounds__(kThreads) class_weight_lookup_kernel(const int64_t* __restrict__ label, int64_t n, int c, int vec,
                                                                       int64_t ignore_label, const float* __restrict__ table,
                                                                       float* __restrict__ out) {
    __shared__ float tab[UEM_MAX_C];
    if (threadIdx.x < c) tab[threadIdx.x] = table[threadIdx.x];
    __syncthreads();
    const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x, nth = (int64_t)gridDim.x * kThreads;
    auto look = [&](int64_t v) { return (v != ignore_label && v >= 0 && v < c) ? tab[v] : 0.f; };  // balance.py:29-32
    if (vec) {
        for (int64_t i = tid; i < n / 4; i += nth) {
            int64_t id[4];
            load_ids<4>(label + 4 * i, id);
            stg_f4(out + 4 * i, make_float4(look(id[0]), look(id[1]), look(id[2]), look(id[3])));
        }
        for (int64_t i = (n / 4) * 4 + tid; i < n; i += nth) out[i] = look(label[i]);
    } else {
        for (int64_t i = tid; i < n; i += nth) out[i] = look(label[i]);
    }
}

// torch.histc semantics: bin = (int)((x - lo) * bins / (hi - lo)), each operation rounded in fp32 in that order, with no
// search against the bin edges (a value on a computed edge may land one bin below it); x == hi lands in the last bin,
// x outside [lo,hi] (or NaN) is dropped.
__global__ void __launch_bounds__(kThreads) hist_f32_kernel(const float* __restrict__ x, int64_t n, int bins, float lo, float hi,
                                                            unsigned long long* __restrict__ hist) {
    extern __shared__ unsigned sh[];
    for (int i = threadIdx.x; i < bins; i += kThreads) sh[i] = 0;
    __syncthreads();
    const float range = __fsub_rn(hi, lo);
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
        const float v = x[i];
        if (!(v >= lo && v <= hi)) continue;
        const int pos = min((int)__fdiv_rn(__fmul_rn(__fsub_rn(v, lo), (float)bins), range), bins - 1);
        atomicAdd(&sh[pos], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += kThreads)
        if (sh[i]) atomicAdd(hist + i, (unsigned long long)sh[i]);
}

// offline regeneration: the label map written to disk is uint8(label + 1), ignore (-1) -> 0
// (pseudo_generation.py:150-151, vis_corrected_pseudo_labels.py:191)
__global__ void __launch_bounds__(kThreads) label_plus1_u8_kernel(const int64_t* __restrict__ label, int64_t n, int vec,
                                                                  uint8_t* __restrict__ out) {
    const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x, nth = (int64_t)gridDim.x * kThreads;
    if (vec) {  // 4 labels (2 x 128-bit) -> one 32-bit store
        for (int64_t i = tid; i < n / 4; i += nth) {
            int64_t a, b2, c2, d;
            ldg_i64x2(label + 4 * i, a, b2);
            ldg_i64x2(label + 4 * i + 2, c2, d);
            const unsigned w = (unsigned)(uint8_t)(a + 1) | ((unsigned)(uint8_t)(b2 + 1) << 8) | ((unsigned)(uint8_t)(c2 + 1) << 16) |
                               ((unsigned)(uint8_t)(d + 1) << 24);
            reinterpret_cast<unsigned*>(out)[i] = w;
        }
        for (int64_t i = (n / 4) * 4 + tid; i < n; i += nth) out[i] = (uint8_t)(label[i] + 1);
    } else {
        for (int64_t i = tid; i < n; i += nth) out[i] = (uint8_t)(label[i] + 1);
    }
}

}  // namespace

extern "C" int uem_class_hist_i64(const int64_t* label, int64_t n, int c, int64_t ignore_label, int64_t* hist, void* stream) {
    UEM_REQUIRE(label && hist && n >= 0, "uem_class_hist_i64: bad arguments");
    if (n == 0) return 0;
    const int grid = (int)min((int64_t)UEM_SMS * 8, (n / 2 + kThreads - 1) / kThreads + 1);
    const int vec = uem_aligned16(label) ? 1 : 0;
    UEM_DISPATCH_C(c, { class_hist_kernel<C><<<grid, kThreads, 0, (cudaStream_t)stream>>>(label, n, vec, ignore_label, (unsigned long long*)hist); });
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_class_weight_lookup_f32(const int64_t* label, int64_t n, int c, int64_t ignore_label, const float* table,
                                           float* out, void* stream) {
    UEM_REQUIRE(label && table && out && n >= 0 && c > 0 && c <= UEM_MAX_C, "uem_class_weight_lookup_f32: bad arguments");
    if (n == 0) return 0;
    const int grid = (int)min((int64_t)UEM_SMS * 8, (n / 4 + kThreads - 1) / kThreads + 1);
    const int vec = (uem_aligned16(label) && uem_aligned16(out)) ? 1 : 0;
    class_weight_lookup_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(label, n, c, vec, ignore_label, table, out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_hist_f32(const float* x, int64_t n, int bins, float lo, float hi, int64_t* hist, void* stream) {
    UEM_REQUIRE(x && hist && n >= 0 && bins > 0 && bins <= 8192, "uem_hist_f32: bad arguments (bins in [1,8192])");
    UEM_REQUIRE(lo < hi, "uem_hist_f32: need lo < hi");
    if (n == 0) return 0;
    const int grid = (int)min((int64_t)UEM_SMS * 4, (n + kThreads - 1) / kThreads);
    hist_f32_kernel<<<grid, kThreads, bins * sizeof(unsigned), (cudaStream_t)stream>>>(x, n, bins, lo, hi, (unsigned long long*)hist);
    UEM_CHECK_LAUNCH();
    return 0;
}

// torch.bucketize(x, boundaries) (right=False), balance.py:194,263: inds[i] = number of boundaries < x[i]
// (NaN and +inf -> nb, -inf -> 0); boundaries sorted ascending, nb <= 1024 (kept in shared memory, binary search)
namespace {
__global__ void __launch_bounds__(256) bucketize_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ bounds, int nb,
                                                        int64_t* __restrict__ inds) {
    extern __shared__ float sb[];
    for (int i = threadIdx.x; i < nb; i += blockDim.x) sb[i] = bounds[i];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = x[i];
        int lo = 0, hi = nb;                     // first index with bounds[idx] >= v (lower_bound); NaN: every test is false -> nb
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (!(sb[mid] >= v)) lo = mid + 1;
            else hi = mid;
        }
        inds[i] = lo;
    }
}
}  // namespace

extern "C" int uem_bucketize_f32(const float* x, int64_t n, const float* boundaries, int nb, int64_t* inds, void* stream) {
    UEM_REQUIRE(x && boundaries && inds && n >= 0 && nb > 0 && nb <= 1024, "uem_bucketize_f32: bad arguments (1..1024 boundaries)");
    if (n == 0) return 0;
    const int grid = (int)min((int64_t)UEM_SMS * 8, (n + 255) / 256);
    bucketize_kernel<<<grid, 256, nb * sizeof(float), (cudaStream_t)stream>>>(x, n, boundaries, nb, inds);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_label_plus1_u8_i64(const int64_t* label, int64_t n, uint8_t* out, void* stream) {
    UEM_REQUIRE(label && out && n > 0, "uem_label_plus1_u8_i64: bad arguments");
    const int vec = uem_aligned16(label) && ((reinterpret_cast<uintptr_t>(out) & 3u) == 0);
    const int grid = (int)min((int64_t)UEM_SMS * 8, (n / 4 + kThreads - 1) / kThreads + 1);
    label_plus1_u8_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(label, n, vec, out);
    UEM_CHECK_LAUNCH();
    return 0;
}
