// a6s/a7 seam: segmented reductions over superpixel ids (replaces torch_scatter.scatter) and
// Aligner.superpixel_expand.
// Reference call sites: uemda/gast/alignment.py:187 (reduce='sum', int64 one-hot), :245 (reduce='max',
// f32 probabilities), :188-190 (majority class per region, gathered back).
//
// HBM-bound scan over (class vector, id) pairs.  Contention control:
//   * every thread owns 4 consecutive pixels per step and keeps a (current id, running reduction) pair
//     in registers; only when the id changes is the table touched (superpixels are spatially coherent);
//   * for MAX the table update is test-then-atomic: an L2-coherent load first, the atomic only if the
//     value would actually raise the slot (a max changes O(log n) times);
//   * the hot id (after 7x7 edge shrinking ~60 % of all pixels carry the ignore id, SURVEY 7) is reduced
//     in registers and flushed once per CTA.
#include "uem_xchg_dev.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kSteps = 4;  // pixel groups per thread

// ---------------------------------------------------------------- int64 min/max (batch-global max id)
__global__ void minmax_init_kernel(int64_t* out) {
    out[0] = INT64_MAX;
    out[1] = INT64_MIN;
}
__global__ void __launch_bounds__(kThreads) minmax_kernel(const int64_t* __restrict__ x, int64_t n, int vec, int64_t* out) {
    int64_t mn = INT64_MAX, mx = INT64_MIN;
    const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x, nth = (int64_t)gridDim.x * kThreads;
    if (vec) {
        const int64_t pairs = n / 2;
        int64_t i = tid;
        for (; i + 3 * nth < pairs; i += 4 * nth) {  // 4 independent 128-bit loads in flight per thread
            int64_t a[8];
#pragma unroll
            for (int u = 0; u < 4; ++u) ldg_i64x2(x + 2 * (i + u * nth), a[2 * u], a[2 * u + 1]);
#pragma unroll
            for (int u = 0; u < 8; ++u) { mn = min(mn, a[u]); mx = max(mx, a[u]); }
        }
        for (; i < pairs; i += nth) {
            int64_t a, b2;
            ldg_i64x2(x + 2 * i, a, b2);
            mn = min(mn, min(a, b2));
            mx = max(mx, max(a, b2));
        }
        if (tid == 0 && (n & 1)) { mn = min(mn, x[n - 1]); mx = max(mx, x[n - 1]); }
    } else {
        for (int64_t i = tid; i < n; i += nth) { int64_t a = x[i]; mn = min(mn, a); mx = max(mx, a); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ int64_t smn[kThreads / 32], smx[kThreads / 32];
    if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < kThreads / 32; ++i) { mn = min(mn, smn[i]); mx = max(mx, smx[i]); }
        atomicMin((long long*)out, (long long)mn);
        atomicMax((long long*)out + 1, (long long)mx);
    }
}

// max only, accumulated with atomicMax into a slot the caller has zeroed (superpixel ids are >= 0): saves the
// init launch on the fused chain
__global__ void __launch_bounds__(kThreads) i64_max_kernel(const int64_t* __restrict__ x, int64_t n, int vec, int64_t* out) {
    int64_t mx = 0;
    const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x, nth = (int64_t)gridDim.x * kThreads;
    if (vec) {
        const int64_t pairs = n / 2;
        int64_t i = tid;
        for (; i + 3 * nth < pairs; i += 4 * nth) {
            int64_t a[8];
#pragma unroll
            for (int u = 0; u < 4; ++u) ldg_i64x2(x + 2 * (i + u * nth), a[2 * u], a[2 * u + 1]);
#pragma unroll
            for (int u = 0; u < 8; ++u) mx = max(mx, a[u]);
        }
        for (; i < pairs; i += nth) {
            int64_t a, b2;
            ldg_i64x2(x + 2 * i, a, b2);
            mx = max(mx, max(a, b2));
        }
        if (tid == 0 && (n & 1)) mx = max(mx, x[n - 1]);
    } else {
        for (int64_t i = tid; i < n; i += nth) mx = max(mx, x[i]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    __shared__ int64_t smx[kThreads / 32];
    if ((threadIdx.x & 31) == 0) smx[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < kThreads / 32; ++i) mx = max(mx, smx[i]);
        if (mx > 0) atomicMax((long long*)out, (long long)mx);
    }
}

// ---------------------------------------------------------------- f32 region reduce
// table slot update
template <int OP> __device__ __forceinline__ void slot_update_f32(unsigned* slot, float v);
template <> __device__ __forceinline__ void slot_update_f32<UEM_REDUCE_MAX>(unsigned* slot, float v) {
    unsigned e = f32_to_ordered(v);
    if (e > ld_cg_u32(slot)) atomicMax(slot, e);
}
template <> __device__ __forceinline__ void slot_update_f32<UEM_REDUCE_SUM>(unsigned* slot, float v) {
    atomicAdd(reinterpret_cast<float*>(slot), v);
}
template <int OP> __device__ __forceinline__ float op_init();
template <> __device__ __forceinline__ float op_init<UEM_REDUCE_MAX>() { return -INFINITY; }
template <> __device__ __forceinline__ float op_init<UEM_REDUCE_SUM>() { return 0.f; }
template <int OP> __device__ __forceinline__ float op_apply(float a, float b);
template <> __device__ __forceinline__ float op_apply<UEM_REDUCE_MAX>(float a, float b) { return fmaxf(a, b); }
template <> __device__ __forceinline__ float op_apply<UEM_REDUCE_SUM>(float a, float b) { return a + b; }

// table: (b,R,C) uint32 slots (MAX: ordered encoding, 0 = untouched; SUM: raw float bits, 0 = 0.0f)
// cnt (optional, MEAN): (b,R) uint32 pixel counts
template <int C, int VEC, int OP>
__global__ void __launch_bounds__(kThreads, 4) region_reduce_f32_kernel(const float* __restrict__ src, int64_t sb, int64_t sn,
                                                                     int64_t sc, const int64_t* __restrict__ index, int64_t N,
                                                                     int64_t R, const int64_t* __restrict__ hot_ptr, int64_t hot_val,
                                                                     int skip_hot, unsigned* __restrict__ table,
                                                                     unsigned* __restrict__ cnt, int* __restrict__ status) {
    const int bi = blockIdx.y;
    const float* s = src + (int64_t)bi * sb;
    const int64_t* idx = index + (int64_t)bi * N;
    unsigned* tab = table + (int64_t)bi * R * C;
    unsigned* cn = cnt ? cnt + (int64_t)bi * R : nullptr;
    const int64_t hot = hot_ptr ? *hot_ptr : hot_val;

    int64_t cur = -1;
    float acc[C], hacc[C];
    unsigned cur_n = 0, hot_n = 0;
#pragma unroll
    for (int ci = 0; ci < C; ++ci) { acc[ci] = op_init<OP>(); hacc[ci] = op_init<OP>(); }

    auto flush = [&]() {
        if (cur >= 0) {
            unsigned* slot = tab + cur * C;
            if (OP == UEM_REDUCE_MAX) {
                // test-then-atomic: the C probes are independent L2 loads issued back to back
                unsigned old[C];
#pragma unroll
                for (int ci = 0; ci < C; ++ci) old[ci] = ld_cg_u32(slot + ci);
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const unsigned e = f32_to_ordered(acc[ci]);
                    if (e > old[ci]) atomicMax(slot + ci, e);
                }
            } else {
#pragma unroll
                for (int ci = 0; ci < C; ++ci) slot_update_f32<OP>(slot + ci, acc[ci]);
            }
            if (cn) atomicAdd(cn + cur, cur_n);
        }
    };

    const int64_t groups = N / VEC;
    const int64_t g0 = (int64_t)blockIdx.x * (kThreads * kSteps);
#pragma unroll 1
    for (int stp = 0; stp < kSteps; ++stp) {
        const int64_t g = g0 + (int64_t)stp * kThreads + threadIdx.x;
        if (g >= groups) break;
        const int64_t n0 = g * VEC;
        int64_t id[VEC];
        load_ids<VEC>(idx + n0, id);
        float v[C][VEC];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            if (VEC == 4) {
                PixVec<VEC> t;
                t.load(s + n0 + (int64_t)ci * sc);  // planar: sn == 1
#pragma unroll
                for (int i = 0; i < VEC; ++i) v[ci][i] = t.v[i];
            } else {
                v[ci][0] = ldg_f1(s + n0 * sn + (int64_t)ci * sc);
            }
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int64_t r = id[i];
            if (r < 0 || r >= R) { if (status) atomicOr(status, 2); continue; }
            if (r == hot) {
                if (!skip_hot) {
#pragma unroll
                    for (int ci = 0; ci < C; ++ci) hacc[ci] = op_apply<OP>(hacc[ci], v[ci][i]);
                    ++hot_n;
                }
                continue;
            }
            if (r != cur) {
                flush();
                cur = r;
                cur_n = 0;
#pragma unroll
                for (int ci = 0; ci < C; ++ci) acc[ci] = op_init<OP>();
            }
#pragma unroll
            for (int ci = 0; ci < C; ++ci) acc[ci] = op_apply<OP>(acc[ci], v[ci][i]);
            ++cur_n;
        }
    }
    flush();

    // hot id: block-level reduction, one table update per CTA
    if (hot >= 0 && !skip_hot) {
        __shared__ float sh[kThreads / 32][C];
        __shared__ unsigned shn[kThreads / 32];
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        unsigned n = __reduce_add_sync(0xffffffffu, hot_n);
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            float x = hacc[ci];
            if (OP == UEM_REDUCE_MAX) x = warp_max(x); else x = warp_sum(x);
            if (lane == 0) sh[warp][ci] = x;
        }
        if (lane == 0) shn[warp] = n;
        __syncthreads();
        if (threadIdx.x < C) {
            float x = sh[0][threadIdx.x];
            unsigned tot = 0;
            for (int i2 = 0; i2 < kThreads / 32; ++i2) tot += shn[i2];
            for (int i2 = 1; i2 < kThreads / 32; ++i2) x = op_apply<OP>(x, sh[i2][threadIdx.x]);
            if (tot && hot >= 0 && hot < R) {
                slot_update_f32<OP>(tab + hot * C + threadIdx.x, x);
                if (cn && threadIdx.x == 0) atomicAdd(cn + hot, tot);
            }
        }
    }
}

// ---------------------------------------------------------------- f32 region MAX, shared-memory privatised
// The hot-path form (region maxima of the soft labels, alignment.py:245): every CTA scans a contiguous pixel range of
// one image and keeps a private (R, C) table of order-encoded maxima in shared memory.  A thread reduces runs of equal
// ids in registers; a finished run is merged test-then-atomic (LDS probe, ATOMS.MAX only when the slot would be
// raised), so the hot "ignored" id costs a probe, not a contended atomic.  Only the regions the CTA touched (byte flags)
// are merged into the global table, again test-then-atomic (ld.cg probe, RED.MAX only when raising).  The batch-global
// max id (alignment.py:241) falls out of the same pass (one atomicMax per CTA), which removes the separate pass over
// the int64 id map.
// Optional fused tail (RegionTail): the last CTA to finish an image turns that image's maxima into the superpixel-view
// weights softmax(max/temp)/(max_c + 1e-7) (alignment.py:252-253) and zeroes the table rows again, so the table is
// clean for the next call and no separate weight kernel / memset sits on the critical path.
struct RegionTail {
    float* sw;           // (b, R+1, CP) weights out (row R = all-ones sentinel); null = no tail
    int* done;           // (b) arrival counters: zero on entry, left zero
    float temp, inv_temp;
    int div_temp;
    unsigned* zero_words;  // cleared by CTA (0,0) on entry (the class-statistics table the refine kernel raises next)
    int n_zero;
};

template <int C, int VEC>
__global__ void __launch_bounds__(1024, 1) region_max_smem_kernel(const float* __restrict__ src, int64_t sb, int64_t sc,
                                                                 const int64_t* __restrict__ index, int64_t N, int64_t R,
                                                                 unsigned* __restrict__ table, long long* __restrict__ maxid,
                                                                 int* __restrict__ status, const RegionTail tail, int l2,
                                                                 const RegionXchg xchg) {
    constexpr int CP = (C + 3) & ~3;   // private rows are padded to CP words: a probe is CP/4 x LDS.128
    const uint64_t pol = l2_policy(l2);   // on the fused chain the refine kernel reads both maps again
    extern __shared__ __align__(16) unsigned tab_s[];  // [R][CP] then [R] touched flags
    __shared__ long long smax[32];
    __shared__ int s_last;
    const int bi = blockIdx.y;
    const float* s = src + (int64_t)bi * sb;
    const int64_t* idx = index + (int64_t)bi * N;
    const int RP = (int)(R * CP);
    const int words = (RP + (int)((R + 3) / 4) + 3) & ~3;
    unsigned char* touched = reinterpret_cast<unsigned char*>(tab_s + RP);
    // the dependent kernel (refine) may start its own prologue now (programmatic dependent launch)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    for (int i = threadIdx.x * 4; i < words; i += blockDim.x * 4) *reinterpret_cast<uint4*>(tab_s + i) = make_uint4(0u, 0u, 0u, 0u);
    if (blockIdx.x == 0 && bi == 0)
        for (int i = threadIdx.x; i < tail.n_zero; i += blockDim.x) tail.zero_words[i] = 0u;
    __syncthreads();

    const int64_t groups = N / VEC;
    const int64_t per = (groups + gridDim.x - 1) / gridDim.x;
    const int64_t g0 = (int64_t)blockIdx.x * per, g1 = min(groups, g0 + per);
    long long mx = 0;
    bool badid = false;
    // Every pixel probes its region's private row (the warp executes the same instructions whatever the ids are, so a
    // per-thread run-length compression only adds divergence); the atomic is issued only when a slot would be raised,
    // which happens O(log n) times per slot.
    for (int64_t g = g0 + threadIdx.x; g < g1; g += blockDim.x) {
        const int64_t n0 = g * VEC;
        int64_t id[VEC];
        load_ids<VEC>(idx + n0, id, pol);
        float v[C][VEC];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            PixVec<VEC> t;
            t.load(s + n0 + (int64_t)ci * sc, pol);
#pragma unroll
            for (int i = 0; i < VEC; ++i) v[ci][i] = t.v[i];
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const long long r64 = id[i];
            if (r64 < 0 || r64 >= R) { badid = true; continue; }
            mx = max(mx, r64);
            const int r = (int)r64;
            if (i == 0 || r64 != id[i > 0 ? i - 1 : 0]) touched[r] = 1;
            unsigned* slot = tab_s + r * CP;
            unsigned old[CP];
#pragma unroll
            for (int q = 0; q < CP / 4; ++q) {
                const uint4 o4 = *reinterpret_cast<const uint4*>(slot + 4 * q);
                old[4 * q] = o4.x; old[4 * q + 1] = o4.y; old[4 * q + 2] = o4.z; old[4 * q + 3] = o4.w;
            }
#pragma unroll
            for (int ci = 0; ci < C; ++ci) {
                const unsigned e = f32_to_ordered(v[ci][i]);
                if (e > old[ci]) atomicMax(slot + ci, e);
            }
        }
    }
    if (badid && status) atomicOr(status, 2);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0 && maxid) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) mx = max(mx, smax[i]);
        if (mx > 0) atomicMax(maxid, mx);
    }
    unsigned* tab = table + (int64_t)bi * R * C;
    for (int r = threadIdx.x; r < (int)R; r += blockDim.x) {
        if (!touched[r]) continue;
        unsigned old[C];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) old[ci] = ld_cg_u32(tab + r * C + ci);
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            const unsigned e = tab_s[r * CP + ci];
            if (e > old[ci]) atomicMax(tab + r * C + ci, e);
        }
    }
    if (tail.sw == nullptr) return;   // (the exchange rides on the fused chain only)
    // ---- last CTA of this image: per-region weights, table rows back to zero
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(tail.done + bi, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (s_last) {
    __threadfence();
    float* swb = tail.sw + (int64_t)bi * (R + 1) * CP;
    for (int r = threadIdx.x; r <= (int)R; r += blockDim.x) {
        float4* dst = reinterpret_cast<float4*>(swb + (int64_t)r * CP);
        if (r == (int)R) {
#pragma unroll
            for (int q = 0; q < CP / 4; ++q) dst[q] = make_float4(1.f, 1.f, 1.f, 1.f);
            continue;
        }
        float z[C];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            const unsigned e = ld_cg_u32(tab + r * C + ci);
            const float v = e ? ordered_to_f32(e) : 0.f;  // untouched slots are 0 like torch_scatter's output
            z[ci] = tail.div_temp ? __fdiv_rn(v, tail.temp) : v * tail.inv_temp;
            tab[r * C + ci] = 0u;
        }
        const float S = exp_shifted<C>(z);
        const float rs = fmaf(-1e-7f, S, 1.0f);
        float o[CP];
#pragma unroll
        for (int ci = 0; ci < CP; ++ci) o[ci] = ci < C ? z[ci < C ? ci : 0] * rs : 0.f;
#pragma unroll
        for (int q = 0; q < CP / 4; ++q) dst[q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    }
    if (threadIdx.x == 0) tail.done[bi] = 0;
    }
    if (xchg.world == 0) return;
    // ---- multi-GPU: the last CTA of the whole launch sends this rank's max id to every rank (and, with global_id_out,
    // waits for theirs): the id part of the step's exchange without a launch of its own
    XHeader* xh = reinterpret_cast<XHeader*>(xchg.peers.base[xchg.rank]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(&xh->region_done, 1u) == gridDim.x * gridDim.y - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const long long local_id = *reinterpret_cast<volatile long long*>(maxid);
    xchg_send_id_from_cta(xchg, local_id);
    if (threadIdx.x == 0) xh->region_done = 0u;
}

// decode the slot table into the dense float output torch_scatter returns (untouched -> 0)
__global__ void region_decode_f32_kernel(const unsigned* __restrict__ table, const unsigned* __restrict__ cnt, int64_t total,
                                         int c, int op, float* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        unsigned e = table[i];
        float v;
        if (op == UEM_REDUCE_MAX) v = e ? ordered_to_f32(e) : 0.f;
        else v = __uint_as_float(e);
        if (op == UEM_REDUCE_MEAN) { unsigned n = cnt[i / c]; v = v / (float)(n ? n : 1u); }
        out[i] = v;
    }
}

// ---------------------------------------------------------------- int64 region reduce (generic strides)
__global__ void fill_i64_kernel(int64_t* p, int64_t n, int64_t v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void __launch_bounds__(kThreads) region_reduce_i64_kernel(const int64_t* __restrict__ src, int64_t sb, int64_t sn,
                                                                     int64_t sc, const int64_t* __restrict__ index, int64_t N,
                                                                     int c, int64_t R, int op, int64_t* __restrict__ out,
                                                                     int* __restrict__ status) {
    const int bi = blockIdx.y;
    const int64_t total = N * c;
    const int64_t hot = R - 1;  // R = index.max()+1 at this seam
    __shared__ unsigned long long hot_sum[64];
    const bool use_hot = (op == UEM_REDUCE_SUM) && c <= 64;
    if (use_hot && threadIdx.x < c) hot_sum[threadIdx.x] = 0ull;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kThreads) {
        const int64_t n = i / c;
        const int ci = (int)(i - n * c);
        const int64_t r = index[(int64_t)bi * N + n];
        if (r < 0 || r >= R) { if (status) atomicOr(status, 2); continue; }
        const int64_t v = src[(int64_t)bi * sb + n * sn + (int64_t)ci * sc];
        long long* slot = (long long*)(out + ((int64_t)bi * R + r) * c + ci);
        if (op == UEM_REDUCE_MAX) { if (v > *(volatile long long*)slot) atomicMax(slot, (long long)v); }
        else if (v != 0) {
            if (use_hot && r == hot) atomicAdd(&hot_sum[ci], (unsigned long long)v);
            else atomicAdd((unsigned long long*)slot, (unsigned long long)v);
        }
    }
    __syncthreads();
    if (use_hot && threadIdx.x < c && hot_sum[threadIdx.x])
        atomicAdd((unsigned long long*)(out + ((int64_t)bi * R + hot) * c + threadIdx.x), hot_sum[threadIdx.x]);
}
__global__ void region_finish_i64_kernel(int64_t* out, int64_t total) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
        if (out[i] == INT64_MIN) out[i] = 0;
}

// ---------------------------------------------------------------- superpixel_expand
// counts (b,R,C) uint32: per-region class histogram of the hard labels (alignment.py:184-187)
template <int C, int VEC>
__global__ void __launch_bounds__(kThreads) region_class_hist_kernel(const int64_t* __restrict__ hard, const int64_t* __restrict__ sup,
                                                                     int64_t N, int64_t R, int64_t ignore_label,
                                                                     unsigned* __restrict__ counts, int* __restrict__ status) {
    const int bi = blockIdx.y;
    const int64_t* hd = hard + (int64_t)bi * N;
    const int64_t* sp = sup + (int64_t)bi * N;
    unsigned* tab = counts + (int64_t)bi * R * C;
    const int64_t hot = R - 1;  // R = sup.max()+1: after edge shrinking the last id is the hot "ignored" region
    int64_t cur = -1;
    unsigned acc[C], hacc[C];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) { acc[ci] = 0; hacc[ci] = 0; }
    auto flush = [&]() {
        if (cur >= 0) {
#pragma unroll
            for (int ci = 0; ci < C; ++ci)
                if (acc[ci]) atomicAdd(tab + cur * C + ci, acc[ci]);
        }
    };
    const int64_t groups = N / VEC;
    const int64_t g0 = (int64_t)blockIdx.x * (kThreads * kSteps);
#pragma unroll 1
    for (int stp = 0; stp < kSteps; ++stp) {
        const int64_t g = g0 + (int64_t)stp * kThreads + threadIdx.x;
        if (g >= groups) break;
        int64_t id[VEC], lb[VEC];
        load_ids<VEC>(sp + g * VEC, id);
        load_ids<VEC>(hd + g * VEC, lb);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int64_t r = id[i], l = lb[i];
            if (r < 0 || r >= R) { if (status) atomicOr(status, 2); continue; }
            if (l != ignore_label && (l < 0 || l >= C)) { if (status) atomicOr(status, 1); continue; }
            if (r == hot) {
#pragma unroll
                for (int ci = 0; ci < C; ++ci) hacc[ci] += (l == ci);
                continue;
            }
            if (r != cur) {
                flush();
                cur = r;
#pragma unroll
                for (int ci = 0; ci < C; ++ci) acc[ci] = 0;
            }
#pragma unroll
            for (int ci = 0; ci < C; ++ci) acc[ci] += (l == ci);
        }
    }
    flush();
    __shared__ unsigned sh[kThreads / 32][C];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
        unsigned x = __reduce_add_sync(0xffffffffu, hacc[ci]);
        if (lane == 0) sh[warp][ci] = x;
    }
    __syncthreads();
    if (threadIdx.x < C) {
        unsigned x = 0;
        for (int i = 0; i < kThreads / 32; ++i) x += sh[i][threadIdx.x];
        if (x) atomicAdd(tab + hot * C + threadIdx.x, x);
    }
}

// Shared-memory privatised form of the per-region class histogram (region table fits shared memory): every CTA
// scans a contiguous pixel range of one image into a private (R, CP) count table with shared-memory atomics (the
// hardware serialises same-address lanes, which is what the hot "ignored" region produces); touched rows are merged into the global
// counts, and the last CTA of an image (arrival counter) takes the first-index majority (alignment.py:188-189).
template <int C, int VEC>
__global__ void __launch_bounds__(1024, 1) region_hist_smem_kernel(const int64_t* __restrict__ hard, const int64_t* __restrict__ sup,
                                                                  int64_t N, int64_t R, int64_t ignore_label,
                                                                  unsigned* __restrict__ counts, int* __restrict__ winner,
                                                                  int* __restrict__ done, int* __restrict__ status) {
    constexpr int CP = (C + 3) & ~3;
    extern __shared__ __align__(16) unsigned cnt_s[];  // [R][CP] then [R] touched flags
    __shared__ int s_last;
    const int bi = blockIdx.y;
    const int64_t* hd = hard + (int64_t)bi * N;
    const int64_t* sp = sup + (int64_t)bi * N;
    const int RP = (int)(R * CP);
    const int words = (RP + (int)((R + 3) / 4) + 3) & ~3;
    unsigned char* touched = reinterpret_cast<unsigned char*>(cnt_s + RP);
    for (int i = threadIdx.x * 4; i < words; i += blockDim.x * 4) *reinterpret_cast<uint4*>(cnt_s + i) = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const int64_t groups = N / VEC;
    const int64_t per = (groups + gridDim.x - 1) / gridDim.x;
    const int64_t g0 = (int64_t)blockIdx.x * per, g1 = min(groups, g0 + per);
    int bad = 0;
    // uniform trip count per warp: match.any needs the whole warp
    const int64_t span = g1 > g0 ? g1 - g0 : 0;
    const int64_t trips = (span + blockDim.x - 1) / blockDim.x;
    // software pipeline: the loads of trip tr+1 are in flight while trip tr updates the table (the trips of a thread were
    // one dependent DRAM round trip each)
    int64_t nid[VEC], nlb[VEC];
    auto fetch = [&](int64_t tr) {
        const int64_t gg = g0 + tr * blockDim.x + threadIdx.x;
#pragma unroll
        for (int i = 0; i < VEC; ++i) { nid[i] = -1; nlb[i] = ignore_label; }
        if (tr < trips && gg < g1) {
            load_ids<VEC>(sp + gg * VEC, nid);
            load_ids<VEC>(hd + gg * VEC, nlb);
        }
    };
    fetch(0);
    for (int64_t tr = 0; tr < trips; ++tr) {
        const int64_t g = g0 + tr * blockDim.x + threadIdx.x;
        int64_t id[VEC], lb[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) { id[i] = nid[i]; lb[i] = nlb[i]; }
        fetch(tr + 1);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int64_t r = id[i], l = lb[i];
            if (g < g1) {
                if (r < 0 || r >= R) bad |= 2;
                else if (l != ignore_label && (l < 0 || l >= C)) bad |= 1;
                else if (l != ignore_label) {
                    // same-address shared atomics resolve at about a lane per cycle: a plain ATOMS on the hot region costs
                    // less than finding the peers first (match.any measured 1.4x slower end to end)
                    atomicAdd(cnt_s + (int)r * CP + (int)l, 1u);
                    touched[r] = 1;
                }
            }
        }
    }
    if (bad && status) atomicOr(status, bad);
    __syncthreads();
    unsigned* tab = counts + (int64_t)bi * R * C;
    for (int r = threadIdx.x; r < (int)R; r += blockDim.x) {
        if (!touched[r]) continue;
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            const unsigned n = cnt_s[r * CP + ci];
            if (n) atomicAdd(tab + r * C + ci, n);
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(done + bi, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int r = threadIdx.x; r < (int)R; r += blockDim.x) {
        unsigned best = ld_cg_u32(tab + r * C);
        int arg = 0;
#pragma unroll
        for (int ci = 1; ci < C; ++ci) {
            const unsigned v = ld_cg_u32(tab + r * C + ci);
            if (v > best) { best = v; arg = ci; }  // first index wins ties (torch.max)
        }
        winner[(int64_t)bi * R + r] = best == 0 ? -1 : arg;  // regions without a labelled pixel -> -1 (alignment.py:189)
    }
}

// majority class per region: first-index argmax, empty -> -1 (alignment.py:188-189); in place:
// counts[(b*R+r)*C + 0] is overwritten by the winner (as int)
template <int C>
__global__ void region_majority_kernel(const unsigned* __restrict__ counts, int64_t regions, int* __restrict__ winner) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < regions; r += (int64_t)gridDim.x * blockDim.x) {
        const unsigned* cnt = counts + r * C;
        unsigned best = cnt[0];
        int arg = 0;
#pragma unroll
        for (int ci = 1; ci < C; ++ci) {
            unsigned v = cnt[ci];
            if (v > best) { best = v; arg = ci; }
        }
        winner[r] = best == 0 ? -1 : arg;
    }
}

template <int VEC>
__global__ void __launch_bounds__(kThreads) region_gather_label_kernel(const int* __restrict__ winner, const int64_t* __restrict__ sup,
                                                                       int64_t N, int64_t R, int64_t* __restrict__ out) {
    const int bi = blockIdx.y;
    const int64_t g = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (g * VEC >= N) return;
    int64_t id[VEC], o[VEC];
    load_ids<VEC>(sup + (int64_t)bi * N + g * VEC, id);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
        const int64_t r = id[i];
        o[i] = (r >= 0 && r < R) ? (int64_t)__ldg(winner + (int64_t)bi * R + r) : -1;
    }
    store_ids<VEC>(out + (int64_t)bi * N + g * VEC, o);
}

}  // namespace

int uem_i64_max_accumulate(const int64_t* x, int64_t n, int64_t* out_max, cudaStream_t st) {
    UEM_REQUIRE(x && out_max && n > 0, "uem_i64_max_accumulate: bad arguments");
    int grid = (int)min((int64_t)UEM_SMS * 8, (n / 8 + kThreads - 1) / kThreads + 1);
    i64_max_kernel<<<grid, kThreads, 0, st>>>(x, n, uem_aligned16(x) ? 1 : 0, out_max);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_i64_minmax(const int64_t* x, int64_t n, int64_t* out_min_max, void* stream) {
    UEM_REQUIRE(x && out_min_max && n > 0, "uem_i64_minmax: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    minmax_init_kernel<<<1, 1, 0, st>>>(out_min_max);
    int grid = (int)min((int64_t)UEM_SMS * 8, (n / 8 + kThreads - 1) / kThreads + 1);
    minmax_kernel<<<grid, kThreads, 0, st>>>(x, n, uem_aligned16(x) ? 1 : 0, out_min_max);
    UEM_CHECK_LAUNCH_N(2);
    return 0;
}

// ws layout: [table b*R*c u32][counts b*R u32][status i32 (+pad)]
extern "C" int64_t uem_region_reduce_ws_bytes(int b, int64_t R, int c) {
    return ((int64_t)b * R * c + (int64_t)b * R + 4) * 4;
}

// Region maxima of a planar map into the encoded table (zero on entry); optionally the batch max id (maxid_out zero on
// entry, ids are >= 0), the fused weight tail (see RegionTail; tail_sw == nullptr: plain reduction) and, on the fused
// chain, the id part of a multi-GPU send from the last CTA (xchg == nullptr: no send).
// Needs R*c*4 + R bytes of shared memory per CTA.
int uem_region_max_f32(const float* src, int64_t sb, int64_t sc, const int64_t* index, int b, int64_t N, int c, int64_t R,
                       unsigned* table, int64_t* maxid_out, int* status, float* tail_sw, int* tail_done, float temp,
                       unsigned* zero_words, int n_zero, const RegionXchg* xchg, cudaStream_t st) {
    const bool vec = (N % 4 == 0) && (sb % 4 == 0) && (sc % 4 == 0) && uem_aligned16(src) && uem_aligned16(index);
    const size_t smem = ((size_t)R * ((c + 3) & ~3) * 4 + (size_t)((R + 3) / 4) * 4 + 15) & ~(size_t)15;
    UEM_REQUIRE(smem <= 200 * 1024, "uem_region_max_f32: region table (%lld x %d) exceeds shared memory", (long long)R, c);
    // the kernel is compiled for <= 64 registers (1024 threads per SM): two CTAs of 512 threads per SM when two private
    // tables fit, otherwise a single 1024-thread CTA; one wave
    const int threads = (2 * (smem + 1024) <= 220 * 1024) ? 512 : 1024;
    int per_sm = threads == 512 ? 2 : 1;
    if (g_uem_region_ctas_per_sm > 0 && per_sm > g_uem_region_ctas_per_sm) per_sm = g_uem_region_ctas_per_sm;
    int chunks = max(1, (UEM_SMS * per_sm) / b);
    const int64_t groups = N / (vec ? 4 : 1);
    chunks = (int)min((int64_t)chunks, max((int64_t)1, groups / threads));
    UEM_REQUIRE(!xchg || (tail_sw && maxid_out), "uem_region_max_f32: the id send rides on the fused chain's region pass only");
    const RegionXchg send = xchg ? *xchg : RegionXchg{};
    RegionTail tail{};
    tail.sw = tail_sw;
    tail.done = tail_done;
    tail.temp = temp;
    tail.inv_temp = 1.0f / temp;
    int ex;
    tail.div_temp = (frexpf(temp, &ex) == 0.5f) ? 0 : 1;
    tail.zero_words = zero_words;
    tail.n_zero = zero_words ? n_zero : 0;
    UEM_DISPATCH_C(c, {
        dim3 grid(chunks, b);
        if (vec) {
            if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(region_max_smem_kernel<C, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            region_max_smem_kernel<C, 4><<<grid, threads, smem, st>>>(src, sb, sc, index, N, R, table, (long long*)maxid_out, status, tail, tail_sw ? g_uem_l2_region : 0, send);
        } else {
            if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(region_max_smem_kernel<C, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            region_max_smem_kernel<C, 1><<<grid, threads, smem, st>>>(src, sb, sc, index, N, R, table, (long long*)maxid_out, status, tail, tail_sw ? g_uem_l2_region : 0, send);
        }
    });
    UEM_CHECK_LAUNCH();
    return 0;
}

// Internal entry shared with the fused refine path (uem_refine.cu): fills the encoded slot table only.
int uem_region_table_f32(const float* src, int64_t sb, int64_t sn, int64_t sc, const int64_t* index, int b, int64_t N,
                         int c, int64_t R, int op, const int64_t* hot_ptr, int64_t hot_val, int skip_hot, unsigned* table,
                         unsigned* cnt, int* status, cudaStream_t st) {
    const int kop = (op == UEM_REDUCE_MAX) ? UEM_REDUCE_MAX : UEM_REDUCE_SUM;
    const bool vec = (sn == 1) && (N % 4 == 0) && (sb % 4 == 0) && (sc % 4 == 0) && uem_aligned16(src) && uem_aligned16(index);
    if (kop == UEM_REDUCE_MAX && !cnt && sn == 1 && R * (((c + 3) & ~3) * 4 + 1) + 64 <= 200 * 1024)
        return uem_region_max_f32(src, sb, sc, index, b, N, c, R, table, nullptr, status, nullptr, nullptr, 1.0f, nullptr, 0, nullptr, st);
    UEM_DISPATCH_C(c, {
        if (vec) {
            dim3 grid(uem_div_up(N / 4, kThreads * kSteps), b);
            if (kop == UEM_REDUCE_MAX)
                region_reduce_f32_kernel<C, 4, UEM_REDUCE_MAX><<<grid, kThreads, 0, st>>>(src, sb, sn, sc, index, N, R, hot_ptr, hot_val, skip_hot, table, cnt, status);
            else
                region_reduce_f32_kernel<C, 4, UEM_REDUCE_SUM><<<grid, kThreads, 0, st>>>(src, sb, sn, sc, index, N, R, hot_ptr, hot_val, skip_hot, table, cnt, status);
        } else {
            dim3 grid(uem_div_up(N, kThreads * kSteps), b);
            if (kop == UEM_REDUCE_MAX)
                region_reduce_f32_kernel<C, 1, UEM_REDUCE_MAX><<<grid, kThreads, 0, st>>>(src, sb, sn, sc, index, N, R, hot_ptr, hot_val, skip_hot, table, cnt, status);
            else
                region_reduce_f32_kernel<C, 1, UEM_REDUCE_SUM><<<grid, kThreads, 0, st>>>(src, sb, sn, sc, index, N, R, hot_ptr, hot_val, skip_hot, table, cnt, status);
        }
    });
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_region_reduce_f32(const float* src, int64_t src_sb, int64_t src_sn, int64_t src_sc, const int64_t* index,
                                     int b, int64_t N, int c, int64_t R, int op, float* out, void* ws, void* stream) {
    UEM_REQUIRE(src && index && out && ws && b > 0 && N > 0 && R > 0, "uem_region_reduce_f32: bad arguments");
    UEM_REQUIRE(op == UEM_REDUCE_SUM || op == UEM_REDUCE_MAX || op == UEM_REDUCE_MEAN, "uem_region_reduce_f32: bad op %d", op);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* table = (unsigned*)ws;
    unsigned* cnt = table + (int64_t)b * R * c;
    UEM_CUDA(cudaMemsetAsync(ws, 0, (size_t)uem_region_reduce_ws_bytes(b, R, c), st));
    // R = index.max()+1 at the torch_scatter seam, so id R-1 exists and (after edge shrinking) is the hot one
    int rc = uem_region_table_f32(src, src_sb, src_sn, src_sc, index, b, N, c, R, op, nullptr, R - 1, 0, table,
                                  op == UEM_REDUCE_MEAN ? cnt : nullptr, (int*)(cnt + (int64_t)b * R), st);
    if (rc) return rc;
    const int64_t total = (int64_t)b * R * c;
    region_decode_f32_kernel<<<(int)min((int64_t)UEM_SMS * 4, (total + 255) / 256), 256, 0, st>>>(table, cnt, total, c, op, out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_region_reduce_i64(const int64_t* src, int64_t src_sb, int64_t src_sn, int64_t src_sc, const int64_t* index,
                                     int b, int64_t N, int c, int64_t R, int op, int64_t* out, void* ws, void* stream) {
    UEM_REQUIRE(src && index && out && b > 0 && N > 0 && R > 0 && c > 0, "uem_region_reduce_i64: bad arguments");
    UEM_REQUIRE(op == UEM_REDUCE_SUM || op == UEM_REDUCE_MAX, "uem_region_reduce_i64: op must be sum or max");
    (void)ws;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t total = (int64_t)b * R * c;
    const int fgrid = (int)min((int64_t)UEM_SMS * 4, (total + 255) / 256);
    if (op == UEM_REDUCE_MAX) fill_i64_kernel<<<fgrid, 256, 0, st>>>(out, total, INT64_MIN);
    else UEM_CUDA(cudaMemsetAsync(out, 0, (size_t)total * 8, st));
    dim3 grid((unsigned)min((int64_t)UEM_SMS * 8, (N * c + kThreads - 1) / kThreads), b);
    region_reduce_i64_kernel<<<grid, kThreads, 0, st>>>(src, src_sb, src_sn, src_sc, index, N, c, R, op, out, nullptr);
    if (op == UEM_REDUCE_MAX) region_finish_i64_kernel<<<fgrid, 256, 0, st>>>(out, total);
    UEM_CHECK_LAUNCH_N(op == UEM_REDUCE_MAX ? 3 : 1);
    return 0;
}

// ws layout: [counts b*R*c u32][winner b*R i32][status i32 (+pad)]
// ws layout: [counts b*R*c u32][winner b*R i32][status i32 (+pad)][done b i32]
extern "C" int64_t uem_superpixel_expand_ws_bytes(int b, int64_t R, int c) {
    return ((int64_t)b * R * c + (int64_t)b * R + 4 + b) * 4;
}

extern "C" int uem_superpixel_expand_i64(const int64_t* hard, const int64_t* sup, int b, int64_t N, int c, int64_t R,
                                         int64_t ignore_label, int64_t* out, void* ws, void* stream) {
    UEM_REQUIRE(hard && sup && out && ws && b > 0 && N > 0 && R > 0, "uem_superpixel_expand_i64: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* counts = (unsigned*)ws;
    int* winner = (int*)(counts + (int64_t)b * R * c);
    int* status = winner + (int64_t)b * R;
    UEM_CUDA(cudaMemsetAsync(ws, 0, (size_t)uem_superpixel_expand_ws_bytes(b, R, c), st));
    const bool vec = (N % 4 == 0) && uem_aligned16(hard) && uem_aligned16(sup) && uem_aligned16(out);
    const int64_t regions = (int64_t)b * R;
    const size_t smem_h = ((size_t)R * ((c + 3) & ~3) * 4 + (size_t)((R + 3) / 4) * 4 + 15) & ~(size_t)15;
    const bool priv = vec && smem_h <= 200 * 1024;
    int launched = 3;
    UEM_DISPATCH_C(c, {
        if (priv) {
            int* done = status + 4;
            const int threads = (2 * (smem_h + 1024) <= 220 * 1024) ? 512 : 1024;
            const int per_sm = threads == 512 ? 2 : 1;
            int chunks = max(1, (UEM_SMS * per_sm) / b);
            chunks = (int)min((int64_t)chunks, max((int64_t)1, (N / 4) / threads));
            if (smem_h > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(region_hist_smem_kernel<C, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_h));
            region_hist_smem_kernel<C, 4><<<dim3(chunks, b), threads, smem_h, st>>>(hard, sup, N, R, ignore_label, counts, winner, done, status);
            launched = 2;
        } else if (vec) {
            dim3 grid(uem_div_up(N / 4, kThreads * kSteps), b);
            region_class_hist_kernel<C, 4><<<grid, kThreads, 0, st>>>(hard, sup, N, R, ignore_label, counts, status);
        } else {
            dim3 grid(uem_div_up(N, kThreads * kSteps), b);
            region_class_hist_kernel<C, 1><<<grid, kThreads, 0, st>>>(hard, sup, N, R, ignore_label, counts, status);
        }
        if (!priv) region_majority_kernel<C><<<(int)min((int64_t)UEM_SMS * 4, (regions + 255) / 256), 256, 0, st>>>(counts, regions, winner);
    });
    if (vec) {
        dim3 grid(uem_div_up(N / 4, kThreads), b);
        region_gather_label_kernel<4><<<grid, kThreads, 0, st>>>(winner, sup, N, R, out);
    } else {
        dim3 grid(uem_div_up(N, kThreads), b);
        region_gather_label_kernel<1><<<grid, kThreads, 0, st>>>(winner, sup, N, R, out);
    }
    UEM_CHECK_LAUNCH_N(launched);
    return 0;
}
