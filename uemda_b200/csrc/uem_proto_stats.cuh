// Format and arithmetic of the prototype statistics (alignment.py:347-353, :463-466), written once for every kernel that
// folds them: the single-GPU fold and fold + EMA (uem_proto.cu), the NCCL pack and the peer exchange (uem_exchange.cu).
// Sharing these helpers is what keeps a one-rank exchange equal to the single-GPU step bit for bit and every rank's
// prototype bank bit-identical.
#pragma once
#include "uem_common.cuh"

namespace {

// The per-image partials uem_proto_accum_nchw_f32 leaves in its workspace: [b*c*k f32 sums | b*c i32 counts]
struct ProtoPartials {
    const float* sums;
    const int* counts;
};
inline ProtoPartials proto_partials(const void* ws, int b, int c, int k) {
    const float* sums = (const float*)ws;
    return {sums, sums ? (const int*)(sums + (int64_t)b * c * k) : nullptr};
}

// Element i of the sums folded over the images in image order (deterministic)
__device__ __forceinline__ float fold_images(const float* __restrict__ sums, int b, int64_t ck, int64_t i) {
    float s = 0.f;
    for (int bi = 0; bi < b; ++bi) s += __ldg(sums + (int64_t)bi * ck + i);
    return s;
}
// Elements 4v .. 4v+3 with one 128-bit load per image (ck % 4 == 0): per element the same additions as fold_images
__device__ __forceinline__ float4 fold_images4(const float* __restrict__ sums, int b, int64_t ck, int64_t v) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int bi = 0; bi < b; ++bi) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(sums + (int64_t)bi * ck) + v);
        s.x += q.x; s.y += q.y; s.z += q.z; s.w += q.w;
    }
    return s;
}
// Pixel count of class ci over the images
__device__ __forceinline__ int64_t fold_image_counts(const int* __restrict__ counts, int b, int c, int ci) {
    int64_t n = 0;
    for (int bi = 0; bi < b; ++bi) n += counts[bi * c + ci];
    return n;
}

// Local prototype from the folded sum and count; a class without samples keeps the old prototype
__device__ __forceinline__ float proto_local(float s, int64_t n, float old, float eps) {
    const float local = s / ((float)n + eps);   // alignment.py:348
    return n < 1 ? old : local;                 // :350
}
// _ema, alignment.py:465: two rounded products, one rounded sum
__device__ __forceinline__ float proto_ema_of(float local, float old, float one_minus_decay, float decay) {
    return __fadd_rn(__fmul_rn(one_minus_decay, local), __fmul_rn(decay, old));
}
__device__ __forceinline__ float proto_ema(float s, int64_t n, float old, float eps, float one_minus_decay, float decay) {
    return proto_ema_of(proto_local(s, n, old, eps), old, one_minus_decay, decay);
}

}  // namespace
