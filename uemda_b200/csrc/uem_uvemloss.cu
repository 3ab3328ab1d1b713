// f3 (SURVEY section 8f, rank 3): the UVEM / UPS target loss fused end to end, forward and backward.
// Reference: uemda/gast/balance.py:437-457 (loss_calc_uvem: bilinear up-sampling of every head's logits to the label
// size, align_corners=True, loss averaged over the heads), :356-394 (UVEMLoss.forward: per-pixel cross-entropy, zeroed
// where the soft label's entropy exceeds the threshold, weighted by get_weight(entropy) [x class-balance weight],
// summed and divided by the number of valid pixels), :321-342 (UPSLoss: the gate without the parabolic weight).
//
// The reference materialises, per head, the up-sampled logits (b,c,H,W), an NHWC copy of them, log-softmax, the
// per-pixel loss, and replays all of it backwards through autograd.  Here:
//   * the detached per-pixel coefficient (weight x gate x class weight, 0 for ignored / gated pixels) comes from the
//     existing entropy/UVEM kernel (uem_uvem_terms_f32) -- it does not depend on the logits;
//   * forward: ONE pass over (target, coef) in the column-walk decomposition of logits_col_kernel: a thread owns an
//     image column, the horizontal half of the interpolation is hoisted out of the row loop, per pixel the logits of
//     all heads are one packed FFMA per class pair, the loss term is coef * (logsumexp - z[target]); per-thread fp32
//     partial sums over its rows, fp64 atomics across warps;
//   * backward: a gather, so the gradient is deterministic (the reference's upsample backward scatters with atomics):
//     ONE WARP per low-res cell (image, i, j) walks the cell's full-resolution footprint (the <= ~2H/h x 2W/w pixels
//     whose interpolation touches it), recomputes the pixel's softmax from the 3x3 low-res neighbourhood held in
//     registers, and accumulates w_y * w_x * coef * (p_c - [c == target]) for all classes and heads; one warp-level
//     reduction, one plain store per (head, class).  Every pixel is visited by the <= 4 cells it interpolates from;
//     (target, coef) are 12 bytes per pixel and stay in L2.
#include "uem_common.cuh"

namespace {

constexpr int kLossMaxHeads = 2;

template <int C, int NM>
__global__ void __launch_bounds__(128, 5) uvem_ce_col_kernel(const float* __restrict__ x1, const float* __restrict__ x2, int b, int h,
                                                             int w, int H, int W, float sy, float sx,
                                                             const int64_t* __restrict__ target, const float* __restrict__ coef,
                                                             double* __restrict__ sums, const int ncols_max) {
    constexpr int NT = 128, CP = (C + 3) & ~3, PC = (C + 1) / 2, TS = NM * CP;
    constexpr float kL2E = 1.4426950408889634f, kLn2 = 0.69314718055994531f;
    extern __shared__ __align__(16) float taps_all[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    float* const taps = taps_all + (size_t)wid * 2 * ncols_max * TS;
    const int64_t HW = (int64_t)H * W;
    const int hw_low = h * w;
    const int nstrips = (W + NT - 1) / NT;
    const int64_t total = (int64_t)b * nstrips * H;
    const int64_t U0 = total * blockIdx.x / gridDim.x, U1 = total * (blockIdx.x + 1) / gridDim.x;
    const int n = (int)(U1 - U0);
    if (n <= 0) return;
    int bs = (int)(U0 / H), y = (int)(U0 - (int64_t)bs * H);
    const float* maps[2] = {x1, x2};

    float2 A[NM][PC], D[NM][PC];
    int cur_bs = -1, cur_i0 = -1, bi = 0;
    int a0 = 0, a1 = 0, abase = 0, ncols = 1;
    float l0x = 0.f, l1x = 0.f;
    bool active = false;
    uint32_t x = 0;
    float acc[NM];
#pragma unroll
    for (int m = 0; m < NM; ++m) acc[m] = 0.f;
    for (int it = 0; it < n; ++it) {
        if (bs != cur_bs) {
            bi = bs / nstrips;
            const int xw = (bs - bi * nstrips) * NT + wid * 32;
            x = (uint32_t)(xw + lane);
            active = (int)x < W;
            const Lerp lx = make_lerp(active ? (int)x : W - 1, w, sx);
            a0 = lx.i0; a1 = lx.i1; l0x = lx.l0; l1x = lx.l1;
            abase = make_lerp(min(xw, W - 1), w, sx).i0;
            ncols = make_lerp(min(xw + 31, W - 1), w, sx).i1 - abase + 1;
            cur_bs = bs;
            cur_i0 = -1;
        }
        const Lerp ly = make_lerp(y, h, sy);
        if (ly.i0 != cur_i0) {
            cur_i0 = ly.i0;
            __syncwarp();
            if (lane < NM * C) {
                const int m = lane / C, ci = lane - m * C;
                const float* plane = maps[m] + ((int64_t)bi * C + ci) * hw_low + abase;
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
                            dst[(j0 + u) * TS] = u0[u] * kL2E;
                            dst[(ncols_max + j0 + u) * TS] = u1[u] * kL2E;
                        }
                }
            }
            __syncwarp();
            const float* t00 = taps + (a0 - abase) * TS;
            const float* t01 = taps + (a1 - abase) * TS;
            const float2 l0 = make_float2(l0x, l0x), l1 = make_float2(l1x, l1x);
#pragma unroll
            for (int m = 0; m < NM; ++m) {
#pragma unroll
                for (int j = 0; j < PC; ++j) {
                    const bool pad = 2 * j + 1 >= C;
                    const int o = m * CP + 2 * j;
                    const float2 p00 = make_float2(t00[o], pad ? 0.f : t00[o + 1]);
                    const float2 p01 = make_float2(t01[o], pad ? 0.f : t01[o + 1]);
                    const float2 p10 = make_float2(t00[ncols_max * TS + o], pad ? 0.f : t00[ncols_max * TS + o + 1]);
                    const float2 p11 = make_float2(t01[ncols_max * TS + o], pad ? 0.f : t01[ncols_max * TS + o + 1]);
                    float2 ta = __ffma2_rn(l1, p01, __fmul2_rn(l0, p00));
                    const float2 tb = __ffma2_rn(l1, p11, __fmul2_rn(l0, p10));
                    float2 td = __fadd2_rn(tb, make_float2(-ta.x, -ta.y));
                    if (pad) { ta.y = -1e30f; td.y = 0.f; }
                    A[m][j] = ta;
                    D[m][j] = td;
                }
            }
        }
        if (active) {
            const int64_t px = (int64_t)bi * HW + (int64_t)y * W + x;
            const float cf = __ldg(coef + px);
            if (cf != 0.f) {   // ignored and gated pixels carry coefficient 0: no term (and no class to select)
                const int t = (int)__ldg(target + px);
                const float2 t2 = make_float2(ly.l1, ly.l1);
#pragma unroll
                for (int m = 0; m < NM; ++m) {
                    float2 z[PC];
                    float mx = -INFINITY, zt = 0.f;
#pragma unroll
                    for (int j = 0; j < PC; ++j) {
                        z[j] = __ffma2_rn(t2, D[m][j], A[m][j]);
                        mx = fmaxf(mx, fmaxf(z[j].x, z[j].y));
                        zt = (t == 2 * j) ? z[j].x : zt;
                        zt = (t == 2 * j + 1) ? z[j].y : zt;
                    }
                    float2 s2;
#pragma unroll
                    for (int j = 0; j < PC; ++j) {
                        const float2 d = __fadd2_rn(z[j], make_float2(-mx, -mx));
                        const float2 e = make_float2(ex2_approx(d.x), ex2_approx(d.y));
                        s2 = j ? __fadd2_rn(s2, e) : e;
                    }
                    // -log softmax[target] = ln2 * (max - z_t) + ln S with z in the log2 domain; S in [1, C] and the term is
                    // small for a confident pixel, so the logarithm is the accurate one
                    acc[m] = fmaf(cf, fmaf(kLn2, mx - zt, logf(s2.x + s2.y)), acc[m]);
                }
            }
        }
        if (++y == H) { y = 0; ++bs; }
    }
#pragma unroll
    for (int m = 0; m < NM; ++m) {
        const float v = warp_sum(acc[m]);
        if (lane == 0 && v != 0.f) atomicAdd(sums + m, (double)v);
    }
}

// first / last output index whose source index i0 (PyTorch arithmetic, make_lerp) is >= / <= a given low-res index
__device__ __forceinline__ int first_with_i0_ge(int i, int in_size, int out_size, float scale) {
    if (i <= 0) return 0;
    int y = scale > 0.f ? (int)((float)i / scale) : out_size;
    y = max(0, min(y, out_size));
    while (y > 0 && make_lerp(y - 1, in_size, scale).i0 >= i) --y;
    while (y < out_size && make_lerp(y, in_size, scale).i0 < i) ++y;
    return y;   // == out_size when no such index
}

// ------------------------------------------------------------------------------------------------
// Backward: every pixel's softmax is evaluated ONCE.
// The full-resolution image splits into h x w "blocks": block (qi, qj) = the pixels whose interpolation starts at low-res
// (qi, qj), i.e. that interpolate from the 2x2 corner cells (qi | qi+1, qj | qj+1).  Pass 1: one warp per block keeps the
// four corners' logits in registers, walks its ~H/h x W/w pixels, and accumulates for the 4 corners x heads x classes
// w_y * w_x * coef * (p_c - [c == target]) in per-lane registers; one warp reduction, then 4 * NM * C plain stores into a
// per-block partial table.  Pass 2: every low-res cell adds the (at most 4 blocks x corners) partials that point at it,
// in a fixed order.  No atomics anywhere: the gradient is bit-reproducible run to run; 4x fewer exponentials than one
// warp per low-res cell gathering its whole footprint (124.7 -> 54.3 us at config 2, profiles/r02_lossbench.txt).
// ------------------------------------------------------------------------------------------------
template <int C, int NM>
__global__ void __launch_bounds__(128) uvem_ce_grad_block_kernel(const float* __restrict__ x1, const float* __restrict__ x2, int b, int h,
                                                                 int w, int H, int W, float sy, float sx,
                                                                 const int64_t* __restrict__ target, const float* __restrict__ coef,
                                                                 float* __restrict__ part) {
    constexpr float kL2E = 1.4426950408889634f;
    const int lane = threadIdx.x & 31;
    const int64_t blk = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int64_t nblk = (int64_t)b * h * w;
    if (blk >= nblk) return;
    const int qj = (int)(blk % w), qi = (int)((blk / w) % h), bi = (int)(blk / ((int64_t)w * h));
    const int hw_low = h * w;
    const int64_t HW = (int64_t)H * W;
    const float* maps[2] = {x1, x2};
    const int y0 = first_with_i0_ge(qi, h, H, sy), y1 = first_with_i0_ge(qi + 1, h, H, sy);
    const int x0 = first_with_i0_ge(qj, w, W, sx), x1e = first_with_i0_ge(qj + 1, w, W, sx);
    const int qi1 = min(qi + 1, h - 1), qj1 = min(qj + 1, w - 1);
    float nb[NM][C][2][2];   // the block's corner logits, pre-scaled by log2 e
#pragma unroll
    for (int m = 0; m < NM; ++m)
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            const float* pl = maps[m] + ((int64_t)bi * C + ci) * hw_low;
            nb[m][ci][0][0] = __ldg(pl + qi * w + qj) * kL2E;
            nb[m][ci][0][1] = __ldg(pl + qi * w + qj1) * kL2E;
            nb[m][ci][1][0] = __ldg(pl + qi1 * w + qj) * kL2E;
            nb[m][ci][1][1] = __ldg(pl + qi1 * w + qj1) * kL2E;
        }
    float acc[2][2][NM][C];
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx)
#pragma unroll
            for (int m = 0; m < NM; ++m)
#pragma unroll
                for (int ci = 0; ci < C; ++ci) acc[dy][dx][m][ci] = 0.f;
    const int fw = x1e - x0, fh = y1 - y0;
    if (fw > 0 && fh > 0) {
        const int npx = fw * fh;
        int fy = 0, fx = lane;
        while (fx >= fw) { fx -= fw; ++fy; }
        for (int q = lane; q < npx; q += 32) {
            const int y = y0 + fy, x = x0 + fx;
            const int64_t px = (int64_t)bi * HW + (int64_t)y * W + x;
            const float cf = __ldg(coef + px);
            if (cf != 0.f) {
                const Lerp ly = make_lerp(y, h, sy), lx = make_lerp(x, w, sx);
                const int t = (int)__ldg(target + px);
                const float w00 = ly.l0 * lx.l0 * cf, w01 = ly.l0 * lx.l1 * cf, w10 = ly.l1 * lx.l0 * cf, w11 = ly.l1 * lx.l1 * cf;
#pragma unroll
                for (int m = 0; m < NM; ++m) {
                    float z[C];
                    float mx = -INFINITY;
#pragma unroll
                    for (int ci = 0; ci < C; ++ci) {   // the forward's interpolation, operation by operation
                        z[ci] = ly.l0 * (lx.l0 * nb[m][ci][0][0] + lx.l1 * nb[m][ci][0][1]) +
                                ly.l1 * (lx.l0 * nb[m][ci][1][0] + lx.l1 * nb[m][ci][1][1]);
                        mx = fmaxf(mx, z[ci]);
                    }
                    float S = 0.f;
#pragma unroll
                    for (int ci = 0; ci < C; ++ci) { z[ci] = ex2_approx(z[ci] - mx); S += z[ci]; }
                    float r = rcp_approx(S);
                    r = fmaf(r, fmaf(-S, r, 1.0f), r);
#pragma unroll
                    for (int ci = 0; ci < C; ++ci) {
                        const float g = fmaf(z[ci], r, (t == ci) ? -1.0f : 0.0f);   // p_c - [c == target]
                        acc[0][0][m][ci] = fmaf(w00, g, acc[0][0][m][ci]);
                        acc[0][1][m][ci] = fmaf(w01, g, acc[0][1][m][ci]);
                        acc[1][0][m][ci] = fmaf(w10, g, acc[1][0][m][ci]);
                        acc[1][1][m][ci] = fmaf(w11, g, acc[1][1][m][ci]);
                    }
                }
            }
            fx += 32;
            while (fx >= fw) { fx -= fw; ++fy; }
        }
    }
    float* dst = part + blk * (4 * NM * C);
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx)
#pragma unroll
            for (int m = 0; m < NM; ++m)
#pragma unroll
                for (int ci = 0; ci < C; ++ci) {
                    const float v = warp_sum(acc[dy][dx][m][ci]);
                    if (lane == 0) dst[((dy * 2 + dx) * NM + m) * C + ci] = v;
                }
}

// Pass 2: cell (i, j) of head m, class ci <- the partials of the blocks qi in {i-1, i}, qj in {j-1, j} whose corner
// (dy, dx) lands on it (min(qi + dy, h-1) == i: the clamped last row / column receives two corners of its own block)
template <int C, int NM>
__global__ void __launch_bounds__(256) uvem_ce_grad_gather_kernel(const float* __restrict__ part, int b, int h, int w,
                                                                  const float* __restrict__ scale, float* __restrict__ g1,
                                                                  float* __restrict__ g2) {
    const int64_t total = (int64_t)b * NM * C * h * w;
    const float sc = __ldg(scale);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(e % w), i = (int)((e / w) % h);
        const int ci = (int)((e / ((int64_t)w * h)) % C), m = (int)((e / ((int64_t)w * h * C)) % NM);
        const int bi = (int)(e / ((int64_t)w * h * C * NM));
        float s = 0.f;
#pragma unroll
        for (int oy = 1; oy >= 0; --oy)        // blocks in the order (i-1, j-1), (i-1, j), (i, j-1), (i, j)
#pragma unroll
            for (int ox = 1; ox >= 0; --ox) {
                const int qi = i - oy, qj = j - ox;
                if (qi < 0 || qj < 0) continue;
                const float* src = part + (((int64_t)bi * h + qi) * w + qj) * (4 * NM * C);
#pragma unroll
                for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 2; ++dx)
                        if (min(qi + dy, h - 1) == i && min(qj + dx, w - 1) == j) s += src[((dy * 2 + dx) * NM + m) * C + ci];
            }
        float* g = m == 0 ? g1 : g2;
        g[((int64_t)bi * C + ci) * h * w + (int64_t)i * w + j] = s * sc;
    }
}

}  // namespace

extern "C" int64_t uem_uvem_loss_backward_ws_bytes(int b, int c, int h, int w, int heads) {
    return (int64_t)b * h * w * 4 * heads * c * 4;
}

// sums: nheads fp64 accumulators, zeroed by the caller.  sum_m = sum_px coef * CE(up(x_m))[target]
extern "C" int uem_uvem_loss_forward_f32(const float* x1, const float* x2, int b, int c, int h, int w, int H, int W,
                                         const int64_t* target, const float* coef, double* sums, void* stream) {
    UEM_REQUIRE(x1 && target && coef && sums && b > 0 && h > 0 && w > 0 && H > 0 && W > 0, "uem_uvem_loss_forward_f32: bad arguments");
    UEM_REQUIRE((int64_t)H * W < ((int64_t)1 << 31), "uem_uvem_loss_forward_f32: image too large");
    cudaStream_t st = (cudaStream_t)stream;
    const float sy = uem_align_corners_scale(h, H), sx = uem_align_corners_scale(w, W);
    int ncols_max = (int)(31.0f * sx) + 3;
    if (ncols_max > w) ncols_max = w;
    const int nm = x2 ? 2 : 1;
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
            sms = UEM_SMS;
    }
    const int64_t total = (int64_t)b * ((W + 127) / 128) * H;
    UEM_DISPATCH_C(c, {
        constexpr int CP = (C + 3) & ~3;
        const size_t smem = (size_t)4 * 2 * ncols_max * nm * CP * 4;
        UEM_REQUIRE(smem <= 200 * 1024, "uem_uvem_loss_forward_f32: low-res width %d too large for the tap scratch", w);
        if (nm == 2) {
            auto kernel = uvem_ce_col_kernel<C, 2>;
            if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int per_sm = 0;
            UEM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, smem));
            const int grid = (int)min(total, (int64_t)sms * max(per_sm, 1));
            kernel<<<grid, 128, smem, st>>>(x1, x2, b, h, w, H, W, sy, sx, target, coef, sums, ncols_max);
        } else {
            auto kernel = uvem_ce_col_kernel<C, 1>;
            if (smem > 48 * 1024) UEM_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int per_sm = 0;
            UEM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, smem));
            const int grid = (int)min(total, (int64_t)sms * max(per_sm, 1));
            kernel<<<grid, 128, smem, st>>>(x1, x2, b, h, w, H, W, sy, sx, target, coef, sums, ncols_max);
        }
    });
    UEM_CHECK_LAUNCH();
    return 0;
}

// g_m (b,c,h,w) = scale[0] * d/dx_m sum_px coef * CE(up(x_m))[target]; every element is written (no zero-init needed)
// ws: uem_uvem_loss_backward_ws_bytes(b, c, h, w, heads) bytes of scratch (the per-block partials)
extern "C" int uem_uvem_loss_backward_f32(const float* x1, const float* x2, int b, int c, int h, int w, int H, int W,
                                          const int64_t* target, const float* coef, const float* scale, float* g1, float* g2,
                                          void* ws, void* stream) {
    UEM_REQUIRE(x1 && g1 && target && coef && scale && b > 0 && h > 0 && w > 0 && H > 0 && W > 0,
                "uem_uvem_loss_backward_f32: bad arguments");
    UEM_REQUIRE(!x2 == !g2, "uem_uvem_loss_backward_f32: second head needs its gradient buffer");
    UEM_REQUIRE(ws, "uem_uvem_loss_backward_f32: ws is required (uem_uvem_loss_backward_ws_bytes bytes)");
    UEM_REQUIRE(h <= 65535 && b <= 65535, "uem_uvem_loss_backward_f32: grid too large");
    cudaStream_t st = (cudaStream_t)stream;
    const float sy = uem_align_corners_scale(h, H), sx = uem_align_corners_scale(w, W);
    const int64_t nblk = (int64_t)b * h * w;
    const int64_t elems = nblk * c * (x2 ? 2 : 1);
    const int ggrid = (int)min((int64_t)UEM_SMS * 8, (elems + 255) / 256);
    UEM_DISPATCH_C(c, {
        if (x2) {
            uvem_ce_grad_block_kernel<C, 2><<<(unsigned)((nblk + 3) / 4), 128, 0, st>>>(x1, x2, b, h, w, H, W, sy, sx, target, coef, (float*)ws);
            uvem_ce_grad_gather_kernel<C, 2><<<ggrid, 256, 0, st>>>((const float*)ws, b, h, w, scale, g1, g2);
        } else {
            uvem_ce_grad_block_kernel<C, 1><<<(unsigned)((nblk + 3) / 4), 128, 0, st>>>(x1, x2, b, h, w, H, W, sy, sx, target, coef, (float*)ws);
            uvem_ce_grad_gather_kernel<C, 1><<<ggrid, 256, 0, st>>>((const float*)ws, b, h, w, scale, g1, g2);
        }
    });
    UEM_CHECK_LAUNCH_N(2);
    return 0;
}
