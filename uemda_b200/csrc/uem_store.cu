// Resident target set: each training batch's soft labels and superpixel maps cut out of tile stores kept in HBM.
// Reference: the self-training loader reads the per-tile soft probabilities written by gener_target_pseudo
// (pseudo_generation.py:135-136 -> basedata.py:87) and the int32 superpixel .tif (basedata.py:77-79), applies the same
// crop / flip / rot90 to both (augmentation.py:150-157) and copies them to the device (train_ssl_uem.py:199-201).
//
// One launch copies every plane of every sample.  A CTA owns a TY x TX tile of the output for all the sample's planes
// (c soft planes, then the id plane).  Codes without a transpose map an output row to one source row (read forwards or
// backwards), so each warp loads and stores 32 consecutive words directly.  Transposing codes map an output row to a
// source column: the CTA loads the TX x TY source block of every plane row by row into shared memory (cp.async, one
// stage per plane, one barrier) and stores it column by column, so both sides stay coalesced.  Loads are 4-byte, so an arbitrary (unaligned) window offset costs nothing extra.
//
// Resident source set: each source batch's labels cut from the label files' own bytes kept in HBM, together with the
// DownscaleLabel cells that update_prototype / update_avg take (train_ssl_uem.py:205,216, train_align_uem.py:147,150,
// alignment.py:86-90,484-509): label_gather_kernel below.
//
// Resident image set: each batch's images cut from the decoded image bytes kept in HBM and mapped through a per-channel
// byte -> value table (the image's crop / flip / rot90 of augmentation.py:150-157 and its normalisation):
// image_gather_kernel below.
#include "uem_common.cuh"
#include "uem_tma.cuh"  // smem_u32

namespace {

constexpr int kThreads = 256;
constexpr int TY = 16;  // output rows per CTA (with 6 CTAs per SM: 40 registers, no spills)
constexpr int TX = 64;  // output columns per CTA
constexpr int kPer = TY * TX / kThreads;

struct Sample {
    bool ok;
    int t, fy, fx;
    int64_t src;  // element offset of the window origin within one (Hs, Ws) plane of the tile
    int64_t tile;
};

__device__ __forceinline__ Sample read_sample(const int64_t* tiles, const int32_t* windows, int s, int64_t num_tiles, int Hs,
                                              int Ws, int Ho, int Wo) {
    Sample r;
    r.tile = tiles[s];
    const int y0 = windows[3 * s], x0 = windows[3 * s + 1], code = windows[3 * s + 2];
    r.t = (code >> 2) & 1;
    r.fy = (code >> 1) & 1;
    r.fx = code & 1;
    const int Hw = r.t ? Wo : Ho, Ww = r.t ? Ho : Wo;
    // 64-bit comparisons: y0 + Hw cannot wrap
    r.ok = r.tile >= 0 && r.tile < num_tiles && code >= 0 && code < 8 && y0 >= 0 && x0 >= 0 && (int64_t)y0 + Hw <= Hs &&
           (int64_t)x0 + Ww <= Ws;
    r.src = r.ok ? (int64_t)y0 * Ws + x0 : 0;
    if (!r.ok) r.tile = 0;  // keeps the plane pointers inside the stores; nothing is read through them
    return r;
}

__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}

// Element i of a thread is row (tid / TX) + i * kRows of the CTA's output tile, column tid % TX (direct and store phases), or
// column (tid / TY) + i * kCols, row tid % TY of the output (transposing load phase): every address is a per-thread base plus
// i times a per-thread step.  W: 32-bit word of a plane (float for the soft labels, int32 for the ids); O: its output type.
constexpr int kRows = kThreads / TX, kCols = kThreads / TY;
constexpr int kStage = TX * (TY + 1);  // words of one plane's stage: [r][q] holds out[oy0 + q, ox0 + r]

struct Geo {
    int Ws, Ho, Wo, oy0, ox0;
};

// codes without a transpose: out[oy, ox] = win[fy ? Ho-1-oy : oy, fx ? Wo-1-ox : ox]; an invalid sample writes zeros
template <typename W, typename O>
__device__ __forceinline__ void copy_plane_direct(const W* __restrict__ in, O* __restrict__ out, const Sample& s, const Geo& g) {
    const int ty = threadIdx.x / TX, ox = g.ox0 + threadIdx.x % TX, oy = g.oy0 + ty;
    if (ox >= g.Wo) return;
    O* o = out + (int64_t)oy * g.Wo + ox;
    const int64_t ostep = (int64_t)kRows * g.Wo;
    const int rows = g.Ho - oy;  // element i is inside the output iff i * kRows < rows
    if (!s.ok) {
#pragma unroll
        for (int i = 0; i < kPer; ++i)
            if (i * kRows < rows) o[i * ostep] = O(0);
        return;
    }
    const int wy = s.fy ? g.Ho - 1 - oy : oy, wx = s.fx ? g.Wo - 1 - ox : ox;
    const W* p = in + (int64_t)wy * g.Ws + wx;
    const int64_t step = s.fy ? -(int64_t)kRows * g.Ws : (int64_t)kRows * g.Ws;
    W v[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i)
        if (i * kRows < rows) v[i] = __ldcs(p + i * step);
#pragma unroll
    for (int i = 0; i < kPer; ++i)
        if (i * kRows < rows) o[i * ostep] = O(v[i]);
}

// transposing codes, load phase: out[oy, ox] = win[fy ? Wo-1-ox : ox, fx ? Ho-1-oy : oy] -> stage (asynchronous copies)
template <typename W>
__device__ __forceinline__ void stage_plane(const W* __restrict__ in, uint32_t* stage, const Sample& s, const Geo& g) {
    const int q = threadIdx.x % TY, r0 = threadIdx.x / TY, oy = g.oy0 + q, ox = g.ox0 + r0;
    if (oy >= g.Ho) return;
    const int wy = s.fy ? g.Wo - 1 - ox : ox, wx = s.fx ? g.Ho - 1 - oy : oy;
    const W* p = in + (int64_t)wy * g.Ws + wx;
    const int64_t step = s.fy ? -(int64_t)kCols * g.Ws : (int64_t)kCols * g.Ws;
    const int cols = g.Wo - ox;
#pragma unroll
    for (int i = 0; i < kPer; ++i)
        if (i * kCols < cols) cp_async_4(stage + (r0 + i * kCols) * (TY + 1) + q, p + i * step);
}

// transposing codes, store phase: the stage read column-wise, conflict-free (row pitch TY + 1)
template <typename W, typename O>
__device__ __forceinline__ void store_plane(const uint32_t* stage, O* __restrict__ out, const Geo& g) {
    const int ty = threadIdx.x / TX, tx = threadIdx.x % TX, ox = g.ox0 + tx, oy = g.oy0 + ty;
    if (ox >= g.Wo) return;
    O* o = out + (int64_t)oy * g.Wo + ox;
    const int64_t ostep = (int64_t)kRows * g.Wo;
    const int rows = g.Ho - oy;
#pragma unroll
    for (int i = 0; i < kPer; ++i)
        if (i * kRows < rows) {
            const uint32_t w = stage[tx * (TY + 1) + ty + i * kRows];
            o[i * ostep] = O(*reinterpret_cast<const W*>(&w));
        }
}

// Transposing codes load every plane of the tile into its own stage before a single barrier, so a CTA keeps
// (c + 1) x 4 loads per thread in flight instead of 4 per barrier.
__global__ void __launch_bounds__(kThreads, 6) tile_gather_kernel(const float* __restrict__ soft_store, const int32_t* __restrict__ id_store,
                                                               int64_t num_tiles, int c, int Hs, int Ws, const int64_t* __restrict__ tiles,
                                                               const int32_t* __restrict__ windows, int Ho, int Wo,
                                                               float* __restrict__ soft_out, int64_t* __restrict__ id_out,
                                                               int32_t* __restrict__ status) {
    extern __shared__ uint32_t stage[];  // (soft planes + id plane) x kStage
    const int n = blockIdx.z;
    const Geo g{Ws, Ho, Wo, (int)blockIdx.y * TY, (int)blockIdx.x * TX};
    const Sample s = read_sample(tiles, windows, n, num_tiles, Hs, Ws, Ho, Wo);
    if (!s.ok && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) atomicOr(status, 1);
    const int64_t plane = (int64_t)Hs * Ws, oplane = (int64_t)Ho * Wo;
    const int cs = soft_store ? c : 0;
    const float* sin = soft_store + s.tile * c * plane + s.src;
    const int32_t* iin = id_store + s.tile * plane + s.src;
    float* sout = soft_out + (int64_t)n * c * oplane;
    int64_t* iout = id_out + (int64_t)n * oplane;
    if (!s.ok || !s.t) {
        for (int ci = 0; ci < cs; ++ci) copy_plane_direct<float, float>(sin + ci * plane, sout + ci * oplane, s, g);
        if (id_store) copy_plane_direct<int32_t, int64_t>(iin, iout, s, g);
        return;
    }
    for (int ci = 0; ci < cs; ++ci) stage_plane<float>(sin + ci * plane, stage + ci * kStage, s, g);
    if (id_store) stage_plane<int32_t>(iin, stage + cs * kStage, s, g);
    cp_async_commit_group();
    cp_async_wait_group<0>();
    __syncthreads();
    for (int ci = 0; ci < cs; ++ci) store_plane<float, float>(stage + ci * kStage, sout + ci * oplane, g);
    if (id_store) store_plane<int32_t, int64_t>(stage + cs * kStage, iout, g);
}

// ------------------------------------------------------------------------------- resident source set
// Label maps stored as the label files' bytes, mapped through a 256-entry LUT.  Every code goes through one byte stage
// in output order (transposing codes load it column-wise like stage_plane), so loads and int64 stores stay coalesced and
// the cell counts read the same stage.  With a power-of-two scale <= TY, the 16-row CTA tile holds whole cells: 4 pixels
// per thread, the s*s/4 threads of a cell consecutive, their packed counts folded by xor-shuffles within a warp and by
// shared memory across the two warps of a 16 x 16 cell.  A cell has at most 256 pixels, so a count fits 9 bits: classes
// 0-6 are fields of a 64-bit word, class 7 and the ignore bin fields of a 32-bit word, and a pixel adds its byte's
// increments from shared memory (no branch on the class).
constexpr int kLabPitch = TX + 4;             // bytes per stage row
constexpr uint32_t kIncBad = 1u << 31;        // in inc_hi: the label is outside {ignore} U [0,n_classes) (not counted; bit 31 of
                                              // a sum is never read)

struct LabelSmem {
    int64_t lut[256];
    uint64_t inc_lo[256];                     // byte -> 1 << 9c for class c < 7
    uint32_t inc_hi[256];                     // byte -> 1 for class 7, 1 << 9 for the ignore label, kIncBad
    uint8_t stage[TY * kLabPitch];            // [row][col] of the CTA's output tile, as stored bytes
    uint64_t lo[kThreads];                    // per lane group: the summed increments
    uint32_t hi[kThreads];
};

// count of bin ci (0..7 = classes, 8 = ignore)
__device__ __forceinline__ unsigned bin_count(uint64_t lo, uint32_t hi, int ci) {
    return ci < 7 ? (unsigned)(lo >> (9 * ci)) & 0x1ffu : (hi >> (9 * (ci - 7))) & 0x1ffu;
}

// check: flag labels outside {ignore} U [0,n_classes) in bit 1 of status.  S: 0, or the power of two <= TY whose cells are
// counted here into down_out (n,1,Ho/S,Wo/S).  An invalid sample writes a zero label and the cells of a zero map.
template <int S>
__global__ void __launch_bounds__(kThreads) label_gather_kernel(const uint8_t* __restrict__ raw, int64_t num_tiles, int Hs, int Ws,
                                                                const int64_t* __restrict__ lut, const int64_t* __restrict__ tiles,
                                                                const int32_t* __restrict__ windows, int Ho, int Wo,
                                                                int64_t* __restrict__ label_out, int check, int n_classes,
                                                                int64_t ignore_label, float min_ratio, int64_t* __restrict__ down_out,
                                                                int32_t* __restrict__ status) {
    static_assert(kThreads == 256, "one thread per LUT entry");
    static_assert(S == 0 || (S >= 2 && S <= TY && (S & (S - 1)) == 0 && TX % S == 0), "cells must lie inside the CTA tile");
    __shared__ LabelSmem sm;
    const int n = blockIdx.z, oy0 = blockIdx.y * TY, ox0 = blockIdx.x * TX;
    const Sample s = read_sample(tiles, windows, n, num_tiles, Hs, Ws, Ho, Wo);
    if (!s.ok && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) atomicOr(status, 1);
    {
        const int64_t v = lut[threadIdx.x];
        const bool ign = v == ignore_label, cls = !ign && v >= 0 && v < n_classes;
        sm.lut[threadIdx.x] = v;
        sm.inc_lo[threadIdx.x] = cls && v < 7 ? 1ull << (9 * v) : 0ull;
        sm.inc_hi[threadIdx.x] = ign ? 1u << 9 : (cls ? (v == 7 ? 1u : 0u) : kIncBad);
    }
    if (s.ok) {
        const uint8_t* in = raw + s.tile * ((int64_t)Hs * Ws) + s.src;
        if (!s.t) {  // out[oy, ox] = win[fy ? Ho-1-oy : oy, fx ? Wo-1-ox : ox]
            const int ty = threadIdx.x / TX, tx = threadIdx.x % TX, ox = ox0 + tx, oy = oy0 + ty;
            if (ox < Wo) {
                const uint8_t* p = in + (int64_t)(s.fy ? Ho - 1 - oy : oy) * Ws + (s.fx ? Wo - 1 - ox : ox);
                const int64_t step = s.fy ? -(int64_t)kRows * Ws : (int64_t)kRows * Ws;
#pragma unroll
                for (int i = 0; i < kPer; ++i)
                    if (oy + i * kRows < Ho) sm.stage[(ty + i * kRows) * kLabPitch + tx] = __ldcs(p + i * step);
            }
        } else {     // out[oy, ox] = win[fy ? Wo-1-ox : ox, fx ? Ho-1-oy : oy]: a warp reads 16 bytes of 2 source rows
            const int q = threadIdx.x % TY, c0 = threadIdx.x / TY, oy = oy0 + q, ox = ox0 + c0;
            if (oy < Ho) {
                const uint8_t* p = in + (int64_t)(s.fy ? Wo - 1 - ox : ox) * Ws + (s.fx ? Ho - 1 - oy : oy);
                const int64_t step = s.fy ? -(int64_t)kCols * Ws : (int64_t)kCols * Ws;
#pragma unroll
                for (int i = 0; i < kPer; ++i)
                    if (ox + i * kCols < Wo) sm.stage[q * kLabPitch + c0 + i * kCols] = __ldcs(p + i * step);
            }
        }
    }
    __syncthreads();
    int bad = 0;
    {   // labels, row-major: a warp stores 32 consecutive int64
        const int ty = threadIdx.x / TX, tx = threadIdx.x % TX, ox = ox0 + tx;
        if (ox < Wo) {
            const int64_t o = ((int64_t)n * Ho + oy0 + ty) * Wo + ox;
#pragma unroll
            for (int i = 0; i < kPer; ++i) {
                const int r = ty + i * kRows;
                if (oy0 + r >= Ho) break;
                int64_t v = 0;
                if (s.ok) {
                    const int b = sm.stage[r * kLabPitch + tx];
                    v = sm.lut[b];
                    bad |= sm.inc_hi[b] == kIncBad;
                }
                if (label_out) label_out[o + (int64_t)i * kRows * Wo] = v;
            }
        }
    }
    // cells, cell-major: thread t counts pixels 4(t % G) .. +3 (row-major within the cell) of cell t / G
    constexpr int G = S * S / 4, kLanes = G < 32 ? G : 32, kCpr = S ? TX / S : 1;
    if (S) {
        const int cell = threadIdx.x / G, k0 = (threadIdx.x % G) * 4;
        const uint8_t* st = sm.stage + (cell / kCpr * S) * kLabPitch + cell % kCpr * S;
        uint64_t lo = 0ull;
        uint32_t hi = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + j;
            // an invalid sample counts its zero map (byte 0 stands in; sm.lut[0] is not used); pixels past the output edge
            // belong to cells that are not written
            const int b = s.ok ? st[(k / S) * kLabPitch + k % S] : 0;
            lo += s.ok ? sm.inc_lo[b] : (ignore_label == 0 ? 0ull : 1ull);
            hi += s.ok ? sm.inc_hi[b] : (ignore_label == 0 ? 1u << 9 : 0u);
        }
#pragma unroll
        for (int o = kLanes >> 1; o > 0; o >>= 1) {
            lo += __shfl_xor_sync(0xffffffffu, lo, o);
            hi += __shfl_xor_sync(0xffffffffu, hi, o);
        }
        if (threadIdx.x % kLanes == 0) {
            sm.lo[threadIdx.x / kLanes] = lo;
            sm.hi[threadIdx.x / kLanes] = hi;
        }
    }
    if (__syncthreads_or(bad) && check && threadIdx.x == 0) atomicOr(status, 2);
    if (!S) return;
    constexpr int kPerCell = S ? G / kLanes : 1;
    const int h = Ho / S, w = Wo / S;
    const int cell = threadIdx.x, cy = oy0 / S + cell / kCpr, cx = ox0 / S + cell % kCpr;
    if (cell >= (S ? TY * TX / (S * S) : 0) || cy >= h || cx >= w) return;
    uint64_t lo = sm.lo[cell * kPerCell];
    uint32_t hi = sm.hi[cell * kPerCell];
#pragma unroll
    for (int g = 1; g < kPerCell; ++g) {
        lo += sm.lo[cell * kPerCell + g];
        hi += sm.hi[cell * kPerCell + g];
    }
    unsigned best = bin_count(lo, hi, 0);
    int arg = 0;
#pragma unroll
    for (int ci = 1; ci < 8; ++ci)
        if (ci < n_classes && bin_count(lo, hi, ci) > best) { best = bin_count(lo, hi, ci); arg = ci; }  // first index wins ties
    if (bin_count(lo, hi, 8) > best) { best = bin_count(lo, hi, 8); arg = 8; }   // the ignore bin is last (alignment.py:497)
    const float ratio = __fdiv_rn((float)best, (float)(S * S));   // avg_pool2d of the one-hot: count / (s*s)
    down_out[((int64_t)n * h + cy) * w + cx] = (arg == 8 || ratio < min_ratio) ? ignore_label : (int64_t)arg;
}

// ------------------------------------------------------------------------------- resident image set
// Images stored as decoded (T,Hs,Ws,C) uint8 (interleaved), each byte mapped through its channel's 256-entry fp32 table.
// A segment is the run of pixels that is contiguous in the source for one CTA tile: an output row (TX pixels) without a
// transpose, an output column (TY pixels) with one; its P * C bytes are read forwards whatever the flip, and a flip only
// reverses the pixel order in which they are staged (the C bytes of a pixel keep their order).  Byte loads: any x0 works.
template <int C>
constexpr int kImgPitch = TX * C + 4;  // bytes per stage row: an odd number of words, so column-wise stage writes spread over banks

template <int C>
struct ImageSmem {
    float table[C][256];
    uint8_t stage[TY * kImgPitch<C>];  // [row q][column x][channel] of the CTA's output tile, as stored bytes
};

// segment k (k < nseg) starts at src + k * seg_step; its pixel p (p < npix) goes to output pixel flip ? npix-1-p : p of the
// segment, staged at k * seg_pitch + pixel * pix_pitch
template <int C, int P>
__device__ __forceinline__ void stage_image(const uint8_t* __restrict__ src, int64_t seg_step, int nseg, int npix, bool flip,
                                            uint8_t* stage, int seg_pitch, int pix_pitch) {
    constexpr int kSeg = P * C;
#pragma unroll
    for (int i = 0; i < TY * TX * C / kThreads; ++i) {
        const int l = threadIdx.x + i * kThreads, k = l / kSeg, j = l % kSeg, p = j / C;
        if (k < nseg && p < npix)
            stage[k * seg_pitch + (flip ? npix - 1 - p : p) * pix_pitch + j % C] = __ldcs(src + k * seg_step + j);
    }
}

// VW = 4: 16-byte stores (Wo % 4 == 0 and out 16-byte aligned); VW = 1: 4-byte stores.  An invalid sample writes zeros.
template <int C, int VW>
__global__ void __launch_bounds__(kThreads) image_gather_kernel(const uint8_t* __restrict__ raw, int64_t num_tiles, int Hs, int Ws,
                                                                const float* __restrict__ table, const int64_t* __restrict__ tiles,
                                                                const int32_t* __restrict__ windows, int Ho, int Wo,
                                                                float* __restrict__ out, int32_t* __restrict__ status) {
    static_assert(C >= 1 && C <= 4 && (VW == 1 || VW == 4), "1 to 4 channels; 4-byte or 16-byte stores");
    __shared__ ImageSmem<C> sm;
    const int n = blockIdx.z;
    const Geo g{Ws, Ho, Wo, (int)blockIdx.y * TY, (int)blockIdx.x * TX};
    const Sample s = read_sample(tiles, windows, n, num_tiles, Hs, Ws, Ho, Wo);
    if (!s.ok && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) atomicOr(status, 1);
#pragma unroll
    for (int ch = 0; ch < C; ++ch) sm.table[ch][threadIdx.x] = table[ch * 256 + threadIdx.x];
    const int rows = min(TY, Ho - g.oy0), cols = min(TX, Wo - g.ox0);
    if (s.ok) {
        const uint8_t* in = raw + (s.tile * Hs * Ws + s.src) * C;
        const int64_t row = (int64_t)Ws * C;
        if (!s.t) {  // segment q = output row oy0 + q: window row fy ? Ho-1-oy : oy, columns of ox0 .. ox0+cols-1
            const int wy = s.fy ? Ho - 1 - g.oy0 : g.oy0, wx = s.fx ? Wo - g.ox0 - cols : g.ox0;
            stage_image<C, TX>(in + wy * row + wx * C, s.fy ? -row : row, rows, cols, s.fx, sm.stage, kImgPitch<C>, C);
        } else {     // segment r = output column ox0 + r: window row fy ? Wo-1-ox : ox, columns of oy0 .. oy0+rows-1
            const int wy = s.fy ? Wo - 1 - g.ox0 : g.ox0, wx = s.fx ? Ho - g.oy0 - rows : g.oy0;
            stage_image<C, TY>(in + wy * row + wx * C, s.fy ? -row : row, cols, rows, s.fx, sm.stage, C, kImgPitch<C>);
        }
    }
    __syncthreads();
    // row-major stores: a warp writes 32 x VW consecutive floats of one plane
    constexpr int kLanes = TX / VW, kStep = kThreads / kLanes;
    const int x = threadIdx.x % kLanes * VW, q0 = threadIdx.x / kLanes;
    if (x >= cols) return;
    const int64_t plane = (int64_t)Ho * Wo;
    float* o = out + (int64_t)n * C * plane + (int64_t)(g.oy0 + q0) * Wo + g.ox0 + x;
#pragma unroll
    for (int i = 0; i < TY / kStep; ++i) {
        const int q = q0 + i * kStep;
        if (q >= rows) break;
        const uint8_t* px = sm.stage + q * kImgPitch<C> + x * C;
#pragma unroll
        for (int ch = 0; ch < C; ++ch) {
            float v[VW];
#pragma unroll
            for (int k = 0; k < VW; ++k) v[k] = s.ok ? sm.table[ch][px[k * C + ch]] : 0.f;
            float* dst = o + ch * plane + (int64_t)i * kStep * Wo;
            if constexpr (VW == 4)
                *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
            else
                *dst = v[0];
        }
    }
}

}  // namespace

extern "C" int uem_tile_gather(const float* soft_store, const int32_t* id_store, int64_t num_tiles, int c, int Hs, int Ws,
                               const int64_t* tiles, const int32_t* windows, int n, int Ho, int Wo, float* soft_out, int64_t* id_out,
                               int32_t* status, void* stream) {
    UEM_REQUIRE(tiles && windows && status && n >= 0 && n <= 65535 && num_tiles >= 0 && Hs > 0 && Ws > 0 && Ho > 0 && Wo > 0,
                "uem_tile_gather: bad arguments");
    UEM_REQUIRE(!soft_store || (soft_out && c >= 1 && c <= UEM_MAX_C), "uem_tile_gather: soft store needs soft_out and c in [1,%d]",
                UEM_MAX_C);
    UEM_REQUIRE(!id_store || id_out, "uem_tile_gather: id store needs id_out");
    if (n == 0 || (!soft_store && !id_store)) return 0;
    const dim3 grid(uem_div_up(Wo, TX), uem_div_up(Ho, TY), n);
    UEM_REQUIRE(grid.y <= 65535, "uem_tile_gather: output height %d too large", Ho);
    const size_t smem = (size_t)((soft_store ? c : 0) + (id_store ? 1 : 0)) * kStage * sizeof(uint32_t);  // <= 39 KiB
    // the whole carveout to shared memory (nothing is re-read through L1): six CTAs of 8 or 9 planes per SM need ~215 KB
    UEM_CUDA(cudaFuncSetAttribute(tile_gather_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    tile_gather_kernel<<<grid, kThreads, smem, (cudaStream_t)stream>>>(soft_store, id_store, num_tiles, c, Hs, Ws, tiles, windows, Ho, Wo,
                                                                    soft_out, id_out, status);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_label_gather_u8(const uint8_t* raw_store, int64_t num_tiles, int Hs, int Ws, const int64_t* lut,
                                   const int64_t* tiles, const int32_t* windows, int n, int Ho, int Wo, int64_t* label_out,
                                   int scale, int n_classes, int64_t ignore_label, float min_ratio, int64_t* down_out,
                                   int32_t* status, void* stream) {
    UEM_REQUIRE((raw_store || num_tiles == 0) && lut && tiles && windows && status && n >= 0 && n <= 65535 && num_tiles >= 0 &&
                    Hs > 0 && Ws > 0 && Ho > 0 && Wo > 0,
                "uem_label_gather_u8: bad arguments");
    UEM_REQUIRE(label_out || down_out, "uem_label_gather_u8: no output (label_out and down_out are both NULL)");
    UEM_REQUIRE(!down_out || (scale > 1 && n_classes >= 1 && n_classes <= UEM_MAX_C),
                "uem_label_gather_u8: down_out needs scale > 1 (got %d) and n_classes in [1,%d] (got %d)", scale, UEM_MAX_C, n_classes);
    // a power-of-two scale <= TY: every cell lies inside one CTA tile and is counted there; any other scale down-scales the
    // written labels with uem_downscale_label_i64 in a second launch
    const bool fused = down_out && scale <= TY && (scale & (scale - 1)) == 0;
    UEM_REQUIRE(!down_out || fused || label_out, "uem_label_gather_u8: scale %d is down-scaled from label_out, which is NULL", scale);
    if (n == 0) return 0;
    const dim3 grid(uem_div_up(Wo, TX), uem_div_up(Ho, TY), n);
    UEM_REQUIRE(grid.y <= 65535, "uem_label_gather_u8: output height %d too large", Ho);
    const cudaStream_t st = (cudaStream_t)stream;
    const int check = down_out ? 1 : 0;
#define UEM_LABEL_GATHER(S_)                                                                                                     \
    label_gather_kernel<S_><<<grid, kThreads, 0, st>>>(raw_store, num_tiles, Hs, Ws, lut, tiles, windows, Ho, Wo, label_out, check, \
                                                       n_classes, ignore_label, min_ratio, down_out, status)
    switch (fused ? scale : 0) {
        case 2: UEM_LABEL_GATHER(2); break;
        case 4: UEM_LABEL_GATHER(4); break;
        case 8: UEM_LABEL_GATHER(8); break;
        case 16: UEM_LABEL_GATHER(16); break;
        default: UEM_LABEL_GATHER(0); break;
    }
#undef UEM_LABEL_GATHER
    UEM_CHECK_LAUNCH();
    if (!down_out || fused) return 0;
    // bit 1 is already set from every label of the window; the down-scale's own check would report the same labels as bit 0
    return uem_downscale_label_i64(label_out, n, Ho, Wo, scale, n_classes, ignore_label, min_ratio, down_out, nullptr, stream);
}

extern "C" int uem_image_gather_u8(const uint8_t* store, int64_t num_tiles, int Hs, int Ws, int C, const float* table,
                                   const int64_t* tiles, const int32_t* windows, int n, int Ho, int Wo, float* out, int32_t* status,
                                   void* stream) {
    UEM_REQUIRE((store || num_tiles == 0) && table && tiles && windows && out && status && n >= 0 && n <= 65535 && num_tiles >= 0 &&
                    Hs > 0 && Ws > 0 && Ho > 0 && Wo > 0,
                "uem_image_gather_u8: bad arguments");
    UEM_REQUIRE(C >= 1 && C <= 4, "uem_image_gather_u8: C = %d channels outside [1,4]", C);
    if (n == 0) return 0;
    const dim3 grid(uem_div_up(Wo, TX), uem_div_up(Ho, TY), n);
    UEM_REQUIRE(grid.y <= 65535, "uem_image_gather_u8: output height %d too large", Ho);
    const cudaStream_t st = (cudaStream_t)stream;
    const bool vec = Wo % 4 == 0 && uem_aligned16(out);
#define UEM_IMAGE_GATHER(C_)                                                                                                     \
    do {                                                                                                                         \
        if (vec)                                                                                                                 \
            image_gather_kernel<C_, 4><<<grid, kThreads, 0, st>>>(store, num_tiles, Hs, Ws, table, tiles, windows, Ho, Wo, out,  \
                                                                  status);                                                       \
        else                                                                                                                     \
            image_gather_kernel<C_, 1><<<grid, kThreads, 0, st>>>(store, num_tiles, Hs, Ws, table, tiles, windows, Ho, Wo, out,  \
                                                                  status);                                                       \
    } while (0)
    switch (C) {
        case 1: UEM_IMAGE_GATHER(1); break;
        case 2: UEM_IMAGE_GATHER(2); break;
        case 3: UEM_IMAGE_GATHER(3); break;
        default: UEM_IMAGE_GATHER(4); break;
    }
#undef UEM_IMAGE_GATHER
    UEM_CHECK_LAUNCH();
    return 0;
}
