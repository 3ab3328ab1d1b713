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
