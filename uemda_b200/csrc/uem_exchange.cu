// Multi-GPU exchange of the per-step statistics as device-side peer stores over NVLink (SURVEY section 8e).
//
// What crosses the fabric per step and rank (reference lines the exchange reproduces for a batch sharded by image):
//   * prototype partial sums (c,k) fp32 + counts (c) int64          alignment.py:347-353 (sums over the WHOLE batch)
//   * class histogram (c) + valid count, int64                      balance.py:45-52 (batch-global label frequencies)
//   * the rank-local max superpixel id, int64                       alignment.py:241 (batch-global "ignored" id)
// ~48 KiB of payload at c = 6, k = 2048.  Instead of a host-issued NCCL all-gather between two CUDA graphs, every rank
// STORES its vector straight into a slot of every peer's symmetric region (peer-mapped device memory: torch symmetric
// memory or cudaIpc handles), and the consumers are kernels of the peer's own graph.
//
// Protocol: every 32-bit payload word travels as ONE 8-byte store {word, sequence number} (the "LL" idea of NCCL's
// low-latency protocol): an 8-byte store is a single transaction, so a reader that sees the expected sequence number in
// the upper half holds valid data in the lower half -- no fences, no separate flags, no arrival counters on the data
// path.  (A first version with __threadfence_system + release flags cost ~18 us per step: system-scope fences issued while
// the other kernels of the step saturate the memory system are slow.)  Payload doubles to ~96 KiB per peer, still latency.
//
//   uem_xchg_send_f32            grid (chunks, world): CTA (ch, p) folds chunk ch of this rank's per-image partials in
//                                image order and stores {value, seq} pairs into peer p's slot [slot][rank].
//   uem_xchg_wait_maxid          one warp: lane r polls rank r's max-id words -> batch-global max id (needed by the
//                                refine kernel, so this heads the step's main branch).
//   uem_xchg_fold_finalize_ema   every thread polls its own words of all ranks (normally already there), folds them in
//                                RANK ORDER (identical fp32 additions on every rank -> the replicated prototype bank stays
//                                bit-identical), local mean, keep-old rule, EMA; the last CTA acknowledges the slot to every
//                                peer (one release store per peer), which is what a sender checks before it overwrites that
//                                slot `depth` steps later.
//   uem_xchg_exchange_fold_ema   the sums part of the send and the fold above in ONE launch.
// Each protocol step (slot addressing, LL stores, acknowledgement wait, id poll, the receiving end) is written once in
// uem_xchg_dev.cuh, and the fold / EMA arithmetic once in uem_proto_stats.cuh.
// No kernel waits for a kernel that is queued behind it on its own GPU: a send of step s waits for the acks of step
// s - depth, the consumers of step s for the sends of step s -- both are upstream in every rank's stream order, so the
// scheme cannot deadlock however the ranks drift.  Every poll is bounded (2 s of %globaltimer): on a timeout status bit 8
// is set in the region header and the kernel carries on, so a lost peer shows up as an error code, not as a hung GPU.
//
// Region layout (same on every rank; all offsets from the region base):
//   [0, 1024)            header, local only: seq_send[4], seq_recv[4], arrive_all[4], fold_arrive[4], status
//   [1280, 1536)         ack_flag[4][16] u32       written by peers
//   [2048, ...)          slots[depth][world][slot_bytes]
// slot (8-byte LL words): [c*k sums | pad to 16 B][c counts lo,hi][c+1 hist lo,hi][max id lo,hi]
#include "uem_xchg_dev.cuh"
#include <string.h>

namespace {

__global__ void __launch_bounds__(256) xchg_send_kernel(const float* __restrict__ partial, const int* __restrict__ cnt_partial, int b,
                                                        int c, int k, const int64_t* __restrict__ max_id,
                                                        const int64_t* __restrict__ hist, const __grid_constant__ Peers peers, int rank, int world,
                                                        int slot, int64_t* __restrict__ global_id_out, int parts) {
    const int ch = blockIdx.x, p = blockIdx.y;
    char* const mine = peers.base[rank];
    XHeader* hdr = reinterpret_cast<XHeader*>(mine);
    __shared__ unsigned s_my;
    // the id-only launch is issued with programmatic stream serialization right behind the region-max kernel (which
    // releases its dependents at entry): its CTAs are resident by the time that kernel ends, the launch latency is hidden
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (threadIdx.x == 0) {
        s_my = *reinterpret_cast<volatile unsigned*>(&hdr->seq_send[slot]) + 1u;
        wait_ack(mine, slot, p, s_my);
    }
    __syncthreads();
    const unsigned my = s_my;
    const int ck = c * k;
    char* dst = peers.base[p] + slot_off(slot, world, rank, c, k);
    // chunk ch of the sums, 4 elements at a time, this rank's partials folded over its images
    const int nvec = (parts & 1) ? (ck + 3) / 4 : 0;   // parts bit 0: sums + counts + histogram; bit 1: max id
    const int v0 = (int)((int64_t)nvec * ch / gridDim.x), v1 = (int)((int64_t)nvec * (ch + 1) / gridDim.x);
    for (int v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        const int64_t e = (int64_t)4 * v;
        if ((ck & 3) == 0) {
            const float4 s = fold_images4(partial, b, ck, v);
            ll_store(dst + e * 8, __float_as_uint(s.x), my);
            ll_store(dst + e * 8 + 8, __float_as_uint(s.y), my);
            ll_store(dst + e * 8 + 16, __float_as_uint(s.z), my);
            ll_store(dst + e * 8 + 24, __float_as_uint(s.w), my);
        } else {
            for (int u = 0; u < 4; ++u)   // ragged last vector (ck % 4 != 0): zero words past the end
                ll_store(dst + (e + u) * 8, __float_as_uint(e + u < ck ? fold_images(partial, b, ck, e + u) : 0.f), my);
        }
    }
    if (ch == 0 && threadIdx.x < 2 * c + 2 && ((threadIdx.x == 2 * c + 1) ? (parts & 2) : (parts & 1))) {
        const int i = threadIdx.x;
        const int64_t v = i < c ? fold_image_counts(cnt_partial, b, c, i) : (i < 2 * c + 1 ? (hist ? hist[i - c] : 0) : (max_id ? max_id[0] : -1));
        ll_store_i64(dst + tail_off(c, k) + (int64_t)i * 16, v, my);
    }
    // optional: the CTA that fills this rank's own slot also polls the other ranks' max ids of the same step and leaves
    // the batch-global id (alignment.py:241) for the refine kernel of the NEXT graph -- no separate wait launch
    if (global_id_out && ch == 0 && p == rank && threadIdx.x < 32) {
        const long long id = poll_max_id(mine, slot, world, c, k, my);
        if (threadIdx.x == 0) global_id_out[0] = id;
    }
    // the last CTA of the FINAL launch of a step (parts bit 2) advances the local sequence number (every CTA has read it by
    // then); an earlier partial launch of the same step leaves it alone, so both tag their words with the same number
    __syncthreads();
    if (threadIdx.x == 0 && (parts & 4)) {
        __threadfence();
        const unsigned old = atomicAdd(&hdr->arrive_all[slot], 1u);
        if (old == gridDim.x * gridDim.y - 1) {
            hdr->arrive_all[slot] = 0u;
            __threadfence();
            *reinterpret_cast<volatile unsigned*>(&hdr->seq_send[slot]) = my;
        }
    }
}

__global__ void __launch_bounds__(32) xchg_wait_maxid_kernel(char* __restrict__ region, int world, int slot, int c, int k,
                                                             int64_t* __restrict__ max_id_out) {
    const unsigned want = *reinterpret_cast<volatile unsigned*>(&reinterpret_cast<XHeader*>(region)->seq_recv[slot]) + 1u;
    const long long id = poll_max_id(region, slot, world, c, k, want);
    if (threadIdx.x == 0 && max_id_out) max_id_out[0] = id;
}

__global__ void __launch_bounds__(256) xchg_fold_finalize_kernel(const __grid_constant__ Peers peers, int rank, int world, int slot, int c, int k,
                                                                 const float* __restrict__ proto_old, float eps, float one_minus_decay,
                                                                 float decay, float* __restrict__ proto_new, float* __restrict__ sums_out,
                                                                 int64_t* __restrict__ counts_out, int64_t* __restrict__ hist_out) {
    XHeader* hdr = reinterpret_cast<XHeader*>(peers.base[rank]);
    const unsigned want = *reinterpret_cast<volatile unsigned*>(&hdr->seq_recv[slot]) + 1u;
    xchg_fold_ema_ack(peers, rank, world, slot, c, k, want, false, proto_old, eps, one_minus_decay, decay, proto_new, sums_out,
                      counts_out, hist_out);
}

// ------------------------------------------------------------------------------------------------
// One launch per step for the sums: local fold -> LL stores into every rank's slot -> the receiving end of
// xchg_fold_finalize_kernel, which here also advances the send sequence number.  Thread i owns element i of the (c,k)
// bank from its own partials to the new prototype; CTA 0 also carries the counts / histogram words.  (The max id travels
// earlier, uem_xchg_send_f32 with parts = 2, tagged with the same sequence number.)  A CTA sends before it polls and its
// peers' CTAs do the same, so no poll waits for anything that is queued behind this launch on any GPU.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) xchg_exchange_fold_kernel(const float* __restrict__ partial, const int* __restrict__ cnt_partial,
                                                                 int b, int c, int k, const int64_t* __restrict__ hist, const __grid_constant__ Peers peers,
                                                                 int rank, int world, int slot, const float* __restrict__ proto_old,
                                                                 float eps, float one_minus_decay, float decay,
                                                                 float* __restrict__ proto_new, float* __restrict__ sums_out,
                                                                 int64_t* __restrict__ counts_out, int64_t* __restrict__ hist_out) {
    char* const mine = peers.base[rank];
    XHeader* hdr = reinterpret_cast<XHeader*>(mine);
    __shared__ unsigned s_my;
    if (threadIdx.x == 0) s_my = *reinterpret_cast<volatile unsigned*>(&hdr->seq_send[slot]) + 1u;
    __syncthreads();
    const unsigned my = s_my;
    if (threadIdx.x < world) wait_ack(mine, slot, threadIdx.x, my);   // every peer must have folded the previous contents
    __syncthreads();
    const int ck = c * k;
    const int64_t my_off = slot_off(slot, world, rank, c, k);
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < ck) {
        const float s = fold_images(partial, b, ck, i);
        for (int p = 0; p < world; ++p) ll_store(peers.base[p] + my_off + (int64_t)i * 8, __float_as_uint(s), my);
    }
    if (blockIdx.x == 0 && threadIdx.x < 2 * c + 1) {
        const int t = threadIdx.x;
        const int64_t v = t < c ? fold_image_counts(cnt_partial, b, c, t) : (hist ? hist[t - c] : 0);
        for (int p = 0; p < world; ++p) ll_store_i64(peers.base[p] + my_off + tail_off(c, k) + (int64_t)t * 16, v, my);
    }
    xchg_fold_ema_ack(peers, rank, world, slot, c, k, my, true, proto_old, eps, one_minus_decay, decay, proto_new, sums_out,
                      counts_out, hist_out);
}

}  // namespace

extern "C" int64_t uem_xchg_region_bytes(int world, int depth, int c, int k) {
    if (world < 1 || world > kMaxWorld || depth < 1 || depth > kMaxDepth || c < 1 || k < 1) return -1;
    return kOffSlots + (int64_t)depth * world * slot_bytes(c, k);
}

extern "C" int uem_xchg_send_f32(const void* partials_ws, int b, int c, int k, const int64_t* max_id, const int64_t* hist,
                                 const void* const* peer_regions, int rank, int world, int depth, int slot, int64_t* global_id_out,
                                 int parts, void* stream) {
    UEM_REQUIRE(b > 0 && c > 0 && c <= UEM_MAX_C && k > 0 && (parts & 3) && !(parts & ~7), "uem_xchg_send_f32: bad arguments");
    UEM_REQUIRE(!(parts & 1) || partials_ws, "uem_xchg_send_f32: the sums part needs the partials");
    Peers P;
    if (int rc = fill_peers(&P, peer_regions, rank, world, depth, slot, "uem_xchg_send_f32")) return rc;
    const ProtoPartials PP = proto_partials(partials_ws, b, c, k);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((parts & 1) ? kSendChunks : 1, world, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (parts == 2) ? 1 : 0;   // id only: overlap the launch with the preceding (region-max) kernel
    UEM_CUDA(cudaLaunchKernelEx(&cfg, xchg_send_kernel, PP.sums, PP.counts, b, c, k, max_id, hist, P, rank, world, slot, global_id_out, parts));
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_xchg_wait_maxid(void* region, int world, int depth, int slot, int c, int k, int64_t* max_id_out, void* stream) {
    UEM_REQUIRE(region && world >= 1 && world <= kMaxWorld && depth >= 1 && depth <= kMaxDepth && slot >= 0 && slot < depth && c > 0 && k > 0,
                "uem_xchg_wait_maxid: bad arguments");
    xchg_wait_maxid_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((char*)region, world, slot, c, k, max_id_out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_xchg_fold_finalize_ema_f32(const void* const* peer_regions, int rank, int world, int depth, int slot, int c, int k,
                                              const float* proto_old, float eps, float one_minus_decay, float decay, float* proto_new,
                                              float* sums_out, int64_t* counts_out, int64_t* hist_out, void* stream) {
    UEM_REQUIRE(c > 0 && c <= UEM_MAX_C && k > 0 && (!proto_new || proto_old), "uem_xchg_fold_finalize_ema_f32: bad arguments");
    Peers P;
    if (int rc = fill_peers(&P, peer_regions, rank, world, depth, slot, "uem_xchg_fold_finalize_ema_f32")) return rc;
    xchg_fold_finalize_kernel<<<uem_div_up((int64_t)c * k, 256), 256, 0, (cudaStream_t)stream>>>(
        P, rank, world, slot, c, k, proto_old, eps, one_minus_decay, decay, proto_new, sums_out, counts_out, hist_out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_xchg_exchange_fold_ema_f32(const void* partials_ws, int b, int c, int k, const int64_t* hist,
                                              const void* const* peer_regions, int rank, int world, int depth, int slot,
                                              const float* proto_old, float eps, float one_minus_decay, float decay, float* proto_new,
                                              float* sums_out, int64_t* counts_out, int64_t* hist_out, void* stream) {
    UEM_REQUIRE(partials_ws && b > 0 && c > 0 && c <= UEM_MAX_C && k > 0 && (!proto_new || proto_old),
                "uem_xchg_exchange_fold_ema_f32: bad arguments");
    Peers P;
    if (int rc = fill_peers(&P, peer_regions, rank, world, depth, slot, "uem_xchg_exchange_fold_ema_f32")) return rc;
    const ProtoPartials PP = proto_partials(partials_ws, b, c, k);
    xchg_exchange_fold_kernel<<<uem_div_up((int64_t)c * k, 256), 256, 0, (cudaStream_t)stream>>>(
        PP.sums, PP.counts, b, c, k, hist, P, rank, world, slot, proto_old, eps, one_minus_decay, decay, proto_new, sums_out, counts_out,
        hist_out);
    UEM_CHECK_LAUNCH();
    return 0;
}

extern "C" int uem_xchg_status(const void* region, int* status_out, void* stream) {
    UEM_REQUIRE(region && status_out, "uem_xchg_status: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    UEM_CUDA(cudaMemcpyAsync(status_out, (const char*)region + offsetof(XHeader, status), sizeof(int), cudaMemcpyDeviceToHost, st));
    UEM_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// ---- cudaIpc plumbing for the symmetric region (used when torch's symmetric memory is unavailable) ----------------------
extern "C" int uem_peer_alloc(int64_t bytes, void** ptr, void* handle64) {
    UEM_REQUIRE(bytes > 0 && ptr && handle64, "uem_peer_alloc: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    UEM_CUDA(cudaMalloc(ptr, (size_t)bytes));
    UEM_CUDA(cudaMemset(*ptr, 0, (size_t)bytes));
    UEM_CUDA(cudaDeviceSynchronize());
    UEM_CUDA(cudaIpcGetMemHandle((cudaIpcMemHandle_t*)handle64, *ptr));
    return 0;
}
extern "C" int uem_peer_open(const void* handle64, void** ptr) {
    UEM_REQUIRE(handle64 && ptr, "uem_peer_open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    UEM_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
extern "C" int uem_peer_close(void* ptr) {
    if (ptr) UEM_CUDA(cudaIpcCloseMemHandle(ptr));
    return 0;
}
extern "C" int uem_peer_free(void* ptr) {
    if (ptr) UEM_CUDA(cudaFree(ptr));
    return 0;
}
