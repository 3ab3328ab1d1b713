// The steps of the exchange protocol (uem_exchange.cu has the description), each written once: slot addressing, LL stores
// and loads, the acknowledgement wait, the id poll and the receive -> rank-ordered fold -> EMA -> acknowledge tail.  They
// are shared by the exchange kernels and the region-max kernel, whose last CTA can carry the id part of a step's send (no
// separate launch between the region pass and its consumers).
#pragma once
#include "uem_proto_stats.cuh"
#include <limits.h>
#include <stddef.h>

// Outside the anonymous namespace: uem_region_max_f32 (uem_region.cu) takes a RegionXchg from uem_refine.cu.
constexpr int kMaxWorld = 16;
struct Peers {
    char* base[kMaxWorld];
};
// The id part of a step's send, carried by the last CTA of the region-max kernel: the rank-local max superpixel id goes
// into slot [slot][rank] of every rank and, with global_id_out, the batch-global id (alignment.py:241) is left there once
// every rank's id of this step has arrived.
struct RegionXchg {
    Peers peers;
    int rank, world, slot, c, k;   // world == 0 in a kernel argument: no send
    long long* global_id_out;
};

namespace {

constexpr int kMaxDepth = 4;
constexpr int kSendChunks = 6;
constexpr int kOffAcks = 1280, kOffSlots = 2048;
constexpr unsigned long long kSpinLimitNs = 2000000000ull;

struct XHeader {
    unsigned seq_send[kMaxDepth];
    unsigned seq_recv[kMaxDepth];
    unsigned arrive_all[kMaxDepth];
    unsigned fold_arrive[kMaxDepth];
    int status;
    unsigned region_done;   // arrival counter of the region-max kernel when it carries the id part of a send (zero between launches)
};
static_assert(sizeof(XHeader) <= kOffAcks, "header overflows its page");

// slot geometry in 8-byte LL words
__host__ __device__ inline int64_t sum_words(int c, int k) { return (((int64_t)c * k) + 3) & ~(int64_t)3; }
__host__ __device__ inline int64_t tail_words(int c) { return (int64_t)(2 * c + 2) * 2; }   // int64 values as (lo, hi)
__host__ __device__ inline int64_t slot_bytes(int c, int k) { return ((sum_words(c, k) + tail_words(c)) * 8 + 127) & ~(int64_t)127; }
// byte offsets: slot [slot][r] from a region base; its tail (counts, histogram, max id) and its id word from the slot start
__host__ __device__ inline int64_t slot_off(int slot, int world, int r, int c, int k) {
    return kOffSlots + ((int64_t)slot * world + r) * slot_bytes(c, k);
}
__host__ __device__ inline int64_t tail_off(int c, int k) { return sum_words(c, k) * 8; }
__host__ __device__ inline int64_t id_off(int c, int k) { return tail_off(c, k) + (int64_t)(2 * c + 1) * 16; }

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// bounded spin until *flag >= want; returns false on timeout
__device__ __forceinline__ bool spin_until(const unsigned* flag, unsigned want) {
    if ((int)(ld_acquire_sys(flag) - want) >= 0) return true;
    const unsigned long long t0 = globaltimer_ns();
    while ((int)(ld_acquire_sys(flag) - want) < 0) {
        __nanosleep(64);
        if (globaltimer_ns() - t0 > kSpinLimitNs) return false;
    }
    return true;
}
// LL word: one 8-byte transaction {payload, sequence number}
__device__ __forceinline__ void ll_store(char* dst, unsigned payload, unsigned seq) {
    asm volatile("st.volatile.global.v2.u32 [%0], {%1,%2};" ::"l"(dst), "r"(payload), "r"(seq) : "memory");
}
__device__ __forceinline__ void ll_store_i64(char* dst, int64_t v, unsigned seq) {
    ll_store(dst, (unsigned)((uint64_t)v & 0xffffffffu), seq);
    ll_store(dst + 8, (unsigned)((uint64_t)v >> 32), seq);
}
// polls (bounded) until the word carries `seq`; *ok = false on timeout
__device__ __forceinline__ unsigned ll_load(const char* src, unsigned seq, bool* ok) {
    unsigned v, f;
    asm volatile("ld.volatile.global.v2.u32 {%0,%1}, [%2];" : "=r"(v), "=r"(f) : "l"(src) : "memory");
    if (f == seq) return v;
    const unsigned long long t0 = globaltimer_ns();
    do {
        __nanosleep(32);
        asm volatile("ld.volatile.global.v2.u32 {%0,%1}, [%2];" : "=r"(v), "=r"(f) : "l"(src) : "memory");
        if (globaltimer_ns() - t0 > kSpinLimitNs) { *ok = false; return v; }
    } while (f != seq);
    return v;
}

__device__ __forceinline__ int64_t ll_load_i64(const char* src, unsigned seq, bool* ok) {
    const unsigned lo = ll_load(src, seq, ok), hi = ll_load(src + 8, seq, ok);
    return (int64_t)(((uint64_t)hi << 32) | lo);
}

// One element of the rank-ordered fold: the words of ALL ranks are requested first (independent loads: one memory latency
// instead of `world` in a row -- the slots were written over NVLink, so every first touch misses), then checked; a word
// whose sequence number is not there yet falls back to the bounded poll.  Same additions in the same order as a plain loop.
__device__ __forceinline__ void ll_raw(const char* src, unsigned& v, unsigned& f) {
    asm volatile("ld.volatile.global.v2.u32 {%0,%1}, [%2];" : "=r"(v), "=r"(f) : "l"(src) : "memory");
}
__device__ __forceinline__ void ll_fold_ranks(const char* sum0, const char* cnt0, int64_t sb, int world, unsigned seq, float* s_out,
                                              int64_t* n_out, bool* ok) {
    float s = 0.f;
    int64_t n = 0;
    for (int r0 = 0; r0 < world; r0 += 8) {
        unsigned v[8], vf[8], lo[8], lf[8], hi[8], hf[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (r0 + u < world) {
                const int64_t off = (int64_t)(r0 + u) * sb;
                ll_raw(sum0 + off, v[u], vf[u]);
                ll_raw(cnt0 + off, lo[u], lf[u]);
                ll_raw(cnt0 + off + 8, hi[u], hf[u]);
            }
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (r0 + u < world) {
                const int r = r0 + u;
                const int64_t off = (int64_t)r * sb;
                if (vf[u] != seq) v[u] = ll_load(sum0 + off, seq, ok);
                if (lf[u] != seq) lo[u] = ll_load(cnt0 + off, seq, ok);
                if (hf[u] != seq) hi[u] = ll_load(cnt0 + off + 8, seq, ok);
                const float x = __uint_as_float(v[u]);
                s = r ? s + x : x;
                n += (int64_t)(((uint64_t)hi[u] << 32) | lo[u]);
            }
    }
    *s_out = s;
    *n_out = n;
}

__device__ __forceinline__ void flag_timeout(char* region) { atomicOr(&reinterpret_cast<XHeader*>(region)->status, 8); }

// Before this rank overwrites its part of `slot` (sequence number seq), peer p must have folded the previous contents
// (seq - 1); p's acknowledgement lands in this rank's own region
__device__ __forceinline__ void wait_ack(char* mine, int slot, int p, unsigned seq) {
    const unsigned* ack = reinterpret_cast<const unsigned*>(mine + kOffAcks) + slot * kMaxWorld + p;
    if (!spin_until(ack, seq - 1u)) flag_timeout(mine);
}

// Called by a whole warp 0: lane r polls rank r's id word of `slot` (tagged seq) in this rank's region; every lane returns
// the max over the ranks, the batch-global id (alignment.py:241)
__device__ __forceinline__ long long poll_max_id(char* mine, int slot, int world, int c, int k, unsigned seq) {
    const int r = threadIdx.x;
    long long id = LLONG_MIN;
    if (r < world) {
        bool ok = true;
        id = ll_load_i64(mine + slot_off(slot, world, r, c, k) + id_off(c, k), seq, &ok);
        if (!ok) flag_timeout(mine);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long other = __shfl_xor_sync(0xffffffffu, id, o);
        id = other > id ? other : id;
    }
    return id;
}

// The id part of a step's send, issued by ONE CTA (every thread calls this; blockDim >= 32), tagged with the slot's next
// send sequence number like xchg_send_kernel's parts = 2
__device__ __forceinline__ void xchg_send_id_from_cta(const RegionXchg& x, long long id) {
    char* const mine = x.peers.base[x.rank];
    const unsigned my = *reinterpret_cast<volatile unsigned*>(&reinterpret_cast<XHeader*>(mine)->seq_send[x.slot]) + 1u;
    if ((int)threadIdx.x < x.world) {
        const int p = threadIdx.x;
        wait_ack(mine, x.slot, p, my);
        ll_store_i64(x.peers.base[p] + slot_off(x.slot, x.world, x.rank, x.c, x.k) + id_off(x.c, x.k), id, my);
    }
    if (x.global_id_out && threadIdx.x < 32) {
        const long long g = poll_max_id(mine, x.slot, x.world, x.c, x.k, my);
        if (threadIdx.x == 0) x.global_id_out[0] = g;
    }
}

// The receiving end of a step, for element i = blockIdx.x * 256 + threadIdx.x of the (c,k) bank (blockDim 256): every
// rank's words of `slot` tagged seq are folded in RANK ORDER (identical fp32 additions on every rank -> the replicated
// prototype bank stays bit-identical), then keep-old rule + EMA; the first 2c+1 threads fold the counts / histogram.
// The last CTA acknowledges the slot to every peer and records seq as received, and also as sent when advance_send
// (a launch that was also the step's send).
__device__ __forceinline__ void xchg_fold_ema_ack(const Peers& peers, int rank, int world, int slot, int c, int k, unsigned seq,
                                                  bool advance_send, const float* __restrict__ proto_old, float eps,
                                                  float one_minus_decay, float decay, float* __restrict__ proto_new,
                                                  float* __restrict__ sums_out, int64_t* __restrict__ counts_out,
                                                  int64_t* __restrict__ hist_out) {
    char* const mine = peers.base[rank];
    XHeader* hdr = reinterpret_cast<XHeader*>(mine);
    const int64_t sb = slot_bytes(c, k);
    const char* slots = mine + slot_off(slot, world, 0, c, k);
    const char* tails = slots + tail_off(c, k);
    const int i = blockIdx.x * 256 + threadIdx.x;
    bool ok = true;
    if (i < c * k) {
        float s;
        int64_t n;
        ll_fold_ranks(slots + (int64_t)i * 8, tails + (int64_t)(i / k) * 16, sb, world, seq, &s, &n, &ok);
        if (sums_out) sums_out[i] = s;
        if (proto_new) proto_new[i] = proto_ema(s, n, proto_old[i], eps, one_minus_decay, decay);
    }
    if (i < 2 * c + 1 && (counts_out || hist_out)) {
        int64_t n = 0;
        for (int r = 0; r < world; ++r) n += ll_load_i64(tails + r * sb + (int64_t)i * 16, seq, &ok);
        if (i < c) { if (counts_out) counts_out[i] = n; }
        else if (hist_out) hist_out[i - c] = n;
    }
    if (!ok) flag_timeout(mine);
    __threadfence();
    __syncthreads();
    __shared__ int s_last;
    if (threadIdx.x == 0) s_last = (atomicAdd(&hdr->fold_arrive[slot], 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        if (threadIdx.x < world)
            st_release_sys(reinterpret_cast<unsigned*>(peers.base[threadIdx.x] + kOffAcks) + slot * kMaxWorld + rank, seq);
        if (threadIdx.x == 0) {
            hdr->fold_arrive[slot] = 0u;
            __threadfence();
            if (advance_send) *reinterpret_cast<volatile unsigned*>(&hdr->seq_send[slot]) = seq;
            *reinterpret_cast<volatile unsigned*>(&hdr->seq_recv[slot]) = seq;
        }
    }
}

inline int fill_peers(Peers* P, const void* const* peer_regions, int rank, int world, int depth, int slot, const char* who) {
    UEM_REQUIRE(peer_regions && world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "%s: bad rank/world (%d/%d, at most %d ranks)",
                who, rank, world, kMaxWorld);
    UEM_REQUIRE(depth >= 1 && depth <= kMaxDepth && slot >= 0 && slot < depth, "%s: bad slot/depth (%d/%d, depth at most %d)", who, slot,
                depth, kMaxDepth);
    for (int r = 0; r < kMaxWorld; ++r) P->base[r] = r < world ? (char*)peer_regions[r] : nullptr;
    for (int r = 0; r < world; ++r) UEM_REQUIRE(P->base[r], "%s: peer region %d is NULL", who, r);
    return 0;
}

}  // namespace
