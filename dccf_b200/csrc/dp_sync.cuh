// dp_sync.cuh — the flag protocol of the data-parallel exchange (dp_exchange.cu), usable from inside OTHER kernels:
// a consumer kernel waits for the peers' segments in its own prologue (no k_dp_wait launch between producer and
// consumer) and its last CTA hands the receive buffers back to the peers (no k_dp_done launches after it).
#pragma once
#include "common.cuh"

namespace dccf {

constexpr int DP_MAX_WORLD = 8;
constexpr int DP_MAX_CTAS = 148;       // CTAs of one push (one arrival flag each)
// Flag area of a symmetric exchange buffer, in int32 words from flag_off:
//   arrival  [DP_MAX_WORLD][DP_MAX_CTAS]   arrival[src][c] = epoch: CTA c of rank src's push of that epoch has landed here
//   consumed [DP_MAX_WORLD]                consumed[dst]   = epoch: rank dst has finished reading what this rank pushed
constexpr int DP_FLAG_CONSUMED = DP_MAX_WORLD * DP_MAX_CTAS;
constexpr int DP_FLAG_WORDS = DP_FLAG_CONSUMED + DP_MAX_WORLD;

__host__ __device__ inline int dp_push_ctas(int64_t seg_floats) {
    int64_t c = (seg_floats / 4 + 255) / 256;
    return (int)(c > DP_MAX_CTAS ? DP_MAX_CTAS : (c < 1 ? 1 : c));
}

__device__ __forceinline__ int32_t ld_acquire_sys(const int32_t* p) {
    int32_t v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int32_t ld_relaxed_sys(const int32_t* p) {
    int32_t v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(int32_t* p, int32_t v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(int32_t* p, int32_t v) {
    asm volatile("st.relaxed.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// System-scope fences are the expensive part of this protocol on B200 (measured on 2 and 8 GPUs, tools/step_timeline
// stamps): an acquire load or release store at .sys scope stalls its thread 3-4 us, and one fence.sc.sys per CTA from
// the three CTAs an SM holds serialises to 3 / 6 / 9 us.  The LEAN protocol (default) therefore keeps exactly the
// ordering each hand-over needs:
//   producer, data -> arrival flag: the bulk copies are waited for (cp.async.bulk.wait_group 0: performed at the peer's
//     L2, the point of coherence of its memory) before a relaxed store of the flag travels the same way;
//   consumer, arrival flag -> data: relaxed polling, CTA barrier, ONE fence.acq_rel.gpu (orders the CTA's later loads and
//     drops the SM's L1 lines), barrier — the peer's writes are already in this GPU's L2 when its flag is;
//   consumer -> producer, consumed flag (write-after-read): the readers' loads have returned before the last CTA's
//     relaxed store is issued (gpu-scope fence + atomic counter between them); the producer polls it relaxed and its
//     copies are control-dependent on what it saw.
// Spin until *p >= want.  A peer that died (or never reaches this step) must not leave this GPU spinning for ever:
// after 60 s — four orders of magnitude beyond any legitimate wait, start-up skew included — the kernel traps, the
// process sees a CUDA error and the job fails loudly instead of hanging the box.
__device__ __forceinline__ void spin_until(const int32_t* p, int32_t want, bool strict = true) {
    const unsigned long long t0 = global_ns();
    while ((strict ? ld_acquire_sys(p) : ld_relaxed_sys(p)) < want) {
        if (global_ns() - t0 > 60ull * 1000000000ull) __trap();
    }
}

// device-side image of dccf_dp_sync (include/dccf_b200.h)
struct DpChannel {
    float* base[DP_MAX_WORLD];   // the symmetric buffer on every rank (own at index rank)
    int64_t flag_off;            // floats: the flag area (see DP_FLAG_*) starts here
    int32_t* epoch_dev;          // completed exchanges on this channel
    int32_t n_ctas;              // CTAs of every rank's push on this channel (dp_push_ctas of its segment)
};
struct DpSync {
    int32_t world, rank, n_wait, n_done;
    DpChannel wait[3];
    DpChannel done[3];
    const float* loss_parts;     // optional: n_loss values loss_stride floats apart, summed into loss_out by the last CTA
    int64_t loss_stride;
    int32_t n_loss;
    int32_t flags;               // dccf_dp_sync.flags
    float* loss_out;
};

// Prologue of a consumer CTA: every CTA of every rank's push of the current exchange has landed, on all wait channels.
// ALL threads of the CTA poll (relaxed loads, a thread's flags of all channels in flight together: at 8 ranks a channel
// has 8 x 148 flags — one warp needed ten dependent rounds of system-scope loads per look, ~8 us even when everything
// had already arrived; 256 threads need one), the CTA agrees through the barrier, ONE thread then issues the system-scope
// fence that orders the CTA's later reads after the observed flags and a second barrier hands that order to the others.
// (A first version fenced in every thread of every CTA: 87 K system fences made the consumer 16 us slower.)
// Call from all threads of the CTA (contains barriers).  mask: bit c set = wait for channel c (CTA-uniform).
__device__ __forceinline__ void dp_wait_inline(const DpSync& s, const uint32_t mask = 7u) {
    if (s.n_wait > 0 && (mask & ((1u << s.n_wait) - 1u)) != 0u) {
        const unsigned long long t0 = global_ns();
        int32_t want[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) want[c] = c < s.n_wait ? __ldg(s.wait[c].epoch_dev) + 1 : 0;
        bool ok;
        do {
            int32_t slack = 0x7fffffff;           // min over the thread's flags of (flag - epoch wanted)
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                if (c >= s.n_wait) break;
                if (!((mask >> c) & 1u)) continue;
                const DpChannel& ch = s.wait[c];
                const int32_t* arrival = reinterpret_cast<const int32_t*>(ch.base[s.rank] + ch.flag_off);
                const int total = s.world * ch.n_ctas;
#pragma unroll 4
                for (int i = threadIdx.x; i < total; i += blockDim.x)
                    slack = min(slack, ld_relaxed_sys(arrival + (i / ch.n_ctas) * DP_MAX_CTAS + (i % ch.n_ctas)) - want[c]);
            }
            ok = slack >= 0;
            if (!ok) {
                if (global_ns() - t0 > 60ull * 1000000000ull) __trap();      // a peer died: fail loudly (see spin_until)
                __nanosleep(64);
            }
        } while (!__syncthreads_and(ok));
        if (threadIdx.x == 0) asm volatile("fence.acq_rel.gpu;" ::: "memory");
        __syncthreads();
    }
}

// Tail of the LAST CTA of the consumer (all other CTAs have finished reading): total loss, then consumed flags to
// every peer (one release store per lane) and the channels' epoch counters.  Call from all threads of that CTA.
__device__ __forceinline__ void dp_done_inline(const DpSync& s) {
    const int t = threadIdx.x;
    if (s.loss_out != nullptr && t == 0) {
        float acc = 0.f;
        for (int i0 = 0; i0 < s.n_loss; i0 += 8) {               // the ranks' terms, loaded together, added in rank order
            float part[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i0 + i < s.n_loss) part[i] = __ldcg(s.loss_parts + (size_t)(i0 + i) * s.loss_stride);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (i0 + i < s.n_loss) acc += part[i];
        }
        s.loss_out[0] = acc;
    }
    if (t < s.n_done * s.world) {
        const DpChannel& c = s.done[t / s.world];
        const int peer = t % s.world;
        int32_t* flag = reinterpret_cast<int32_t*>(c.base[peer] + c.flag_off) + DP_FLAG_CONSUMED + s.rank;
        st_relaxed_sys(flag, *c.epoch_dev + 1);
    }
    __syncthreads();
    if (t < s.n_done) *s.done[t].epoch_dev += 1;
}

}  // namespace dccf
