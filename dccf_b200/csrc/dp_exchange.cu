// dp_exchange.cu — the data-parallel gradient exchange as plain kernels over NVLink peer memory.
//
// Every rank owns a symmetric buffer [ recv: world x seg floats | arrival flags | consumed flags ] whose
// address on every peer is known (torch symmetric memory / CUDA IPC mappings).  Per training step:
//   k_dp_push : wait until every peer has consumed the previous step's data, then store this rank's packed
//               gradient segment (records, dW, db, keys, loss) straight into slot `rank` of EVERY peer's recv
//               buffer with 128-bit stores over NVLink (an all-gather written by the producers), fence, and
//               publish the step number in each peer's arrival flag
//   k_dp_wait : spin until all world arrival flags show this step (the peers run their own k_dp_push)
//   ...the Adam kernels read recv...
//   k_dp_done : tell every peer this rank is done reading, advance the step counter
// No NCCL call and no host involvement: the whole step, exchange included, is capturable in one CUDA graph.
#include "common.cuh"
#include "dp_sync.cuh"
#include "tc_common.cuh"

namespace dccf {

struct DpPeers {
    float* base[DP_MAX_WORLD];
};

// Up to two ranges of the segment are not copied from `send` but summed on the fly from row-split partial buffers
// (the dW / db partials of the backward, ascending split order — the fold dccf_sum_parts would do in two more launches).
struct DpFold {
    const float* parts;      // [n_parts][stride]
    int32_t n_parts;
    int64_t stride;          // floats between partial buffers
    int64_t off4, n4;        // range of the segment in float4 units: [off4, off4 + n4)
};
struct DpFolds {
    DpFold f[2];
    int32_t n;
};

// shared -> global bulk copy (TMA engine), completion tracked by bulk async-groups
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(tc::smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// float4 per piece staged in shared memory: 4 KB.  Not more: the push of the gradient records runs BESIDE the dW kernel
// (96 KB of shared memory per CTA) and the side-stream Adam sweep (120 KB) — with a 16 KB piece the three no longer fit
// an SM together and the dW kernel started 7 us later.
constexpr int DP_PIECE4 = 256;

// Each CTA owns a CONTIGUOUS range of the segment: it reads (or folds from the partial buffers) the range piece by piece
// into shared memory and ships every piece to every peer with ONE bulk copy per peer issued by one lane — the TMA engine
// writes to the peers' memory over NVLink in large transactions.  (The first version stored from the SMs, one 16-byte
// store per thread and peer: measured on 8 x B200, a rank's 7 MB of outgoing segments drained at ~115 GB/s and the last
// peer saw the dW / db segment 24 us after the push kernel had ended.)  Lane p then waits for ITS copies to complete and
// publishes the CTA's arrival on peer p with a relaxed store (lean protocol, dp_sync.cuh): one arrival flag per (source
// rank, source CTA) on every peer, no grid-wide counter, no second fence.  The consumer waits for all of a push's flags.
// FOLD: some ranges of the segment are sums of partial buffers (dW / db): sixteen float4 loads in flight per thread — a
// register budget the plain pushes (ids, gradient records: they run beside the dW kernel and the sweep) do not pay for
template <bool FOLD>
__global__ void __launch_bounds__(256) k_dp_push(const float* __restrict__ send, int64_t seg, DpPeers peers, int world,
                                                 int rank, int64_t flag_off, const int32_t* __restrict__ epoch_dev,
                                                 int32_t* cta_counter, const DpFolds folds) {
    __shared__ __align__(128) float4 piece[DP_PIECE4];
    // debug timeline slot by what is pushed: 8 ids (small segment), 10 gradient records, 11 dW / db / loss (folded partials)
    const int tl_slot = folds.n > 0 ? 11 : (seg < 16384 ? 8 : 10);
    tl_begin(tl_slot);
    (void)cta_counter;
    // (the peers' consumed flags are requested together with the epoch: one round trip instead of two on the way to the
    // first copy)
    const int32_t* consumed = reinterpret_cast<const int32_t*>(peers.base[rank] + flag_off) + DP_FLAG_CONSUMED;
    // (world <= DP_MAX_WORLD already; the constant bound, tested first, keeps ptxas at 23 / 112 registers instead of 26 / 114)
    const int32_t seen = ((int)threadIdx.x < DP_MAX_WORLD && (int)threadIdx.x < world) ? ld_relaxed_sys(consumed + threadIdx.x)
                                                                                       : (int32_t)0x80000000;
    const int32_t epoch = __ldg(epoch_dev) + 1;
    // a consumer launched as a programmatic dependent (dccf_adam_touched, DCCF_DP_SYNC_OVERLAP_PUSH) may start once every
    // CTA of this push is resident and has read the channel's epoch (the consumer's last CTA advances it)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int64_t n4 = seg >> 2;
    const int64_t per = (n4 + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * per, hi = min(lo + per, n4);
    const float4* src = reinterpret_cast<const float4*>(send);
    bool waited = false;
    for (int64_t base = lo; base < hi || !waited; base += DP_PIECE4) {
        const int64_t m = max((int64_t)0, min((int64_t)DP_PIECE4, hi - base));
        for (int64_t i = base + threadIdx.x; i < base + m; i += blockDim.x) {
            int which = -1;
            if (FOLD)
                for (int k = 0; k < folds.n; ++k)
                    if (i >= folds.f[k].off4 && i < folds.f[k].off4 + folds.f[k].n4) which = k;
            float4 v;
            if (which < 0) {
                v = src[i];
            } else {
                const DpFold& f = folds.f[which];
                const float* pp = f.parts + (i - f.off4) * 4;
                v = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int32_t p0 = 0; p0 < f.n_parts; p0 += 16) {      // up to sixteen loads in flight, added in ascending order
                    float4 t16[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (p0 + j < f.n_parts) t16[j] = __ldg(reinterpret_cast<const float4*>(pp + (size_t)(p0 + j) * f.stride));
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (p0 + j < f.n_parts) { v.x += t16[j].x; v.y += t16[j].y; v.z += t16[j].z; v.w += t16[j].w; }
                }
            }
            piece[i - base] = v;
        }
        if (!waited) {
            // peers have finished reading what this rank pushed last step (checked once per CTA, after the first loads)
            if ((int)threadIdx.x < world && seen < epoch - 1) spin_until(consumed + threadIdx.x, epoch - 1, false);
            waited = true;
        }
        tc::fence_proxy_async_smem();        // this thread's shared-memory writes -> visible to the bulk-copy engine
        __syncthreads();
        if ((int)threadIdx.x < world && m > 0) {
            bulk_s2g(peers.base[threadIdx.x] + (int64_t)rank * seg + base * 4, piece, (uint32_t)(m * 16));
            bulk_commit();
            bulk_wait_read0();               // the piece has been read out: the buffer may be refilled
        }
        __syncthreads();
    }
    if (FOLD) { tl_begin(14); tl_end(14); }  // (debug timeline: every piece folded and handed to the copy engine)
    if ((int)threadIdx.x < world) {
        bulk_wait0();                        // this lane's copies to its peer are complete
        if (FOLD) { tl_begin(15); tl_end(15); }
        asm volatile("fence.proxy.async;" ::: "memory");
        int32_t* flag = reinterpret_cast<int32_t*>(peers.base[threadIdx.x] + flag_off) + rank * DP_MAX_CTAS + blockIdx.x;
        st_relaxed_sys(flag, epoch);         // (the copies it announces are complete: lean protocol, dp_sync.cuh)
    }
    tl_end(tl_slot);
}

__global__ void k_dp_wait(const float* my_base, int world, int64_t flag_off, const int32_t* __restrict__ epoch_dev, int n_ctas) {
    tl_begin(9);
    const int32_t epoch = __ldg(epoch_dev) + 1;
    const int32_t* arrival = reinterpret_cast<const int32_t*>(my_base + flag_off);
    for (int i = threadIdx.x; i < world * n_ctas; i += blockDim.x)
        spin_until(arrival + (i / n_ctas) * DP_MAX_CTAS + (i % n_ctas), epoch);
    __syncthreads();
    tl_end(9);
}

__global__ void k_dp_done(DpPeers peers, int world, int rank, int64_t flag_off, int32_t* epoch_dev) {
    const int32_t epoch = *epoch_dev + 1;
    __syncthreads();
    if ((int)threadIdx.x < world)
        st_release_sys(reinterpret_cast<int32_t*>(peers.base[threadIdx.x] + flag_off) + DP_FLAG_CONSUMED + rank, epoch);
    __syncthreads();
    if (threadIdx.x == 0) *epoch_dev = epoch;
}

static int fill_peers(DpPeers* out, const uint64_t* peer_bases, int world, const char* who) {
    DCCF_CHECK_ARG(peer_bases != nullptr && world >= 1 && world <= DP_MAX_WORLD, "%s: world size must be in [1,%d]", who, DP_MAX_WORLD);
    for (int p = 0; p < DP_MAX_WORLD; ++p) out->base[p] = p < world ? reinterpret_cast<float*>(peer_bases[p]) : nullptr;
    for (int p = 0; p < world; ++p) DCCF_CHECK_ARG(out->base[p] != nullptr, "%s: peer %d has a null buffer", who, p);
    return DCCF_OK;
}

}  // namespace dccf

using namespace dccf;

extern "C" int dccf_debug_timeline_dp(unsigned long long* slots) {
    cudaError_t e = cudaMemcpyToSymbol(g_timeline, &slots, sizeof(slots));
    if (e != cudaSuccess) {
        set_error("dccf_debug_timeline: %s", cudaGetErrorString(e));
        return DCCF_ERR_CUDA;
    }
    return DCCF_OK;
}

// peer_bases: HOST array of `world` device addresses (this rank's own buffer at index `rank`)
static int dp_push_impl(const float* send, int64_t seg_floats, const uint64_t* peer_bases, int32_t world, int32_t rank,
                        int64_t flag_off, const int32_t* epoch_dev, int32_t* cta_counter, const DpFolds& folds,
                        cudaStream_t stream) {
    DpPeers peers;
    int rc = fill_peers(&peers, peer_bases, world, "dccf_dp_push");
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(send && epoch_dev && cta_counter, "dccf_dp_push: null buffer");
    DCCF_CHECK_ARG(seg_floats > 0 && seg_floats % 4 == 0, "dccf_dp_push: segment length must be a positive multiple of 4 floats");
    DCCF_CHECK_ARG(rank >= 0 && rank < world, "dccf_dp_push: rank %d outside [0,%d)", rank, world);
    const int64_t ctas = dp_push_ctas(seg_floats);
    static PerDeviceOnce carve_once;      // (same carveout as its neighbours in the step, see dccf_adam_link_ids)
    if (carve_once.need()) {
        cudaFuncSetAttribute(k_dp_push<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(k_dp_push<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carve_once.mark();
    }
    if (folds.n > 0)
        k_dp_push<true><<<(unsigned)ctas, 256, 0, stream>>>(send, seg_floats, peers, world, rank, flag_off, epoch_dev, cta_counter, folds);
    else
        k_dp_push<false><<<(unsigned)ctas, 256, 0, stream>>>(send, seg_floats, peers, world, rank, flag_off, epoch_dev, cta_counter, folds);
    DCCF_CHECK_LAUNCH("k_dp_push");
    return DCCF_OK;
}

// peer_bases: HOST array of `world` device addresses (this rank's own buffer at index `rank`)
extern "C" int dccf_dp_push(const float* send, int64_t seg_floats, const uint64_t* peer_bases, int32_t world,
                            int32_t rank, int64_t flag_off, const int32_t* epoch_dev, int32_t* cta_counter,
                            void* stream_) {
    DpFolds folds;
    folds.n = 0;
    return dp_push_impl(send, seg_floats, peer_bases, world, rank, flag_off, epoch_dev, cta_counter, folds,
                        (cudaStream_t)stream_);
}

extern "C" int dccf_dp_push_fold(const float* send, int64_t seg_floats, const uint64_t* peer_bases, int32_t world,
                                 int32_t rank, int64_t flag_off, const int32_t* epoch_dev, int32_t* cta_counter,
                                 const float* parts_a, int32_t n_parts_a, int64_t stride_a, int64_t off_a, int64_t n_a,
                                 const float* parts_b, int32_t n_parts_b, int64_t stride_b, int64_t off_b, int64_t n_b,
                                 void* stream_) {
    DpFolds folds;
    folds.n = 0;
    const float* parts[2] = {parts_a, parts_b};
    const int32_t n_parts[2] = {n_parts_a, n_parts_b};
    const int64_t stride[2] = {stride_a, stride_b}, off[2] = {off_a, off_b}, n[2] = {n_a, n_b};
    for (int k = 0; k < 2; ++k) {
        if (parts[k] == nullptr || n[k] <= 0) continue;
        DCCF_CHECK_ARG(n_parts[k] >= 1 && off[k] % 4 == 0 && n[k] % 4 == 0 && stride[k] % 4 == 0 && off[k] + n[k] <= seg_floats &&
                           (reinterpret_cast<uintptr_t>(parts[k]) & 15) == 0,
                       "dccf_dp_push_fold: range %d must be 16-byte aligned and inside the segment", k);
        DpFold& f = folds.f[folds.n++];
        f.parts = parts[k]; f.n_parts = n_parts[k]; f.stride = stride[k]; f.off4 = off[k] / 4; f.n4 = n[k] / 4;
    }
    return dp_push_impl(send, seg_floats, peer_bases, world, rank, flag_off, epoch_dev, cta_counter, folds,
                        (cudaStream_t)stream_);
}

extern "C" int64_t dccf_dp_flag_floats(void) { return DP_FLAG_WORDS; }

extern "C" int dccf_dp_wait(const float* my_base, int64_t seg_floats, int32_t world, int64_t flag_off, const int32_t* epoch_dev,
                            void* stream_) {
    DCCF_CHECK_ARG(my_base && epoch_dev && world >= 1 && world <= DP_MAX_WORLD && seg_floats > 0, "dccf_dp_wait: bad argument");
    k_dp_wait<<<1, 256, 0, (cudaStream_t)stream_>>>(my_base, world, flag_off, epoch_dev, dp_push_ctas(seg_floats));
    DCCF_CHECK_LAUNCH("k_dp_wait");
    return DCCF_OK;
}

extern "C" int dccf_dp_done(const uint64_t* peer_bases, int32_t world, int32_t rank, int64_t flag_off, int32_t* epoch_dev,
                            void* stream_) {
    DpPeers peers;
    int rc = fill_peers(&peers, peer_bases, world, "dccf_dp_done");
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(epoch_dev != nullptr && rank >= 0 && rank < world, "dccf_dp_done: bad argument");
    k_dp_done<<<1, 32, 0, (cudaStream_t)stream_>>>(peers, world, rank, flag_off, epoch_dev);
    DCCF_CHECK_LAUNCH("k_dp_done");
    return DCCF_OK;
}
