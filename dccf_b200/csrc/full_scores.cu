// full_scores.cu — full-catalogue scoring: the one place on this path where the work is a dense
// user x item GEMM, so it runs on the tcgen05 tensor cores.
//
//   score[u,i] = ( <A[u,:], B[i,:]> + row_bias[u] + col_bias[i] + g ) * col_scale[i]        A [U,64], B [I,64]
//
// Instances:
//   * the IPSBiasedMF exposure matrix (src/models/IPSBiasedMF.py:37-57; README.md:27-29: the full U x I
//     prediction matrix of that model IS <ds>.ips_expo_prob.npy): A = user factors, B = item factors,
//     row/col bias = user/item bias, g = global bias, col_scale = 1 / max(propensity, M);
//   * deterministic DCCF scoring of the whole catalogue (std 0, no confounders): A = E_user,
//     B = relu(PI + PF) (the per-item hidden vector), no biases.
// Two outputs: the materialised [U,I] matrix (HBM-write-bound: 4 B per score) and/or a fused per-user
// top-k (score desc, item id asc) that never writes the matrix — each epilogue thread owns one user row
// and keeps its running top-k in registers while the item tiles stream through TMEM.
//
// Two kernels:
//   k_fs_prep_b   once per call: the item side B'[i] = cs_i * [B[i,:], 1, col_bias[i], 0..] split into its TF32 hi / lo
//                 parts and written as the K-major core-matrix images the MMA reads, one 36 KB block per 64-item tile.
//                 (The first version re-did this split in every CTA for every tile: 250 user tiles x 594 item tiles on
//                 the Yelp shape, four staging warps per CTA — the epilogue and the staging, not the tensor pipe, set its
//                 2.2 us per tile; ncu: tensor pipe 26 %.)
//   k_full_scores CTA = 128 users x a range of 64-item tiles, 10 warps:
//     warps 0-7  epilogue: warp w reads TMEM lanes 32*(w%4).. (its quarter of the user rows) and the columns
//                32*(w/4).. of the tile — thread = (user row, half of the tile's items); double-buffered accumulators
//     warp  8    one thread issues tcgen05.mma.kind::tf32 (M=128, N=64, K=8) x 9 k-steps x 3 products, A from TMEM
//     warp  9    one thread streams the pre-split item-tile images with cp.async.bulk (TMA engine) through a
//                three-stage mbarrier ring
#include "common.cuh"
#include "tc_common.cuh"

namespace dccf {

constexpr int FS_BM = 128, FS_BN = 64;
constexpr int FS_NT = 320;
constexpr int FS_KMAX = 16;                              // largest fused top-k
constexpr int FS_BSTAGES = 3;                            // item-tile ring
// The biases and the column scale ride inside the GEMM: K is augmented from 64 to 72,
//   A'[u] = [ A[u,:], row_bias[u] + g, 1, 0.. ]      B'[i] = cs_i * [ B[i,:], 1, col_bias[i], 0.. ]
// so that <A'[u], B'[i]> = cs_i * (<A[u],B[i]> + row_bias[u] + g + col_bias[i]) and the epilogue is a bare
// accumulator read.  Operand images ([rows x 32] / [rows x 8], K-major core matrices, hi and lo parts):
constexpr uint32_t FS_B_IMG = FS_BN * 32 * 4;            //  8 KB
constexpr uint32_t FS_B_AUG = FS_BN * 8 * 4;             //  2 KB
constexpr int FS_KAUG = 72;                              // augmented K
constexpr uint32_t FS_TM_AHI = 256, FS_TM_ALO = 384;     // TMEM columns of the user tile (hi / lo), 72 each
constexpr uint32_t FS_B_HALF = 2 * FS_B_IMG + FS_B_AUG;
constexpr uint32_t FS_STAGE = 2 * FS_B_HALF;             // 36 KB per item tile: [hi: img0 img1 aug | lo: img0 img1 aug]
constexpr int FS_OUT_LD = 32 + 4;                        // padded row of a warp's 32 x 32 store-staging tile
constexpr uint32_t FS_OUT_BYTES = 8 * 32 * FS_OUT_LD * 4;   // one tile per epilogue warp
constexpr uint32_t FS_SMEM = FS_BSTAGES * FS_STAGE + FS_OUT_BYTES + 256;
constexpr uint32_t FS_TMEM_COLS = 512;                   // accumulators: 2 buffers x (main + correction) x 64; A: 2 x 72
constexpr uint32_t FS_LBO = 128, FS_SBO = 1024, FS_SBO_AUG = 256;

__device__ __forceinline__ float fs_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

struct FsParams {
    const float* A;          // [U,64]
    const float* row_bias;   // [U] or null
    const float* Bimg;       // pre-split item-tile images (k_fs_prep_b): n_tiles x FS_STAGE bytes
    float g;
    float* out;              // [U,I] or null
    float* topk_score;       // [2*splits,U,k] or null (one list per item split and column half)
    int64_t* topk_id;        // [2*splits,U,k]
    int32_t n_users, n_items, k;
    int32_t tiles_per_split, n_tiles;
    const int64_t* excl_off;     // [U+1] CSR over the rows of A (EXCL only)
    const int32_t* excl_items;   // each row's excluded items, ascending, unique, < n_items
};

// byte offset of 4 consecutive k values of row r inside a hi (or lo) half of an item-tile image
__device__ __forceinline__ uint32_t fs_b_offset(int r, int k) {
    if (k < 64) return (uint32_t)(k >> 5) * FS_B_IMG + (uint32_t)((r >> 3) * FS_SBO + ((k & 31) >> 2) * FS_LBO + (r & 7) * 16);
    return 2 * FS_B_IMG + (uint32_t)((r >> 3) * FS_SBO_AUG + ((k - 64) >> 2) * FS_LBO + (r & 7) * 16);
}

// The item side, once per call: thread = (item of the tile, half of K).  One CTA of 128 threads per 64-item tile.
__global__ void __launch_bounds__(128) k_fs_prep_b(const float* __restrict__ B, const float* __restrict__ col_bias,
                                                   const float* __restrict__ col_scale, int32_t n_items,
                                                   float* __restrict__ Bimg) {
    const int item = threadIdx.x & 63, khalf = threadIdx.x >> 6;
    const int64_t i_raw = (int64_t)blockIdx.x * FS_BN + item;
    const bool live = i_raw < n_items;
    const int64_t i = live ? i_raw : (int64_t)n_items - 1;
    const float cs = live ? (col_scale ? __ldg(col_scale + i) : 1.f) : 0.f;      // dead columns score 0
    uint8_t* hi_base = reinterpret_cast<uint8_t*>(Bimg) + (size_t)blockIdx.x * FS_STAGE;
    uint8_t* lo_base = hi_base + FS_B_HALF;
    auto put = [&](int k, float4 v) {
        float4 hi, lo;
        hi.x = fs_hi(v.x); hi.y = fs_hi(v.y); hi.z = fs_hi(v.z); hi.w = fs_hi(v.w);
        lo.x = __fsub_rn(v.x, hi.x); lo.y = __fsub_rn(v.y, hi.y); lo.z = __fsub_rn(v.z, hi.z); lo.w = __fsub_rn(v.w, hi.w);
        const uint32_t off = fs_b_offset(item, k);
        *reinterpret_cast<float4*>(hi_base + off) = hi;
        *reinterpret_cast<float4*>(lo_base + off) = lo;
    };
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        float4 v = ldg4(B + (size_t)i * D + khalf * 32 + q * 4);
        v.x *= cs; v.y *= cs; v.z *= cs; v.w *= cs;
        put(khalf * 32 + q * 4, v);
    }
    // augmentation columns: khalf 0 writes k 64..67, khalf 1 writes k 68..71
    const float cb = (live && col_bias) ? __ldg(col_bias + i) : 0.f;
    put(64 + khalf * 4, (khalf == 0) ? make_float4(cs, cs * cb, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f));
}

// TOPK: fused per-user top-k (k <= KCAP); the matrix is written when prm.out is given (either or both).
// EXCL (with TOPK, without the matrix): each row's items in prm.excl_off / prm.excl_items score -inf and never rank.
template <bool TOPK, int KCAP, bool EXCL>
__global__ void __launch_bounds__(FS_NT, 1) k_full_scores(const FsParams prm) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* stage0 = smem;
    float* out_s = reinterpret_cast<float*>(smem + FS_BSTAGES * FS_STAGE);
    uint64_t* b_full = reinterpret_cast<uint64_t*>(smem + FS_BSTAGES * FS_STAGE + FS_OUT_BYTES);
    uint64_t* b_empty = b_full + FS_BSTAGES;
    uint64_t* acc_full = b_empty + FS_BSTAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t u0 = (int64_t)blockIdx.x * FS_BM;
    const int split = blockIdx.y;
    const int t_lo = split * prm.tiles_per_split;
    const int t_hi = min(t_lo + prm.tiles_per_split, prm.n_tiles);

    if (tid == 0) {
        for (int s = 0; s < FS_BSTAGES; ++s) {
            tc::mbar_init(&b_full[s], 1);      // the expect_tx arrival of the bulk copy
            tc::mbar_init(&b_empty[s], 1);     // tcgen05.commit
        }
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&acc_full[s], 1);    // tcgen05.commit
            tc::mbar_init(&acc_empty[s], 8);   // eight epilogue warps
        }
        tc::fence_barrier_init();
    }
    if (warp == 8) tc::tmem_alloc(tmem_slot, FS_TMEM_COLS);

    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    // user tile -> tensor memory, once: A'[u] = [A[u,:], row_bias[u] + g, 1, 0..] as 72 columns of lane u;
    // warps 0-3 write the hi parts, warps 4-7 the lo parts (a warp reaches the 32 lanes of its quarter)
    if (warp < 8) {
        const int r = (warp & 3) * 32 + lane;
        const bool lo_part = warp >= 4;
        const int64_t u = min(u0 + r, (int64_t)prm.n_users - 1);
        const uint32_t col0 = lo_part ? FS_TM_ALO : FS_TM_AHI;
#pragma unroll
        for (int c8 = 0; c8 < FS_KAUG / 8; ++c8) {
            float v[8];
            if (c8 < 8) {
                const float4 x0 = ldg4(prm.A + (size_t)u * D + c8 * 8), x1 = ldg4(prm.A + (size_t)u * D + c8 * 8 + 4);
                v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
            } else {
                v[0] = (prm.row_bias ? __ldg(prm.row_bias + u) : 0.f) + prm.g;
                v[1] = 1.f;
                v[2] = v[3] = v[4] = v[5] = v[6] = v[7] = 0.f;
            }
            uint32_t w[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float hi = fs_hi(v[j]);
                w[j] = __float_as_uint(lo_part ? __fsub_rn(v[j], hi) : hi);
            }
            tc::tmem_st_32x8(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + col0 + c8 * 8, w);
        }
        tc::tmem_wait_st();
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();

    if (warp == 9) {
        // ===== item-tile streamer: one bulk copy of the pre-split image per tile =====
        if (lane == 0) {
            for (int t = t_lo; t < t_hi; ++t) {
                const int n = t - t_lo, s = n % FS_BSTAGES;
                const uint32_t ph = (uint32_t)(n / FS_BSTAGES) & 1u;
                tc::mbar_wait(&b_empty[s], ph ^ 1u);
                tc::mbar_arrive_expect_tx(&b_full[s], FS_STAGE);
                tc::bulk_g2s(stage0 + s * FS_STAGE, reinterpret_cast<const uint8_t*>(prm.Bimg) + (size_t)t * FS_STAGE,
                             FS_STAGE, &b_full[s]);
            }
        }
        __syncwarp();
    } else if (warp == 8) {
        // ===== MMA issuer =====
        if (lane == 0) {
            constexpr uint32_t idesc = tc::make_idesc_tf32(FS_BM, FS_BN);
            for (int t = t_lo; t < t_hi; ++t) {
                const int n = t - t_lo, s = n % FS_BSTAGES, a = n & 1;
                const uint32_t ph_b = (uint32_t)(n / FS_BSTAGES) & 1u, ph_a = (uint32_t)(n >> 1) & 1u;
                tc::mbar_wait(&b_full[s], ph_b);
                tc::mbar_wait(&acc_empty[a], ph_a ^ 1u);   // the epilogue has drained this accumulator pair
                tc::tc_fence_after_sync();
                const uint32_t b_hi0 = tc::smem_u32(stage0 + s * FS_STAGE), b_lo0 = b_hi0 + FS_B_HALF;
                const uint32_t d_main = tmem_base + (uint32_t)(a * 2) * FS_BN;
                const uint32_t d_corr = d_main + FS_BN;
#pragma unroll
                for (int ks = 0; ks < 9; ++ks) {
                    // k-steps 0..7: the two [rows x 32] images; k-step 8: the [rows x 8] augmentation image
                    const uint32_t b_off = ks < 8 ? (uint32_t)(ks >> 2) * FS_B_IMG + (uint32_t)(ks & 3) * 2 * FS_LBO : 2 * FS_B_IMG;
                    const uint32_t sbo = ks < 8 ? FS_SBO : FS_SBO_AUG;
                    const uint32_t a_hi = tmem_base + FS_TM_AHI + (uint32_t)ks * 8;     // 8 K columns per MMA
                    const uint32_t a_lo = tmem_base + FS_TM_ALO + (uint32_t)ks * 8;
                    const uint64_t b_hi = tc::make_smem_desc(b_hi0 + b_off, FS_LBO, sbo);
                    const uint64_t b_lo = tc::make_smem_desc(b_lo0 + b_off, FS_LBO, sbo);
                    tc::umma_tf32_ts(d_corr, a_lo, b_hi, idesc, ks != 0);
                    tc::umma_tf32_ts(d_corr, a_hi, b_lo, idesc, 1u);
                    tc::umma_tf32_ts(d_main, a_hi, b_hi, idesc, ks != 0);
                }
                tc::umma_commit(&b_empty[s]);
                tc::umma_commit(&acc_full[a]);
            }
        }
        __syncwarp();
    } else {
        // ===== epilogue: thread = (user row, half of the tile's 64 items) =====
        const int quarter = warp & 3, chalf = warp >> 2;
        const int64_t u = u0 + quarter * 32 + lane;
        const bool valid = u < prm.n_users;
        // running top-k of this (row, column half), ASCENDING: top_s[0] is the worst kept score = the threshold an item
        // must beat (-inf until k items are in), top_s[k-1] the best.  Every index below is a compile-time constant
        // (a first version kept the list descending and read its k-th entry: the compiler put the list in local
        // memory, and the insertion path — taken by some lane in 61 % of the tiles — was most of the kernel's 660 M
        // instructions).
        float top_s[KCAP];
        int32_t top_i[KCAP];
#pragma unroll
        for (int j = 0; j < KCAP; ++j) { top_s[j] = -INFINITY; top_i[j] = -1; }
        const int k = prm.k;
        float* my_out = out_s + warp * 32 * FS_OUT_LD;
        // exclusion cursor: this thread's items arrive in ascending id order, so the row's sorted list is merged
        // against them.  nxt = the first listed item not yet passed; one binary search places it at the split's
        // first item, and every read stays inside [c, c_end) whatever the list holds.
        int64_t c = 0, c_end = 0;
        int32_t nxt = INT32_MAX;
        if (EXCL && valid) {
            c = __ldg(prm.excl_off + u);
            c_end = __ldg(prm.excl_off + u + 1);
            const int32_t first = t_lo * FS_BN;
            int64_t hi = c_end;
            while (c < hi) {
                const int64_t mid = (c + hi) >> 1;
                if (__ldg(prm.excl_items + mid) < first) c = mid + 1; else hi = mid;
            }
            if (c < c_end) nxt = __ldg(prm.excl_items + c);
        }
        for (int t = t_lo; t < t_hi; ++t) {
            const int n = t - t_lo, a = n & 1;
            const uint32_t ph = (uint32_t)(n >> 1) & 1u;
            tc::mbar_wait(&acc_full[a], ph);
            tc::tc_fence_after_sync();
            const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(a * 2) * FS_BN + chalf * 32;
            const int64_t i0 = (int64_t)t * FS_BN + chalf * 32;       // first item of this warp's 32 columns
            // main and correction accumulators of this warp's 32 columns: two TMEM loads in flight, one wait
            uint32_t rm[32], rc[32];
            tc::tmem_ld_32x32_issue(lane_addr, rm);
            tc::tmem_ld_32x32_issue(lane_addr + FS_BN, rc);
            tc::tmem_wait_ld();
            // every TMEM read of this warp is done: hand the accumulator pair back to the MMA warp
            tc::tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&acc_empty[a]);
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(rm[j]) + __uint_as_float(rc[j]);
            uint32_t excl_mask = 0;     // bit j: item i0 + j is excluded
            if (EXCL) {
                const int32_t lo32 = (int32_t)i0;
                while (nxt < lo32 + 32) {                   // items below i0 (the other column half's) are passed over
                    if (nxt >= lo32) excl_mask |= 1u << (nxt - lo32);
                    ++c;
                    nxt = (c < c_end) ? __ldg(prm.excl_items + c) : INT32_MAX;
                }
            }
            if (TOPK) {
                // columns beyond the catalogue (last tile only) never rank; NaN never compares greater and stays out
                const int64_t live = (int64_t)prm.n_items - i0;
                float best = -INFINITY;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (live < 32 && j >= live) v[j] = -INFINITY;
                    if (EXCL && (excl_mask >> j & 1u)) v[j] = -INFINITY;   // compile-time j: v stays in registers
                    best = fmaxf(best, v[j]);
                }
                if (best > top_s[0]) {
                    // some item of this row's 32 beats the threshold: items arrive in ascending id, so an equal score
                    // never displaces an earlier one (strict comparisons)
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        if (v[j] > top_s[0]) {
                            top_s[0] = v[j];
                            top_i[0] = (int32_t)(i0 + j);
#pragma unroll
                            for (int q = 0; q + 1 < KCAP; ++q) {
                                if (q + 1 < k && top_s[q] > top_s[q + 1]) {
                                    const float ts = top_s[q]; top_s[q] = top_s[q + 1]; top_s[q + 1] = ts;
                                    const int32_t ti = top_i[q]; top_i[q] = top_i[q + 1]; top_i[q + 1] = ti;
                                }
                            }
                        }
                    }
                }
            }
            if (prm.out != nullptr) {
                // this row's scores go through the warp's staging tile: coalesced write-out of the 32 x 32 tile, four
                // rows (4 x 128 B) per instruction
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    st4(my_out + lane * FS_OUT_LD + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
                __syncwarp();
                const int rsub = lane >> 3, c4 = (lane & 7) * 4;
                const bool vec_ok = ((prm.n_items & 3) == 0);
#pragma unroll 4
                for (int rr = 0; rr < 32; rr += 4) {
                    const int r = rr + rsub;
                    const int64_t uu = u0 + quarter * 32 + r;
                    const int64_t i = i0 + c4;
                    if (uu < prm.n_users) {
                        const float4 w = ld4(my_out + r * FS_OUT_LD + c4);
                        float* dst = prm.out + (size_t)uu * prm.n_items + i;
                        if (vec_ok && i + 3 < prm.n_items) {
                            st4(dst, w);
                        } else {
                            const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e)
                                if (i + e < prm.n_items) dst[e] = wv[e];
                        }
                    }
                }
                __syncwarp();
            }
        }
        if (TOPK && valid) {
            // best first (the merge kernel reads descending lists, unfilled slots last)
            const size_t list = (size_t)(split * 2 + chalf);
            float* ds = prm.topk_score + (list * prm.n_users + u) * k;
            int64_t* di = prm.topk_id + (list * prm.n_users + u) * k;
#pragma unroll
            for (int q = 0; q < KCAP; ++q)
                if (q < k) { ds[k - 1 - q] = top_s[q]; di[k - 1 - q] = top_i[q]; }
        }
    }

    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 8) tc::tmem_dealloc(tmem_base, FS_TMEM_COLS);
}

// merge the per-split partial top-k lists: one thread per user
__global__ void k_topk_merge(const float* __restrict__ ps, const int64_t* __restrict__ pi, int32_t n_splits,
                             int32_t n_users, int32_t k, float* __restrict__ out_s, int64_t* __restrict__ out_i) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_users) return;
    float last_s = INFINITY;
    int64_t last_i = -1;
    for (int q = 0; q < k; ++q) {
        float bs = -INFINITY;
        int64_t bi = -1;
        for (int s = 0; s < n_splits; ++s)
            for (int j = 0; j < k; ++j) {
                const size_t o = ((size_t)s * n_users + u) * k + j;
                const float sc = ps[o];
                const int64_t id = pi[o];
                if (id < 0) continue;
                const bool below = (q == 0) || sc < last_s || (sc == last_s && id > last_i);
                if (below && (bi < 0 || sc > bs || (sc == bs && id < bi))) { bs = sc; bi = id; }
            }
        out_s[(size_t)u * k + q] = bs;
        out_i[(size_t)u * k + q] = bi;
        last_s = bs;
        last_i = bi;
    }
}

}  // namespace dccf

using namespace dccf;

extern "C" int32_t dccf_full_scores_splits(int32_t n_users, int32_t n_items) {
    // number of partial top-k lists per user the caller's workspaces must hold: item splits x 2 column halves
    const int ut = (n_users + FS_BM - 1) / FS_BM, it = (n_items + FS_BN - 1) / FS_BN;
    if (ut <= 0 || it <= 0) return 2;
    int splits = (2 * 148 + ut - 1) / ut;      // about two CTAs' worth of work per SM
    if (splits > it) splits = it;
    if (splits < 1) splits = 1;
    return 2 * splits;
}

extern "C" int64_t dccf_full_scores_ws_floats(int32_t n_items) {
    const int64_t n_tiles = (n_items + FS_BN - 1) / FS_BN;
    return n_tiles * (int64_t)(FS_STAGE / 4);
}

extern "C" int dccf_full_scores(int32_t n_users, int32_t n_items, const float* A, const float* B,
                                const float* row_bias, const float* col_bias, const float* col_scale, float g,
                                float* out, int32_t k, float* topk_score, int64_t* topk_id, float* ws_score,
                                int64_t* ws_id, float* ws_items, const int64_t* excl_off, const int32_t* excl_items,
                                void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DCCF_CHECK_ARG(A && B, "dccf_full_scores: null factor matrix");
    DCCF_CHECK_ARG(out || (topk_score && topk_id), "dccf_full_scores: nothing to produce (out and top-k both null)");
    DCCF_CHECK_ARG((topk_score == nullptr) == (topk_id == nullptr), "dccf_full_scores: top-k needs both score and id outputs");
    DCCF_CHECK_ARG(topk_score == nullptr || (k >= 1 && k <= FS_KMAX), "dccf_full_scores: fused top-k supports 1 <= k <= %d, got %d", FS_KMAX, k);
    DCCF_CHECK_ARG(ws_items != nullptr && (reinterpret_cast<uintptr_t>(ws_items) & 127) == 0,
                   "dccf_full_scores: ws_items (dccf_full_scores_ws_floats(n_items) floats, 128-byte aligned) is required");
    DCCF_CHECK_ARG((excl_off == nullptr) == (excl_items == nullptr), "dccf_full_scores: exclusion needs both excl_off and excl_items");
    DCCF_CHECK_ARG(excl_off == nullptr || (topk_score != nullptr && out == nullptr),
                   "dccf_full_scores: known-item exclusion applies to the fused top-k only (out must be NULL)");
    if (n_users <= 0 || n_items <= 0) return DCCF_OK;
    const int lists = dccf_full_scores_splits(n_users, n_items);
    const int splits = lists / 2;
    DCCF_CHECK_ARG(topk_score == nullptr || (ws_score && ws_id), "dccf_full_scores: top-k needs the [%d,U,k] workspaces (dccf_full_scores_splits)", lists);
    FsParams prm;
    prm.A = A; prm.row_bias = row_bias; prm.Bimg = ws_items; prm.g = g;
    prm.out = out; prm.n_users = n_users; prm.n_items = n_items; prm.k = topk_score ? k : 1;
    prm.n_tiles = (n_items + FS_BN - 1) / FS_BN;
    prm.tiles_per_split = (prm.n_tiles + splits - 1) / splits;
    prm.topk_score = topk_score ? ws_score : nullptr;
    prm.topk_id = topk_score ? ws_id : nullptr;
    prm.excl_off = excl_off;
    prm.excl_items = excl_items;
    static PerDeviceOnce attr_once;
    if (attr_once.need()) {
        cudaError_t e = cudaFuncSetAttribute(k_full_scores<false, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_full_scores<true, 8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_full_scores<true, 16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_full_scores<true, 8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_full_scores<true, 16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FS_SMEM);
        if (e != cudaSuccess) {
            set_error("dccf_full_scores: cannot opt in to %u bytes of shared memory: %s", FS_SMEM, cudaGetErrorString(e));
            return DCCF_ERR_CUDA;
        }
        attr_once.mark();
    }
    k_fs_prep_b<<<(unsigned)prm.n_tiles, 128, 0, stream>>>(B, col_bias, col_scale, n_items, ws_items);
    DCCF_CHECK_LAUNCH("k_fs_prep_b");
    dim3 grid((unsigned)((n_users + FS_BM - 1) / FS_BM), (unsigned)splits);
    if (!topk_score) k_full_scores<false, 1, false><<<grid, FS_NT, FS_SMEM, stream>>>(prm);
    else if (excl_off) {
        if (k <= 8) k_full_scores<true, 8, true><<<grid, FS_NT, FS_SMEM, stream>>>(prm);
        else k_full_scores<true, 16, true><<<grid, FS_NT, FS_SMEM, stream>>>(prm);
    } else if (k <= 8) k_full_scores<true, 8, false><<<grid, FS_NT, FS_SMEM, stream>>>(prm);
    else k_full_scores<true, 16, false><<<grid, FS_NT, FS_SMEM, stream>>>(prm);
    DCCF_CHECK_LAUNCH("k_full_scores");
    if (topk_score) {
        k_topk_merge<<<(unsigned)((n_users + 127) / 128), 128, 0, stream>>>(ws_score, ws_id, lists, n_users, k, topk_score, topk_id);
        DCCF_CHECK_LAUNCH("k_topk_merge");
    }
    return DCCF_OK;
}
