// tc_train.cu — the two large contractions of a TRAINING step on the tensor cores (tcgen05 / TMEM), spread over
// every SM although a step has few rows (256 pairs = 5 632 predictor rows = 44 row tiles for 148 SMs).
//
// Forward (replaces src/models/DCCF.py:84-96 for the step's rows):
//   pre[r,:] = W · [E_item[item_r] | Feat[i_r] + eps_r] + b
//   grid = (row tiles of 128) x (K splits): CTA (t, ks) multiplies its 128 rows by the K range of split ks
//   (32-wide chunks of the 832 columns) as an error-compensated 3xTF32 product and writes a PARTIAL
//   pre-activation tile; k_train_fwd_finish (one CTA per pair) adds the partials and the bias, applies
//   ReLU + dropout, saves h, dots with the user row and runs the backdoor-adjusted softmax sum of the pair.
//
// Backward (replaces the addmm backward of autograd, src/runners/BaseRunner.py:183):
//   gW[c, k] = sum_r dpre[r, c] · x[r, k]          gb[c] = sum_r dpre[r, c]
//   grid = (tiles of 128 columns of [x | 1]) x (row splits): the contraction index is the ROW, so the
//   producers regenerate x (same Philox stream as the forward) and store it TRANSPOSED — a 4x4 register
//   transpose across four lanes turns "4 columns of one row" into "4 rows of one column", which is one
//   16-byte store into the same K-major core-matrix layout the forward uses (no MN-major descriptors).
//   dpre comes from the record role of k_bpr_bwd (bpr_bwd.cu), which also produces the embedding-gradient
//   records and the loss.  The bias gradient falls out of the same GEMM through a column of ones at k = K.
#include "backdoor.cuh"
#include "common.cuh"
#include "tc_common.cuh"
#include "tc_layout.cuh"

namespace dccf {

// Ring depth of the two training contractions: the evaluation scorer's depth.  (A third stage, with the side-stream
// sweep's shared-memory limiter shrunk to make room for its 144 KB, was measured and rejected: DESIGN.md §8.)
constexpr int TT_STAGES = TC_STAGES;
constexpr uint32_t TT_SMEM_BYTES = TT_STAGES * TC_STAGE_BYTES + 256;
static_assert(TT_SMEM_BYTES <= 227 * 1024, "training ring does not fit the shared memory of an SM");

// ---------------------------------------------------------------------------------------------
// W [D, K] -> per-chunk operand images [chunk][ hi 8 KB | lo 8 KB ], all K = D + F columns
// ---------------------------------------------------------------------------------------------
__global__ void k_prep_w_image(const float* __restrict__ W, int K, float* __restrict__ img) {
    const int total = D * K;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int n = i / K, k = i - n * K;
        const float w = __ldg(W + i);
        const float hi = tf32_hi(w);
        const int c = k / TC_KC, kk = k - c * TC_KC;
        float* base = img + (size_t)c * (2 * TC_B_BYTES / 4);
        const uint32_t off = core_offset(n, kk) / 4;
        base[off] = hi;
        base[TC_B_BYTES / 4 + off] = __fsub_rn(w, hi);
    }
}

// store a float4 as its TF32 hi part and the exact remainder
__device__ __forceinline__ void store_hi_lo(uint8_t* hi_base, uint8_t* lo_base, uint32_t off, const float4& v) {
    float4 hi, lo;
    hi.x = tf32_hi(v.x); hi.y = tf32_hi(v.y); hi.z = tf32_hi(v.z); hi.w = tf32_hi(v.w);
    lo.x = __fsub_rn(v.x, hi.x); lo.y = __fsub_rn(v.y, hi.y);
    lo.z = __fsub_rn(v.z, hi.z); lo.w = __fsub_rn(v.w, hi.w);
    *reinterpret_cast<float4*>(hi_base + off) = hi;
    *reinterpret_cast<float4*>(lo_base + off) = lo;
}

// issue the 3xTF32 MMAs of one 32-wide stage (see tc_scores.cu for the accumulator rotation)
__device__ __forceinline__ void issue_stage_mmas(uint32_t stage_addr, uint32_t tmem_base, int stage_index) {
    constexpr uint32_t idesc = tc::make_idesc_tf32(TC_BM, D);
    const uint32_t a_hi = stage_addr;
    const uint32_t a_lo = a_hi + TC_A_BYTES;
    const uint32_t b_hi = a_hi + 2 * TC_A_BYTES;
    const uint32_t b_lo = b_hi + TC_B_BYTES;
#pragma unroll
    for (int j = 0; j < TC_KC / 8; ++j) {
        const uint32_t ko = (uint32_t)j * 2 * TC_LBO;   // two core matrices per K=8 step
        const uint64_t da_hi = tc::make_smem_desc(a_hi + ko, TC_LBO, TC_SBO);
        const uint64_t da_lo = tc::make_smem_desc(a_lo + ko, TC_LBO, TC_SBO);
        const uint64_t db_hi = tc::make_smem_desc(b_hi + ko, TC_LBO, TC_SBO);
        const uint64_t db_lo = tc::make_smem_desc(b_lo + ko, TC_LBO, TC_SBO);
        const int ks = stage_index * (TC_KC / 8) + j;
        const uint32_t main_acc = tmem_base + (uint32_t)(1 + ks % (TC_NACC - 1)) * D;
        tc::umma_tf32(tmem_base, da_lo, db_hi, idesc, ks != 0);
        tc::umma_tf32(tmem_base, da_hi, db_lo, idesc, 1u);
        tc::umma_tf32(main_acc, da_hi, db_hi, idesc, ks >= TC_NACC - 1);
    }
}

// accumulator columns [16*quarter, 16*quarter + 16) of this thread's TMEM lane: three main accumulators,
// then the small correction terms, added in round-to-nearest FP32
__device__ __forceinline__ void load_acc_quarter(uint32_t tmem_base, int lane_quarter, int quarter, float (&acc)[16]) {
    float part[16];
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lane_quarter * 32) << 16) + (uint32_t)(quarter * 16);
    tc::tmem_ld_32x16(lane_addr + 1 * D, acc);
    tc::tmem_ld_32x16(lane_addr + 2 * D, part);
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] += part[j];
    tc::tmem_ld_32x16(lane_addr + 3 * D, part);
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] += part[j];
    tc::tmem_ld_32x16(lane_addr, part);
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] += part[j];
}

// =============================================================================================
// forward
// =============================================================================================
struct TrainFwdParams {
    const float* E_item;
    const float* Feat;
    const float* gWimg;          // operand images of W, one per 32-wide chunk of K
    const int64_t* X;
    const int64_t* sample_item;
    const uint64_t* batch_ptrs;  // optional (with batch_cursor): X / sample_item are batch *batch_cursor of the epoch arrays
    const int64_t* batch_cursor; //   whose base addresses are batch_ptrs[0..1] (the staged copies are written concurrently)
    const float* noise;          // mode 1
    float* pre_part;             // [n_ksplits][N][D]
    int32_t* err_flag;
    int64_t n_rows;
    int32_t n_items, F, S, A, R;
    int32_t n_chunks;            // (D + F) / 32
    float noise_std;
    RngSpec rng;
};

template <int NOISE_MODE>
__global__ void __launch_bounds__(TC_NT, 2) k_train_fwd_tc(const TrainFwdParams prm) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + TT_STAGES * TC_STAGE_BYTES);
    uint64_t* empty_bar = full_bar + TT_STAGES;
    uint64_t* accum_bar = empty_bar + TT_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    tl_begin(2);
    tl_end(7);        // slot 7, "end" field: the LATEST CTA start of this kernel
    const int64_t row_base = (int64_t)blockIdx.x * TC_BM;
    const int ks = (int)blockIdx.y, n_ks = (int)gridDim.y;
    const int c_lo = (int)(((int64_t)ks * prm.n_chunks) / n_ks);
    const int c_hi = (int)(((int64_t)(ks + 1) * prm.n_chunks) / n_ks);
    const int n_local = c_hi - c_lo;

    // producers: thread = (row, quarter of the 32-wide K chunk); the id lookups overlap the barrier / TMEM set-up
    const int row = tid & (TC_BM - 1), kq = (tid >> 7) & 3;
    const int64_t grow = min(row_base + row, prm.n_rows - 1);
    int32_t fi = 0, it = 0;
    if (warp < TC_PRODUCERS / 32) {
        const uint32_t p = (uint32_t)grow / (uint32_t)prm.R;
        const int z = (int)((uint32_t)grow - p * (uint32_t)prm.R) / prm.A;
        const int64_t *X = prm.X, *si = prm.sample_item;
        if (prm.batch_cursor != nullptr) {
            // the ids straight from the device-resident epoch: the launch that stages them (k_link_ids) runs beside this one
            const int64_t b = *prm.batch_cursor, n_pairs = (int64_t)((uint32_t)prm.n_rows / (uint32_t)prm.R);
            X = reinterpret_cast<const int64_t*>(prm.batch_ptrs[0]) + b * n_pairs * 2;
            si = reinterpret_cast<const int64_t*>(prm.batch_ptrs[1]) + b * n_pairs * prm.S;
        }
        fi = checked_id(X[2 * (int64_t)p + 1], prm.n_items, prm.err_flag);
        it = (z == 0) ? fi : checked_id(si[(int64_t)p * prm.S + (z - 1)], prm.n_items, prm.err_flag);
    }

    if (tid == 0) {
        for (int s = 0; s < TT_STAGES; ++s) {
            tc::mbar_init(&full_bar[s], TC_PRODUCERS / 32 + 1);   // producer warps + the expect_tx arrival
            tc::mbar_init(&empty_bar[s], 1);                      // one tcgen05.commit
        }
        tc::mbar_init(accum_bar, 1);
        tc::fence_barrier_init();
    }
    if (warp == TC_PRODUCERS / 32) tc::tmem_alloc(tmem_slot, TC_TMEM_COLS);
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;
    // The middle kernel may be launched as a programmatic dependent of this one (phases bit 16): its CTAs may be placed
    // from here on.  They read this grid's outputs only after their griddepcontrol.wait, which returns when this grid has
    // COMPLETED — and this grid does not complete before the kernel before it has (the wait at the end).
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp < TC_PRODUCERS / 32) {
        // ===== producers =====
        const float* item_ptr = prm.E_item + (size_t)it * D + kq * 8;
        const float* feat_ptr = prm.Feat + (size_t)fi * prm.F + kq * 8;
        const float* nptr = (NOISE_MODE == 1) ? prm.noise + (size_t)grow * prm.F + kq * 8 : nullptr;
        RngKey key_noise = make_rng_key(0, 0, DOMAIN_NOISE);
        if (NOISE_MODE == 2) key_noise = resolve_rng_key(prm.rng, DOMAIN_NOISE);
        // the table values of chunk c (this thread's 8 columns of its row): E_item columns for c < D / 32, Feat after
        auto fetch = [&](int c, float4 (&v)[2]) {
            const int k0 = c * TC_KC;                 // first column of the chunk in [E_item | Feat]
            const float* src = (k0 < D) ? item_ptr + k0 : feat_ptr + (k0 - D);
#pragma unroll
            for (int q = 0; q < 2; ++q) v[q] = ldg4(src + 4 * q);
        };
        // chunk c's noise added to its table values
        auto add_noise = [&](int c, float4 (&v)[2]) {
            const int k0 = c * TC_KC;
            if (k0 < D) return;
            const int f0 = k0 - D;
            if (NOISE_MODE != 0) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    float4 e;
                    if (NOISE_MODE == 1) e = ldg4(nptr + f0 + 4 * q);
                    else e = noise_quad(key_noise, (uint32_t)grow, (uint32_t)(f0 / 4 + kq * 2 + q), prm.noise_std);
                    v[q].x = __fadd_rn(v[q].x, e.x); v[q].y = __fadd_rn(v[q].y, e.y);
                    v[q].z = __fadd_rn(v[q].z, e.z); v[q].w = __fadd_rn(v[q].w, e.w);
                }
            }
        };
        // stage i of this CTA's sequence: wait until the MMAs that read its slot have completed, store, publish
        auto commit = [&](int i, const float4 (&v)[2]) {
            const int s = i % TT_STAGES;
            const uint32_t ph = (uint32_t)(i / TT_STAGES) & 1u;
            tc::mbar_wait(&empty_bar[s], ph ^ 1u);
            uint8_t* a_hi = smem + s * TC_STAGE_BYTES;
            uint8_t* a_lo = a_hi + TC_A_BYTES;
#pragma unroll
            for (int q = 0; q < 2; ++q) store_hi_lo(a_hi, a_lo, core_offset(row, kq * 8 + 4 * q), v[q]);
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&full_bar[s]);
        };
        float4 v[2];
        if (n_local > 0) fetch(c_lo, v);
        for (int i = 0; i < n_local; ++i) {
            // the next chunk's loads are in flight while this chunk's noise is generated
            float4 vn[2];
            if (i + 1 < n_local) fetch(c_lo + i + 1, vn);
            add_noise(c_lo + i, v);
            commit(i, v);
            if (i + 1 < n_local) { v[0] = vn[0]; v[1] = vn[1]; }
        }
    } else if (warp == TC_PRODUCERS / 32) {
        // ===== MMA issuer =====
        if (lane == 0) {
            for (int i = 0; i < n_local; ++i) {
                const int s = i % TT_STAGES;
                const uint32_t ph = (uint32_t)(i / TT_STAGES) & 1u;
                tc::mbar_wait(&full_bar[s], ph);
                tc::tc_fence_after_sync();
                issue_stage_mmas(tc::smem_u32(smem + s * TC_STAGE_BYTES), tmem_base, i);
                tc::umma_commit(&empty_bar[s]);   // frees the stage when these MMAs have read it
            }
            tc::umma_commit(accum_bar);           // accumulators complete
        }
        __syncwarp();
    } else {
        // ===== W streamer (TMA engine bulk copies) =====
        if (lane == 0) {
            for (int i = 0; i < n_local; ++i) {
                const int c = c_lo + i;
                const int s = i % TT_STAGES;
                const uint32_t ph = (uint32_t)(i / TT_STAGES) & 1u;
                tc::mbar_wait(&empty_bar[s], ph ^ 1u);
                tc::mbar_arrive_expect_tx(&full_bar[s], 2 * TC_B_BYTES);
                tc::bulk_g2s(smem + s * TC_STAGE_BYTES + 2 * TC_A_BYTES, prm.gWimg + (size_t)c * (2 * TC_B_BYTES / 4),
                             2 * TC_B_BYTES, &full_bar[s]);
            }
        }
        __syncwarp();
    }

    // ===== epilogue: the 16 producer warps; warp w reads TMEM lanes 32*(w%4).. (the only ones it may touch) and
    // columns 16*(w/4)..: one 16-column slice of 32 rows of the partial pre-activations of this K split =====
    if (warp < TC_PRODUCERS / 32) {
        const int lq = warp & 3, cq = warp >> 2;
        const int64_t orow = row_base + lq * 32 + lane;
        const bool valid = orow < prm.n_rows;
        float* out = prm.pre_part + ((size_t)ks * (size_t)prm.n_rows + (size_t)(valid ? orow : 0)) * D + cq * 16;
        float acc[16];
        if (n_local > 0) {
            tc::mbar_wait(accum_bar, 0u);
            tc::tc_fence_after_sync();
            load_acc_quarter(tmem_base, lq, cq, acc);
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[j] = 0.f;
        }
        if (valid) {
#pragma unroll
            for (int j = 0; j < 16; j += 4) st4(out + j, make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]));
        }
    }

    tc::tc_fence_before_sync();
    __syncthreads();
    tl_end(2);
    if (warp == TC_PRODUCERS / 32) tc::tmem_dealloc(tmem_base, TC_TMEM_COLS);
    // Launched as a programmatic dependent of the kernel before it on the stream (dccf_train_fwd_bwd_tc, phases bit 8):
    // this grid started while that kernel was still running and read nothing it writes; it must not COMPLETE before that
    // kernel has, because the next kernel on the stream depends on both.  (A no-op in a plain launch.)
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// One CTA per pair: 8 half-warps take the pair's R rows (lane = 4 columns), then warp 0 runs the backdoor sum.
struct TrainFinishParams {
    dccf_expo ex;
    const float* E_user;
    const float* bias;
    const int64_t* X;
    const int64_t* sample_item;
    const float* mask;           // mode 1
    const float* pre_part;
    float* ws_rows;
    float* save_h;
    float* save_w;
    float* out_pred;
    int32_t* err_flag;
    int64_t n_pairs, n_rows;
    int32_t n_users, user_base, n_items, S, A, R;
    int32_t n_ksplits, mask_mode;
    float keep_prob, drop_scale;
    RngSpec rng;
};

__global__ void __launch_bounds__(128) k_train_fwd_finish(const TrainFinishParams prm) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int hw = tid >> 4, sub = tid & 15;
    const int64_t p = blockIdx.x;
    const int32_t u = checked_id(prm.X[2 * p] - prm.user_base, prm.n_users, prm.err_flag);
    const float4 e = ldg4(prm.E_user + (size_t)u * D + sub * 4);
    const float4 b = ldg4(prm.bias + sub * 4);
    RngKey key_drop = make_rng_key(0, 0, DOMAIN_DROPOUT);
    if (prm.mask_mode == 2) key_drop = resolve_rng_key(prm.rng, DOMAIN_DROPOUT);
    const uint32_t half_mask = (lane & 16) ? 0xffff0000u : 0x0000ffffu;
    const size_t part_stride = (size_t)prm.n_rows * D;

    for (int l = hw; l < prm.R; l += 8) {
        const int64_t r = p * prm.R + l;
        const float* src = prm.pre_part + (size_t)r * D + sub * 4;
        float4 acc = ldg4(src);
        for (int k = 1; k < prm.n_ksplits; ++k) {
            const float4 t = ldg4(src + (size_t)k * part_stride);
            acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
        }
        float4 h = make_float4(fmaxf(acc.x + b.x, 0.f), fmaxf(acc.y + b.y, 0.f), fmaxf(acc.z + b.z, 0.f),
                               fmaxf(acc.w + b.w, 0.f));
        if (prm.mask_mode == 1) {
            const float4 m = ldg4(prm.mask + (size_t)r * D + sub * 4);
            h.x *= m.x; h.y *= m.y; h.z *= m.z; h.w *= m.w;
        } else if (prm.mask_mode == 2) {
            const float4 m = dropout_quad(key_drop, (uint32_t)r, (uint32_t)sub, prm.keep_prob, prm.drop_scale);
            h.x *= m.x; h.y *= m.y; h.z *= m.z; h.w *= m.w;
        }
        if (prm.save_h != nullptr) st4(prm.save_h + (size_t)r * D + sub * 4, h);
        float dot = h.x * e.x;
        dot = fmaf(h.y, e.y, dot);
        dot = fmaf(h.z, e.z, dot);
        dot = fmaf(h.w, e.w, dot);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(half_mask, dot, o);
        if (sub == 0) prm.ws_rows[r] = dot;
    }
    __syncthreads();   // the pair's row scores (global memory, written by this CTA) are visible to warp 0
    if (tid < 32)
        backdoor_pair(prm.ex, prm.X, prm.sample_item, p, lane, prm.n_users, prm.user_base, prm.n_items, prm.S, prm.A,
                      prm.ws_rows + p * prm.R, prm.out_pred + p,
                      prm.save_w != nullptr ? prm.save_w + p * (prm.S + 1) : nullptr, prm.err_flag);
}

// =============================================================================================
// fused middle of the step (BPR / MSE loss): per-pair forward epilogue, backdoor sum, loss term, d loss / d pred,
// dpre rows and the embedding-gradient records in ONE kernel.  A CTA owns one loss term: with BPR the positive
// pair j and its negative j + b (src/models/DCCF.py:116-120), so d loss / d pred needs no second pass over
// global memory and the activations h never leave shared memory.
// =============================================================================================
constexpr int TM_NT = 768;   // 48 half-warps: every phase below is a single pass at the reference shapes (2 x 22 rows)

struct TrainMidParams {
    dccf_expo ex;
    const float* E_user;
    const float* W;
    const float* bias;
    const int64_t* X;
    const int64_t* sample_item;
    const float* Y;
    const float* mask;           // mode 1
    const float* pre_part;
    const float* expo_e;         // optional [P, Z] + expo_den [P]: the exposure softmax of every pair, precomputed from
    const float* expo_den;       // the ids on another stream (dccf_adam_link_ids); null: evaluated here
    const uint64_t* batch_ptrs;  // optional (with batch_cursor): the user ids read before griddepcontrol.wait come from
    const int64_t* batch_cursor; //   batch *batch_cursor of the device-resident epoch, as in k_train_fwd_tc
    float* out_pred;
    float* loss_terms;
    float* dpre_rows;
    float* gu_rec;
    float* gi_rec;
    int32_t* rec_keys_u;
    int32_t* rec_keys_i;
    float* save_h;               // optional
    float* save_w;               // optional
    int32_t* err_flag;
    int64_t n_pairs, n_rows;
    int64_t mse_pairs;           // MSE: the pairs the mean is over (world * n_pairs in a data-parallel step)
    int32_t n_users, user_base, n_items, S, A, R, Z, K;
    int32_t n_ksplits, mask_mode, loss_mode;
    float keep_prob, drop_scale, inv_A;
    RngSpec rng;
};

__host__ __device__ inline size_t train_mid_smem_floats(int R, int Z, int npc) {
    return (size_t)D * D + (size_t)npc * R * D + (size_t)npc * Z * D + (size_t)npc * R + (size_t)npc * Z + 8;
}

// (no launch bound: the default 1024-thread bound caps the kernel at 64 registers, so that a 256-thread CTA of the
// side-stream Adam sweep still fits beside its 768 threads)
// 64 registers x 768 threads = 3/4 of the SM's register file: the side sweep's CTA (7 warps x 64 registers) stays resident
// beside this kernel.  (At 70 registers a sweep CTA wider than 128 threads kept every CTA of this kernel off its SM
// until the sweep had finished.)
__global__ void __maxnreg__(64) k_train_mid(const TrainMidParams prm) {
    extern __shared__ __align__(16) float sm[];
    const int R = prm.R, Z = prm.Z, A = prm.A;
    const int npc = (prm.loss_mode == 0) ? 2 : 1;   // pairs per CTA
    float* Wi_s = sm;                               // [D][D]   Wi_s[j*D + k] = W[j][k], k < D
    float* h_s = Wi_s + D * D;                      // [npc*R][D] post-dropout activations
    float* dsum_s = h_s + (size_t)npc * R * D;      // [npc*Z][D] sum_a dpre
    float* score_s = dsum_s + (size_t)npc * Z * D;  // [npc*R]
    float* w_s = score_s + npc * R;                 // [npc*Z]  softmax exposure weights
    float* pred_s = w_s + npc * Z;                  // [2]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    tl_begin(3);
    const int hw = tid >> 4, sub = tid & 15;
    const int64_t jt = blockIdx.x;
    const int64_t b = prm.n_pairs >> 1;
    const int64_t p_second = (prm.loss_mode == 0) ? jt + b : jt;
    auto pair_of = [&](int q) { return q == 0 ? jt : p_second; };
    const uint32_t half_mask = (lane & 16) ? 0xffff0000u : 0x0000ffffu;

    // Launched as a programmatic dependent of the partial-product kernel (phases bit 16), this CTA may start while that
    // kernel runs (only on an SM without one of its CTAs: 768 x 64 registers do not fit beside its 576 x 56).  Until
    // griddepcontrol.wait it reads only state that existed before the step: W, b, E_user (the user rows are touched
    // rows, which only k_adam_touched writes, after the step's dW kernel), the RNG key and, through the batch cursor,
    // the ids of a device-resident epoch.  The staged X, expo_e / expo_den and pre_part are read after the wait, which
    // returns when the partial-product kernel has completed — and that kernel does not complete before k_adam_link_ids,
    // which writes them, has (its own wait).  Both instructions are no-ops in a plain launch.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // W_i: loaded now, parked in registers, stored to shared memory after the first phase (only the last one reads it)
    float4 wreg[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
        const int i = tid + t * TM_NT;
        if (i < D * D / 4) wreg[t] = ldg4(prm.W + (size_t)(i / (D / 4)) * prm.K + (i % (D / 4)) * 4);
    }
    const float4 bia = ldg4(prm.bias + sub * 4);
    RngKey key_drop = make_rng_key(0, 0, DOMAIN_DROPOUT);
    if (prm.mask_mode == 2) key_drop = resolve_rng_key(prm.rng, DOMAIN_DROPOUT);
    const size_t part_stride = (size_t)prm.n_rows * D;
    // the user rows of the CTA's (at most two) pairs, columns 4*sub .. 4*sub+3
    const int64_t* Xu = prm.X;
    if (prm.batch_cursor != nullptr) Xu = reinterpret_cast<const int64_t*>(prm.batch_ptrs[0]) + *prm.batch_cursor * prm.n_pairs * 2;
    else asm volatile("griddepcontrol.wait;" ::: "memory");
    const int32_t u0 = checked_id(Xu[2 * jt] - prm.user_base, prm.n_users, prm.err_flag);
    const int32_t u1 = checked_id(Xu[2 * p_second] - prm.user_base, prm.n_users, prm.err_flag);
    const float4 eu0 = ldg4(prm.E_user + (size_t)u0 * D + sub * 4);
    const float4 eu1 = ldg4(prm.E_user + (size_t)u1 * D + sub * 4);
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // ---- A: rows of the CTA's pairs: partial sums + bias, ReLU, dropout, dot with the user row -------------
    for (int rr = hw; rr < npc * R; rr += TM_NT / 16) {
        const int q = rr / R, l = rr - q * R;
        const int64_t p = pair_of(q);
        const int64_t r = p * R + l;
        const float4 e = q == 0 ? eu0 : eu1;
        const float* src = prm.pre_part + (size_t)r * D + sub * 4;
        // the K-split partials (at most 8, fwd_ksplits_for) in two groups of four loads in flight, added in ascending
        // order (a rolled loop waited for them one L2 round trip after the other; all eight at once spill at 64 registers)
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k0 = 0; k0 < 8; k0 += 4) {
            float4 part[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k0 + k < prm.n_ksplits) part[k] = ldg4(src + (size_t)(k0 + k) * part_stride);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k0 + k == 0) acc = part[0];
                else if (k0 + k < prm.n_ksplits) { acc.x += part[k].x; acc.y += part[k].y; acc.z += part[k].z; acc.w += part[k].w; }
            }
        }
        float4 h = make_float4(fmaxf(acc.x + bia.x, 0.f), fmaxf(acc.y + bia.y, 0.f), fmaxf(acc.z + bia.z, 0.f),
                               fmaxf(acc.w + bia.w, 0.f));
        if (prm.mask_mode == 1) {
            const float4 m = ldg4(prm.mask + (size_t)r * D + sub * 4);
            h.x *= m.x; h.y *= m.y; h.z *= m.z; h.w *= m.w;
        } else if (prm.mask_mode == 2) {
            const float4 m = dropout_quad(key_drop, (uint32_t)r, (uint32_t)sub, prm.keep_prob, prm.drop_scale);
            h.x *= m.x; h.y *= m.y; h.z *= m.z; h.w *= m.w;
        }
        if (prm.save_h != nullptr) st4(prm.save_h + (size_t)r * D + sub * 4, h);
        st4(h_s + (size_t)rr * D + sub * 4, h);
        float dot = h.x * e.x;
        dot = fmaf(h.y, e.y, dot);
        dot = fmaf(h.z, e.z, dot);
        dot = fmaf(h.w, e.w, dot);
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(half_mask, dot, o);
        if (sub == 0) score_s[rr] = dot;
    }
#pragma unroll
    for (int t = 0; t < 2; ++t) {
        const int i = tid + t * TM_NT;
        if (i < D * D / 4) st4(&Wi_s[(i / (D / 4)) * D + (i % (D / 4)) * 4], wreg[t]);
    }
    __syncthreads();

    // ---- B: backdoor-adjusted sum of each pair (one warp per pair) ------------------------------------------
    if (warp < npc) {
        const int64_t p = pair_of(warp);
        if (prm.expo_e != nullptr) {
            backdoor_apply(prm.expo_e + p * Z, __ldg(prm.expo_den + p), lane, prm.S, A, score_s + warp * R, pred_s + warp,
                           w_s + warp * Z);
        } else {
            backdoor_pair(prm.ex, prm.X, prm.sample_item, p, lane, prm.n_users, prm.user_base, prm.n_items, prm.S, A,
                          score_s + warp * R, pred_s + warp, w_s + warp * Z, prm.err_flag);
        }
        __syncwarp();
        if (lane == 0) prm.out_pred[p] = pred_s[warp];
        if (prm.save_w != nullptr)
            for (int z = lane; z < Z; z += 32) prm.save_w[p * Z + z] = w_s[warp * Z + z];
    }
    __syncthreads();

    // loss term and d loss / d pred of the CTA's pairs (every thread evaluates the two scalars it needs itself)
    float dp0, dp1 = 0.f;
    if (prm.loss_mode == 0) {
        const float d = pred_s[0] - pred_s[1];
        const float sg = 1.f / (1.f + expf(-d));
        const float g = -(1.f - sg);
        dp0 = g;
        dp1 = -g;
        // -log(sigmoid(d)) = softplus(-d), evaluated the stable way
        if (tid == 0) prm.loss_terms[jt] = (d > 0.f) ? log1pf(expf(-d)) : (-d + log1pf(expf(d)));
    } else {
        const float d = pred_s[0] - __ldg(prm.Y + jt);
        dp0 = 2.f * d / (float)prm.mse_pairs;
        if (tid == 0) prm.loss_terms[jt] = d * d;
    }

    // ---- C1: dpre rows (to global memory for the dW kernel) and their sum over the attribute copies ---------
    for (int qz = hw; qz < npc * Z; qz += TM_NT / 16) {
        const int q = qz / Z, z = qz - q * Z;
        const int64_t p = pair_of(q);
        const float4 e = q == 0 ? eu0 : eu1;
        const float ds = (q == 0 ? dp0 : dp1) * w_s[qz] * prm.inv_A;
        float4 dsum = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int a = 0; a < A; ++a) {
            const int l = z * A + a;
            const int64_t r = p * R + l;
            const float4 h = ld4(h_s + (size_t)(q * R + l) * D + sub * 4);
            float4 g;
            if (prm.mask_mode == 1) {
                const float4 m = ldg4(prm.mask + (size_t)r * D + sub * 4);
                g = make_float4(h.x > 0.f ? m.x : 0.f, h.y > 0.f ? m.y : 0.f, h.z > 0.f ? m.z : 0.f, h.w > 0.f ? m.w : 0.f);
            } else {
                const float sc = (prm.mask_mode == 2) ? prm.drop_scale : 1.f;
                g = make_float4(h.x > 0.f ? sc : 0.f, h.y > 0.f ? sc : 0.f, h.z > 0.f ? sc : 0.f, h.w > 0.f ? sc : 0.f);
            }
            const float4 dv = make_float4(ds * e.x * g.x, ds * e.y * g.y, ds * e.z * g.z, ds * e.w * g.w);
            st4(prm.dpre_rows + (size_t)r * D + sub * 4, dv);
            dsum.x += dv.x; dsum.y += dv.y; dsum.z += dv.z; dsum.w += dv.w;
        }
        st4(dsum_s + (size_t)qz * D + sub * 4, dsum);
    }
    // user-row record: gu[c] = sum_{z,a} ds * h[.,c], rows in ascending order (thread = column; the warps at the
    // top of the CTA, which have no C1 work at the reference shapes)
    if (tid >= TM_NT - npc * D) {
        const int t2 = tid - (TM_NT - npc * D);
        const int q = t2 >> 6, c = t2 & (D - 1);
        const int64_t p = pair_of(q);
        const float dpq = q == 0 ? dp0 : dp1;
        float gu = 0.f;
        for (int l = 0; l < R; ++l) {
            const float ds = dpq * w_s[q * Z + l / A] * prm.inv_A;
            gu = fmaf(ds, h_s[(size_t)(q * R + l) * D + c], gu);
        }
        prm.gu_rec[(size_t)p * D + c] = gu;
        if (c == 0) prm.rec_keys_u[p] = q == 0 ? u0 : u1;
    }
    __syncthreads();

    // ---- C2: item-row records gi[k] = sum_j W[j][k] * dsum[j]  (thread = column k, ascending j; four records
    // per thread at a time so that four independent FMA chains share each W value) ------------------------------
    {
        const int k = tid & (D - 1);
        const int n_qz = npc * Z;
        for (int base = (tid >> 6) * 4; base < n_qz; base += (TM_NT / D) * 4) {
            const float* d0 = dsum_s + (size_t)min(base + 0, n_qz - 1) * D;
            const float* d1 = dsum_s + (size_t)min(base + 1, n_qz - 1) * D;
            const float* d2 = dsum_s + (size_t)min(base + 2, n_qz - 1) * D;
            const float* d3 = dsum_s + (size_t)min(base + 3, n_qz - 1) * D;
            float g0 = 0.f, g1 = 0.f, g2 = 0.f, g3 = 0.f;
#pragma unroll 8
            for (int j = 0; j < D; ++j) {
                const float w = Wi_s[j * D + k];
                g0 = fmaf(w, d0[j], g0);
                g1 = fmaf(w, d1[j], g1);
                g2 = fmaf(w, d2[j], g2);
                g3 = fmaf(w, d3[j], g3);
            }
            const float gv[4] = {g0, g1, g2, g3};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int qz = base + i;
                if (qz < n_qz) {
                    const int q = qz / Z, z = qz - q * Z;
                    const int64_t rec = pair_of(q) * Z + z;
                    prm.gi_rec[(size_t)rec * D + k] = gv[i];
                    if (k == 0)
                        prm.rec_keys_i[rec] = checked_id(slot_item(prm.X, prm.sample_item, pair_of(q), z, prm.S), prm.n_items, nullptr);
                }
            }
        }
    }
    __syncthreads();
    tl_end(3);
}

// =============================================================================================
// backward: gW / gb partial tiles
// =============================================================================================
// 16 producer warps + the MMA warp + 2 idle warps that only take part in the CTA-wide barriers.  They fix the kernel's
// occupancy at ONE CTA per SM: at 56 registers (the __maxnreg__ below) a CTA takes 608 x 56 = 34 048 registers, more than
// half of the SM's 65 536, so two do not fit — as a programmatic dependent of the middle kernel (phases bit 32) the CTAs
// placed early would otherwise double up on the few free SMs and unbalance the grid.  One CTA still fits beside a CTA of
// the side-stream sweep (224 x 64 = 14 336 registers, 120 KB of shared memory + this kernel's 96 KB), and none beside a
// middle-kernel CTA (768 x 64 = 49 152 registers).  tests/test_occupancy.py checks these facts on the built library.
constexpr int TB_NT = TC_PRODUCERS + 32 + 64;

struct TrainBwdParams {
    const float* E_item;
    const float* Feat;
    const int64_t* X;
    const int64_t* sample_item;
    const uint64_t* batch_ptrs;  // optional (with batch_cursor): the ids come from batch *batch_cursor of the
    const int64_t* batch_cursor; //   device-resident epoch, as in k_train_fwd_tc (so they can be read before the wait)
    const float* noise;          // mode 1
    const float* dpre_rows;      // [N, D]
    float* gW_part;              // [n_splits][D][K]
    float* gb_part;              // [n_splits][D]
    const float* loss_terms;     // optional [n_loss_terms]: summed into out_loss by CTA (0,0) (fused step)
    float* out_loss;
    int64_t n_loss_terms;
    float loss_scale;
    int64_t n_rows;
    int32_t n_items, F, S, A, R, K;
    int32_t rows_per_split;      // multiple of 32
    float noise_std;
    RngSpec rng;
};

// 4x4 transpose across the four lanes of a quad: in: lane j holds a[0..3] = M[j][0..3]; out: lane j holds M[0..3][j]
__device__ __forceinline__ void quad_transpose(float4& a, int j) {
    const bool odd = (j & 1) != 0, up = (j & 2) != 0;
    float s0 = odd ? a.x : a.y, s1 = odd ? a.z : a.w;
    s0 = __shfl_xor_sync(0xffffffffu, s0, 1);
    s1 = __shfl_xor_sync(0xffffffffu, s1, 1);
    if (odd) { a.x = s0; a.z = s1; } else { a.y = s0; a.w = s1; }
    float t0 = up ? a.x : a.z, t1 = up ? a.y : a.w;
    t0 = __shfl_xor_sync(0xffffffffu, t0, 2);
    t1 = __shfl_xor_sync(0xffffffffu, t1, 2);
    if (up) { a.x = t0; a.y = t1; } else { a.z = t0; a.w = t1; }
}

template <int NOISE_MODE>
__global__ void __maxnreg__(56) k_train_bwd_tc(const TrainBwdParams prm) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + TT_STAGES * TC_STAGE_BYTES);
    uint64_t* empty_bar = full_bar + TT_STAGES;
    uint64_t* accum_bar = empty_bar + TT_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    tl_begin(4);
    const int mt = (int)blockIdx.x, sp = (int)blockIdx.y;
    const int64_t row_lo = (int64_t)sp * prm.rows_per_split;
    const int64_t row_hi = min(row_lo + prm.rows_per_split, prm.n_rows);
    const int n_st = row_hi > row_lo ? (int)((row_hi - row_lo + TC_KC - 1) / TC_KC) : 0;

    if (tid == 0) {
        for (int s = 0; s < TT_STAGES; ++s) {
            tc::mbar_init(&full_bar[s], TC_PRODUCERS / 32);
            tc::mbar_init(&empty_bar[s], 1);
        }
        tc::mbar_init(accum_bar, 1);
        tc::fence_barrier_init();
    }
    if (warp == TC_PRODUCERS / 32) tc::tmem_alloc(tmem_slot, TC_TMEM_COLS);
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < TC_PRODUCERS / 32) {
        // ===== producers =====
        // x tile (the A operand, M = column of [x | 1], K = row): a quad of lanes owns 4 rows x 4 columns
        const int j = lane & 3, g = lane >> 2;
        const int rq = warp & 7;            // which 4 of the stage's 32 rows
        const int cb0 = warp >> 3;          // 32-column blocks cb0 and cb0 + 2 of the 128-column tile
        // dpre tile (the B operand, N = output channel, K = row): thread owns channel bc, rows 4*brq .. 4*brq+3
        const int bc = tid & 63, brq = tid >> 6;
        RngKey key_noise = make_rng_key(0, 0, DOMAIN_NOISE);
        if (NOISE_MODE == 2) key_noise = resolve_rng_key(prm.rng, DOMAIN_NOISE);
        const int64_t *X = prm.X, *si = prm.sample_item;
        if (prm.batch_cursor != nullptr) {
            const int64_t b = *prm.batch_cursor, n_pairs = (int64_t)((uint32_t)prm.n_rows / (uint32_t)prm.R);
            X = reinterpret_cast<const int64_t*>(prm.batch_ptrs[0]) + b * n_pairs * 2;
            si = reinterpret_cast<const int64_t*>(prm.batch_ptrs[1]) + b * n_pairs * prm.S;
        }

        // the B operand of stage st: dpre values, thread = channel bc, rows 4*brq .. 4*brq+3
        auto fetch_dpre = [&](int st, float4& dv) {
            const int64_t r0 = row_lo + (int64_t)st * TC_KC + brq * 4;
            const float* src = prm.dpre_rows + (size_t)r0 * D + bc;
            dv.x = (r0 + 0 < row_hi) ? __ldg(src) : 0.f;
            dv.y = (r0 + 1 < row_hi) ? __ldg(src + D) : 0.f;
            dv.z = (r0 + 2 < row_hi) ? __ldg(src + 2 * D) : 0.f;
            dv.w = (r0 + 3 < row_hi) ? __ldg(src + 3 * D) : 0.f;
        };
        // the A operand of stage st: this lane's 4 columns of x for its row (before the transpose)
        auto fetch_x = [&](int st, float4 (&v)[2]) {
            const int64_t r = row_lo + (int64_t)st * TC_KC + rq * 4 + j;
            const bool live = r < row_hi;
            int32_t fi = 0, it = 0;
            if (live) {
                const uint32_t p = (uint32_t)r / (uint32_t)prm.R;
                fi = checked_id(X[2 * (int64_t)p + 1], prm.n_items, nullptr);
                if (mt == 0) {
                    const int z = (int)((uint32_t)r - p * (uint32_t)prm.R) / prm.A;
                    it = (z == 0) ? fi : checked_id(si[(int64_t)p * prm.S + (z - 1)], prm.n_items, nullptr);
                }
            }
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int col = mt * TC_BM + (cb0 + 2 * t) * 32 + g * 4;   // first of this lane's 4 columns of [x | 1]
                v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (live) {
                    if (col < D) {
                        v[t] = ldg4(prm.E_item + (size_t)it * D + col);
                    } else if (col < prm.K) {
                        const int f = col - D;
                        v[t] = ldg4(prm.Feat + (size_t)fi * prm.F + f);
                        if (NOISE_MODE != 0) {
                            float4 e;
                            if (NOISE_MODE == 1) e = ldg4(prm.noise + (size_t)r * prm.F + f);
                            else e = noise_quad(key_noise, (uint32_t)r, (uint32_t)(f / 4), prm.noise_std);
                            v[t].x = __fadd_rn(v[t].x, e.x); v[t].y = __fadd_rn(v[t].y, e.y);
                            v[t].z = __fadd_rn(v[t].z, e.z); v[t].w = __fadd_rn(v[t].w, e.w);
                        }
                    } else if (col == prm.K) {
                        v[t].x = 1.f;                 // the column of ones: its output row is the bias gradient
                    }
                }
            }
        };

        // stage st of this CTA, A operand: transpose, wait until the MMAs that read its slot have completed, store
        auto store_x = [&](int st, float4 (&v)[2]) {
            const int s = st % TT_STAGES;
            const uint32_t ph = (uint32_t)(st / TT_STAGES) & 1u;
            quad_transpose(v[0], j);
            quad_transpose(v[1], j);
            tc::mbar_wait(&empty_bar[s], ph ^ 1u);
            uint8_t* a_hi = smem + s * TC_STAGE_BYTES;
            uint8_t* a_lo = a_hi + TC_A_BYTES;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int m = (cb0 + 2 * t) * 32 + g * 4 + j;      // after the transpose this lane holds column m,
                store_hi_lo(a_hi, a_lo, core_offset(m, rq * 4), v[t]);   // rows 4*rq .. 4*rq+3 of the stage
            }
        };
        // ... B operand (after its A operand): store, publish the stage
        auto store_dpre = [&](int st, const float4& dv) {
            const int s = st % TT_STAGES;
            uint8_t* b_hi = smem + s * TC_STAGE_BYTES + 2 * TC_A_BYTES;
            uint8_t* b_lo = b_hi + TC_B_BYTES;
            store_hi_lo(b_hi, b_lo, core_offset(bc, brq * 4), dv);
            tc::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&full_bar[s]);
        };
        // Launched as a programmatic dependent of the middle kernel (phases bit 32), this CTA may start while that kernel
        // runs.  Only dpre and the loss terms come from it: with the ids of a device-resident epoch (batch cursor) the A
        // operands of the first TT_STAGES stages (free ring slots) are built before griddepcontrol.wait, from tables the
        // step has not written yet.  The wait returns when the middle kernel has completed, which it does only after the
        // partial-product kernel has (its own wait).  A no-op in a plain launch.
        const int n_pre = (prm.batch_cursor != nullptr) ? min(n_st, TT_STAGES) : 0;
        {
            float4 xp[TT_STAGES][2];
#pragma unroll
            for (int st = 0; st < TT_STAGES; ++st)
                if (st < n_pre) fetch_x(st, xp[st]);
#pragma unroll
            for (int st = 0; st < TT_STAGES; ++st)
                if (st < n_pre) store_x(st, xp[st]);
        }
        asm volatile("griddepcontrol.wait;" ::: "memory");
        float4 v[2], dv;
        {
            float4 dp[TT_STAGES];
#pragma unroll
            for (int st = 0; st < TT_STAGES; ++st)
                if (st < n_pre) fetch_dpre(st, dp[st]);
            if (n_pre < n_st) { fetch_x(n_pre, v); fetch_dpre(n_pre, dv); }
#pragma unroll
            for (int st = 0; st < TT_STAGES; ++st)
                if (st < n_pre) store_dpre(st, dp[st]);
        }
        for (int st = n_pre; st < n_st; ++st) {
            // the next stage's operands are in flight while this one is transposed, stored and multiplied
            float4 vn[2], dvn;
            if (st + 1 < n_st) { fetch_x(st + 1, vn); fetch_dpre(st + 1, dvn); }
            store_x(st, v);
            store_dpre(st, dv);
            if (st + 1 < n_st) {
                v[0] = vn[0]; v[1] = vn[1]; dv = dvn;
            }
        }
        // the scalar loss of the fused step: per-term values summed in a fixed order (lane-strided, then a shuffle
        // tree) by one warp that is idle during the epilogue
        if (warp == 4 && mt == 0 && sp == 0 && prm.loss_terms != nullptr) {
            float acc = 0.f;
            for (int64_t i = lane; i < prm.n_loss_terms; i += 32) acc += __ldg(prm.loss_terms + i);
            acc = warp_sum(acc);
            if (lane == 0) prm.out_loss[0] = acc * prm.loss_scale;
        }
    } else if (warp == TC_PRODUCERS / 32) {
        // ===== MMA issuer =====
        if (lane == 0) {
            for (int st = 0; st < n_st; ++st) {
                const int s = st % TT_STAGES;
                const uint32_t ph = (uint32_t)(st / TT_STAGES) & 1u;
                tc::mbar_wait(&full_bar[s], ph);
                tc::tc_fence_after_sync();
                issue_stage_mmas(tc::smem_u32(smem + s * TC_STAGE_BYTES), tmem_base, st);
                tc::umma_commit(&empty_bar[s]);
            }
            tc::umma_commit(accum_bar);
        }
        __syncwarp();
    }

    // ===== epilogue: the 16 producer warps; warp w owns TMEM lanes 32*(w%4).. = 32 consecutive columns m of the
    // tile and the output channels 16*(w/4)..; lanes of a warp are consecutive columns of gW, so every store below
    // is one coalesced 128-byte line =====
    if (warp < TC_PRODUCERS / 32) {
        const int lq = warp & 3, cq = warp >> 2;
        const int col = mt * TC_BM + lq * 32 + lane;
        float acc[16];
        if (n_st > 0) {
            tc::mbar_wait(accum_bar, 0u);
            tc::tc_fence_after_sync();
            load_acc_quarter(tmem_base, lq, cq, acc);
        } else {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) acc[jj] = 0.f;
        }
        float* gw = prm.gW_part + (size_t)sp * D * prm.K;
        float* gb = prm.gb_part + (size_t)sp * D;
        if (col < prm.K) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) gw[(size_t)(cq * 16 + jj) * prm.K + col] = acc[jj];
        } else if (col == prm.K) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) gb[cq * 16 + jj] = acc[jj];
        }
    }

    tc::tc_fence_before_sync();
    __syncthreads();
    tl_end(4);
    if (warp == TC_PRODUCERS / 32) tc::tmem_dealloc(tmem_base, TC_TMEM_COLS);
}

// defined in bpr_bwd.cu
int bpr_bwd_launch(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat, const float* W,
                   const int64_t* X, const int64_t* sample_item, const float* Y, int64_t n_pairs, const dccf_rng* rng,
                   int32_t loss_mode, const float* pred, const float* save_h, const float* save_w, float* out_loss,
                   float* gW_part, float* gb_part, float* gu_rec, float* gi_rec, int32_t* rec_keys_u, int32_t* rec_keys_i,
                   float* dpre_rows, bool with_gw, cudaStream_t stream);

static int32_t fwd_ksplits_for(int64_t n_rows, int n_chunks) {
    if (n_rows <= 0) return 1;
    const int64_t tiles = (n_rows + TC_BM - 1) / TC_BM;
    int64_t ks = 148 / tiles;                      // about one CTA per SM
    if (ks > 8) ks = 8;
    if (ks > n_chunks) ks = n_chunks;
    if (ks < 1) ks = 1;
    return (int32_t)ks;
}

static void bwd_geometry(int64_t n_rows, int K, int32_t* n_mtiles, int32_t* n_splits, int32_t* rows_per_split) {
    const int mt = (K + 1 + TC_BM - 1) / TC_BM;    // columns of [x | 1]
    int64_t want = 148 / mt;
    if (want < 1) want = 1;
    int64_t rps = (n_rows + want - 1) / want;
    rps = ((rps + TC_KC - 1) / TC_KC) * TC_KC;
    if (rps < TC_KC) rps = TC_KC;
    *n_mtiles = mt;
    *rows_per_split = (int32_t)rps;
    *n_splits = (int32_t)((n_rows + rps - 1) / rps);
    if (*n_splits < 1) *n_splits = 1;
}

template <typename Kern>
static int opt_in_smem(Kern k, const char* name) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TT_SMEM_BYTES);
    // always the largest shared-memory carveout: a CTA of the side-stream Adam sweep (120 KB) and a tensor-core CTA
    // (96 KB) share an SM only if neither launch shrinks the carveout under the other
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) {
        set_error("%s: cannot opt in to %u bytes of shared memory: %s", name, TT_SMEM_BYTES, cudaGetErrorString(e));
        return DCCF_ERR_CUDA;
    }
    return DCCF_OK;
}

}  // namespace dccf

using namespace dccf;

extern "C" int64_t dccf_train_w_image_floats(int32_t feat_dim) {
    return (int64_t)((D + feat_dim) / TC_KC) * (2 * TC_B_BYTES / 4);
}

extern "C" int dccf_debug_timeline_train(unsigned long long* slots) {
    cudaError_t e = cudaMemcpyToSymbol(g_timeline, &slots, sizeof(slots));
    if (e != cudaSuccess) {
        set_error("dccf_debug_timeline: %s", cudaGetErrorString(e));
        return DCCF_ERR_CUDA;
    }
    return DCCF_OK;
}

extern "C" int dccf_train_prep_w_image(const float* W, int32_t feat_dim, float* w_image, void* stream_) {
    DCCF_CHECK_ARG(W && w_image && feat_dim > 0 && feat_dim % 64 == 0, "dccf_train_prep_w_image: bad argument");
    k_prep_w_image<<<104, 256, 0, (cudaStream_t)stream_>>>(W, D + feat_dim, w_image);
    DCCF_CHECK_LAUNCH("k_prep_w_image");
    return DCCF_OK;
}

extern "C" int32_t dccf_train_fwd_ksplits(int64_t n_rows, int32_t feat_dim) {
    return fwd_ksplits_for(n_rows, (D + feat_dim) / TC_KC);
}

extern "C" int32_t dccf_train_bwd_splits(int64_t n_rows, int32_t feat_dim) {
    int32_t mt, ns, rps;
    bwd_geometry(n_rows, D + feat_dim, &mt, &ns, &rps);
    return ns;
}

// W images + partial products of every (row tile, K split)
static int launch_fwd_tc(const dccf_dims* dims, const float* E_item, const float* Feat, const float* W, const int64_t* X,
                         const int64_t* sample_item, int64_t n_pairs, const dccf_rng* rng, float* ws_wimg,
                         bool w_image_valid, float* ws_pre_part, int32_t* err_flag, int32_t* n_ks_out,
                         cudaStream_t stream, const dccf_batch_ref* batch = nullptr, bool programmatic = false) {
    const int F = dims->feat_dim, K = D + F, Z = dims->n_samples + 1, R = Z * dims->n_attr;
    const int64_t n_rows = n_pairs * R;
    static PerDeviceOnce attr_once;
    if (attr_once.need()) {
        int rc = opt_in_smem(k_train_fwd_tc<0>, "dccf_train_fwd_tc");
        if (rc == DCCF_OK) rc = opt_in_smem(k_train_fwd_tc<1>, "dccf_train_fwd_tc");
        if (rc == DCCF_OK) rc = opt_in_smem(k_train_fwd_tc<2>, "dccf_train_fwd_tc");
        if (rc != DCCF_OK) return rc;
        attr_once.mark();
    }
    if (!w_image_valid) {
        k_prep_w_image<<<104, 256, 0, stream>>>(W, K, ws_wimg);
        DCCF_CHECK_LAUNCH("k_prep_w_image");
    }
    TrainFwdParams prm;
    prm.E_item = E_item; prm.Feat = Feat; prm.gWimg = ws_wimg; prm.X = X; prm.sample_item = sample_item;
    prm.batch_ptrs = batch ? batch->epoch_ptrs_dev : nullptr; prm.batch_cursor = batch ? batch->cursor_dev : nullptr;
    prm.noise = rng->noise; prm.pre_part = ws_pre_part; prm.err_flag = err_flag; prm.n_rows = n_rows;
    prm.n_items = dims->n_items; prm.F = F; prm.S = dims->n_samples; prm.A = dims->n_attr; prm.R = R;
    prm.n_chunks = K / TC_KC; prm.noise_std = rng->noise_std;
    prm.rng.seed = rng->seed; prm.rng.offset = rng->offset; prm.rng.offset_dev = rng->offset_dev;
    const int32_t n_ks = fwd_ksplits_for(n_rows, prm.n_chunks);
    *n_ks_out = n_ks;
    const dim3 grid((unsigned)((n_rows + TC_BM - 1) / TC_BM), (unsigned)n_ks);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(TC_NT); cfg.dynamicSmemBytes = TT_SMEM_BYTES; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = (programmatic && w_image_valid) ? 1 : 0;     // (never over k_prep_w_image: its output is read)
    cudaError_t le;
    switch (rng->noise_mode) {
        case 0: le = cudaLaunchKernelEx(&cfg, k_train_fwd_tc<0>, prm); break;
        case 1: le = cudaLaunchKernelEx(&cfg, k_train_fwd_tc<1>, prm); break;
        default: le = cudaLaunchKernelEx(&cfg, k_train_fwd_tc<2>, prm); break;
    }
    if (le != cudaSuccess) {
        set_error("k_train_fwd_tc: launch failed: %s", cudaGetErrorString(le));
        return DCCF_ERR_CUDA;
    }
    DCCF_CHECK_LAUNCH("k_train_fwd_tc");
    return DCCF_OK;
}

// gW / gb partial tiles from the dpre rows (+ the scalar loss of the fused step)
static int launch_bwd_tc(const dccf_dims* dims, const float* E_item, const float* Feat, const int64_t* X,
                         const int64_t* sample_item, int64_t n_pairs, const dccf_rng* rng, const float* ws_dpre,
                         float* gW_part, float* gb_part, const float* loss_terms, int64_t n_loss_terms,
                         float loss_scale, float* out_loss, cudaStream_t stream, const dccf_batch_ref* batch = nullptr,
                         bool programmatic = false) {
    static PerDeviceOnce attr_once;
    if (attr_once.need()) {
        int rc = opt_in_smem(k_train_bwd_tc<0>, "dccf_train_bwd_tc");
        if (rc == DCCF_OK) rc = opt_in_smem(k_train_bwd_tc<1>, "dccf_train_bwd_tc");
        if (rc == DCCF_OK) rc = opt_in_smem(k_train_bwd_tc<2>, "dccf_train_bwd_tc");
        if (rc != DCCF_OK) return rc;
        attr_once.mark();
    }
    const int F = dims->feat_dim, K = D + F, Z = dims->n_samples + 1, R = Z * dims->n_attr;
    TrainBwdParams prm;
    prm.E_item = E_item; prm.Feat = Feat; prm.X = X; prm.sample_item = sample_item; prm.noise = rng->noise;
    prm.batch_ptrs = batch ? batch->epoch_ptrs_dev : nullptr; prm.batch_cursor = batch ? batch->cursor_dev : nullptr;
    prm.dpre_rows = ws_dpre; prm.gW_part = gW_part; prm.gb_part = gb_part; prm.n_rows = n_pairs * R;
    prm.loss_terms = loss_terms; prm.out_loss = out_loss; prm.n_loss_terms = n_loss_terms; prm.loss_scale = loss_scale;
    prm.n_items = dims->n_items; prm.F = F; prm.S = dims->n_samples; prm.A = dims->n_attr; prm.R = R; prm.K = K;
    prm.noise_std = rng->noise_std;
    prm.rng.seed = rng->seed; prm.rng.offset = rng->offset; prm.rng.offset_dev = rng->offset_dev;
    int32_t n_mtiles, n_splits;
    bwd_geometry(prm.n_rows, K, &n_mtiles, &n_splits, &prm.rows_per_split);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)n_mtiles, (unsigned)n_splits); cfg.blockDim = dim3(TB_NT);
    cfg.dynamicSmemBytes = TT_SMEM_BYTES; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = programmatic ? 1 : 0;
    cudaError_t le;
    switch (rng->noise_mode) {
        case 0: le = cudaLaunchKernelEx(&cfg, k_train_bwd_tc<0>, prm); break;
        case 1: le = cudaLaunchKernelEx(&cfg, k_train_bwd_tc<1>, prm); break;
        default: le = cudaLaunchKernelEx(&cfg, k_train_bwd_tc<2>, prm); break;
    }
    if (le != cudaSuccess) {
        set_error("k_train_bwd_tc: launch failed: %s", cudaGetErrorString(le));
        return DCCF_ERR_CUDA;
    }
    DCCF_CHECK_LAUNCH("k_train_bwd_tc");
    return DCCF_OK;
}

static int check_fwd_args(const char* who, const dccf_dims* dims, const dccf_expo* expo, const dccf_rng* rng,
                          const int64_t* sample_item, int64_t n_pairs) {
    DCCF_CHECK_ARG(dims && expo && rng, "%s: null struct argument", who);
    DCCF_CHECK_ARG(dims->dim == D, "%s: dim=%d but this build has D=%d", who, dims->dim, D);
    DCCF_CHECK_ARG(dims->feat_dim > 0 && dims->feat_dim % 64 == 0, "%s: feat_dim=%d must be a positive multiple of 64", who, dims->feat_dim);
    DCCF_CHECK_ARG(dims->n_samples >= 0 && dims->n_attr >= 1, "%s: bad n_samples/n_attr", who);
    DCCF_CHECK_ARG(dims->n_samples == 0 || sample_item, "%s: sample_item is null", who);
    DCCF_CHECK_ARG(rng->noise_mode >= 0 && rng->noise_mode <= 2 && rng->mask_mode >= 0 && rng->mask_mode <= 2, "%s: bad rng mode", who);
    DCCF_CHECK_ARG(rng->noise_mode != 1 || rng->noise, "%s: noise_mode 1 needs a noise tensor", who);
    DCCF_CHECK_ARG(rng->mask_mode != 1 || rng->mask, "%s: mask_mode 1 needs a mask tensor", who);
    DCCF_CHECK_ARG(expo->mode == 0 ? expo->dense != nullptr
                                   : (expo->mode == 1 && expo->mf_user && expo->mf_item && expo->mf_user_bias && expo->mf_item_bias && expo->propensity),
                   "%s: exposure source incomplete (mode %d)", who, expo->mode);
    const int64_t R = (int64_t)(dims->n_samples + 1) * dims->n_attr;
    DCCF_CHECK_ARG(n_pairs * R < (int64_t)1 << 31, "%s: %lld rows in one call (max 2^31-1)", who, (long long)(n_pairs * R));
    return DCCF_OK;
}

extern "C" int dccf_train_fwd_tc(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat,
                                 const float* W, const float* b, const dccf_expo* expo, const int64_t* X,
                                 const int64_t* sample_item, int64_t n_pairs, const dccf_rng* rng, float* out_pred,
                                 float* ws_rows, float* ws_wimg, float* ws_pre_part, float* save_h, float* save_w,
                                 int32_t* err_flag, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int rc = check_fwd_args("dccf_train_fwd_tc", dims, expo, rng, sample_item, n_pairs);
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(E_user && E_item && Feat && W && b && X && out_pred && ws_rows && ws_wimg && ws_pre_part, "dccf_train_fwd_tc: null buffer");
    if (n_pairs <= 0) return DCCF_OK;
    const int Z = dims->n_samples + 1, R = Z * dims->n_attr;
    int32_t n_ks = 1;
    rc = launch_fwd_tc(dims, E_item, Feat, W, X, sample_item, n_pairs, rng, ws_wimg, false, ws_pre_part, err_flag,
                       &n_ks, stream);
    if (rc != DCCF_OK) return rc;

    TrainFinishParams fin;
    fin.ex = *expo; fin.E_user = E_user; fin.bias = b; fin.X = X; fin.sample_item = sample_item; fin.mask = rng->mask;
    fin.pre_part = ws_pre_part; fin.ws_rows = ws_rows; fin.save_h = save_h; fin.save_w = save_w; fin.out_pred = out_pred;
    fin.err_flag = err_flag; fin.n_pairs = n_pairs; fin.n_rows = n_pairs * R; fin.n_users = dims->n_users;
    fin.user_base = dims->user_base; fin.n_items = dims->n_items; fin.S = dims->n_samples; fin.A = dims->n_attr; fin.R = R;
    fin.n_ksplits = n_ks; fin.mask_mode = rng->mask_mode; fin.keep_prob = 1.0f - rng->p_drop;
    fin.drop_scale = (rng->p_drop < 1.0f) ? 1.0f / (1.0f - rng->p_drop) : 0.0f;
    fin.rng.seed = rng->seed; fin.rng.offset = rng->offset; fin.rng.offset_dev = rng->offset_dev;
    k_train_fwd_finish<<<(unsigned)n_pairs, 128, 0, stream>>>(fin);
    DCCF_CHECK_LAUNCH("k_train_fwd_finish");
    return DCCF_OK;
}

extern "C" int dccf_train_bwd_tc(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat,
                                 const float* W, const int64_t* X, const int64_t* sample_item, const float* Y,
                                 int64_t n_pairs, const dccf_rng* rng, int32_t loss_mode, const float* pred,
                                 const float* save_h, const float* save_w, float* out_loss, float* gW_part,
                                 float* gb_part, float* gu_rec, float* gi_rec, int32_t* rec_keys_u, int32_t* rec_keys_i,
                                 float* ws_dpre, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DCCF_CHECK_ARG(dims && rng, "dccf_train_bwd_tc: null struct argument");
    DCCF_CHECK_ARG(gW_part && gb_part && ws_dpre, "dccf_train_bwd_tc: null buffer");
    // records (embedding gradients), loss and the dpre rows: the record / loss roles of k_bpr_bwd (validates the rest)
    int rc = bpr_bwd_launch(dims, E_user, E_item, Feat, W, X, sample_item, Y, n_pairs, rng, loss_mode, pred, save_h,
                            save_w, out_loss, nullptr, nullptr, gu_rec, gi_rec, rec_keys_u, rec_keys_i, ws_dpre, false,
                            stream);
    if (rc != DCCF_OK || n_pairs <= 0) return rc;
    return launch_bwd_tc(dims, E_item, Feat, X, sample_item, n_pairs, rng, ws_dpre, gW_part, gb_part, nullptr, 0,
                         1.f, nullptr, stream);
}

extern "C" int64_t dccf_train_fused_smem_bytes(int32_t n_samples, int32_t n_attr, int32_t loss_mode) {
    const int Z = n_samples + 1, R = Z * n_attr;
    return (int64_t)(train_mid_smem_floats(R, Z, loss_mode == 0 ? 2 : 1) * sizeof(float));
}

extern "C" int dccf_train_fwd_bwd_tc(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat,
                                     const float* W, const float* b, const dccf_expo* expo, const int64_t* X,
                                     const int64_t* sample_item, const float* Y, int64_t n_pairs, int64_t mse_pairs,
                                     const dccf_rng* rng, int32_t loss_mode, float* out_pred, float* out_loss, float* ws_wimg,
                                     int32_t w_image_valid, float* ws_pre_part, float* ws_dpre, float* ws_loss_terms,
                                     float* gW_part, float* gb_part, float* gu_rec, float* gi_rec, int32_t* rec_keys_u,
                                     int32_t* rec_keys_i, float* save_h, float* save_w, const float* expo_e,
                                     const float* expo_den, const dccf_batch_ref* batch, int32_t phases, int32_t* err_flag,
                                     void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int rc = check_fwd_args("dccf_train_fwd_bwd_tc", dims, expo, rng, sample_item, n_pairs);
    DCCF_CHECK_ARG(batch == nullptr || (batch->epoch_ptrs_dev != nullptr && batch->cursor_dev != nullptr), "dccf_train_fwd_bwd_tc: batch needs both pointers");
    DCCF_CHECK_ARG(phases >= 1 && phases <= 63 && (phases & 7) != 0, "dccf_train_fwd_bwd_tc: phases is a mask of 1 (partial products), 2 (middle kernel), 4 (dW / db), + 8 / 16 / 32 (programmatic launch of phase 1 / 2 / 4)");
    DCCF_CHECK_ARG(!(phases & 16) || (phases & 3) == 3, "dccf_train_fwd_bwd_tc: phases + 16 needs phases 1 and 2 in the same call");
    DCCF_CHECK_ARG(!(phases & 32) || (phases & 6) == 6, "dccf_train_fwd_bwd_tc: phases + 32 needs phases 2 and 4 in the same call");
    DCCF_CHECK_ARG((expo_e == nullptr) == (expo_den == nullptr), "dccf_train_fwd_bwd_tc: expo_e and expo_den go together");
    DCCF_CHECK_ARG(mse_pairs == 0 || mse_pairs >= n_pairs, "dccf_train_fwd_bwd_tc: mse_pairs=%lld is below n_pairs=%lld (0: n_pairs)", (long long)mse_pairs, (long long)n_pairs);
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(loss_mode == 0 || loss_mode == 1, "dccf_train_fwd_bwd_tc: loss_mode must be 0 (BPR) or 1 (MSE)");
    DCCF_CHECK_ARG(E_user && E_item && Feat && W && b && X && out_pred && out_loss && ws_wimg && ws_pre_part && ws_dpre &&
                       ws_loss_terms && gW_part && gb_part && gu_rec && gi_rec && rec_keys_u && rec_keys_i,
                   "dccf_train_fwd_bwd_tc: null buffer");
    DCCF_CHECK_ARG(loss_mode != 1 || Y, "dccf_train_fwd_bwd_tc: MSE needs Y");
    DCCF_CHECK_ARG(loss_mode != 0 || n_pairs % 2 == 0, "dccf_train_fwd_bwd_tc: BPR needs an even number of pairs, got %lld", (long long)n_pairs);
    if (n_pairs <= 0) return DCCF_OK;
    const int Z = dims->n_samples + 1, R = Z * dims->n_attr, K = D + dims->feat_dim;
    const size_t smem = train_mid_smem_floats(R, Z, loss_mode == 0 ? 2 : 1) * sizeof(float);
    DCCF_CHECK_ARG(smem <= 200 * 1024, "dccf_train_fwd_bwd_tc: S=%d A=%d need %zu bytes of shared memory per CTA; use dccf_train_fwd_tc + dccf_train_bwd_tc", dims->n_samples, dims->n_attr, smem);
    // the middle kernel's carveout and the largest dynamic shared memory opted in so far, per device (indexed as
    // PerDeviceOnce): an opt-in made on one GPU does not carry over to the next one a process drives
    struct MidSmemOptIn { bool carveout; size_t bytes; };
    static MidSmemOptIn mid_opted[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    MidSmemOptIn& opted = mid_opted[dev & 63];
    if (!opted.carveout) {
        cudaFuncSetAttribute(k_train_mid, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        opted.carveout = true;
        opted.bytes = 48 * 1024;
    }
    if (smem > opted.bytes) {
        cudaError_t e = cudaFuncSetAttribute(k_train_mid, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            set_error("dccf_train_fwd_bwd_tc: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
            return DCCF_ERR_CUDA;
        }
        opted.bytes = smem;
    }
    int32_t n_ks = fwd_ksplits_for(n_pairs * R, K / TC_KC);
    if (phases & 1) {
        rc = launch_fwd_tc(dims, E_item, Feat, W, X, sample_item, n_pairs, rng, ws_wimg, w_image_valid != 0, ws_pre_part,
                           err_flag, &n_ks, stream, batch, (phases & 8) != 0);
        if (rc != DCCF_OK) return rc;
    }
    if (!(phases & 6)) return DCCF_OK;

    TrainMidParams mid;
    mid.ex = *expo; mid.E_user = E_user; mid.W = W; mid.bias = b; mid.X = X; mid.sample_item = sample_item; mid.Y = Y;
    mid.mask = rng->mask; mid.pre_part = ws_pre_part; mid.expo_e = expo_e; mid.expo_den = expo_den;
    mid.batch_ptrs = batch ? batch->epoch_ptrs_dev : nullptr; mid.batch_cursor = batch ? batch->cursor_dev : nullptr;
    mid.out_pred = out_pred; mid.loss_terms = ws_loss_terms;
    mid.dpre_rows = ws_dpre; mid.gu_rec = gu_rec; mid.gi_rec = gi_rec; mid.rec_keys_u = rec_keys_u; mid.rec_keys_i = rec_keys_i;
    mid.save_h = save_h; mid.save_w = save_w; mid.err_flag = err_flag; mid.n_pairs = n_pairs; mid.n_rows = n_pairs * R;
    mid.mse_pairs = mse_pairs > 0 ? mse_pairs : n_pairs;
    mid.n_users = dims->n_users; mid.user_base = dims->user_base; mid.n_items = dims->n_items; mid.S = dims->n_samples;
    mid.A = dims->n_attr; mid.R = R; mid.Z = Z; mid.K = K; mid.n_ksplits = n_ks; mid.mask_mode = rng->mask_mode;
    mid.loss_mode = loss_mode; mid.keep_prob = 1.0f - rng->p_drop;
    mid.drop_scale = (rng->p_drop < 1.0f) ? 1.0f / (1.0f - rng->p_drop) : 0.0f;
    mid.inv_A = 1.0f / (float)dims->n_attr;
    mid.rng.seed = rng->seed; mid.rng.offset = rng->offset; mid.rng.offset_dev = rng->offset_dev;
    const int64_t n_terms = (loss_mode == 0) ? n_pairs / 2 : n_pairs;
    if (phases & 2) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)n_terms); cfg.blockDim = dim3(TM_NT); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = (phases & 16) ? 1 : 0;
        const cudaError_t le = cudaLaunchKernelEx(&cfg, k_train_mid, mid);
        if (le != cudaSuccess) {
            set_error("k_train_mid: launch failed: %s", cudaGetErrorString(le));
            return DCCF_ERR_CUDA;
        }
        DCCF_CHECK_LAUNCH("k_train_mid");
    }
    if (!(phases & 4)) return DCCF_OK;

    return launch_bwd_tc(dims, E_item, Feat, X, sample_item, n_pairs, rng, ws_dpre, gW_part, gb_part, ws_loss_terms,
                         n_terms, loss_mode == 0 ? 1.f : 1.f / (float)mid.mse_pairs, out_loss, stream, batch, (phases & 32) != 0);
}
