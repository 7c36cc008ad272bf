// mf.cu — training and scoring of the exposure models BiasedMF / IPSBiasedMF (the producer of <ds>.ips_expo_prob.npy,
// README.md:27-29 of the reference):
//   pred = (<p_u, q_i> + b_u + b_i + g) / max(propensity_i, M)        (BiasedMF: propensity 1, M = 1)
// The optimizer step reuses the split step of adam.cu unchanged: dccf_adam_link_ids (record p = user row / item row of
// pair p), dccf_adam_untouched, dccf_adam_csr_build, then the kernels below, then dccf_adam_touched with the embedding
// tables and three dense tensors (user_bias, item_bias, global_bias).
#include "common.cuh"
#include "backdoor.cuh"

namespace dccf {

constexpr int MF_THREADS = 256;
constexpr int MF_PAIRS_PER_CTA = MF_THREADS / 16;     // one half-warp per pair

struct MfStepArgs {
    const float *E_user, *E_item, *user_bias, *item_bias, *global_bias, *propensity;
    float M;
    const int64_t* X;
    const float* Y;
    int64_t n_pairs;
    int32_t n_users, n_items, loss_mode;
    float* pred;
    float *gu_rec, *gi_rec, *gb_rec;
    int32_t *keys_u, *keys_i;
    float *g_part, *loss_part;
    int32_t* err_flag;
};

// Forward, loss and backward of one batch.  Half-warp per pair, lane = 4 columns.  BPR (loss_mode 0): warp w owns the
// positive pair w (half 0) and its negative w + P/2 (half 1, same user); MSE (loss_mode 1): pairs 2w and 2w + 1.
// Per pair: records d pred-loss / d p_u, d / d q_i (64 wide) and the scalar bias record r = dL/dpred / max(prop, M);
// per CTA: the sum of r (the global_bias gradient) and of the loss terms, both in half-warp order.
__global__ void __launch_bounds__(MF_THREADS) k_mf_step(const MfStepArgs a) {
    __shared__ float s_r[MF_PAIRS_PER_CTA], s_l[MF_PAIRS_PER_CTA];
    const int sub = threadIdx.x & 15, half = (threadIdx.x >> 4) & 1, hw = threadIdx.x >> 4;
    const uint32_t half_mask = half ? 0xffff0000u : 0x0000ffffu;
    const int64_t warp = ((int64_t)blockIdx.x * MF_THREADS + threadIdx.x) >> 5;
    const bool bpr = a.loss_mode == 0;
    const int64_t p = bpr ? warp + half * (a.n_pairs / 2) : 2 * warp + half;
    const bool live = bpr ? warp < a.n_pairs / 2 : p < a.n_pairs;
    float r = 0.f, term = 0.f, pred = 0.f;
    int32_t u = 0, it = 0;
    float4 pu = make_float4(0.f, 0.f, 0.f, 0.f), qi = pu;
    float scale = 1.f;
    if (live) {
        u = checked_id(a.X[2 * p], a.n_users, sub == 0 ? a.err_flag : nullptr);
        it = checked_id(a.X[2 * p + 1], a.n_items, sub == 0 ? a.err_flag : nullptr);
        pu = ldg4(a.E_user + (size_t)u * D + sub * 4);
        qi = ldg4(a.E_item + (size_t)it * D + sub * 4);
        float dot = fmaf(pu.x, qi.x, fmaf(pu.y, qi.y, fmaf(pu.z, qi.z, __fmul_rn(pu.w, qi.w))));
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(half_mask, dot, o);
        scale = fmaxf(__ldg(a.propensity + it), a.M);
        pred = (dot + __ldg(a.user_bias + u) + __ldg(a.item_bias + it) + __ldg(a.global_bias)) / scale;
    }
    float dl = 0.f;
    if (bpr) {
        // -log sigmoid(pos - neg) and its derivative; every lane of a half-warp holds the same pred (butterfly sum)
        const float x = __shfl_sync(0xffffffffu, pred, sub) - __shfl_sync(0xffffffffu, pred, 16 + sub);
        const float sig_neg = 1.f / (1.f + expf(x));                                // sigmoid(-(pos - neg))
        dl = half ? sig_neg : -sig_neg;
        term = (half == 0) ? (x > 0.f ? log1pf(expf(-x)) : log1pf(expf(x)) - x) : 0.f;
    } else if (live) {
        const float e = pred - __ldg(a.Y + p);
        dl = 2.f * e / (float)a.n_pairs;
        term = e * e;
    }
    if (live) {
        r = dl / scale;
        const float4 gu = make_float4(r * qi.x, r * qi.y, r * qi.z, r * qi.w);
        const float4 gi = make_float4(r * pu.x, r * pu.y, r * pu.z, r * pu.w);
        st4(a.gu_rec + (size_t)p * D + sub * 4, gu);
        st4(a.gi_rec + (size_t)p * D + sub * 4, gi);
        if (sub == 0) {
            a.gb_rec[p] = r;
            a.keys_u[p] = u;
            a.keys_i[p] = it;
            a.pred[p] = pred;
        }
    } else {
        r = 0.f;
        term = 0.f;
    }
    if (sub == 0) { s_r[hw] = r; s_l[hw] = term; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float gs = 0.f, ls = 0.f;
        for (int k = 0; k < MF_PAIRS_PER_CTA; ++k) { gs += s_r[k]; ls += s_l[k]; }
        a.g_part[blockIdx.x] = gs;
        a.loss_part[blockIdx.x] = ls;
    }
}

struct MfBiasArgs {
    int32_t n_users, n_items;
    const int32_t *head_u, *off_u, *csr_u;
    const int32_t *head_i, *off_i, *csr_i;
    const float* gb_rec;
    float *g_user, *g_item;
    const float* loss_part;
    int32_t n_loss_part;
    float loss_scale;
    float* out_loss;
};

// sum of the scalar records of one row in ascending record index: n rounds of "smallest id above the last one" over the
// row's CSR range (the arrival order of the ids depends on atomics timing; this order does not)
__device__ __forceinline__ float row_bias_grad(const int32_t* head, const int32_t* off, const int32_t* csr, const float* rec,
                                               int32_t row) {
    const int32_t n = head[row] + 1;
    if (n <= 0) return 0.f;
    const int32_t o = off[row];
    if (n == 1) return __ldg(rec + __ldcg(csr + o));
    float g = 0.f;
    int32_t last = -1;
    for (int32_t k = 0; k < n; ++k) {
        int32_t best = 0x7fffffff;
        for (int32_t e = 0; e < n; ++e) {
            const int32_t q = __ldcg(csr + o + e);
            if (q > last && q < best) best = q;
        }
        g += __ldg(rec + best);
        last = best;
    }
    return g;
}

// dense [U] and [I] bias gradients from the CSR of the embedding tables (thread per row, zero for untouched rows); block 0
// also sums the CTA loss partials of k_mf_step in index order
__global__ void __launch_bounds__(256) k_mf_bias_grad(const MfBiasArgs a) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n_users) {
        a.g_user[i] = row_bias_grad(a.head_u, a.off_u, a.csr_u, a.gb_rec, (int32_t)i);
    } else if (i < (int64_t)a.n_users + a.n_items) {
        const int32_t row = (int32_t)(i - a.n_users);
        a.g_item[row] = row_bias_grad(a.head_i, a.off_i, a.csr_i, a.gb_rec, row);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        float l = 0.f;
        for (int32_t k = 0; k < a.n_loss_part; ++k) l += a.loss_part[k];
        a.out_loss[0] = l * a.loss_scale;
    }
}

// predictions of evaluation pairs with the arithmetic of expo_value (the exposure source of the DCCF kernels); global_bias
// read from device memory
__global__ void __launch_bounds__(256) k_mf_scores(dccf_expo ex, const float* global_bias, const int64_t* X, int64_t n_pairs,
                                                   int32_t n_users, int32_t n_items, float* out, int32_t* err_flag) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    ex.mf_global_bias = __ldg(global_bias);
    const int32_t u = checked_id(X[2 * p], n_users, err_flag);
    const int32_t it = checked_id(X[2 * p + 1], n_items, err_flag);
    out[p] = expo_value(ex, u, it, n_items);
}

}  // namespace dccf

using namespace dccf;

extern "C" int32_t dccf_mf_step_ctas(int64_t n_pairs) {
    return n_pairs <= 0 ? 0 : (int32_t)((n_pairs + MF_PAIRS_PER_CTA - 1) / MF_PAIRS_PER_CTA);
}

extern "C" int dccf_mf_step(int32_t n_users, int32_t n_items, const float* E_user, const float* E_item,
                            const float* user_bias, const float* item_bias, const float* global_bias,
                            const float* propensity, float min_propensity, const int64_t* X, const float* Y,
                            int64_t n_pairs, int32_t loss_mode, float* out_pred, float* gu_rec, float* gi_rec,
                            float* gb_rec, int32_t* rec_keys_u, int32_t* rec_keys_i, float* g_part, float* loss_part,
                            int32_t* err_flag, void* stream) {
    DCCF_CHECK_ARG(n_users > 0 && n_items > 0 && n_pairs >= 0, "dccf_mf_step: bad sizes");
    DCCF_CHECK_ARG(loss_mode == 0 || loss_mode == 1, "dccf_mf_step: loss_mode must be 0 (BPR) or 1 (MSE)");
    DCCF_CHECK_ARG(loss_mode != 0 || n_pairs % 2 == 0, "dccf_mf_step: BPR needs an even number of pairs");
    DCCF_CHECK_ARG(loss_mode != 1 || Y, "dccf_mf_step: MSE needs Y");
    if (n_pairs == 0) return DCCF_OK;
    DCCF_CHECK_ARG(E_user && E_item && user_bias && item_bias && global_bias && propensity && X && out_pred && gu_rec &&
                   gi_rec && gb_rec && rec_keys_u && rec_keys_i && g_part && loss_part,
                   "dccf_mf_step: null argument");
    MfStepArgs a;
    a.E_user = E_user; a.E_item = E_item; a.user_bias = user_bias; a.item_bias = item_bias;
    a.global_bias = global_bias; a.propensity = propensity; a.M = min_propensity;
    a.X = X; a.Y = Y; a.n_pairs = n_pairs; a.n_users = n_users; a.n_items = n_items; a.loss_mode = loss_mode;
    a.pred = out_pred; a.gu_rec = gu_rec; a.gi_rec = gi_rec; a.gb_rec = gb_rec; a.keys_u = rec_keys_u;
    a.keys_i = rec_keys_i; a.g_part = g_part; a.loss_part = loss_part; a.err_flag = err_flag;
    k_mf_step<<<(unsigned)dccf_mf_step_ctas(n_pairs), MF_THREADS, 0, (cudaStream_t)stream>>>(a);
    DCCF_CHECK_LAUNCH("k_mf_step");
    return DCCF_OK;
}

extern "C" int dccf_mf_bias_grad(const dccf_adam_table* user, const dccf_adam_table* item, const float* gb_rec,
                                 float* g_user_bias, float* g_item_bias, const float* loss_part, int32_t n_loss_part,
                                 float loss_scale, float* out_loss, void* stream) {
    DCCF_CHECK_ARG(user && item && g_user_bias && g_item_bias && out_loss, "dccf_mf_bias_grad: null argument");
    DCCF_CHECK_ARG(user->head && user->csr_off && user->csr && item->head && item->csr_off && item->csr,
                   "dccf_mf_bias_grad: the tables need their CSR record lists (dccf_adam_csr_build)");
    DCCF_CHECK_ARG(n_loss_part >= 0 && (n_loss_part == 0 || loss_part), "dccf_mf_bias_grad: bad loss partials");
    DCCF_CHECK_ARG(user->n_rows > 0 && item->n_rows > 0 && user->n_rows + item->n_rows < ((int64_t)1 << 31),
                   "dccf_mf_bias_grad: bad table sizes");
    DCCF_CHECK_ARG(gb_rec || ((int64_t)user->n_seg * user->seg_len == 0 && (int64_t)item->n_seg * item->seg_len == 0),
                   "dccf_mf_bias_grad: null bias records");
    MfBiasArgs a;
    a.n_users = (int32_t)user->n_rows; a.n_items = (int32_t)item->n_rows;
    a.head_u = user->head; a.off_u = user->csr_off; a.csr_u = user->csr;
    a.head_i = item->head; a.off_i = item->csr_off; a.csr_i = item->csr;
    a.gb_rec = gb_rec; a.g_user = g_user_bias; a.g_item = g_item_bias;
    a.loss_part = loss_part; a.n_loss_part = n_loss_part; a.loss_scale = loss_scale; a.out_loss = out_loss;
    const int64_t blocks = ((int64_t)a.n_users + a.n_items + 255) / 256;
    k_mf_bias_grad<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    DCCF_CHECK_LAUNCH("k_mf_bias_grad");
    return DCCF_OK;
}

extern "C" int dccf_mf_scores(int32_t n_users, int32_t n_items, const dccf_expo* factors, const float* global_bias,
                              const int64_t* X, int64_t n_pairs, float* out, int32_t* err_flag, void* stream) {
    DCCF_CHECK_ARG(factors && factors->mode == 1 && factors->mf_user && factors->mf_item && factors->mf_user_bias &&
                   factors->mf_item_bias && factors->propensity && global_bias,
                   "dccf_mf_scores: needs IPS-MF factors (mode 1) and the global bias");
    DCCF_CHECK_ARG(n_users > 0 && n_items > 0 && n_pairs >= 0, "dccf_mf_scores: bad sizes");
    if (n_pairs == 0) return DCCF_OK;
    DCCF_CHECK_ARG(X && out, "dccf_mf_scores: null argument");
    k_mf_scores<<<(unsigned)((n_pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*factors, global_bias, X, n_pairs,
                                                                                     n_users, n_items, out, err_flag);
    DCCF_CHECK_LAUNCH("k_mf_scores");
    return DCCF_OK;
}
