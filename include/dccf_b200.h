/*
 * dccf_b200.h — C-ABI of the B200-native DCCF hot path (libdccf_b200.so).
 *
 * The reference (rutgerswiselab/DCCF) has no FFI of its own: its hot path is eager PyTorch
 * inside Python classes.  Each entry point below replaces a span of reference Python, cited
 * as `file:line` relative to the reference root.  All pointers are DEVICE pointers unless a
 * parameter is documented as host; buffers are owned by the caller (PyTorch allocator on the
 * Python side); nothing is allocated or freed by the library; every call is asynchronous on
 * `stream` (a cudaStream_t passed as void*).
 *
 * Return value: 0 on success, negative dccf_status otherwise; dccf_last_error() returns a
 * thread-local message for the last failure.
 *
 * Shapes use the reference's names: U users, I items, D = u_vector_size (= 64 in this build),
 * F = feature width (768), S = --sample-num, A = --attribute-num, Z = S+1 slots,
 * R = Z*A predictor rows per (user,item) pair, P pairs per call, N = P*R rows.
 * Row r of a call is (p, z, a) with r = (p*Z + z)*A + a   (src/models/DCCF.py:76-82).
 */
#ifndef DCCF_B200_H
#define DCCF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCCF_ABI_VERSION 40
#define DCCF_DIM 64 /* u_vector_size == i_vector_size compiled into the kernels */

typedef enum dccf_status {
    DCCF_OK = 0,
    DCCF_ERR_ARG = -1,     /* bad argument (null pointer, unsupported size) */
    DCCF_ERR_CUDA = -2,    /* a CUDA runtime call failed; see dccf_last_error() */
    DCCF_ERR_UNSUPPORTED = -3
} dccf_status;

/* Model geometry (src/models/DCCF.py:23-34 ctor arguments). */
typedef struct dccf_dims {
    int32_t n_users;   /* U */
    int32_t n_items;   /* I */
    int32_t dim;       /* D, must equal DCCF_DIM */
    int32_t feat_dim;  /* F, multiple of 64 */
    int32_t n_samples; /* S  (--sample-num) */
    int32_t n_attr;    /* A  (--attribute-num) */
    int32_t user_base; /* row-sharded user table: this rank owns global users [user_base, user_base + n_users);
                          E_user, the dense expo rows / IPS-MF user factors and the user gradient records are
                          indexed by uid - user_base.  0 when the table is not sharded. */
    int32_t _pad;
} dccf_dims;

/* Exposure source for softmax_z(expo_prob[u, item_z])  (src/models/DCCF.py:64,98). */
typedef struct dccf_expo {
    int32_t mode;            /* 0: dense [U,I] f32 matrix (ips_expo_prob.npy);
                                1: on the fly from IPSBiasedMF factors (src/models/IPSBiasedMF.py:37-57) */
    int32_t _pad;
    const float* dense;      /* mode 0 */
    const float* mf_user;    /* mode 1: [U,D] */
    const float* mf_item;    /* mode 1: [I,D] */
    const float* mf_user_bias; /* [U] */
    const float* mf_item_bias; /* [I] */
    const float* propensity; /* [I] */
    float mf_global_bias;
    float mf_min_propensity; /* M */
} dccf_expo;

/* Random inputs of one predict call (src/models/DCCF.py:87 noise, :94 dropout).
 * mode 0: absent (std == 0 / p == 0); mode 1: explicit tensor supplied by the caller (parity
 * runs feed the reference's own draws); mode 2: counter-based Philox4x32-10 generated in
 * registers — bit-identical to what dccf_noise_fill / dccf_dropout_mask_fill materialise for
 * the same (seed, offset). */
typedef struct dccf_rng {
    int32_t noise_mode;
    int32_t mask_mode;
    const float* noise; /* mode 1: [N,F] = eps (already scaled by std) */
    const float* mask;  /* mode 1: [N,D] = bernoulli(1-p)/(1-p)       */
    float noise_std;    /* mode 2 */
    float p_drop;       /* mode 2 */
    uint64_t seed;      /* mode 2 */
    uint64_t offset;    /* mode 2: call counter, distinct per predict call */
    const uint64_t* offset_dev; /* mode 2, optional DEVICE pointer: when non-NULL the kernels read the
                                   call counter from here instead of `offset` (lets a captured CUDA
                                   graph be replayed; see dccf_state_advance) */
} dccf_rng;

const char* dccf_last_error(void);
int dccf_abi_version(void);

/* ---- RNG materialisers (host-visible definition of the mode-2 streams) ------------------ */
/* out[r,f] = std * normal(seed, offset, row0 + r, f)          replaces DCCF.py:87 `normal_` */
int dccf_noise_fill(float* out, int64_t n_rows, int32_t feat_dim, float std,
                    uint64_t seed, uint64_t offset, int64_t row0, void* stream);
/* out[r,j] = (uniform(seed, offset, row0 + r, j) < 1-p) / (1-p)   replaces DCCF.py:94 Dropout */
int dccf_dropout_mask_fill(float* out, int64_t n_rows, int32_t dim, float p_drop,
                           uint64_t seed, uint64_t offset, int64_t row0, void* stream);

/* ---- (a)+(b): fused gather + predictor rows + backdoor-adjusted score ------------------- */
/* Replaces DCCF.predict lines 74-100 (src/models/DCCF.py).
 *   X            [P,2] int64, col 0 = uid, col 1 = iid           (feed_dict['X'])
 *   sample_item  [P,S] int64 confounder items                    (DCCF.py:72, drawn by caller)
 *   W            [D, D+F] row-major  (mlp.0.weight),  b [D]      (mlp.0.bias)
 *   out_pred     [P]
 *   ws_rows      [N] workspace: s[r] = <E_user[u], dropout(relu(W x_r + b))>
 *   ws_wt        [(D+F)*D] workspace: W transposed (k-major)
 *   save_h       [N,D] or NULL: post-dropout activations kept for the backward pass
 *   save_w       [P,Z] or NULL: softmax exposure weights
 *   err_flag     int32[1]: set to 1 if any id was out of range (ids are clamped, never faulting)
 */
int dccf_score_fwd(const dccf_dims* dims, const float* E_user, const float* E_item,
                   const float* Feat, const float* W, const float* b, const dccf_expo* expo,
                   const int64_t* X, const int64_t* sample_item, int64_t n_pairs,
                   const dccf_rng* rng, float* out_pred, float* ws_rows, float* ws_wt,
                   float* save_h, float* save_w, int32_t* err_flag, void* stream);

/* ---- (a)+(b), tensor-core variant for evaluation batches ------------------------------------ */
/* Same result as dccf_score_fwd (no save_h / save_w: inference only) with the W_f·eps product on the
 * tcgen05 tensor cores as an error-compensated 3xTF32 product (FP32-level accuracy) and the noise-free terms
 * taken from two projected tables.  dccf_tc_prepare must be called again whenever E_item, W or b change:
 *   PI [I,D] = E_item·W_i^T     PF [I,D] = Feat·W_f^T + b     gB [dccf_tc_operand_floats(F)] = split W_f
 *   dbg_pre [N,D] or NULL: the raw tensor-core accumulator W_f·eps (tests)
 */
int64_t dccf_tc_operand_floats(int32_t feat_dim);
int dccf_tc_prepare(const dccf_dims* dims, const float* E_item, const float* Feat, const float* W,
                    const float* b, float* ws_wt, float* PI, float* PF, float* gB, void* stream);
int dccf_score_fwd_tc(const dccf_dims* dims, const float* E_user, const float* PI, const float* PF,
                      const float* gB, const dccf_expo* expo, const int64_t* X, const int64_t* sample_item,
                      int64_t n_pairs, const dccf_rng* rng, float* out_pred, float* ws_rows, float* dbg_pre,
                      int32_t* err_flag, void* stream);

/* ---- (a)+(b), gather variant for noise-free scoring ------------------------------------------ */
/* src/models/DCCF.py:74-100 when --std 0 and dropout 0 (evaluation of a model trained without feature noise; the
 * parity configuration): the attribute copies coincide and the predictor input has no per-row random part, so
 *   pred[p] = sum_z softmax_z(expo[u_p, item(p,z)]) · < E_user[u_p], relu(PI[item(p,z)] + PF[i_p]) >
 * with the two projected tables of dccf_tc_prepare — Z + 2 row gathers per pair instead of a contraction over the
 * D + F inputs: the HBM / L2-bound regime of the scorer (SURVEY.md §8d).  No workspace, no random inputs.
 *   out_pred [P] */
int dccf_score_gather(const dccf_dims* dims, const float* E_user, const float* PI, const float* PF,
                      const dccf_expo* expo, const int64_t* X, const int64_t* sample_item, int64_t n_pairs,
                      float* out_pred, int32_t* err_flag, void* stream);

/* ---- (c) part 1: pairwise loss forward + full backward ---------------------------------- */
/* Replaces DCCF.forward lines 116-125 (src/models/DCCF.py) + autograd backward
 * (src/runners/BaseRunner.py:183).  One launch.
 *   loss_mode 0: BPR  -sum_j log sigmoid(pred[j]-pred[j+P/2])   (rank==1, P even)
 *   loss_mode 1: MSE  mean_p (pred[p]-Y[p])^2                    (rank==0)
 *   loss_mode 2: no loss: Y[p] holds d loss/d pred[p] computed by the caller (autograd path);
 *                out_loss may be NULL
 *   pred [P], save_h [N,D], save_w [P,Z] from dccf_score_fwd called with the SAME rng.
 *   out_loss     float[1]
 *   gW_part      [n_splits, D, D+F], gb_part [n_splits, D]: per-row-split partial sums of
 *                d loss/d W and d loss/d b, summed in ascending split order by dccf_adam_dense
 *   gu_rec       [P,D]    gradient record for user row X[p,0]
 *   gi_rec       [P*Z,D]  gradient record for item row items[p,z]
 *   rec_keys_u   [P] int32, rec_keys_i [P*Z] int32: the table rows those records belong to
 * n_splits must equal dccf_bwd_splits(N) with N = P*Z*A.
 */
int32_t dccf_bwd_splits(int64_t n_rows);
int dccf_bpr_bwd(const dccf_dims* dims, const float* E_user, const float* E_item,
                 const float* Feat, const float* W, const int64_t* X, const int64_t* sample_item,
                 const float* Y, int64_t n_pairs, const dccf_rng* rng, int32_t loss_mode,
                 const float* pred, const float* save_h, const float* save_w, float* out_loss,
                 float* gW_part, float* gb_part, float* gu_rec, float* gi_rec,
                 int32_t* rec_keys_u, int32_t* rec_keys_i, void* stream);

/* ---- training step on the tensor cores (tcgen05, 3xTF32) --------------------------------- */
/* Same results as dccf_score_fwd (with save_h / save_w) and dccf_bpr_bwd, for the rows of ONE training step
 * (src/runners/BaseRunner.py:175-188), with both large contractions on the tensor cores and spread over all
 * SMs: the forward as (128-row tiles) x (K splits) partial products, the backward dW / db as (128-column
 * tiles of [x | 1]) x (row splits) with the row as the contraction index.
 *   ws_wimg      [dccf_train_w_image_floats(F)] workspace: hi/lo operand images of W (rebuilt per call)
 *   ws_pre_part  [dccf_train_fwd_ksplits(N, F), N, D] workspace: partial pre-activations
 *   gW_part      [dccf_train_bwd_splits(N, F), D, D+F], gb_part [same, D]
 *   ws_dpre      [N, D] workspace: d loss / d pre-activation rows
 * All other arguments as in dccf_score_fwd / dccf_bpr_bwd; both calls must use the SAME rng. */
int64_t dccf_train_w_image_floats(int32_t feat_dim);
int32_t dccf_train_fwd_ksplits(int64_t n_rows, int32_t feat_dim);
int32_t dccf_train_bwd_splits(int64_t n_rows, int32_t feat_dim);
int dccf_train_fwd_tc(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat,
                      const float* W, const float* b, const dccf_expo* expo, const int64_t* X,
                      const int64_t* sample_item, int64_t n_pairs, const dccf_rng* rng, float* out_pred,
                      float* ws_rows, float* ws_wimg, float* ws_pre_part, float* save_h, float* save_w,
                      int32_t* err_flag, void* stream);
int dccf_train_bwd_tc(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat,
                      const float* W, const int64_t* X, const int64_t* sample_item, const float* Y,
                      int64_t n_pairs, const dccf_rng* rng, int32_t loss_mode, const float* pred,
                      const float* save_h, const float* save_w, float* out_loss, float* gW_part,
                      float* gb_part, float* gu_rec, float* gi_rec, int32_t* rec_keys_u, int32_t* rec_keys_i,
                      float* ws_dpre, void* stream);

/* Forward + loss + backward of one training step in three launches (BPR loss_mode 0 or MSE loss_mode 1): the
 * partial products, then ONE fused kernel per loss term (forward epilogue, backdoor sum, loss term,
 * d loss / d pred, dpre rows, embedding-gradient records — with BPR a CTA owns the positive pair j and its
 * negative j + P/2), then the dW / db tiles (whose CTA (0,0) also sums the loss terms in a fixed order).
 *   w_image_valid != 0: ws_wimg already holds the operand images of the current W (dccf_adam_step wrote them)
 *   the dW kernel regenerates the rows Feat[i] + eps the forward multiplied (same noise stream), it stores none
 *   ws_loss_terms [P/2] (BPR) or [P] (MSE) workspace;  save_h / save_w optional (NULL: not written)
 *   expo_e [P, Z] / expo_den [P] optional: the exposure softmax precomputed by dccf_adam_link_ids
 *   phases: mask of 1 = the partial products, 2 = the middle kernel, 4 = the dW / db tiles (7 = everything; same
 *        arguments every time) — lets the caller wait for / signal other streams between the kernels (the stream
 *        that produced expo_e before the middle kernel; the stream that ships the gradient records after it).
 *        + 8: the partial-product kernel is launched as a PROGRAMMATIC DEPENDENT of the kernel before it on the stream
 *        (cudaLaunchAttributeProgrammaticStreamSerialization): it starts as soon as that kernel — dccf_adam_link_ids,
 *        which signals griddepcontrol.launch_dependents first thing — has started, reads nothing it writes (use
 *        `batch` when the ids are being staged by it) and does not complete before it has; needs w_image_valid.
 *        + 16: the middle kernel is a programmatic dependent of the partial-product kernel (needs phases 1 and 2):
 *        its barrier-free prologue (W_i, b, the RNG key; with `batch` the user rows) runs before it waits.
 *        + 32: the dW / db kernel is a programmatic dependent of the middle kernel (needs phases 2 and 4): barriers,
 *        tensor memory and, with `batch`, the x operand of its first stages are set up before it waits for dpre.
 *        Each kernel completes only after the kernel it depends on has, so the chain stays ordered
 *   batch (optional): the partial-product kernel (phase 1) takes its ids from batch *cursor_dev of a device-resident
 *        epoch (epoch_ptrs_dev[0..1] = base addresses of X_epoch [n, P, 2] / sample_epoch [n, P, S], the arrays
 *        dccf_link_extra's staging reads) instead of X / sample_item — it then does not have to wait for the launch
 *        that stages them (dccf_adam_link_ids), which runs beside it (phases + 8); phases 2 and 4 read the same ids
 *        through it before their wait (phases + 16 / + 32) and X / sample_item, the staged copies, after it
 *   mse_pairs: the number of pairs the MSE mean is taken over (0: n_pairs).  A data-parallel step passes world * n_pairs,
 *        so that d loss / d pred = 2 (pred - Y) / mse_pairs and the loss term is the rank's share of the mean over the
 *        global batch; counts below n_pairs are rejected.  BPR ignores it.  The middle kernel reads Y after its wait
 *        (Y may be the staged copy of a device-resident label epoch, dccf_link_extra.Y_out)
 * Needs dccf_train_fused_smem_bytes(S, A, loss_mode) <= 200 KB of shared memory per CTA (else use the two calls
 * above). */
typedef struct dccf_batch_ref { const uint64_t* epoch_ptrs_dev; const int64_t* cursor_dev; } dccf_batch_ref;
int64_t dccf_train_fused_smem_bytes(int32_t n_samples, int32_t n_attr, int32_t loss_mode);
int dccf_train_fwd_bwd_tc(const dccf_dims* dims, const float* E_user, const float* E_item, const float* Feat,
                          const float* W, const float* b, const dccf_expo* expo, const int64_t* X,
                          const int64_t* sample_item, const float* Y, int64_t n_pairs, int64_t mse_pairs,
                          const dccf_rng* rng, int32_t loss_mode, float* out_pred, float* out_loss, float* ws_wimg,
                          int32_t w_image_valid, float* ws_pre_part, float* ws_dpre, float* ws_loss_terms,
                          float* gW_part, float* gb_part, float* gu_rec, float* gi_rec, int32_t* rec_keys_u,
                          int32_t* rec_keys_i, float* save_h, float* save_w, const float* expo_e,
                          const float* expo_den, const dccf_batch_ref* batch, int32_t phases, int32_t* err_flag,
                          void* stream);

/* ---- (c) part 2: l2 + clip + optimizer (Adam, GD, Adagrad), dense over every row ---------- */
/* Replaces model.l2()*l2 (BaseRunner.py:181, BaseModel.py:179-187), clip_grad_value_
 * (BaseRunner.py:185) and the optimizer step (BaseRunner.py:83-107,187), every optimizer with
 * weight_decay = l2:
 *   g = clamp(g_sparse + 2*l2*p, -clip, clip) + wd*p
 * then, by dccf_adam.rule:
 *   0 Adam     m,v,p updated as torch 2.11 optim/adam.py (_multi_tensor_adam, non-capturable branch)
 *   1 GD       torch.optim.SGD, momentum 0:   p = p - lr*g                        (no state)
 *   2 Adagrad  torch.optim.Adagrad, lr_decay 0, initial_accumulator_value 0:
 *              s = s + g*g ; p = p - lr*g / (sqrt(s) + eps)                       (state_sum s in `m`)
 * The update is dense: rows without gradient records step with g_sparse = 0.  A rule reads and
 * writes only its own state; the state pointers it does not have may be NULL.  Only
 * dccf_adam_step, dccf_adam_untouched and dccf_adam_touched take rule != 0.
 * Embedding-table variant: the gradient arrives as n_rec records (row id + D floats); records
 * with equal ids are summed in ascending record order (deterministic).
 *   head  int32[n_table_rows], persistent, must be -1 everywhere on entry; is -1 again on exit
 *   next  int32[n_rec] workspace
 */
typedef struct dccf_adam {
    double lr, beta1, beta2, eps; /* Python doubles, as torch.optim.Adam receives them */
    double l2;          /* weight of sum p^2 in the loss  (--l2) */
    double weight_decay;/* Adam weight_decay               (--l2) */
    double clip;        /* clip_grad_value_ bound, 50; <= 0 disables */
    int32_t step;       /* t = 1,2,... */
    int32_t rule;       /* 0 Adam (a zero-initialised struct), 1 GD, 2 Adagrad */
    const int32_t* step_dev; /* optional DEVICE pointer overriding `step` (graph replay) */
} dccf_adam;

int dccf_adam_sweep(float* table, float* m, float* v, int64_t n_table_rows,
                    const int32_t* rec_keys, const float* rec_grads, int64_t n_rec,
                    int32_t* head, int32_t* next, const dccf_adam* hp, void* stream);
/* Same, with the records in n_seg segments of seg_len records (one segment per data-parallel rank after
 * the gradient all-gather): segment s has its keys at rec_keys + s*key_seg_stride (int32 units) and its
 * gradients at rec_grads + s*grad_seg_stride (float units).  Records are summed in ascending global index
 * (segment-major), so every rank computes bit-identical updates. */
int dccf_adam_sweep_seg(float* table, float* m, float* v, int64_t n_table_rows,
                        const int32_t* rec_keys, const float* rec_grads, int32_t n_seg, int64_t seg_len,
                        int64_t key_seg_stride, int64_t grad_seg_stride,
                        int32_t* head, int32_t* next, const dccf_adam* hp, void* stream);
/* out[i] = sum_k parts[k*part_stride + i], ascending k: folds the row-split partials of dccf_bpr_bwd into one
 * [D, D+F] gradient before it is exchanged between ranks. */
int dccf_sum_parts(const float* parts, int32_t n_parts, int64_t part_stride, int64_t n, float* out, void* stream);
/* Dense variant for mlp.0.weight / mlp.0.bias: g = sum over n_parts partial buffers of n floats. */
int dccf_adam_dense(float* p, float* m, float* v, int64_t n, const float* g_parts,
                    int32_t n_parts, int64_t part_stride, const dccf_adam* hp, void* stream);
/* The whole optimizer step in two launches (record linking + one sweep over every tensor): up to 4
 * embedding tables with segmented records and up to 4 dense tensors with partial-sum gradients.  Same
 * arithmetic and summation order as the per-tensor entry points above. */
typedef struct dccf_adam_table {
    float* table; float* m; float* v;  /* m / v: the rule's state (see dccf_adam.rule) */
    int64_t n_rows;
    const int32_t* rec_keys; const float* rec_grads;
    int32_t n_seg; int32_t _pad;
    int64_t seg_len, key_seg_stride, grad_seg_stride;
    int32_t* head; int32_t* next;      /* next: n_seg*seg_len entries, private to this table */
    /* CSR record lists (all four NULL: linked lists through head / next).  With them dccf_adam_link_ids COUNTS instead of
     * linking — head[row] = (records of the row) - 1, next[r] = arrival position of record r in its row, rec_row[r] = the
     * row — dccf_adam_csr_build groups the record ids by row (csr_off [n_rows]; csr [2 * n_seg*seg_len]: the grouped
     * record ids, then the compact list of the step's touched rows; csr_pool: int32[2] = {ids used, rows touched}, zero
     * between steps), and dccf_adam_touched runs one half-warp per TOUCHED ROW, reading its records with parallel
     * loads instead of walking a list (the walk of the hottest item's list was the critical path of the data-parallel
     * step).  Same summation order (ascending record index), same bits. */
    int32_t* rec_row; int32_t* csr_off; int32_t* csr; int32_t* csr_pool;
} dccf_adam_table;
typedef struct dccf_adam_tensor {
    float* p; float* m; float* v;
    int64_t n;
    const float* g_parts;
    int32_t n_parts; int32_t _pad;
    int64_t part_stride;
} dccf_adam_tensor;
int dccf_adam_step(const dccf_adam_table* tables, int32_t n_tables, const dccf_adam_tensor* dense,
                   int32_t n_dense, const dccf_adam* hp, void* stream);
/* Host only, no CUDA call: the CTA ranges one launch of the optimizer step gives its tensors — tables first (n_rows,
 * n_rec records each), then dense tensors (n_dense_elems each).  mode 0: dccf_adam_step; 1: dccf_adam_untouched
 * (threads_per_cta >= 0); 2: dccf_adam_touched and dccf_adam_csr_build; 3: dccf_adam_untouched (threads_per_cta < 0,
 * the wide sweep).  Only mode 2 reads n_rec; modes 0, 1 and 3 share the CTAs by n_rows.  Writes block_lo / block_n
 * [n_tables + n_dense] and returns the grid size; -1 on a bad argument (a negative count among them). */
int32_t dccf_adam_blocks(int32_t mode, const int64_t* n_rows, const int64_t* n_rec, int32_t n_tables,
                         const int64_t* n_dense_elems, int32_t n_dense, int32_t* block_lo, int32_t* block_n);
/* The same optimizer step split around the backward pass: the rows a step does not touch (99 % of both
 * embedding tables; their gradient is the l2 / weight-decay term only) are swept by dccf_adam_untouched on a
 * second stream WHILE the forward and backward run; the touched rows, W and b follow the backward.
 *   dccf_adam_link_ids      builds the record lists of the step from the ids alone (record p = user row of pair
 *                           p, record p*Z + z = item row of slot z; out-of-range ids are clamped to row 0 exactly as
 *                           the kernels that write the records do): afterwards head[row] >= 0 marks a touched row
 *                           Data parallel: the ids of all n_seg ranks (gathered at the start of the step), segment s
 *                           at X + s*seg_stride / sample_item + s*seg_stride (int64 elements), records numbered
 *                           segment-major like the gathered gradient records; user_seg >= 0: only that segment
 *                           has user records (row-sharded user table), numbered locally.  n_seg == 0: no linking,
 *                           only the exposure softmax below.
 *                           expo (optional): the same launch also evaluates the exposure softmax of every pair of
 *                           this rank's own batch (X_local / sample_item_local; NULL: segment 0)
 *                           (src/models/DCCF.py:98, a function of the ids only): expo_e [P, Z] = exp(expo - max),
 *                           expo_den [P] = A * sum_z, consumed by dccf_train_fwd_bwd_tc
 *   dccf_adam_untouched     rows whose head is -1; at most 148 CTAs of threads_per_cta threads (0 = 224) so that a
 *                           tensor-core CTA fits beside each
 *   dccf_adam_touched       the head record of each list updates its row (records summed in ascending index) and
 *                           resets head to -1; dense tensors as in dccf_adam_step.  already_linked = 0: links the
 *                           records first (dccf_adam_link_ids was not used).  w_image (optional): operand images
 *                           of the UPDATED W [D, w_image_K] = dense[w_image_tensor] for the next step's
 *                           dccf_train_fwd_bwd_tc(w_image_valid = 1); dccf_train_prep_w_image builds them from
 *                           scratch.  cta_counter (optional, int32 zero on entry / exit): the last CTA to finish does
 *                           advance_step_dev[0] += 1, advance_offset_dev[0] += 1 and advance_cursor_dev[0] += 1 — the
 *                           batch cursor of a device-resident epoch — each when non-NULL (replaces dccf_state_advance
 *                           in a captured step; every other reader of the counters must have completed).
 *                           sync (optional, needs cta_counter): data-parallel step — every CTA first waits for the peers'
 *                           gradient segments, the last CTA sums the ranks' loss terms and hands the buffers back.
 * Every row is updated exactly once, with the arithmetic of dccf_adam_step. */
/* Data-parallel synchronisation folded into a consumer kernel (NULL: none).  A channel is one symmetric exchange buffer
 * of dccf_dp_push.  The kernel that receives a dccf_dp_sync
 *   - waits in the prologue of every CTA until all `world` arrival flags of each wait channel show the current exchange
 *     (what dccf_dp_wait does in a launch of its own between producer and consumer);
 *   - in its LAST CTA: sums n_loss values loss_stride floats apart into loss_out (the ranks' loss terms), marks every
 *     done channel as consumed on every peer and advances its epoch counter (what dccf_dp_done does, one launch per
 *     channel, after the consumer). */
typedef struct dccf_dp_channel {
    uint64_t peer_bases[8];      /* device address of the buffer on every rank (this rank's own at index rank) */
    int64_t flag_off;            /* floats */
    int32_t* epoch_dev;
    int64_t seg_floats;          /* segment length of the channel's pushes (fixes the number of arrival flags) */
} dccf_dp_channel;
typedef struct dccf_dp_sync {
    int32_t world, rank, n_wait, n_done;
    dccf_dp_channel wait[3];
    dccf_dp_channel done[3];
    const float* loss_parts; int64_t loss_stride; int32_t n_loss; int32_t flags; float* loss_out;
} dccf_dp_sync;
/* dccf_dp_sync.flags, dccf_adam_touched only: wait[0] is the channel of the gradient records, wait[1] the channel of
 * dW / db / loss, and the kernel launched just before dccf_adam_touched on its stream is this rank's push of the latter.
 * The CTAs that sweep table rows then wait for wait[0] only, the CTAs of the dense tensors for wait[1]; the launch is a
 * programmatic dependent of that push (it starts when every CTA of the push is resident, and does not complete before
 * the push has): the table rows are swept WHILE dW / db travel. */
#define DCCF_DP_SYNC_OVERLAP_PUSH 1
/* Optional extras of dccf_adam_link_ids (NULL: none), all device pointers:
 *   staging (epoch_ptrs_dev != NULL): the step reads its batch from a device-resident epoch — what dccf_stage_batch does
 *     in a launch of its own: X / sample_item arguments are ignored, the batch is [*cursor] of the arrays whose
 *     addresses sit in epoch_ptrs_dev {X_epoch [n,P,2], sample_epoch [n,P,S]}; every id is copied into X_out /
 *     sample_item_out (the buffers the later kernels of the step read) by the thread that links it.  Y_out (optional,
 *     rating prediction): the labels of the batch, float32 from the label epoch Y_epoch [n,P] whose address sits in
 *     epoch_ptrs_dev[6], are copied into Y_out [P] by the thread that copies the pair's user id.  The cursor is NOT
 *     moved here: the partial-product kernel may be reading the same batch beside this launch (dccf_batch_ref);
 *     dccf_adam_touched (advance_cursor_dev) moves it when the step is over.  Needs n_seg <= 1.
 *   L2 prefetch (any pointer may be NULL): the rows this step will touch — the pairs' user rows, the slot items' rows
 *     and their Adam moments, the true items' feature rows — and up to four dense ranges (W, its moments, its operand
 *     images) are requested into L2 (prefetch.global.L2) while the step's first kernels run, so that the forward, the
 *     middle kernel and the touched-row sweep find them there instead of in DRAM.  No effect on results.
 *   sync: data-parallel link of the GLOBAL step — wait for the peers' ids in the prologue, hand the id buffer back in
 *     the last CTA (stage_counter: int32 CTA counter, zero on entry / exit). */
typedef struct dccf_link_extra {
    const uint64_t* epoch_ptrs_dev; int64_t* cursor_dev; int64_t* X_out; int64_t* sample_item_out; float* Y_out;
    int32_t* stage_counter;
    const float* pf_user[3];     /* E_user, exp_avg, exp_avg_sq   [n_users, D] */
    const float* pf_item[3];     /* E_item, exp_avg, exp_avg_sq   [n_items, D] */
    const float* pf_feat;        /* Feat [n_items, feat_dim] */
    const void* pf_dense[4]; int64_t pf_dense_bytes[4];
    const dccf_dp_sync* sync;    /* HOST pointer, copied at launch */
    int32_t* rec_row_user; int32_t* rec_row_item;   /* counting mode (CSR lists, see dccf_adam_table): both non-NULL */
} dccf_link_extra;
int dccf_adam_link_ids(const dccf_dims* dims, const int64_t* X, const int64_t* sample_item, int64_t n_pairs,
                       int32_t n_seg, int64_t seg_stride, int32_t user_seg, int32_t* head_user, int32_t* next_user,
                       int32_t* head_item, int32_t* next_item, const dccf_expo* expo, const int64_t* X_local,
                       const int64_t* sample_item_local, float* expo_e, float* expo_den,
                       const dccf_link_extra* extra, void* stream);
int dccf_adam_untouched(const dccf_adam_table* tables, int32_t n_tables, const dccf_adam* hp,
                        int32_t threads_per_cta, void* stream);
/* Between dccf_adam_link_ids (counting mode) and dccf_adam_touched, any stream: record ids grouped by row (2 launches). */
int dccf_adam_csr_build(const dccf_adam_table* tables, int32_t n_tables, void* stream);
int dccf_adam_touched(const dccf_adam_table* tables, int32_t n_tables, const dccf_adam_tensor* dense,
                      int32_t n_dense, const dccf_adam* hp, int32_t already_linked, float* w_image,
                      int32_t w_image_tensor, int32_t w_image_K, int32_t* cta_counter, int32_t* advance_step_dev,
                      uint64_t* advance_offset_dev, int64_t* advance_cursor_dev, const dccf_dp_sync* sync, void* stream);
int dccf_train_prep_w_image(const float* W, int32_t feat_dim, float* w_image, void* stream);
/* First node of a captured training step that reads its inputs from a device-resident epoch:
 * epoch_ptrs_dev = device array {address of X_epoch [n_batches,P,2], address of sample_epoch [n_batches,P,S]; with
 * Y_out also slot 6 = address of the label epoch Y_epoch [n_batches,P] float32}, cursor_dev = device int64 batch
 * counter (copied batch *cursor, then incremented).  Y_out (optional): the batch's labels (rating prediction). */
int dccf_stage_batch(const uint64_t* epoch_ptrs_dev, int64_t* cursor_dev, int64_t n_pairs, int32_t n_samples,
                     int64_t* X_out, int64_t* sample_item_out, float* Y_out, void* stream);
/* step_dev[0] += 1 ; offset_dev[0] += offset_inc  (either pointer may be NULL) — the last node
 * of a captured training step, so that a replay sees t+1 and a fresh rng counter. */
int dccf_state_advance(int32_t* step_dev, uint64_t* offset_dev, uint64_t offset_inc, void* stream);

/* ---- debug ------------------------------------------------------------------------------- */
/* Install (or remove, with NULL) a device buffer of 2 x 16 uint64 slots in which the kernels of the fused training
 * step record {earliest CTA start, latest CTA end} in nanoseconds of %globaltimer: slot 0 k_link_ids,
 * 1 k_adam_untouched, 2 k_train_fwd_tc, 3 k_train_mid, 4 k_train_bwd_tc, 5 k_adam_touched, 6 k_stage_batch,
 * 8 k_dp_push (ids), 9 k_dp_wait, 10 k_dp_push (records), 11 k_dp_push (dW / db / loss), 12 the moment the peers'
 * segments had arrived in k_adam_touched, 13 k_csr_build.
 * The caller initialises every slot to {UINT64_MAX, 0} (tools/step_timeline.py).  One entry point per
 * translation unit that owns instrumented kernels. */
int dccf_debug_timeline_train(unsigned long long* slots);
int dccf_debug_timeline_adam(unsigned long long* slots);
int dccf_debug_timeline_dp(unsigned long long* slots);

/* ---- (d): evaluation ranker -------------------------------------------------------------- */
/* Replaces BaseModel.evaluate_method ranking branch (src/models/BaseModel.py:82-126) and
 * src/utils/rank_metrics.py:61-87,130-201.
 *   scores [n_rows] f32, labels [n_rows] f32, iids [n_rows] int64, all in data order
 *   cand_rows [n_cand] int32: row indices grouped by user; user g owns cand_rows[off[g]..off[g+1]).
 *             NULL: the rows are already grouped by user (the evaluation set is built user-major), candidate c
 *             IS row c and the scores / labels are read contiguously
 *   user_off  [n_users+1] int64
 * Ranking order: score descending, ties by item id ascending, then by row index ascending; NaN last.
 *   out_topk_iid [n_users,k] int64 (-1 padded), out_topk_row [n_users,k] int32 (may be NULL)
 *   out_metrics  [n_users,5] f64: ndcg@k, hit@k, precision@k, recall@k, f1@k
 * k <= 16: one streaming pass per user (per-lane top-k in registers); larger k: k selection rounds. */
int dccf_rank_eval(const float* scores, const float* labels, const int64_t* iids,
                   const int32_t* cand_rows, const int64_t* user_off, int64_t n_users, int32_t k,
                   int64_t* out_topk_iid, int32_t* out_topk_row, double* out_metrics,
                   void* stream);
/* Every '<name>@k' metric of a metric list in ONE launch (the reference loops over the users once per metric,
 * src/models/BaseModel.py:90-126): ks = HOST array of n_k (1..4) strictly ascending values of k, each <= 16.
 *   out_topk_iid / out_topk_row [n_users, ks[n_k-1]]  (may be NULL)
 *   out_metrics [n_users, n_k, 5] f64 (may be NULL when out_sums is given)
 *   out_sums    [n_k, 5] f64: the per-user values summed over users in a fixed order (warp, CTA, then the CTAs in
 *               index order by the last CTA to finish) — what np.average over users needs; may be NULL
 *   ws          device workspace of dccf_rank_eval_ws_bytes() bytes, ZERO on first use (the kernel leaves its
 *               counter at zero); required with out_sums */
int64_t dccf_rank_eval_ws_bytes(int64_t n_users);
int dccf_rank_eval_multi(const float* scores, const float* labels, const int64_t* iids, const int32_t* cand_rows,
                         const int64_t* user_off, int64_t n_users, const int32_t* ks, int32_t n_k,
                         int64_t* out_topk_iid, int32_t* out_topk_row, double* out_metrics, void* ws,
                         double* out_sums, void* stream);
/* Ranking metrics of full-catalogue top-k lists (dccf_full_scores with known-item exclusion) against held-out
 * positives, with the definitions of dccf_rank_eval_multi applied to the ranked list of every rankable item (label 1
 * for a positive):
 *   topk_id  [n_users, k_list] int64: score descending, ties by item id ascending, -1 padded; 1 <= k_list <= 16
 *   pos_off  [n_users+1] int64, pos_items int32: each user's positives, ascending and unique (a CSR over the same rows)
 *   ks       HOST array of n_k (1..4) strictly ascending values of k, each <= k_list
 *   ndcg = DCG / IDCG with IDCG = sum_{j < min(n_pos, k)} 1 / log2(j + 2); hit; precision = hits / k;
 *   recall = hits / n_pos; f1 = 2 hits / (k + n_pos).  Users with n_pos == 0 are not counted.
 *   out_metrics [n_users, n_k, 5] f64 (may be NULL; NaN in the rows of users not counted)
 *   out_sums    [n_k, 5] f64, summed in a fixed order as dccf_rank_eval_multi does (may be NULL)
 *   out_count   device int64: the number of users counted (may be NULL)
 *   ws          the workspace of dccf_rank_eval_multi (dccf_rank_eval_ws_bytes, zero on first use); required with
 *               out_sums */
int dccf_topk_metrics(const int64_t* topk_id, int64_t n_users, int32_t k_list, const int64_t* pos_off,
                      const int32_t* pos_items, const int32_t* ks, int32_t n_k, double* out_metrics, void* ws,
                      double* out_sums, int64_t* out_count, void* stream);

/* ---- data-parallel gradient exchange over NVLink peer memory (new: the reference is single-GPU) ----- */
/* Every rank owns a symmetric buffer of floats: [ recv: world*seg | flag area of dccf_dp_flag_floats() words ] mapped on
 * all peers; peer_bases is a HOST array with its device address on each rank.  Flag area: one ARRIVAL flag per (source
 * rank, CTA of its push) + one CONSUMED flag per reader.
 *   dccf_dp_push: stores `send` (seg floats) into slot `rank` of every peer's recv region with 128-bit stores after the
 *                 peers have consumed the previous step; every CTA publishes its own arrival on every peer (a release
 *                 store per peer after the CTA barrier — no grid-wide counter)
 *   dccf_dp_wait: spins until every CTA of every rank's push of the current step has arrived (or fold it into the
 *                 consumer kernel: dccf_dp_sync)
 *   dccf_dp_done: marks this rank's recv region as consumed on every peer and advances epoch_dev (device int32,
 *                 the number of completed exchanges; starts at 0)
 * flag_off: offset of the flag area in floats (>= world*seg, multiple of 4).  cta_counter: unused (kept for ABI). */
int64_t dccf_dp_flag_floats(void);
int dccf_dp_push(const float* send, int64_t seg_floats, const uint64_t* peer_bases, int32_t world, int32_t rank,
                 int64_t flag_off, const int32_t* epoch_dev, int32_t* cta_counter, void* stream);
/* Same as dccf_dp_push, but up to two ranges [off, off + n) (floats) of the segment are not read from `send`: they
 * are the sum over n_parts partial buffers parts[q*stride + .], ascending q — the dW / db row-split partials of the
 * backward folded on the way out (what dccf_sum_parts would do in two extra launches).  Ranges and strides must be
 * multiples of 4 floats, the partial buffers 16-byte aligned; a NULL `parts` skips that range. */
int dccf_dp_push_fold(const float* send, int64_t seg_floats, const uint64_t* peer_bases, int32_t world,
                      int32_t rank, int64_t flag_off, const int32_t* epoch_dev, int32_t* cta_counter,
                      const float* parts_a, int32_t n_parts_a, int64_t stride_a, int64_t off_a, int64_t n_a,
                      const float* parts_b, int32_t n_parts_b, int64_t stride_b, int64_t off_b, int64_t n_b,
                      void* stream);
int dccf_dp_wait(const float* my_base, int64_t seg_floats, int32_t world, int64_t flag_off, const int32_t* epoch_dev,
                 void* stream);
int dccf_dp_done(const uint64_t* peer_bases, int32_t world, int32_t rank, int64_t flag_off, int32_t* epoch_dev,
                 void* stream);

/* ---- full-catalogue scoring (tcgen05 GEMM) -------------------------------------------------- */
/* score[u,i] = ( <A[u,:], B[i,:]> + row_bias[u] + col_bias[i] + g ) * col_scale[i],  A [U,D], B [I,D] f32,
 * 3xTF32 on the tensor cores (FP32-level accuracy).  Replaces IPSBiasedMF.predict over the whole catalogue
 * (src/models/IPSBiasedMF.py:37-57 with col_scale = 1/max(propensity, M); README.md:27-29: that matrix is
 * <ds>.ips_expo_prob.npy) and serves deterministic full-catalogue DCCF scoring.  Bias / scale vectors may be
 * NULL.  Outputs, either or both:
 *   out        [U,I]  the materialised matrix (or NULL)
 *   topk_score [U,k] f32, topk_id [U,k] int64 (-1 padded): fused per-user top-k, score descending, ties by
 *              item id ascending, NaN last; 1 <= k <= 16 (or NULL)
 *   ws_score / ws_id: [dccf_full_scores_splits(U,I), U, k] workspaces of the fused top-k (one partial list per item
 *              split and half of an item tile, merged by a second launch); required with topk_score
 *   ws_items:  dccf_full_scores_ws_floats(n_items) floats, 128-byte aligned: the item side pre-split into the TF32 hi / lo
 *              operand images the tensor cores read (written once per call by k_fs_prep_b, streamed by the GEMM's
 *              CTAs with cp.async.bulk)
 *   excl_off [U+1] int64, excl_items int32: known-item exclusion for the fused top-k, a CSR over the rows of A (each
 *              row's items ascending, unique, < n_items); those items never enter the row's list, and a row with fewer
 *              than k other items is -1 padded.  Both NULL: no exclusion.  Rejected together with `out`.  A list
 *              that is not sorted may fail to exclude some of its items but is never read outside [off[u], off[u+1]). */
int32_t dccf_full_scores_splits(int32_t n_users, int32_t n_items);
int64_t dccf_full_scores_ws_floats(int32_t n_items);
int dccf_full_scores(int32_t n_users, int32_t n_items, const float* A, const float* B, const float* row_bias,
                     const float* col_bias, const float* col_scale, float g, float* out, int32_t k,
                     float* topk_score, int64_t* topk_id, float* ws_score, int64_t* ws_id, float* ws_items,
                     const int64_t* excl_off, const int32_t* excl_items, void* stream);

/* ---- exposure models: BiasedMF / IPSBiasedMF training and scoring ------------------------------- */
/* The model whose U x I prediction is <ds>.ips_expo_prob.npy (README.md:27-29; src/models/IPSBiasedMF.py:37-57):
 *   pred = (<p_u, q_i> + b_u + b_i + g) / max(propensity_i, M)      (BiasedMF: propensity 1, M = 1)
 * One training step is the split optimizer step above with S = 0 (record p = user row and item row of pair p):
 *   dccf_adam_link_ids (CSR counting mode) -> dccf_adam_untouched -> dccf_adam_csr_build -> dccf_mf_step ->
 *   dccf_mf_bias_grad -> dccf_adam_touched(tables: E_user, E_item; dense: user_bias [U], item_bias [I] with one partial
 *   each, global_bias [1] with the dccf_mf_step_ctas(P) CTA partials, part_stride 1).
 * dccf_mf_step: forward, loss and backward of one batch in one launch (loss_mode 0 BPR over [pos ; neg] halves, P even;
 *   1 MSE mean against Y [P]).  global_bias is a DEVICE pointer to the 0-d parameter (graph replay).
 *   out_pred [P]; gu_rec / gi_rec [P, D]: d loss / d p_u, d loss / d q_i of pair p; gb_rec [P]: d loss / d pred / max(prop, M)
 *   (the gradient of b_u, b_i and g from pair p); rec_keys_u / rec_keys_i [P] int32: the rows (out-of-range ids are
 *   clamped to row 0 and raise err_flag, as dccf_adam_link_ids clamps them); g_part / loss_part
 *   [dccf_mf_step_ctas(P)]: per-CTA sums of gb_rec and of the loss terms.
 * dccf_mf_bias_grad: dense d loss / d b_u [U] and d loss / d b_i [I] — the scalar records of each row summed in ascending
 *   record index through the CSR that dccf_adam_csr_build built for `user` / `item` (0 for untouched rows) — and
 *   out_loss[0] = loss_scale * sum of the loss partials in index order.  Between dccf_adam_csr_build and dccf_adam_touched.
 * dccf_mf_scores: out[p] = pred of pair X[p] with the arithmetic of the DCCF kernels' exposure mode 1; factors->
 *   mf_global_bias is ignored, the value is read from global_bias (device). */
int32_t dccf_mf_step_ctas(int64_t n_pairs);
int dccf_mf_step(int32_t n_users, int32_t n_items, const float* E_user, const float* E_item, const float* user_bias,
                 const float* item_bias, const float* global_bias, const float* propensity, float min_propensity,
                 const int64_t* X, const float* Y, int64_t n_pairs, int32_t loss_mode, float* out_pred, float* gu_rec,
                 float* gi_rec, float* gb_rec, int32_t* rec_keys_u, int32_t* rec_keys_i, float* g_part, float* loss_part,
                 int32_t* err_flag, void* stream);
int dccf_mf_bias_grad(const dccf_adam_table* user, const dccf_adam_table* item, const float* gb_rec, float* g_user_bias,
                      float* g_item_bias, const float* loss_part, int32_t n_loss_part, float loss_scale, float* out_loss,
                      void* stream);
int dccf_mf_scores(int32_t n_users, int32_t n_items, const dccf_expo* factors, const float* global_bias, const int64_t* X,
                   int64_t n_pairs, float* out, int32_t* err_flag, void* stream);

/* ---- host side: exact replay of the reference's negative sampler ---------------------------- */
/* Replaces the Python loop of src/data_processor/DataProcessor.py:446-524 draw for draw.  HOST pointers.
 *   mt_key[624], mt_pos: numpy's legacy MT19937 state (np.random.get_state()[1:3]); advanced in place
 *   uids [n]: users in sampling order; neg_n negatives each; train != 0: avoid the train history and the
 *             negatives already drawn for that user in this call; train == 0: avoid train U validation/test
 *             history, per-row draw memory only
 *   *_off [n_users+1], *_items: CSR of sorted, de-duplicated per-user item lists
 *   out_iid [n*neg_n] */
int dccf_sample_negatives(uint32_t* mt_key, int32_t* mt_pos, const int64_t* uids, int64_t n, int32_t neg_n,
                          int32_t train, int64_t item_num, int64_t n_users, const int64_t* train_off,
                          const int64_t* train_items, const int64_t* vt_off, const int64_t* vt_items,
                          int64_t* out_iid);

/* ---- host side: exact replay of the confounder draw ------------------------------------------- */
/* Replaces `torch.randint(item_num, size=(P, S))` of src/models/DCCF.py:72 (torch CPU generator, at::mt19937):
 * out[k] = next_u32 % high for k = 0..n-1, the generator advanced in place exactly as torch would.  HOST pointers.
 *   mt_state[624], *mt_left: words and `left_` counter of at::mt19937 as serialised by torch.get_rng_state()
 *                            (CPUGeneratorImplStateLegacy: `state` at byte 24, one word per uint64; `left` at byte 8)
 *   *mt_next:                receives the matching `next_` index (byte 16 of the same blob)
 *   0 < high < 2^32; torch 2.11 itself takes this 32-bit path only for high < 2^28 (64-bit words above), which is
 *   the range the Python binding routes here (dccf_b200/host_rng.py) */
int dccf_confounder_draw(uint32_t* mt_state, int32_t* mt_left, int32_t* mt_next, int64_t high, int64_t n, int64_t* out);
/* The same stream continued on the device: state_dev = uint32[625] in DEVICE memory (the 624 words + the index of the
 * next unread word, 624 = regenerate first; i.e. 625 - left), advanced in place by one single-CTA kernel per call
 * (three barriers per generation of 624 words); out_dev [n] int64 in device memory — the scorer's sample_item buffer.
 * An evaluation pass uploads torch's generator once and reads it back once. */
int dccf_confounder_draw_dev(uint32_t* state_dev, int64_t high, int64_t n, int64_t* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DCCF_B200_H */
