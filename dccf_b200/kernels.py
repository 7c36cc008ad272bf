"""Tensor-level wrappers over the C-ABI (dccf_b200/_lib.py).  Each function launches hand-written
sm_100a kernels on the current CUDA stream; none has a CPU implementation.
"""
import ctypes

import torch

from . import _lib
from ._lib import Adam, AdamTable, AdamTensor, Dims, DpSync, Expo, LinkExtra, Rng, check, ptr, stream_ptr

D = _lib.DIM

# number of kernels of this library launched so far (bench.py reports it as gpu_launches)
LAUNCHES = [0]


def make_dims(n_users, n_items, feat_dim, n_samples, n_attr, dim=D, user_base=0):
    """n_users = rows of the (local) user table; user_base = first global uid it holds (row-sharded tables)."""
    return Dims(int(n_users), int(n_items), int(dim), int(feat_dim), int(n_samples), int(n_attr), int(user_base), 0)


def make_expo(dense=None, ipsmf=None):
    """Exposure source: a dense [U,I] matrix (src/models/DCCF.py:64) or IPSBiasedMF factors
    (src/models/IPSBiasedMF.py:37-57) as a dict of CUDA tensors + two floats."""
    e = Expo()
    if ipsmf is not None:
        e.mode = 1
        e.mf_user = ptr(ipsmf['mf_user']).value
        e.mf_item = ptr(ipsmf['mf_item']).value
        e.mf_user_bias = ptr(ipsmf['mf_user_bias']).value
        e.mf_item_bias = ptr(ipsmf['mf_item_bias']).value
        e.propensity = ptr(ipsmf['propensity']).value
        e.mf_global_bias = float(ipsmf['mf_global_bias'])
        e.mf_min_propensity = float(ipsmf['mf_min_propensity'])
    else:
        e.mode = 0
        e.dense = ptr(dense).value
    return e


def make_rng(noise=None, mask=None, noise_std=0.0, p_drop=0.0, seed=0, offset=0, offset_dev=None,
             generate_noise=False, generate_mask=False):
    """mode 1 when a tensor is given, mode 2 when generate_* is set, else mode 0 (absent)."""
    r = Rng()
    r.noise_mode = 1 if noise is not None else (2 if generate_noise else 0)
    r.mask_mode = 1 if mask is not None else (2 if generate_mask else 0)
    r.noise = ptr(noise).value if noise is not None else None
    r.mask = ptr(mask).value if mask is not None else None
    r.noise_std = float(noise_std)
    r.p_drop = float(p_drop)
    r.seed = int(seed) & 0xffffffffffffffff
    r.offset = int(offset) & 0xffffffffffffffff
    r.offset_dev = ptr(offset_dev).value if offset_dev is not None else None
    return r


RULE_ADAM, RULE_GD, RULE_ADAGRAD = 0, 1, 2


def make_adam(lr, l2, weight_decay, step=1, step_dev=None, beta1=0.9, beta2=0.999, eps=1e-8, clip=50.0, rule=RULE_ADAM):
    """dccf_adam: hyper-parameters of the optimizer step; rule 0 Adam, 1 GD, 2 Adagrad (include/dccf_b200.h)."""
    a = Adam()
    a.lr, a.beta1, a.beta2, a.eps = float(lr), float(beta1), float(beta2), float(eps)
    a.l2, a.weight_decay, a.clip = float(l2), float(weight_decay), float(clip)
    a.step = int(step)
    a.rule = int(rule)
    a.step_dev = ptr(step_dev).value if step_dev is not None else None
    return a


def noise_fill(out, std, seed, offset, row0=0):
    lib = _lib.load()
    n_rows, F = out.shape
    check(lib.dccf_noise_fill(ptr(out), n_rows, F, float(std), int(seed), int(offset), int(row0), stream_ptr()),
          'dccf_noise_fill')
    LAUNCHES[0] += 1
    return out


def dropout_mask_fill(out, p_drop, seed, offset, row0=0):
    lib = _lib.load()
    n_rows, dim = out.shape
    check(lib.dccf_dropout_mask_fill(ptr(out), n_rows, dim, float(p_drop), int(seed), int(offset), int(row0),
                                     stream_ptr()), 'dccf_dropout_mask_fill')
    LAUNCHES[0] += 1
    return out


def score_fwd(dims, E_user, E_item, Feat, W, b, expo, X, sample_item, rng, out_pred, ws_rows, ws_wt, save_h=None,
              save_w=None, err_flag=None):
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_score_fwd(ctypes.byref(dims), ptr(E_user), ptr(E_item), ptr(Feat), ptr(W), ptr(b),
                             ctypes.byref(expo), ptr(X), ptr(sample_item), n_pairs, ctypes.byref(rng), ptr(out_pred),
                             ptr(ws_rows), ptr(ws_wt), ptr(save_h), ptr(save_w), ptr(err_flag), stream_ptr()),
          'dccf_score_fwd')
    LAUNCHES[0] += 3 if n_pairs > 0 else 0      # k_transpose_w, k_row_scores, k_backdoor
    return out_pred


def tc_operand_floats(feat_dim):
    return int(_lib.load().dccf_tc_operand_floats(int(feat_dim)))


def tc_prepare(dims, E_item, Feat, W, b, ws_wt, PI, PF, gB):
    """Project the item tables and split W_f for the tensor-core scorer (4 launches)."""
    lib = _lib.load()
    check(lib.dccf_tc_prepare(ctypes.byref(dims), ptr(E_item), ptr(Feat), ptr(W), ptr(b), ptr(ws_wt), ptr(PI), ptr(PF),
                              ptr(gB), stream_ptr()), 'dccf_tc_prepare')
    LAUNCHES[0] += 4


def score_fwd_tc(dims, E_user, PI, PF, gB, expo, X, sample_item, rng, out_pred, ws_rows, dbg_pre=None, err_flag=None):
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_score_fwd_tc(ctypes.byref(dims), ptr(E_user), ptr(PI), ptr(PF), ptr(gB), ctypes.byref(expo), ptr(X),
                                ptr(sample_item), n_pairs, ctypes.byref(rng), ptr(out_pred), ptr(ws_rows), ptr(dbg_pre),
                                ptr(err_flag), stream_ptr()), 'dccf_score_fwd_tc')
    LAUNCHES[0] += 2 if n_pairs > 0 else 0      # k_row_scores_tc, k_backdoor
    return out_pred


def score_gather(dims, E_user, PI, PF, expo, X, sample_item, out_pred, err_flag=None):
    """Noise-free scoring from the projected tables (dccf_score_gather): one gather kernel, no workspace."""
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_score_gather(ctypes.byref(dims), ptr(E_user), ptr(PI), ptr(PF), ctypes.byref(expo), ptr(X),
                                ptr(sample_item), n_pairs, ptr(out_pred), ptr(err_flag), stream_ptr()),
          'dccf_score_gather')
    LAUNCHES[0] += 1 if n_pairs > 0 else 0
    return out_pred


def bwd_splits(n_rows):
    return int(_lib.load().dccf_bwd_splits(int(n_rows)))


def bpr_bwd(dims, E_user, E_item, Feat, W, X, sample_item, Y, rng, loss_mode, pred, save_h, save_w, out_loss, gW_part,
            gb_part, gu_rec, gi_rec, rec_keys_u, rec_keys_i):
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_bpr_bwd(ctypes.byref(dims), ptr(E_user), ptr(E_item), ptr(Feat), ptr(W), ptr(X), ptr(sample_item),
                           ptr(Y), n_pairs, ctypes.byref(rng), int(loss_mode), ptr(pred), ptr(save_h), ptr(save_w),
                           ptr(out_loss), ptr(gW_part), ptr(gb_part), ptr(gu_rec), ptr(gi_rec), ptr(rec_keys_u),
                           ptr(rec_keys_i), stream_ptr()), 'dccf_bpr_bwd')
    LAUNCHES[0] += 1 if n_pairs > 0 else 0


def train_w_image_floats(feat_dim):
    return int(_lib.load().dccf_train_w_image_floats(int(feat_dim)))


def train_fwd_ksplits(n_rows, feat_dim):
    return int(_lib.load().dccf_train_fwd_ksplits(int(n_rows), int(feat_dim)))


def train_bwd_splits(n_rows, feat_dim):
    return int(_lib.load().dccf_train_bwd_splits(int(n_rows), int(feat_dim)))


def train_fwd_tc(dims, E_user, E_item, Feat, W, b, expo, X, sample_item, rng, out_pred, ws_rows, ws_wimg, ws_pre_part,
                 save_h, save_w, err_flag=None):
    """Forward of a training step on the tensor cores (3 launches: W operand images, partial products per
    (row tile, K split), per-pair epilogue + backdoor sum)."""
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_train_fwd_tc(ctypes.byref(dims), ptr(E_user), ptr(E_item), ptr(Feat), ptr(W), ptr(b),
                                ctypes.byref(expo), ptr(X), ptr(sample_item), n_pairs, ctypes.byref(rng), ptr(out_pred),
                                ptr(ws_rows), ptr(ws_wimg), ptr(ws_pre_part), ptr(save_h), ptr(save_w), ptr(err_flag),
                                stream_ptr()), 'dccf_train_fwd_tc')
    LAUNCHES[0] += 3 if n_pairs > 0 else 0
    return out_pred


def train_bwd_tc(dims, E_user, E_item, Feat, W, X, sample_item, Y, rng, loss_mode, pred, save_h, save_w, out_loss,
                 gW_part, gb_part, gu_rec, gi_rec, rec_keys_u, rec_keys_i, ws_dpre):
    """Loss + backward of a training step, dW / db on the tensor cores (2 launches)."""
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_train_bwd_tc(ctypes.byref(dims), ptr(E_user), ptr(E_item), ptr(Feat), ptr(W), ptr(X),
                                ptr(sample_item), ptr(Y), n_pairs, ctypes.byref(rng), int(loss_mode), ptr(pred),
                                ptr(save_h), ptr(save_w), ptr(out_loss), ptr(gW_part), ptr(gb_part), ptr(gu_rec),
                                ptr(gi_rec), ptr(rec_keys_u), ptr(rec_keys_i), ptr(ws_dpre), stream_ptr()),
          'dccf_train_bwd_tc')
    LAUNCHES[0] += 2 if n_pairs > 0 else 0


def train_fused_supported(n_samples, n_attr, loss_mode):
    return int(_lib.load().dccf_train_fused_smem_bytes(int(n_samples), int(n_attr), int(loss_mode))) <= 200 * 1024


def train_fwd_bwd_tc(dims, E_user, E_item, Feat, W, b, expo, X, sample_item, Y, rng, loss_mode, out_pred, out_loss,
                     ws_wimg, w_image_valid, ws_pre_part, ws_dpre, ws_loss_terms, gW_part, gb_part, gu_rec, gi_rec,
                     rec_keys_u, rec_keys_i, save_h=None, save_w=None, expo_e=None, expo_den=None, err_flag=None, phases=7,
                     batch=None, mse_pairs=0):
    """Forward + BPR/MSE loss + backward of a training step: partial products, fused per-loss-term middle kernel,
    dW / db tiles (3 launches, 4 when the W operand images must be rebuilt).  batch = (epoch_ptrs_dev, cursor_dev): the
    partial-product kernel takes its ids from the device-resident epoch itself (X / sample_item are then the staged
    copies another launch is writing; the later kernels read those).  phases + 8 / 16 / 32: the partial-product /
    middle / dW kernel starts as a programmatic dependent of the kernel launched before it on the stream (see
    include/dccf_b200.h).  mse_pairs: the pairs the MSE mean is over (0: this call's; world * P data parallel)."""
    lib = _lib.load()
    n_pairs = X.shape[0]
    ref = None
    if batch is not None:
        ref = _lib.BatchRef()
        ref.epoch_ptrs_dev, ref.cursor_dev = ptr(batch[0]).value, ptr(batch[1]).value
    check(lib.dccf_train_fwd_bwd_tc(ctypes.byref(dims), ptr(E_user), ptr(E_item), ptr(Feat), ptr(W), ptr(b),
                                    ctypes.byref(expo), ptr(X), ptr(sample_item), ptr(Y), n_pairs, int(mse_pairs),
                                    ctypes.byref(rng),
                                    int(loss_mode), ptr(out_pred), ptr(out_loss), ptr(ws_wimg), int(bool(w_image_valid)),
                                    ptr(ws_pre_part), ptr(ws_dpre), ptr(ws_loss_terms), ptr(gW_part), ptr(gb_part),
                                    ptr(gu_rec), ptr(gi_rec), ptr(rec_keys_u), ptr(rec_keys_i), ptr(save_h), ptr(save_w),
                                    ptr(expo_e), ptr(expo_den), ctypes.byref(ref) if ref is not None else None, int(phases),
                                    ptr(err_flag), stream_ptr()),
          'dccf_train_fwd_bwd_tc')
    if n_pairs > 0:
        LAUNCHES[0] += ((1 if w_image_valid else 2) if phases & 1 else 0) + (1 if phases & 2 else 0) + (1 if phases & 4 else 0)



def adam_sweep(table, m, v, rec_keys, rec_grads, n_rec, head, nxt, hp):
    lib = _lib.load()
    check(lib.dccf_adam_sweep(ptr(table), ptr(m), ptr(v), table.shape[0], ptr(rec_keys), ptr(rec_grads), int(n_rec),
                              ptr(head), ptr(nxt), ctypes.byref(hp), stream_ptr()), 'dccf_adam_sweep')
    LAUNCHES[0] += 2 if n_rec > 0 else 1        # k_link_records, k_adam_sweep


def adam_sweep_seg(table, m, v, rec_keys, rec_grads, n_seg, seg_len, key_seg_stride, grad_seg_stride, head, nxt, hp):
    """Records in n_seg segments (one per data-parallel rank); strides in elements of the key / gradient arrays."""
    lib = _lib.load()
    check(lib.dccf_adam_sweep_seg(ptr(table), ptr(m), ptr(v), table.shape[0], ptr(rec_keys), ptr(rec_grads),
                                  int(n_seg), int(seg_len), int(key_seg_stride), int(grad_seg_stride), ptr(head),
                                  ptr(nxt), ctypes.byref(hp), stream_ptr()), 'dccf_adam_sweep_seg')
    LAUNCHES[0] += 2 if n_seg * seg_len > 0 else 1


def sum_parts(parts, n_parts, part_stride, n, out):
    lib = _lib.load()
    check(lib.dccf_sum_parts(ptr(parts), int(n_parts), int(part_stride), int(n), ptr(out), stream_ptr()),
          'dccf_sum_parts')
    LAUNCHES[0] += 1


def adam_dense(p, m, v, g_parts, n_parts, part_stride, hp):
    lib = _lib.load()
    check(lib.dccf_adam_dense(ptr(p), ptr(m), ptr(v), p.numel(), ptr(g_parts), int(n_parts), int(part_stride),
                              ctypes.byref(hp), stream_ptr()), 'dccf_adam_dense')
    LAUNCHES[0] += 1


def adam_table(table, m, v, rec_keys, rec_grads, n_seg, seg_len, key_seg_stride, grad_seg_stride, head, nxt, csr=None):
    """m / v: the optimizer rule's state (None where the rule has none).  csr = (rec_row [n_rec], csr_off [n_rows],
    csr [2 * n_rec], csr_pool [2]) int32 tensors: CSR record lists (counting link + dccf_adam_csr_build) instead of
    linked lists."""
    t = AdamTable()
    if csr is not None:
        t.rec_row, t.csr_off, t.csr, t.csr_pool = (ptr(x).value for x in csr)
    t.table = ptr(table).value
    t.m = ptr(m).value if m is not None else None
    t.v = ptr(v).value if v is not None else None
    t.n_rows = table.shape[0]
    t.rec_keys = ptr(rec_keys).value if rec_keys is not None else None
    t.rec_grads = ptr(rec_grads).value if rec_grads is not None else None
    t.n_seg, t.seg_len = int(n_seg), int(seg_len)
    t.key_seg_stride, t.grad_seg_stride = int(key_seg_stride), int(grad_seg_stride)
    t.head = ptr(head).value
    t.next = ptr(nxt).value if nxt is not None else None
    return t


def adam_tensor(p, m, v, g_parts, n_parts, part_stride):
    t = AdamTensor()
    t.p = ptr(p).value
    t.m = ptr(m).value if m is not None else None
    t.v = ptr(v).value if v is not None else None
    t.n = p.numel()
    t.g_parts = ptr(g_parts).value if g_parts is not None else None
    t.n_parts, t.part_stride = int(n_parts), int(part_stride)
    return t


def adam_step(tables, dense, hp):
    """l2 + clip + the optimizer rule of `hp` over every tensor of the model in two launches (dccf_adam_step)."""
    lib = _lib.load()
    ta = (AdamTable * max(1, len(tables)))(*tables)
    da = (AdamTensor * max(1, len(dense)))(*dense)
    check(lib.dccf_adam_step(ta, len(tables), da, len(dense), ctypes.byref(hp), stream_ptr()), 'dccf_adam_step')
    LAUNCHES[0] += 2 if any(t.n_seg * t.seg_len > 0 for t in tables) else 1


DP_SYNC_OVERLAP_PUSH = 1


def make_dp_sync(world, rank, wait=(), done=(), loss=None, flags=0):
    """dccf_dp_sync: `wait` / `done` = exchange channels (objects with peer_bases, flag_off, epoch_dev: the p2p
    SegmentExchange of dccf_b200/dist.py) a consumer kernel waits on in its prologue / hands back from its last CTA;
    loss = (parts tensor, stride in floats, n, out tensor): the ranks' loss terms summed by that last CTA."""
    s = DpSync()
    s.world, s.rank, s.n_wait, s.n_done = int(world), int(rank), len(wait), len(done)
    s.flags = int(flags)
    for arr, chans in ((s.wait, wait), (s.done, done)):
        for k, c in enumerate(chans):
            for p in range(world):
                arr[k].peer_bases[p] = int(c.peer_bases[p])
            arr[k].flag_off = int(c.flag_off)
            arr[k].epoch_dev = ptr(c.epoch_dev).value
            arr[k].seg_floats = int(c.seg)
    if loss is not None:
        parts, stride, n, out = loss
        s.loss_parts, s.loss_stride, s.n_loss, s.loss_out = ptr(parts).value, int(stride), int(n), ptr(out).value
    return s


def adam_csr_build(tables):
    """Record ids grouped by row after a counting link (dccf_adam_csr_build, 2 launches)."""
    lib = _lib.load()
    ta = (AdamTable * max(1, len(tables)))(*tables)
    check(lib.dccf_adam_csr_build(ta, len(tables), stream_ptr()), 'dccf_adam_csr_build')
    LAUNCHES[0] += 2 if any(t.n_seg * t.seg_len > 0 for t in tables) else 0


def make_link_extra(stage=None, prefetch_user=None, prefetch_item=None, prefetch_feat=None, prefetch_dense=None,
                    sync=None, counter=None, rec_rows=None, epoch_global=None):
    """Extras of dccf_adam_link_ids.  stage = (epoch_ptrs_dev, cursor_dev, X_out, si_out, counter[, Y_out]): the batch
    is read from a device-resident epoch (replaces dccf_stage_batch); with Y_out also its labels (epoch_ptrs_dev slot 6).
    prefetch_user / prefetch_item = up to three [rows, D] tensors each (parameter and the optimizer state it has),
    prefetch_feat = Feat, prefetch_dense = up to four tensors: what the step will touch, requested into L2 ahead of its
    use.  epoch_global = (epoch_ptrs_dev, cursor_dev): the
    data-parallel link reads every rank's ids of the current batch from an epoch-wide gather (no per-step id exchange)."""
    e = LinkExtra()
    if stage is not None:
        ep, cur, X_out, si_out, counter = stage[:5]
        e.epoch_ptrs_dev, e.cursor_dev = ptr(ep).value, ptr(cur).value
        e.X_out, e.sample_item_out, e.stage_counter = ptr(X_out).value, ptr(si_out).value, ptr(counter).value
        if len(stage) > 5 and stage[5] is not None:
            e.Y_out = ptr(stage[5]).value
    if epoch_global is not None:        # data-parallel link from the epoch-wide gather of every rank's ids
        ep, cur = epoch_global
        e.epoch_ptrs_dev, e.cursor_dev = ptr(ep).value, ptr(cur).value
    for k, t in enumerate(prefetch_user or ()):
        e.pf_user[k] = ptr(t).value
    for k, t in enumerate(prefetch_item or ()):
        e.pf_item[k] = ptr(t).value
    if prefetch_feat is not None:
        e.pf_feat = ptr(prefetch_feat).value
    for k, t in enumerate(prefetch_dense or ()):
        e.pf_dense[k] = ptr(t).value
        e.pf_dense_bytes[k] = t.numel() * t.element_size()
    if rec_rows is not None:            # counting link (CSR record lists): (rec_row_user, rec_row_item)
        e.rec_row_user, e.rec_row_item = ptr(rec_rows[0]).value, ptr(rec_rows[1]).value
    if sync is not None:                # (data parallel) wait for the ids / hand the id buffer back inside the kernel
        e.sync = ctypes.pointer(sync)
        e._keep_sync = sync
        e.stage_counter = ptr(counter).value
    return e


def adam_link_ids(dims, X, sample_item, head_user, next_user, head_item, next_item, expo=None, expo_e=None,
                  expo_den=None, n_pairs=None, n_seg=1, seg_stride=0, user_seg=-1, X_local=None, si_local=None,
                  extra=None):
    """Record lists of the step from the ids alone (before any gradient exists); with `expo` also the exposure
    softmax of every local pair (expo_e [P, Z], expo_den [P]).  Data parallel: X / sample_item point at segment 0
    of the gathered ids, n_seg segments seg_stride int64 apart.  extra: make_link_extra(...)."""
    lib = _lib.load()
    n_pairs = X.shape[0] if n_pairs is None else int(n_pairs)
    check(lib.dccf_adam_link_ids(ctypes.byref(dims), ptr(X), ptr(sample_item), n_pairs, int(n_seg), int(seg_stride),
                                 int(user_seg), ptr(head_user), ptr(next_user), ptr(head_item), ptr(next_item),
                                 ctypes.byref(expo) if expo is not None else None, ptr(X_local), ptr(si_local),
                                 ptr(expo_e), ptr(expo_den), ctypes.byref(extra) if extra is not None else None,
                                 stream_ptr()), 'dccf_adam_link_ids')
    LAUNCHES[0] += 1 if n_pairs > 0 else 0


def adam_untouched(tables, hp, threads=0):
    """l2 + clip + the optimizer rule over the rows no record of this step refers to (head == -1): one launch, <= 148 CTAs of
    `threads` threads (0 = the library's default)."""
    lib = _lib.load()
    ta = (AdamTable * max(1, len(tables)))(*tables)
    check(lib.dccf_adam_untouched(ta, len(tables), ctypes.byref(hp), int(threads), stream_ptr()), 'dccf_adam_untouched')
    LAUNCHES[0] += 1


def adam_touched(tables, dense, hp, already_linked=False, w_image=None, w_image_tensor=0, w_image_K=0, cta_counter=None,
                 advance_step_dev=None, advance_offset_dev=None, sync=None, advance_cursor_dev=None):
    """The optimizer rule over the touched rows and the dense tensors (one launch, two when the records still need linking).
    sync (make_dp_sync): data-parallel step — wait for the peers' gradient segments in the kernel's prologue, total loss
    and hand-back of the exchange buffers by its last CTA."""
    lib = _lib.load()
    ta = (AdamTable * max(1, len(tables)))(*tables)
    da = (AdamTensor * max(1, len(dense)))(*dense)
    check(lib.dccf_adam_touched(ta, len(tables), da, len(dense), ctypes.byref(hp), int(bool(already_linked)),
                                ptr(w_image), int(w_image_tensor), int(w_image_K), ptr(cta_counter),
                                ptr(advance_step_dev), ptr(advance_offset_dev), ptr(advance_cursor_dev),
                                ctypes.byref(sync) if sync is not None else None, stream_ptr()), 'dccf_adam_touched')
    LAUNCHES[0] += 1 if already_linked or not any(t.n_seg * t.seg_len > 0 for t in tables) else 2


def train_prep_w_image(W, feat_dim, w_image):
    lib = _lib.load()
    check(lib.dccf_train_prep_w_image(ptr(W), int(feat_dim), ptr(w_image), stream_ptr()), 'dccf_train_prep_w_image')
    LAUNCHES[0] += 1


def stage_batch(epoch_ptrs_dev, cursor_dev, n_pairs, n_samples, X_out, si_out, Y_out=None):
    lib = _lib.load()
    check(lib.dccf_stage_batch(ptr(epoch_ptrs_dev), ptr(cursor_dev), int(n_pairs), int(n_samples), ptr(X_out), ptr(si_out),
                               ptr(Y_out), stream_ptr()), 'dccf_stage_batch')
    LAUNCHES[0] += 1


def state_advance(step_dev, offset_dev, offset_inc=1):
    lib = _lib.load()
    check(lib.dccf_state_advance(ptr(step_dev), ptr(offset_dev), int(offset_inc), stream_ptr()), 'dccf_state_advance')
    LAUNCHES[0] += 1


def mf_step_ctas(n_pairs):
    """Number of CTA partials (global_bias gradient, loss) of dccf_mf_step for a batch of n_pairs."""
    return int(_lib.load().dccf_mf_step_ctas(int(n_pairs)))


def mf_step(E_user, E_item, user_bias, item_bias, global_bias, propensity, M, X, Y, loss_mode, out_pred, gu_rec, gi_rec,
            gb_rec, keys_u, keys_i, g_part, loss_part, err_flag=None):
    """Forward, loss and backward of one BiasedMF / IPSBiasedMF batch (dccf_mf_step, one launch)."""
    lib = _lib.load()
    n_pairs = X.shape[0]
    check(lib.dccf_mf_step(E_user.shape[0], E_item.shape[0], ptr(E_user), ptr(E_item), ptr(user_bias), ptr(item_bias),
                           ptr(global_bias), ptr(propensity), float(M), ptr(X), ptr(Y), n_pairs, int(loss_mode),
                           ptr(out_pred), ptr(gu_rec), ptr(gi_rec), ptr(gb_rec), ptr(keys_u), ptr(keys_i), ptr(g_part),
                           ptr(loss_part), ptr(err_flag), stream_ptr()), 'dccf_mf_step')
    LAUNCHES[0] += 1 if n_pairs > 0 else 0


def mf_bias_grad(user_table, item_table, gb_rec, g_user_bias, g_item_bias, loss_part, n_loss_part, loss_scale, out_loss):
    """Dense bias gradients from the CSR record lists of the two embedding tables (AdamTable descriptors) and the loss
    (dccf_mf_bias_grad, one launch)."""
    lib = _lib.load()
    check(lib.dccf_mf_bias_grad(ctypes.byref(user_table), ctypes.byref(item_table), ptr(gb_rec), ptr(g_user_bias),
                                ptr(g_item_bias), ptr(loss_part), int(n_loss_part), float(loss_scale), ptr(out_loss),
                                stream_ptr()), 'dccf_mf_bias_grad')
    LAUNCHES[0] += 1


def mf_scores(factors, global_bias, X, out, err_flag=None):
    """Predictions of the pairs X [P, 2] from IPS-MF factors (make_expo keys; global_bias a device tensor)."""
    lib = _lib.load()
    e = make_expo(ipsmf=dict(factors, mf_global_bias=0.0))
    n_pairs = X.shape[0]
    check(lib.dccf_mf_scores(factors['mf_user'].shape[0], factors['mf_item'].shape[0], ctypes.byref(e), ptr(global_bias),
                             ptr(X), n_pairs, ptr(out), ptr(err_flag), stream_ptr()), 'dccf_mf_scores')
    LAUNCHES[0] += 1 if n_pairs > 0 else 0
    return out


def rank_eval(scores, labels, iids, cand_rows, user_off, k, out_metrics, out_topk_iid=None, out_topk_row=None):
    """One k; cand_rows None = rows already grouped by user (candidate c is row c)."""
    lib = _lib.load()
    n_users = user_off.shape[0] - 1
    check(lib.dccf_rank_eval(ptr(scores), ptr(labels), ptr(iids), ptr(cand_rows), ptr(user_off), n_users, int(k),
                             ptr(out_topk_iid), ptr(out_topk_row), ptr(out_metrics), stream_ptr()), 'dccf_rank_eval')
    LAUNCHES[0] += 1 if n_users > 0 else 0
    return out_metrics


RANK_MAX_NK, RANK_STREAM_MAX_K = 4, 16
_RANK_WS = {}


def rank_workspace(device):
    """Zero-initialised workspace of dccf_rank_eval_multi (partial sums + CTA counter), one per device and stream."""
    key = (torch.device(device).index, torch.cuda.current_stream().cuda_stream)
    ws = _RANK_WS.get(key)
    if ws is None:
        ws = _RANK_WS[key] = torch.zeros(int(_lib.load().dccf_rank_eval_ws_bytes(0)), dtype=torch.uint8, device=device)
    return ws


def rank_eval_multi(scores, labels, iids, cand_rows, user_off, ks, out_metrics=None, out_sums=None, out_topk_iid=None,
                    out_topk_row=None):
    """Every metric at every k of `ks` (ascending, <= 4 values, each <= 16) in one launch: per-user values
    [n_users, n_k, 5] and / or their sums over users [n_k, 5] (dccf_rank_eval_multi)."""
    lib = _lib.load()
    n_users = user_off.shape[0] - 1
    arr = (ctypes.c_int32 * len(ks))(*[int(k) for k in ks])
    ws = rank_workspace(scores.device) if out_sums is not None else None
    check(lib.dccf_rank_eval_multi(ptr(scores), ptr(labels), ptr(iids), ptr(cand_rows), ptr(user_off), n_users, arr,
                                   len(ks), ptr(out_topk_iid), ptr(out_topk_row), ptr(out_metrics), ptr(ws),
                                   ptr(out_sums), stream_ptr()), 'dccf_rank_eval_multi')
    LAUNCHES[0] += 1 if n_users > 0 else 0


_FS_WS = {}


def full_scores(A, B, row_bias=None, col_bias=None, col_scale=None, g=0.0, materialise=True, k=0, exclude=None):
    """Full-catalogue scoring on the tensor cores (dccf_full_scores).  Returns (matrix [U,I] or None,
    topk_score [U,k] or None, topk_id [U,k] or None).  exclude = (off int64 [U+1], items int32) CUDA tensors: each
    row's known items, dropped from its top-k (not with the matrix)."""
    lib = _lib.load()
    U, I = A.shape[0], B.shape[0]
    dev = A.device
    out = torch.empty((U, I), dtype=torch.float32, device=dev) if materialise else None
    ts = ti = ws = wi = None
    if k > 0:
        ts = torch.empty((U, k), dtype=torch.float32, device=dev)
        ti = torch.empty((U, k), dtype=torch.int64, device=dev)
        lists = int(lib.dccf_full_scores_splits(U, I))
        ws = torch.empty((lists, U, k), dtype=torch.float32, device=dev)
        wi = torch.empty((lists, U, k), dtype=torch.int64, device=dev)
    # pre-split operand images of the item side: one workspace per (device, catalogue size), rewritten by every call
    key = (dev.index, I)
    items = _FS_WS.get(key)
    if items is None:
        items = _FS_WS[key] = torch.empty(int(lib.dccf_full_scores_ws_floats(I)), dtype=torch.float32, device=dev)
    eo, ei = exclude if exclude is not None else (None, None)
    if ei is not None and ei.numel() == 0:      # no listed item anywhere: a valid address that is never read
        ei = torch.zeros(1, dtype=torch.int32, device=dev)
    check(lib.dccf_full_scores(U, I, ptr(A), ptr(B), ptr(row_bias), ptr(col_bias), ptr(col_scale), float(g), ptr(out),
                               int(k), ptr(ts), ptr(ti), ptr(ws), ptr(wi), ptr(items), ptr(eo), ptr(ei), stream_ptr()),
          'dccf_full_scores')
    LAUNCHES[0] += 3 if k > 0 else 2
    return out, ts, ti


def topk_metrics(topk_id, pos_off, pos_items, ks, out_metrics=None, out_sums=None, out_count=None):
    """Every metric at every k of `ks` (ascending, <= 4 values, each <= the list length) of ranked top-k lists against
    each user's sorted positives (dccf_topk_metrics, one launch): per-user values [n_users, n_k, 5], their sums over the
    users with a positive [n_k, 5] and / or the number of those users (int64 [1])."""
    lib = _lib.load()
    n_users, k_list = topk_id.shape
    arr = (ctypes.c_int32 * len(ks))(*[int(k) for k in ks])
    ws = rank_workspace(topk_id.device) if out_sums is not None else None
    check(lib.dccf_topk_metrics(ptr(topk_id), int(n_users), int(k_list), ptr(pos_off), ptr(pos_items), arr, len(ks),
                                ptr(out_metrics), ptr(ws), ptr(out_sums), ptr(out_count), stream_ptr()),
          'dccf_topk_metrics')
    LAUNCHES[0] += 1 if n_users > 0 else 0


def dp_push(send, seg, peer_bases, world, rank, flag_off, epoch_dev, cta_counter):
    """Store this rank's gradient segment into every peer's receive buffer (NVLink P2P stores)."""
    lib = _lib.load()
    arr = (ctypes.c_uint64 * world)(*[int(b) for b in peer_bases])
    check(lib.dccf_dp_push(ptr(send), int(seg), arr, int(world), int(rank), int(flag_off), ptr(epoch_dev),
                           ptr(cta_counter), stream_ptr()), 'dccf_dp_push')
    LAUNCHES[0] += 1


def dp_push_fold(send, seg, peer_bases, world, rank, flag_off, epoch_dev, cta_counter, folds):
    """dp_push with up to two ranges of the segment summed on the fly from partial buffers:
    folds = [(parts, n_parts, stride, offset, n), ...]."""
    lib = _lib.load()
    arr = (ctypes.c_uint64 * world)(*[int(b) for b in peer_bases])
    f = list(folds) + [(None, 0, 0, 0, 0)] * (2 - len(folds))
    check(lib.dccf_dp_push_fold(ptr(send), int(seg), arr, int(world), int(rank), int(flag_off), ptr(epoch_dev),
                                ptr(cta_counter), ptr(f[0][0]), int(f[0][1]), int(f[0][2]), int(f[0][3]), int(f[0][4]),
                                ptr(f[1][0]), int(f[1][1]), int(f[1][2]), int(f[1][3]), int(f[1][4]), stream_ptr()),
          'dccf_dp_push_fold')
    LAUNCHES[0] += 1


def dp_flag_floats():
    return int(_lib.load().dccf_dp_flag_floats())


def dp_wait(my_buf, seg, world, flag_off, epoch_dev):
    lib = _lib.load()
    check(lib.dccf_dp_wait(ptr(my_buf), int(seg), int(world), int(flag_off), ptr(epoch_dev), stream_ptr()), 'dccf_dp_wait')
    LAUNCHES[0] += 1


def dp_done(peer_bases, world, rank, flag_off, epoch_dev):
    lib = _lib.load()
    arr = (ctypes.c_uint64 * world)(*[int(b) for b in peer_bases])
    check(lib.dccf_dp_done(arr, int(world), int(rank), int(flag_off), ptr(epoch_dev), stream_ptr()), 'dccf_dp_done')
    LAUNCHES[0] += 1
