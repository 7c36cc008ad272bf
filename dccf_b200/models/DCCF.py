"""DCCF with the reference's model protocol (src/models/DCCF.py:14-127) on hand-written sm_100a kernels.

`predict` / `forward` keep the reference's feed_dict contract and outputs.  The device work of
DCCF.predict lines 74-100 (index expansion, three gathers, noise, cat, Linear+ReLU+Dropout, dot,
exposure softmax, backdoor sum) is one call of dccf_score_fwd; the backward of the whole graph is one
call of dccf_bpr_bwd; l2 + clip + Adam is dccf_adam_sweep / dccf_adam_dense.  Two ways to train:

  * `train_step(feed_dict, ...)` — the fused path used by dccf_b200's BaseRunner (no autograd at all);
  * `forward(feed_dict)` under autograd — the prediction is a torch.autograd.Function whose backward
    calls the same CUDA kernel, so an unmodified reference-style runner (loss.backward(), any torch
    optimizer) also works.

Random inputs.  The reference draws confounder items on the torch CPU generator (DCCF.py:72), noise
and dropout on the CUDA generator (DCCF.py:87,94).  Here: confounders are drawn by the same
`torch.randint` call on the CPU generator (bit-identical indices); noise and dropout come from the
library's counter-based Philox stream generated inside the kernels (seed = random_seed, one counter
per predict call) unless the feed_dict carries explicit tensors under 'sample_item', 'noise',
'dropout_mask' — that is how the parity tests inject the reference's own draws.

There is no CPU implementation: calling predict without CUDA raises.
"""
import os

import numpy as np
import torch

from .. import host_rng, kernels
from .DMF import DMF


class FusedAdamState(object):
    """Optimizer state of the fused path: the rule's state per parameter, step count, and the persistent per-row
    list heads of the gradient-record scatter.  Stands where the reference keeps its torch optimizer in
    `model.optimizer` (src/runners/BaseRunner.py:83-107,168-169).  kind: 'adam' (exp_avg / exp_avg_sq), 'gd'
    (torch.optim.SGD without momentum: no state) or 'adagrad' (state_sum); eps defaults to torch's value per kind."""

    RULES = {'adam': kernels.RULE_ADAM, 'gd': kernels.RULE_GD, 'adagrad': kernels.RULE_ADAGRAD}

    def __init__(self, model, lr, l2, weight_decay, kind='adam', beta1=0.9, beta2=0.999, eps=None, clip=50.0):
        if kind not in self.RULES:
            raise ValueError('unknown fused optimizer %r (adam, gd, adagrad)' % (kind,))
        self.kind, self.rule = kind, self.RULES[kind]
        self.lr, self.l2, self.weight_decay = lr, l2, weight_decay
        self.beta1, self.beta2, self.clip = beta1, beta2, clip
        self.eps = eps if eps is not None else (1e-10 if kind == 'adagrad' else 1e-8)
        self.step_count = 0
        self.params = {'E_user': model.uid_embeddings.weight, 'E_item': model.iid_embeddings.weight,
                       'W': model.mlp[0].weight, 'b': model.mlp[0].bias}
        if kind == 'adam':
            self.exp_avg = {k: torch.zeros_like(p.data) for k, p in self.params.items()}
            self.exp_avg_sq = {k: torch.zeros_like(p.data) for k, p in self.params.items()}
        elif kind == 'adagrad':
            self.state_sum = {k: torch.zeros_like(p.data) for k, p in self.params.items()}
        dev = model.uid_embeddings.weight.device
        self.head_u = torch.full((model.uid_embeddings.weight.shape[0],), -1, dtype=torch.int32, device=dev)
        self.head_i = torch.full((model.item_num,), -1, dtype=torch.int32, device=dev)

    def _state_names(self):
        return {'adam': ('exp_avg', 'exp_avg_sq'), 'gd': (), 'adagrad': ('state_sum',)}[self.kind]

    def state_of(self, k):
        """(m, v) of parameter k as the kernels take them (dccf_adam_table / _tensor), None where the rule has none."""
        if self.kind == 'adam':
            return self.exp_avg[k], self.exp_avg_sq[k]
        if self.kind == 'adagrad':
            return self.state_sum[k], None
        return None, None

    def hp(self, step=None, step_dev=None):
        return kernels.make_adam(self.lr, self.l2, self.weight_decay, step=self.step_count if step is None else step,
                                 step_dev=step_dev, beta1=self.beta1, beta2=self.beta2, eps=self.eps, clip=self.clip,
                                 rule=self.rule)

    def zero_grad(self):
        pass

    def state_dict(self):
        sd = {'step': self.step_count, 'kind': self.kind, 'lr': self.lr, 'l2': self.l2,
              'weight_decay': self.weight_decay}
        for n in self._state_names():
            sd[n] = getattr(self, n)
        return sd

    def load_state_dict(self, sd):
        """Resume: state and step count of a saved run (SURVEY.md §8f-4; the reference resumes weights only)."""
        kind = sd.get('kind', 'adam')
        if kind != self.kind:
            raise ValueError('cannot load the state of a fused %s optimizer into a fused %s optimizer' % (kind, self.kind))
        for n in self._state_names():
            for k, t in getattr(self, n).items():
                t.copy_(sd[n][k])
        self.step_count = int(sd['step'])
        self.lr, self.l2, self.weight_decay = sd['lr'], sd['l2'], sd['weight_decay']


class _ScoreFn(torch.autograd.Function):
    """pred = DCCF score; backward through dccf_bpr_bwd with the upstream gradient (loss_mode 2)."""

    @staticmethod
    def forward(ctx, E_user, E_item, W, b, model, call):
        pred = model._launch_fwd(call, save=True)
        ctx.model, ctx.call = model, call
        return pred

    @staticmethod
    def backward(ctx, dpred):
        model, call = ctx.model, ctx.call
        rec = model._launch_bwd(call, loss_mode=2, Y=dpred.contiguous().float())
        gE_user = torch.zeros_like(model.uid_embeddings.weight)
        gE_item = torch.zeros_like(model.iid_embeddings.weight)
        gE_user.index_add_(0, rec['keys_u'].long(), rec['gu_rec'])
        gE_item.index_add_(0, rec['keys_i'].long(), rec['gi_rec'])
        gW = rec['gW_part'].sum(dim=0)
        gb = rec['gb_part'].sum(dim=0)
        return gE_user, gE_item, gW, gb, None, None


class DCCF(DMF):
    @staticmethod
    def parse_model_args(parser, model_name='DCCF'):
        """Flags and defaults of DCCF.py:15-21 (note the dashes)."""
        parser.add_argument('--sentence-model', type=str, default='paraphrase-distilroberta-base-v1',
                            help='the name of sentence model')
        parser.add_argument('--sample-num', type=int, default=10, help='the number of sampled items')
        parser.add_argument('--attribute-num', type=int, default=2, help='the number of item features')
        parser.add_argument('--std', type=float, default=0.1, help='std of feature distribution')
        return DMF.parse_model_args(parser, model_name)

    def __init__(self, path, dataset, sentence_model, sample_num, attribute_num, std, label_min, label_max,
                 feature_num, user_num, item_num, u_vector_size, i_vector_size, n_layers, random_seed, model_path,
                 feature_embedding=None, expo_prob=None, expo_factors=None, user_shard=None):
        """Reference constructor arguments (src/main.py:137-145).  The three trailing keyword arguments
        are additions: in-memory tables instead of the .npy files, and IPSBiasedMF factors for
        on-the-fly exposure (scaled config) instead of the dense user x item matrix."""
        self.path = path
        self.dataset = dataset
        self.sentence_model = sentence_model
        self.sample_num = sample_num
        self.attribute_num = attribute_num
        self.std = std
        self._given = (feature_embedding, expo_prob, expo_factors)
        # row-sharded user table (scaled config, SURVEY.md §8e): this rank owns global users [lo, hi); the
        # embedding, its Adam state, the exposure rows / IPS-MF user factors hold only those rows and every
        # batch it is given must contain only those users
        self.user_shard = None if user_shard is None else (int(user_shard[0]), int(user_shard[1]))
        if int(n_layers) != 1:
            # src/models/DCCF.py:58-60 sizes extra Linear(64 -> 64) layers from --n_layers (default 1, the value of the
            # reference's README run): the fused kernels implement the single Linear(D + F -> D) predictor only
            raise ValueError('--n_layers %d: the B200 DCCF kernels implement the reference default --n_layers 1 (one '
                             'Linear(64 + F -> 64) + ReLU + Dropout); other depths are not supported' % int(n_layers))
        DMF.__init__(self, label_min=label_min, label_max=label_max, feature_num=feature_num, user_num=user_num,
                     item_num=item_num, u_vector_size=u_vector_size, i_vector_size=i_vector_size, n_layers=n_layers,
                     random_seed=random_seed, model_path=model_path)
        self._rng_offset = 0
        self._ws = {}
        self._err_flag = None
        self._dp = None
        self._param_epoch = 0          # bumped whenever the fused kernels change the parameters in place
        self._tc_cache = None

    # ---- construction ------------------------------------------------------------------------
    @staticmethod
    def _table_device():
        return torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else torch.device('cpu')

    def _init_weights(self):
        """Same modules in the same order as DCCF.py:47-64, so the torch CPU generator is consumed
        identically and `apply(init_paras)` yields the reference's initial weights for a given seed."""
        feature_embedding, expo_prob, expo_factors = self._given
        dev = self._table_device()
        lo, hi = self.user_shard if self.user_shard is not None else (0, self.user_num)
        self.uid_embeddings = torch.nn.Embedding(hi - lo, self.ui_vector_size)
        self.iid_embeddings = torch.nn.Embedding(self.item_num, self.ui_vector_size)
        if feature_embedding is None:
            feature_embedding = np.load(os.path.join(self.path, self.dataset + '_' + self.sentence_model + '.npy'))
        # plain attributes, not parameters/buffers: absent from state_dict like in the reference (DCCF.py:55,64)
        self.feature_embedding = torch.as_tensor(feature_embedding, dtype=torch.float32).to(dev).contiguous()
        self.mlp = torch.nn.ModuleList([torch.nn.Linear(self.ui_vector_size + self.feature_embedding.shape[1],
                                                        self.ui_vector_size)])
        for _ in range(self.n_layers - 1):
            self.mlp.append(torch.nn.Linear(self.ui_vector_size, self.ui_vector_size))
        self.expo_factors = None
        self.expo_prob = None
        def local_rows(t):      # a per-user array given for ALL users is cut down to this rank's rows
            return t[lo:hi] if (self.user_shard is not None and t.shape[0] == self.user_num) else t

        if expo_factors is not None:
            self.expo_factors = {}
            for k, v in expo_factors.items():
                if k in ('mf_global_bias', 'mf_min_propensity'):
                    self.expo_factors[k] = float(v)
                else:
                    v = torch.as_tensor(v, dtype=torch.float32)
                    if k in ('mf_user', 'mf_user_bias'):
                        v = local_rows(v)
                    self.expo_factors[k] = v.to(dev).contiguous()
        else:
            if expo_prob is None:
                expo_prob = np.load(os.path.join(self.path, self.dataset + '.ips_expo_prob.npy'), mmap_mode='r')
            expo_prob = local_rows(expo_prob)
            if not torch.is_tensor(expo_prob):
                expo_prob = torch.from_numpy(np.ascontiguousarray(expo_prob, dtype=np.float32))
            self.expo_prob = expo_prob.to(dev, torch.float32).contiguous()

    # ---- kernel plumbing ---------------------------------------------------------------------
    def _dims(self):
        lo = self.user_shard[0] if self.user_shard is not None else 0
        return kernels.make_dims(self.uid_embeddings.weight.shape[0], self.item_num, self.feature_embedding.shape[1],
                                 self.sample_num, self.attribute_num, dim=self.ui_vector_size, user_base=lo)

    def _expo(self):
        if self.expo_factors is not None:
            return kernels.make_expo(ipsmf=self.expo_factors)
        return kernels.make_expo(dense=self.expo_prob)

    def _buf(self, name, shape, dtype):
        """Grow-only workspace tensor on the parameters' device."""
        n = 1
        for s in shape:
            n *= int(s)
        cur = self._ws.get(name)
        if cur is None or cur.numel() < n or cur.dtype != dtype:
            cur = torch.empty(max(n, 1), dtype=dtype, device=self.uid_embeddings.weight.device)
            self._ws[name] = cur
        return cur[:n].view(*shape) if n > 0 else cur[:0].view(*shape)

    def _check_ready(self):
        w = self.uid_embeddings.weight
        if not w.is_cuda:
            raise RuntimeError('DCCF (dccf_b200) runs on CUDA only: move the model with .cuda() on a B200; there is no '
                               'CPU fallback')
        if w.device.index is not None and w.device.index != torch.cuda.current_device():
            # launches go to the current device's stream (dccf_b200/_lib.py: stream_ptr)
            raise RuntimeError('the model lives on %s but the current CUDA device is %d: call torch.cuda.set_device(%d) '
                               '(one process per GPU)' % (w.device, torch.cuda.current_device(), w.device.index))
        if self.ui_vector_size != kernels.D:
            raise NotImplementedError('the kernels are compiled for u_vector_size = i_vector_size = %d' % kernels.D)
        if self.feature_embedding.device != w.device:
            self.feature_embedding = self.feature_embedding.to(w.device)
            if self.expo_prob is not None:
                self.expo_prob = self.expo_prob.to(w.device)
            if self.expo_factors is not None:
                self.expo_factors = {k: (v.to(w.device) if torch.is_tensor(v) else v)
                                     for k, v in self.expo_factors.items()}
        if self._err_flag is None or self._err_flag.device != w.device:
            self._err_flag = torch.zeros(1, dtype=torch.int32, device=w.device)

    def _make_call(self, feed_dict):
        """Resolve the inputs of one predict call: ids, confounder draw, rng modes."""
        self._check_ready()
        dev = self.uid_embeddings.weight.device
        X = feed_dict['X']
        if not torch.is_tensor(X):
            X = torch.as_tensor(np.asarray(X))
        X = X.to(dev, torch.int64)
        if X.dim() != 2 or X.shape[1] < 2:
            raise ValueError("feed_dict['X'] must be [P, >=2] with uid in column 0 and iid in column 1")
        if X.shape[1] != 2 or not X.is_contiguous():
            X = X[:, :2].contiguous()
        P = X.shape[0]
        S, A = self.sample_num, self.attribute_num
        sample_item = feed_dict.get('sample_item')
        if sample_item is None:
            # DCCF.py:72 — same call on the same (CPU) generator as the reference
            sample_item = torch.randint(self.item_num, size=(P, S))
        sample_item = sample_item.to(dev, torch.int64, non_blocking=True).contiguous()
        p_drop = float(feed_dict.get('dropout', 0.0))
        noise, mask = feed_dict.get('noise'), feed_dict.get('dropout_mask')
        if noise is not None:
            noise = noise.to(dev, torch.float32).contiguous()
        if mask is not None:
            mask = mask.to(dev, torch.float32).contiguous()
        self._rng_offset += 1
        seed = self.random_seed
        if self._dp is not None:                       # decorrelate the ranks' noise / dropout streams
            seed = (seed + 0x9E3779B97F4A7C15 * self._dp['rank']) & 0xffffffffffffffff
        rng = kernels.make_rng(noise=noise, mask=mask, noise_std=self.std, p_drop=p_drop, seed=seed,
                               offset=self._rng_offset, generate_noise=(noise is None and self.std > 0),
                               generate_mask=(mask is None and p_drop > 0))
        return {'X': X, 'sample_item': sample_item, 'rng': rng, 'noise': noise, 'mask': mask, 'P': P,
                'N': P * (S + 1) * A, 'force_tc': feed_dict.get('force_tc'), 'dbg_pre': feed_dict.get('dbg_pre')}

    # evaluation batches with feature noise go to the tcgen05 scorer (dccf_score_fwd_tc) when they are large
    # enough to fill the machine; training steps and noise-free scoring use the FP32 SIMT kernels
    use_tensor_cores = True
    # training steps: both large contractions (forward W·x, backward dW = dpre^T·x) on the tensor cores, spread over
    # all SMs by (row tile, K split) / (column tile, row split) — dccf_train_fwd_tc / dccf_train_bwd_tc.  False:
    # the FP32 SIMT kernels (k_row_scores_splitk, k_bpr_bwd), kept as the cross-check of the tensor-core path.
    use_tensor_cores_train = True
    # forward + loss + backward as dccf_train_fwd_bwd_tc (one fused kernel between the two contractions)
    use_fused_step = True
    tc_min_rows = 128 * 148
    # noise-free inference (--std 0, dropout 0, no explicit noise / mask) as a pure gather over the projected item
    # tables (dccf_score_gather) instead of the K = D + F contraction: 1.9e-7 from the general FP32 scorer and green
    # against the reference fixture on a B200 (tests/test_gpu_zz_gather.py, round-1 driver run).  On by default;
    # DCCF_GATHER=0 falls back to the general scorer (the cross-check).
    use_gather_scorer = os.environ.get('DCCF_GATHER', '1') != '0'
    # How inference draws the feature noise the library generates itself (--std > 0, no explicit noise tensor):
    #   'exact'     eps ~ N(0, std^2 I_F) per predictor row, multiplied into W_f — the reference's formulation
    #               (src/models/DCCF.py:87-92), F normals per row;
    #   'projected' the only thing the predictor sees of eps is W_f·eps ~ N(0, std^2 W_f W_f^T): draw g ~ N(0, std^2 I_D)
    #               and multiply by a D x D factor M with M M^T = W_f W_f^T.  Identically distributed predictions from
    #               D = 64 instead of F = 768 normals per row, through the same tcgen05 kernel with a D-wide operand.
    # Explicit noise tensors (the parity path) always take the exact formulation.  Default 'exact'; 'projected' is
    # opt-in (also: DCCF_EVAL_NOISE=projected) and was first run on hardware by the round-end run of round 1.
    eval_noise = os.environ.get('DCCF_EVAL_NOISE', 'exact')
    # predict_many: draw the confounders of an evaluation pass on the device (k_confounder_draw continues torch's CPU
    # generator there; bit-identical ids, no per-batch host draw or host->device copy).  Opt-in until seen on hardware.
    device_confounders = os.environ.get('DCCF_DEVICE_DRAW', '0') != '0'

    def _tc_tables(self):
        """PI = E_item·W_i^T, PF = Feat·W_f^T + b and the split W_f operand, rebuilt when a parameter changed."""
        W, b, ei = self.mlp[0].weight, self.mlp[0].bias, self.iid_embeddings.weight
        key = (self._param_epoch, W._version, b._version, ei._version, W.data_ptr(), ei.data_ptr(),
               self.feature_embedding.data_ptr())
        if self._tc_cache is not None and self._tc_cache['key'] == key:
            return self._tc_cache
        D, F = self.ui_vector_size, self.feature_embedding.shape[1]
        dev = W.device
        c = self._tc_cache or {}
        if c.get('PI') is None or c['PI'].shape[0] != self.item_num:
            c = {'PI': torch.empty((self.item_num, D), dtype=torch.float32, device=dev),
                 'PF': torch.empty((self.item_num, D), dtype=torch.float32, device=dev),
                 'gB': torch.empty(kernels.tc_operand_floats(F), dtype=torch.float32, device=dev)}
        kernels.tc_prepare(self._dims(), ei.data, self.feature_embedding, W.data, b.data,
                           self._buf('ws_wt', ((D + F) * D,), torch.float32), c['PI'], c['PF'], c['gB'])
        c['key'] = key
        self._tc_cache = c
        return c

    def projection_factor(self):
        """M [D, D] (float64, CPU) with M·M^T = W_f·W_f^T, from the symmetric eigendecomposition (any rank):
        W_f·eps with eps ~ N(0, std^2 I_F) and M·g with g ~ N(0, std^2 I_D) have the same distribution."""
        D = self.ui_vector_size
        Wf = self.mlp[0].weight.detach()[:, D:].to('cpu', torch.float64)
        lam, V = torch.linalg.eigh(Wf @ Wf.T)
        return V * lam.clamp_min(0.0).sqrt()

    def _projected_operand(self, t):
        """The tensor-core operand image of M (in place of W_f) for the current parameters, cached with the tables."""
        if t.get('gBp_key') == t['key']:
            return t['gBp']
        D = self.ui_vector_size
        dev = self.mlp[0].weight.device
        Wfake = torch.zeros((D, 2 * D), dtype=torch.float32)
        Wfake[:, D:] = self.projection_factor().to(torch.float32)
        Wfake = Wfake.to(dev)
        if t.get('gBp') is None:
            t['gBp'] = torch.empty(kernels.tc_operand_floats(D), dtype=torch.float32, device=dev)
        # dccf_tc_prepare on a stand-in problem with F = D and 8 zero items: only its split of "W_f" (= M) is kept
        z = torch.zeros((8, D), dtype=torch.float32, device=dev)
        kernels.tc_prepare(kernels.make_dims(8, 8, D, 0, 1, dim=D), z, z, Wfake, torch.zeros(D, device=dev),
                           torch.empty(2 * D * D, dtype=torch.float32, device=dev), torch.empty_like(z),
                           torch.empty_like(z), t['gBp'])
        t['gBp_key'] = t['key']
        return t['gBp']

    def _launch_fwd(self, call, save):
        P, N = call['P'], call['N']
        D, Z = self.ui_vector_size, self.sample_num + 1
        K = D + self.feature_embedding.shape[1]
        dev = self.uid_embeddings.weight.device
        pred = torch.empty(P, dtype=torch.float32, device=dev)
        if P == 0:
            return pred
        if not save and self.use_gather_scorer and call['rng'].noise_mode == 0 and call['rng'].mask_mode == 0:
            t = self._tc_tables()
            kernels.score_gather(self._dims(), self.uid_embeddings.weight.data, t['PI'], t['PF'], self._expo(),
                                 call['X'], call['sample_item'], pred, self._err_flag)
            call['pred'] = pred
            return pred
        ws_rows = self._buf('ws_rows', (N,), torch.float32)
        if not save and self.use_tensor_cores and call['rng'].noise_mode != 0 and \
                (N >= self.tc_min_rows or call.get('force_tc')):
            t = self._tc_tables()
            dbg = call.get('dbg_pre')
            dims, gB = self._dims(), t['gB']
            if self.eval_noise == 'projected' and call['rng'].noise_mode == 2:
                gB = self._projected_operand(t)             # M in place of W_f, D normals per row in place of F
                dims.feat_dim = D
            kernels.score_fwd_tc(dims, self.uid_embeddings.weight.data, t['PI'], t['PF'], gB, self._expo(),
                                 call['X'], call['sample_item'], call['rng'], pred, ws_rows, dbg, self._err_flag)
            call['pred'] = pred
            return pred
        ws_wt = self._buf('ws_wt', (K * D,), torch.float32)
        save_h = save_w = None
        if save:
            call['save_h'] = save_h = torch.empty((N, D), dtype=torch.float32, device=dev)
            call['save_w'] = save_w = torch.empty((P, Z), dtype=torch.float32, device=dev)
            if self.use_tensor_cores and self.use_tensor_cores_train:
                F = K - D
                n_ks = kernels.train_fwd_ksplits(N, F)
                kernels.train_fwd_tc(
                    self._dims(), self.uid_embeddings.weight.data, self.iid_embeddings.weight.data,
                    self.feature_embedding, self.mlp[0].weight.data, self.mlp[0].bias.data, self._expo(), call['X'],
                    call['sample_item'], call['rng'], pred, ws_rows,
                    self._buf('ws_wimg', (kernels.train_w_image_floats(F),), torch.float32),
                    self._buf('ws_pre_part', (n_ks, N, D), torch.float32), save_h, save_w, self._err_flag)
                call['pred'] = pred
                call['tc_train'] = True
                return pred
        kernels.score_fwd(self._dims(), self.uid_embeddings.weight.data, self.iid_embeddings.weight.data,
                          self.feature_embedding, self.mlp[0].weight.data, self.mlp[0].bias.data, self._expo(),
                          call['X'], call['sample_item'], call['rng'], pred, ws_rows, ws_wt, save_h, save_w,
                          self._err_flag)
        call['pred'] = pred
        return pred

    def _rec_buffers(self, call, loss_mode, n_splits):
        """Outputs of the backward: row-split partials of dW / db, gradient records + keys, loss.  Under data
        parallelism the records, keys and loss live directly in the rank's send segment."""
        P = call['P']
        D, Z = self.ui_vector_size, self.sample_num + 1
        K = D + self.feature_embedding.shape[1]
        rec = {
            'gW_part': self._buf('gW_part', (n_splits, D, K), torch.float32),
            'gb_part': self._buf('gb_part', (n_splits, D), torch.float32),
            'n_splits': n_splits,
        }
        if self._dp is not None and loss_mode != 2:
            ex = self._exchange_for(P)
            v = ex.send_views()
            rec.update({'gu_rec': v['gu_rec'], 'gi_rec': v['gi_rec'], 'keys_u': v['keys_u'], 'keys_i': v['keys_i'],
                        'loss': v['loss'], 'exchange': ex, 'send': v})
            if not ex.user_records:      # row-sharded user table: user-row gradients stay on this rank
                rec['gu_rec'] = self._buf('gu_rec', (P, D), torch.float32)
                rec['keys_u'] = self._buf('keys_u', (P,), torch.int32)
        else:
            rec.update({'gu_rec': self._buf('gu_rec', (P, D), torch.float32),
                        'gi_rec': self._buf('gi_rec', (P * Z, D), torch.float32),
                        'keys_u': self._buf('keys_u', (P,), torch.int32),
                        'keys_i': self._buf('keys_i', (P * Z,), torch.int32),
                        'loss': self._buf('loss', (1,), torch.float32)})
        return rec

    def _launch_bwd(self, call, loss_mode, Y):
        if loss_mode == 1 and self._dp is not None:
            # this backward divides by the local batch: a data-parallel MSE step takes the fused step's global divisor
            raise RuntimeError('data-parallel --rank 0 training needs the fused step (dccf_train_fwd_bwd_tc)')
        N = call['N']
        D = self.ui_vector_size
        F = self.feature_embedding.shape[1]
        tc = bool(call.get('tc_train'))
        rec = self._rec_buffers(call, loss_mode, kernels.train_bwd_splits(N, F) if tc else kernels.bwd_splits(N))
        args = (self._dims(), self.uid_embeddings.weight.data, self.iid_embeddings.weight.data,
                self.feature_embedding, self.mlp[0].weight.data, call['X'], call['sample_item'], Y,
                call['rng'], loss_mode, call['pred'], call['save_h'], call['save_w'], rec['loss'],
                rec['gW_part'], rec['gb_part'], rec['gu_rec'], rec['gi_rec'], rec['keys_u'], rec['keys_i'])
        if tc:
            kernels.train_bwd_tc(*args, self._buf('ws_dpre', (N, D), torch.float32))
        else:
            kernels.bpr_bwd(*args)
        return rec

    def _fused_step_ok(self, loss_mode):
        return self.use_tensor_cores and self.use_tensor_cores_train and self.use_fused_step and \
            loss_mode in (0, 1) and kernels.train_fused_supported(self.sample_num, self.attribute_num, loss_mode)

    def _launch_fwd_bwd(self, call, loss_mode, Y, rec=None, w_image_valid=False, expo_e=None, expo_den=None,
                        between=None, batch=None, programmatic=False):
        """Forward + loss + backward of one step through dccf_train_fwd_bwd_tc (three launches; the activations
        never leave shared memory).  Data parallel, the MSE mean is over the global batch of world * P pairs: the ranks'
        gradients and loss terms then sum to those of one GPU on the concatenated batch.  Returns (prediction, gradient
        buffers)."""
        P, N = call['P'], call['N']
        D = self.ui_vector_size
        F = self.feature_embedding.shape[1]
        dev = self.uid_embeddings.weight.device
        pred = torch.empty(P, dtype=torch.float32, device=dev)
        if rec is None:
            rec = self._rec_buffers(call, loss_mode, kernels.train_bwd_splits(N, F))
        if P == 0:
            rec['loss'].zero_()
            return pred, rec
        n_ks = kernels.train_fwd_ksplits(N, F)
        args = (
            self._dims(), self.uid_embeddings.weight.data, self.iid_embeddings.weight.data, self.feature_embedding,
            self.mlp[0].weight.data, self.mlp[0].bias.data, self._expo(), call['X'], call['sample_item'], Y, call['rng'],
            loss_mode, pred, rec['loss'], self._buf('ws_wimg', (kernels.train_w_image_floats(F),), torch.float32),
            w_image_valid, self._buf('ws_pre_part', (n_ks, N, D), torch.float32), self._buf('ws_dpre', (N, D), torch.float32),
            self._buf('ws_loss_terms', (P,), torch.float32), rec['gW_part'], rec['gb_part'], rec['gu_rec'],
            rec['gi_rec'], rec['keys_u'], rec['keys_i'], None, None, expo_e, expo_den, self._err_flag)
        mse_pairs = rec['exchange'].world * P if 'exchange' in rec else 0
        pdl = 8 if (programmatic and w_image_valid) else 0     # phase 1 beside the kernel launched just before it
        if between is None:
            # one chain: the middle and dW kernels are programmatic dependents of the kernel before them, and do their
            # prologues while it runs.  (The data-parallel step records an event between them: plain launches.)
            kernels.train_fwd_bwd_tc(*args, phases=7 | pdl | (16 | 32 if pdl else 0), batch=batch, mse_pairs=mse_pairs)
        else:                       # kernel by kernel, with the caller's stream plumbing after each
            for phase in (1, 2, 4):
                kernels.train_fwd_bwd_tc(*args, phases=phase | (pdl if phase == 1 else 0), batch=batch, mse_pairs=mse_pairs)
                between(phase)
        call['pred'] = pred
        return pred, rec

    def save_training_state(self, path=None):
        """Weights (the reference's state_dict keys) + fused-optimizer moments / step + the position of the library's
        noise / dropout streams: everything a run needs to continue bit-identically (SURVEY.md §8f-4)."""
        path = path or (self.model_path + '.train_state')
        dir_path = os.path.dirname(path)
        if dir_path and not os.path.exists(dir_path):
            os.makedirs(dir_path)
        opt = self.optimizer.state_dict() if isinstance(self.optimizer, FusedAdamState) else None
        torch.save({'model': self.state_dict(), 'optimizer': opt, 'rng_offset': self._rng_offset}, path)
        return path

    def load_training_state(self, path=None):
        path = path or (self.model_path + '.train_state')
        st = torch.load(path, map_location=self.uid_embeddings.weight.device)
        self.load_state_dict(st['model'])
        if st['optimizer'] is not None:
            if not isinstance(self.optimizer, FusedAdamState):
                self.optimizer = self.make_fused_optimizer(lr=st['optimizer']['lr'], l2=st['optimizer']['l2'],
                                                           weight_decay=st['optimizer']['weight_decay'],
                                                           kind=st['optimizer'].get('kind', 'adam'))
            self.optimizer.load_state_dict(st['optimizer'])
        self._rng_offset = int(st['rng_offset'])
        self._param_epoch += 1                      # projected tables / operand images of the old weights are stale
        return self

    # ---- checkpoints with a row-sharded user table --------------------------------------------------------
    def save_model(self, model_path=None):
        """BaseModel.save_model (src/models/BaseModel.py:224-236).  With a row-sharded user table (`user_shard`) the
        replicas are NOT identical: every rank sends its user rows to rank 0, which writes ONE state_dict with the full
        [user_num, D] table under the reference's keys — the file is interchangeable with an unsharded run's."""
        import logging
        import torch.distributed as dist
        if self.user_shard is None or not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return DMF.save_model(self, model_path)
        model_path = model_path or self.model_path
        rank, world = dist.get_rank(), dist.get_world_size()
        w = self.uid_embeddings.weight.data
        bounds = [None] * world
        dist.all_gather_object(bounds, self.user_shard)
        if rank == 0:
            full = torch.empty((self.user_num, w.shape[1]), dtype=w.dtype, device=w.device)
            full[bounds[0][0]:bounds[0][1]] = w
            for r in range(1, world):
                dist.recv(full[bounds[r][0]:bounds[r][1]], src=r)
            sd = {k: v for k, v in self.state_dict().items()}
            sd['uid_embeddings.weight'] = full
            dir_path = os.path.dirname(model_path)
            if dir_path and not os.path.exists(dir_path):
                os.makedirs(dir_path)
            torch.save(sd, model_path)
        else:
            dist.send(w.contiguous(), dst=0)
        dist.barrier()
        logging.info('Save model to ' + model_path)

    def load_model(self, model_path=None):
        """BaseModel.load_model; a rank that owns users [lo, hi) keeps only those rows of the saved user table."""
        import logging
        if self.user_shard is None:
            return DMF.load_model(self, model_path)
        model_path = model_path or self.model_path
        sd = torch.load(model_path, map_location='cpu')
        lo, hi = self.user_shard
        if sd['uid_embeddings.weight'].shape[0] == self.user_num:
            sd['uid_embeddings.weight'] = sd['uid_embeddings.weight'][lo:hi].clone()
        self.load_state_dict(sd)
        self._param_epoch += 1
        self.eval()
        logging.info('Load model from ' + model_path)

    def check_ids(self):
        """Raise if any kernel since the last check met a user/item id outside the tables (the kernels clamp
        such ids and raise a device flag instead of faulting; the reference would raise an IndexError)."""
        if self._err_flag is not None and int(self._err_flag.item()) != 0:
            self._err_flag.zero_()
            raise IndexError('user or item id out of range in feed_dict[\'X\'] / sample_item')

    # ---- reference protocol ------------------------------------------------------------------
    def predict(self, feed_dict):
        """{'prediction': Tensor[P], 'check': [('prediction', Tensor)]} (DCCF.py:66-107)."""
        call = self._make_call(feed_dict)
        need_grad = torch.is_grad_enabled() and bool(feed_dict.get('train', False)) and \
            any(p.requires_grad for p in self.parameters())
        if need_grad:
            prediction = _ScoreFn.apply(self.uid_embeddings.weight, self.iid_embeddings.weight, self.mlp[0].weight,
                                        self.mlp[0].bias, self, call)
        else:
            prediction = self._launch_fwd(call, save=False)
        return {'prediction': prediction, 'check': [('prediction', prediction)]}

    def draw_confounders(self, n_pairs):
        """The confounder draw of one predict call — `torch.randint(item_num, (P, S))` on the torch CPU generator
        exactly as src/models/DCCF.py:72 — into pinned memory.  A caller that knows its next batch (the runner's
        fit loop) draws it right after launching the current step, so the host generator overlaps the device;
        the generator is consumed in the same order as without the prefetch."""
        buf = torch.empty((n_pairs, self.sample_num), dtype=torch.int64, pin_memory=torch.cuda.is_available())
        if self.sample_num > 0 and n_pairs > 0:
            host_rng.randint(self.item_num, (n_pairs, self.sample_num), out=buf)
        return buf

    def predict_many(self, feed_dicts, depth=2):
        """Predictions for a list of feed dicts (an evaluation pass).  Identical to calling `predict` on each
        in turn — including the order in which the torch CPU generator is consumed (DCCF.py:72) — but the
        confounder draw of batch k+1 is made by a worker thread into pinned memory while batch k runs on the
        GPU, so the host generator no longer serialises with the device."""
        import queue
        import threading
        S = self.sample_num
        if self.device_confounders and S > 0 and self.item_num < (1 << 28) and host_rng.available() and \
                any('sample_item' not in fd for fd in feed_dicts):
            # the torch CPU generator continued on the device for the length of the pass: every batch's draw is one
            # kernel writing straight into device memory (host_rng.DeviceStream), same ids in the same order
            self._check_ready()
            stream = host_rng.DeviceStream(self.uid_embeddings.weight.device)
            outs = []
            try:
                for fd in feed_dicts:
                    if 'sample_item' not in fd:
                        fd = dict(fd)
                        fd['sample_item'] = stream.draw(self.item_num, (fd['X'].shape[0], S))
                    outs.append(self.predict(fd)['prediction'])
            finally:
                stream.finish()
            return outs
        pin = torch.cuda.is_available()
        q = queue.Queue(maxsize=max(1, depth))
        stop = threading.Event()

        def put(item):
            # never block for ever on the bounded queue: a consumer that failed stops reading it
            while not stop.is_set():
                try:
                    q.put(item, timeout=0.1)
                    return True
                except queue.Full:
                    continue
            return False

        def produce():
            try:
                for fd in feed_dicts:
                    if stop.is_set():
                        return
                    if 'sample_item' in fd or S == 0:
                        if not put(None):
                            return
                        continue
                    buf = torch.empty((fd['X'].shape[0], S), dtype=torch.int64, pin_memory=pin)
                    host_rng.randint(self.item_num, (fd['X'].shape[0], S), out=buf)
                    if not put(buf):
                        return
            except BaseException as e:      # surface the failure in the consumer
                put(e)

        worker = threading.Thread(target=produce, daemon=True)
        worker.start()
        outs = []
        try:
            for fd in feed_dicts:
                draw = q.get()
                if isinstance(draw, BaseException):
                    raise draw
                if draw is not None:
                    fd = dict(fd)
                    fd['sample_item'] = draw
                outs.append(self.predict(fd)['prediction'])
        finally:
            stop.set()                      # a failed predict: release the producer, then wait for it (bounded)
            worker.join(timeout=30)
        return outs

    def forward(self, feed_dict):
        """predict + BPR (rank 1; first half positives, second half their negatives) or MSE loss
        (DCCF.py:109-127)."""
        out_dict = self.predict(feed_dict)
        if feed_dict['rank'] == 1:
            b = int(feed_dict['Y'].shape[0] / 2)
            pos, neg = out_dict['prediction'][:b], out_dict['prediction'][b:]
            loss = -(pos - neg).sigmoid().log().sum()
        else:
            loss = torch.nn.MSELoss()(out_dict['prediction'], feed_dict['Y'].to(out_dict['prediction'].device))
        out_dict['loss'] = loss
        return out_dict

    # ---- data parallel ----------------------------------------------------------------------
    def enable_data_parallel(self, group=None, p2p=True):
        """Replicated parameters, per-rank batches, gradients exchanged once per step (dccf_b200/dist.py):
        by this rank's own kernels over NVLink peer memory (p2p=True, default) or by an NCCL all-gather.
        Requires an initialised torch.distributed process group."""
        import torch.distributed as dist
        self._dp = {'world': dist.get_world_size(group), 'rank': dist.get_rank(group), 'group': group, 'ex': {},
                    'p2p': p2p}
        return self

    def data_parallel_suspended(self):
        """Context manager: steps inside run as on one GPU (no exchange; every rank must then feed the SAME batch and
        random inputs, so the replicas remain bit-identical) — the tail of an epoch that does not fill a global step."""
        import contextlib

        @contextlib.contextmanager
        def cm():
            saved, self._dp = self._dp, None
            try:
                yield self
            finally:
                self._dp = saved
        return cm()

    def _exchange_for(self, P):
        from ..dist import GradExchange
        ex = self._dp['ex'].get(P)
        if ex is None:
            D, Z = self.ui_vector_size, self.sample_num + 1
            ex = GradExchange(P, Z, D, D + self.feature_embedding.shape[1], self._dp['world'], self._dp['rank'],
                              self.uid_embeddings.weight.device, group=self._dp['group'],
                              use_p2p=self._dp.get('p2p', True), user_records=self.user_shard is None)
            self._dp['ex'][P] = ex
        return ex

    # ---- fused training step -----------------------------------------------------------------
    def make_fused_optimizer(self, lr, l2, weight_decay=None, kind='adam', **kw):
        """State of the fused step for kind 'adam', 'gd' or 'adagrad' (torch.optim.Adam / SGD / Adagrad with
        weight_decay, as src/runners/BaseRunner.py:83-107 builds them)."""
        self._check_ready()
        return FusedAdamState(self, lr=lr, l2=l2, weight_decay=l2 if weight_decay is None else weight_decay, kind=kind,
                              **kw)

    # record lists of the split optimizer step as CSR ranges (counting link + dccf_adam_csr_build off the critical path)
    # instead of linked lists: DCCF_ADAM_CSR=0 restores the lists (A/B; same summation order, same bits)
    use_csr_lists = os.environ.get('DCCF_ADAM_CSR', '1') != '0'

    def _csr_bufs(self, which, n_rec, n_rows, opt):
        if opt.__dict__.get('csr_pool') is None:
            opt.csr_pool = torch.zeros(4, dtype=torch.int32, device=self.uid_embeddings.weight.device)
        k = 0 if which == 'u' else 2
        return (self._buf('rec_row_' + which, (n_rec,), torch.int32), self._buf('csr_off_' + which, (n_rows,), torch.int32),
                self._buf('csr_' + which, (2 * n_rec,), torch.int32), opt.csr_pool[k:k + 2])

    def _step_tables(self, rec, P, opt, csr=False):
        """Descriptors of the optimizer step's tensors: the two embedding tables with their gradient records and W, b
        with their partial sums.  Data parallel: records / dW / db of every rank, read from the receive buffer of the
        gradient exchange (static addresses, so the descriptors can be built before the exchange runs).  csr: record
        lists as CSR ranges (the split step)."""
        Z, D = self.sample_num + 1, self.ui_vector_size
        W, b = self.mlp[0].weight.data, self.mlp[0].bias.data
        eu, ei = self.uid_embeddings.weight.data, self.iid_embeddings.weight.data
        su, si, sW, sb = (opt.state_of(k) for k in ('E_user', 'E_item', 'W', 'b'))
        dp = 'exchange' in rec
        world = rec['exchange'].world if dp else 1
        n_u = (world if (dp and rec['exchange'].user_records) else 1) * P
        n_i = world * P * Z
        next_u, next_i = self._buf('next_u', (n_u,), torch.int32), self._buf('next_i', (n_i,), torch.int32)
        csr_u = self._csr_bufs('u', n_u, eu.shape[0], opt) if csr else None
        csr_i = self._csr_bufs('i', n_i, ei.shape[0], opt) if csr else None
        if dp:
            ex = rec['exchange']
            rseg, dseg = ex.seg_of('gi'), ex.seg_of('gW')
            if ex.user_records:
                user = kernels.adam_table(eu, *su, ex.recv_part('keys_u'), ex.recv_part('gu'), world, P,
                                          rseg, rseg, opt.head_u, next_u, csr=csr_u)
            else:
                user = kernels.adam_table(eu, *su, rec['keys_u'], rec['gu_rec'], 1, P, P, P * D,
                                          opt.head_u, next_u, csr=csr_u)
            tables = [user,
                      kernels.adam_table(ei, *si, ex.recv_part('keys_i'), ex.recv_part('gi'),
                                         world, P * Z, rseg, rseg, opt.head_i, next_i, csr=csr_i)]
            dense = [kernels.adam_tensor(W, *sW, ex.recv_part('gW'), world, dseg),
                     kernels.adam_tensor(b, *sb, ex.recv_part('gb'), world, dseg)]
            return tables, dense
        tables = [kernels.adam_table(eu, *su, rec['keys_u'], rec['gu_rec'], 1, P, P, P * D,
                                     opt.head_u, next_u, csr=csr_u),
                  kernels.adam_table(ei, *si, rec['keys_i'], rec['gi_rec'], 1, P * Z, P * Z,
                                     P * Z * D, opt.head_i, next_i, csr=csr_i)]
        dense = [kernels.adam_tensor(W, *sW, rec['gW_part'], rec['n_splits'], W.numel()),
                 kernels.adam_tensor(b, *sb, rec['gb_part'], rec['n_splits'], b.numel())]
        return tables, dense

    def _exchange_dense(self, rec, push_only=False):
        """Data parallel: all-gather dW / db / loss; the row-split partials of dW / db are folded into the segment by
        the push kernel itself (peer-memory mode) or by two dccf_sum_parts launches.  push_only: the consumer kernel
        waits for the peers itself."""
        ex, v = rec['exchange'], rec['send']
        W, b = self.mlp[0].weight.data, self.mlp[0].bias.data
        if ex.mode == 'p2p':
            folds = [(rec['gW_part'], rec['n_splits'], W.numel(), ex.off['gW'][0], W.numel()),
                     (rec['gb_part'], rec['n_splits'], b.numel(), ex.off['gb'][0], b.numel())]
            if push_only:
                ex.dense.push(folds=folds)
            else:
                ex.exchange_dense(folds=folds)
            return
        kernels.sum_parts(rec['gW_part'], rec['n_splits'], W.numel(), W.numel(), v['gW'])
        kernels.sum_parts(rec['gb_part'], rec['n_splits'], b.numel(), b.numel(), v['gb'])
        ex.exchange_dense()

    def _apply_adam(self, rec, P, opt, hp):
        """l2 + clip + Adam over both tables, W and b (two launches); under data parallelism preceded by the
        fold of the row-split partials and ONE all-gather of the packed gradient segment."""
        tables, dense = self._step_tables(rec, P, opt)
        if 'exchange' in rec:
            rec['exchange'].exchange_records()
            self._exchange_dense(rec)
            kernels.adam_step(tables, dense, hp)
            loss = rec['exchange'].total_loss()
            rec['exchange'].done()
            return loss
        kernels.adam_step(tables, dense, hp)
        return rec['loss'][0]

    # fused step with the optimizer split around the backward: the Adam sweep of the rows the (global) batch does not
    # touch runs on a second stream while the forward and backward run (dccf_adam_link_ids / _untouched / _touched)

    def _sweep_threads(self, dp, opt):
        """Launch shape of the untouched-row sweep: one small CTA per SM hidden beside the tensor-core kernels and
        the middle kernel (0 = the library's default, 224 threads: the widest CTA whose registers fit beside the middle
        kernel's) while the tables are small enough for that to finish in time; -1 = the wide, full-occupancy sweep once
        the sweep itself bounds the step (scaled configuration with Adam: 24 B x 64 x 10^6..10^7 rows per step — at the
        ~3 TB/s of the narrow launch that is milliseconds).  Bytes per parameter: the parameter and each state tensor
        of the rule, read and written (Adam 24, Adagrad 16, GD 8)."""
        rows = self.uid_embeddings.weight.shape[0] + self.item_num
        bytes_per_param = 8 * (1 + sum(t is not None for t in opt.state_of('E_item')))
        if rows * self.ui_vector_size * bytes_per_param > 400e6:
            return -1
        return 0

    def _wimg_key(self):
        W = self.mlp[0].weight
        return (W._version, W.data_ptr(), self._param_epoch)

    def _split_step_ok(self, loss_mode, P=None):
        if not self._fused_step_ok(loss_mode):
            return False
        if self._dp is None:
            return True
        # data parallel: needs the ids of every rank at the start of the step, exchanged by plain kernels
        return P is not None and self._exchange_for(P).mode == 'p2p' and self._id_exchange_for(P).mode == 'p2p'

    def _id_exchange_for(self, P):
        from ..dist import IdExchange
        ix = self._dp.setdefault('ids', {}).get(P)
        if ix is None:
            ix = IdExchange(P, self.sample_num, self._dp['world'], self._dp['rank'], self.uid_embeddings.weight.device,
                            group=self._dp['group'], use_p2p=self._dp.get('p2p', True))
            self._dp['ids'][P] = ix
        return ix

    def _fused_split_step(self, call, loss_mode, Y, opt, hp, w_image_valid, overlap, counters=None, stage=None,
                          epoch_ids=None):
        """Forward + loss + backward + optimizer with the optimizer split around the backward.  overlap=True: the
        sweep of the untouched rows goes to a side stream (forked from / joined to the current stream with events,
        so it is also legal under CUDA-graph capture).  Data parallel: the ranks first gather each other's ids
        (call['X'] / call['sample_item'] must then be the send buffers of the id exchange), and the gradients are
        exchanged between the backward and the sweep of the touched rows.  counters = (step_dev, offset_dev): the
        last CTA of the step advances them.  Returns (prediction, loss)."""
        P, N = call['P'], call['N']
        D, F = self.ui_vector_size, self.feature_embedding.shape[1]
        rec = self._rec_buffers(call, loss_mode, kernels.train_bwd_splits(N, F))
        csr = self.use_csr_lists
        tables, dense = self._step_tables(rec, P, opt, csr=csr)
        world = rec['exchange'].world if 'exchange' in rec else 1
        next_u = self._buf('next_u', ((world if ('exchange' in rec and rec['exchange'].user_records) else 1) * P,), torch.int32)
        next_i = self._buf('next_i', (world * P * (self.sample_num + 1),), torch.int32)
        wimg = self._buf('ws_wimg', (kernels.train_w_image_floats(F),), torch.float32)
        if opt.__dict__.get('cta_counter') is None:
            opt.cta_counter = torch.zeros(1, dtype=torch.int32, device=self.uid_embeddings.weight.device)
        main = torch.cuda.current_stream()
        expo_e = self._buf('ws_expo_e', (P, self.sample_num + 1), torch.float32)
        expo_den = self._buf('ws_expo_den', (P,), torch.float32)
        dp = 'exchange' in rec
        if dp:
            ex, ix = rec['exchange'], self._id_exchange_for(P)
            assert call['X'].data_ptr() == ix.send_X.data_ptr() and call['sample_item'].data_ptr() == ix.send_si.data_ptr()

        # The exposure softmax of the local pairs (read by the middle kernel) and, on one GPU, the record lists: first,
        # on the main stream.  (On the side stream this kernel would run beside the first CTAs of the partial-product
        # kernel — measured: that kernel then takes 22 us instead of 13.)  k_link_ids also requests what the step will
        # touch into L2: rows of the tables and their optimizer state, the true items' feature rows, W with its state and
        # operand images.
        eu, ei = self.uid_embeddings.weight.data, self.iid_embeddings.weight.data
        W = self.mlp[0].weight.data
        # (only the tensors the optimizer rule has)
        pf_user = tuple(t for t in (eu,) + opt.state_of('E_user') if t is not None)
        pf_item = tuple(t for t in (ei,) + opt.state_of('E_item') if t is not None)
        pf_W = tuple(t for t in (W,) + opt.state_of('W') if t is not None)
        rec_rows = (self._ws['rec_row_u'], self._ws['rec_row_i']) if csr else None      # (allocated by _step_tables)
        if not dp:
            extra = kernels.make_link_extra(
                stage=stage, prefetch_user=pf_user, prefetch_item=pf_item, rec_rows=rec_rows,
                prefetch_feat=self.feature_embedding, prefetch_dense=(wimg,) + pf_W)
        else:
            # data parallel: the local launch stages the batch (device-resident epoch) and evaluates the exposure softmax;
            # the record lists of the GLOBAL step are linked on the side stream
            extra = kernels.make_link_extra(stage=stage, prefetch_feat=self.feature_embedding, prefetch_dense=(wimg,))

        # The forward needs nothing this launch produces except — with a device-resident epoch — the staged ids, and
        # those it can read from the epoch arrays itself (dccf_batch_ref): it is launched as a PROGRAMMATIC DEPENDENT of
        # this kernel and starts beside it (the 5 us of k_link_ids were the head of every step's critical path).  The
        # forward does not complete before this kernel has, so the middle kernel still finds the exposure softmax and
        # the staged ids.  (A first version put this launch on the side stream: same overlap, but a graph with two root
        # nodes and a cross-stream edge into the middle kernel started 3 us later and left 2 us wider gaps.)
        beside = overlap and w_image_valid
        batch = (stage[0], stage[1]) if (stage is not None and beside) else None
        kernels.adam_link_ids(self._dims(), call['X'], call['sample_item'], opt.head_u, next_u, opt.head_i, next_i,
                              self._expo(), expo_e, expo_den, n_seg=0 if dp else 1, extra=extra)

        def link_global():
            # data parallel: every rank's ids, then the record lists of the GLOBAL step.  The synchronisation is folded
            # into the consumers: they wait for the peers' segments in their own prologue and their last CTA hands the
            # buffers back.
            pf = dict(prefetch_user=pf_user, prefetch_item=pf_item,
                      prefetch_dense=pf_W)
            if epoch_ids is not None:
                # every rank's ids of the whole epoch were gathered once (begin_resident_epoch): no id exchange in the step
                kernels.adam_link_ids(self._dims(), None, None, opt.head_u, next_u, opt.head_i, next_i, n_pairs=P,
                                      n_seg=ex.world, seg_stride=0, user_seg=-1 if ex.user_records else ex.rank,
                                      extra=kernels.make_link_extra(epoch_global=epoch_ids, rec_rows=rec_rows, **pf))
                return
            ix.push()
            if opt.__dict__.get('link_counter') is None:
                opt.link_counter = torch.zeros(1, dtype=torch.int32, device=eu.device)
            ids = ix.recv.view(torch.int64)
            extra_g = kernels.make_link_extra(sync=kernels.make_dp_sync(ix.world, ix.rank, wait=(ix,), done=(ix,)),
                                              counter=opt.link_counter, rec_rows=rec_rows, **pf)
            kernels.adam_link_ids(self._dims(), ids, ids[ix.si_off_i64:], opt.head_u, next_u, opt.head_i, next_i,
                                  n_pairs=P, n_seg=ix.world, seg_stride=ix.seg_i64,
                                  user_seg=-1 if ex.user_records else ix.rank, extra=extra_g)

        between = None
        if overlap:
            d = self.__dict__
            if d.get('_side_stream') is None:
                d['_side_stream'] = torch.cuda.Stream(device=main.device)
                d['_ship_stream'] = torch.cuda.Stream(device=main.device)
            side, ship = d['_side_stream'], d['_ship_stream']
            fork, done = torch.cuda.Event(), torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)
            with torch.cuda.stream(side):
                if dp:                      # the id exchange waits for the peers: never on the critical path
                    link_global()
                if csr:
                    linked = torch.cuda.Event()
                    linked.record(side)
                kernels.adam_untouched(tables, hp, self._sweep_threads(dp and epoch_ids is None, opt))
                done.record(side)
            # The CSR ranges of the step's record lists (two small launches; the touched-row sweep that needs them runs
            # after the backward): on a third stream as soon as the lists are linked, beside the sweep and the forward —
            # done before the middle kernel starts at 1-2 ranks.  At 8 ranks they are still resident when the middle
            # kernel wants its SMs and that kernel ends 7 us later than on one GPU; the other placements measured on
            # 8 x B200 moved that cost instead of removing it (DESIGN.md §8).
            csr_done = None
            if csr:
                csr_done = torch.cuda.Event()
                ship.wait_event(linked)
                with torch.cuda.stream(ship):
                    kernels.adam_csr_build(tables)
                    csr_done.record(ship)
            if dp:
                mid_done, shipped = torch.cuda.Event(), torch.cuda.Event()

                def between(phase):        # noqa: E306  the gradient records leave while the dW kernel runs
                    if phase == 2:
                        mid_done.record(main)
                        ship.wait_event(mid_done)
                        with torch.cuda.stream(ship):
                            ex.rec.push()
                            shipped.record(ship)
        else:
            if dp:
                link_global()
            kernels.adam_untouched(tables, hp, self._sweep_threads(dp and epoch_ids is None, opt))
            if csr:
                kernels.adam_csr_build(tables)
        pred, rec = self._launch_fwd_bwd(call, loss_mode, Y, rec=rec, w_image_valid=w_image_valid, expo_e=expo_e,
                                         expo_den=expo_den, between=between, batch=batch, programmatic=beside)
        sync = None
        if dp:
            if overlap:
                # The touched-row sweep is launched as a programmatic dependent of the dW / db push and starts beside it:
                # everything else it depends on (record push, side sweep, CSR ranges) is joined BEFORE the push, which
                # is then its only — programmatic — predecessor.  (All three end long before the dW kernel does.)
                main.wait_event(shipped)
                main.wait_event(done)
                if csr_done is not None:
                    main.wait_event(csr_done)
            else:
                ex.rec.push()
            self._exchange_dense(rec, push_only=True)
            total = self._buf('dp_total_loss', (1,), torch.float32)
            a_loss, _ = ex.off['loss']
            sync = kernels.make_dp_sync(ex.world, ex.rank, wait=(ex.rec, ex.dense), done=(ex.rec, ex.dense),
                                        loss=(ex.dense.recv[a_loss:], ex.dense.seg, ex.world, total),
                                        flags=kernels.DP_SYNC_OVERLAP_PUSH if overlap else 0)
        elif overlap:
            main.wait_event(done)
            if csr_done is not None:
                main.wait_event(csr_done)
        step_dev, offset_dev = counters if counters is not None else (None, None)
        kernels.adam_touched(tables, dense, hp, True, wimg, 0, D + F, opt.cta_counter, step_dev, offset_dev, sync=sync,
                             advance_cursor_dev=stage[1] if stage is not None else None)
        if dp:
            return pred, total[0]
        return pred, rec['loss'][0]

    def train_step(self, feed_dict, opt=None, stage_events=None):
        """One iteration of BaseRunner.fit (src/runners/BaseRunner.py:175-188): forward, loss, l2 term,
        backward, clip, Adam — no autograd, no host sync.  Steps whose random inputs come from the library's
        own streams are captured once into a CUDA graph per batch shape and replayed (one graph launch instead
        of six kernel launches; the step counter and the rng call counter then live in device memory).
        Returns the reference's out_dict (prediction, check, loss); under graph replay the tensors are the
        graph's static outputs, valid until the next train_step."""
        opt = opt or self.optimizer
        if not isinstance(opt, FusedAdamState):
            raise RuntimeError('train_step needs the fused optimizer state (model.make_fused_optimizer)')
        if stage_events is None and self.use_cuda_graph and 'noise' not in feed_dict and \
                'dropout_mask' not in feed_dict:
            out = self._train_step_graph(feed_dict, opt)
            if out is not None:
                return out
        call = self._make_call(feed_dict)
        loss_mode = 0 if feed_dict['rank'] == 1 else 1
        Y = feed_dict['Y'].to(call['X'].device, torch.float32).contiguous() if loss_mode == 1 else None
        if stage_events is None and call['P'] > 0 and self._split_step_ok(loss_mode, call['P']):
            if self._dp is not None:        # the ids travel to the peers from the id exchange's send buffers
                ix = self._id_exchange_for(call['P'])
                ix.send_X.copy_(call['X'])
                ix.send_si.copy_(call['sample_item'])
                call['X'], call['sample_item'] = ix.send_X, ix.send_si
            valid = self.__dict__.get('_wimg_valid_key') == self._wimg_key()
            opt.step_count += 1
            self._param_epoch += 1
            pred, loss = self._fused_split_step(call, loss_mode, Y, opt, opt.hp(), valid, overlap=False)
            self.__dict__['_wimg_valid_key'] = self._wimg_key()
            return {'prediction': pred, 'check': [('prediction', pred)], 'loss': loss.clone()}
        if stage_events is not None:
            stage_events[0].record()
        if stage_events is None and self._fused_step_ok(loss_mode):
            pred, rec = self._launch_fwd_bwd(call, loss_mode, Y)
        else:
            pred = self._launch_fwd(call, save=True)
            if stage_events is not None:
                stage_events[1].record()
            rec = self._launch_bwd(call, loss_mode=loss_mode, Y=Y)
        if stage_events is not None:
            stage_events[2].record()
        opt.step_count += 1
        self._param_epoch += 1
        loss = self._apply_adam(rec, call['P'], opt, opt.hp())
        if stage_events is not None:
            stage_events[3].record()
        return {'prediction': pred, 'check': [('prediction', pred)], 'loss': loss.clone()}

    # ---- CUDA-graph replay of the fused step -----------------------------------------------------
    use_cuda_graph = True
    def _build_step_graph(self, P, rank_mode, p_drop, opt, staged):
        """Capture forward + backward + (exchange) + Adam + counter advance for a batch of P pairs.  `staged`:
        the batch is copied from a device-resident epoch (by k_link_ids, or dccf_stage_batch as the graph's first
        node) — with rank_mode 0 its labels too."""
        dev = self.uid_embeddings.weight.device
        S = self.sample_num
        # ids and confounder draws of the step in ONE buffer [X (P x 2) | sample_item (P x S)]: a batch that arrives from
        # the host is staged in pinned memory with the same layout and uploaded by a single copy
        ids = torch.zeros(2 * P + P * S, dtype=torch.int64, device=dev)
        g = {'ids': ids, 'X': ids[:2 * P].view(P, 2), 'si': ids[2 * P:].view(P, S),
             'Y': torch.zeros(P, dtype=torch.float32, device=dev),
             'step_dev': torch.zeros(1, dtype=torch.int32, device=dev),
             'offset_dev': torch.zeros(1, dtype=torch.int64, device=dev), 'synced': None}
        if staged:
            # [X, si, X_all, si_all, stride_X, stride_si, Y (rank_mode 0)]
            g['epoch_ptrs'] = torch.zeros(7, dtype=torch.int64, device=dev)
            g['cursor'] = torch.zeros(1, dtype=torch.int64, device=dev)
            g['stage_counter'] = torch.zeros(1, dtype=torch.int32, device=dev)
        if self._dp is not None and self._split_step_ok(0 if rank_mode == 1 else 1, P):
            ix = self._id_exchange_for(P)       # the step's input buffers ARE the send segment of the id exchange
            g['X'], g['si'] = ix.send_X, ix.send_si
            g['ids'] = ix.send[:4 * P + 2 * P * S].view(torch.int64)
        seed = self.random_seed
        if self._dp is not None:
            seed = (seed + 0x9E3779B97F4A7C15 * self._dp['rank']) & 0xffffffffffffffff
        rng = kernels.make_rng(noise_std=self.std, p_drop=p_drop, seed=seed, offset_dev=g['offset_dev'],
                               generate_noise=self.std > 0, generate_mask=p_drop > 0)
        call = {'X': g['X'], 'sample_item': g['si'], 'rng': rng, 'noise': None, 'mask': None, 'P': P,
                'N': P * (S + 1) * self.attribute_num}
        hp = opt.hp(step=1, step_dev=g['step_dev'])
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        launches_before = kernels.LAUNCHES[0]
        with torch.cuda.graph(graph, capture_error_mode='thread_local'):
            loss_mode = 0 if rank_mode == 1 else 1
            Yg = g['Y'] if rank_mode != 1 else None
            split = self._split_step_ok(loss_mode, P)
            # a batch read from a device-resident epoch: fetched by k_link_ids itself in the split step (each linking
            # thread copies the id it links; data parallel, every rank's ids of the whole epoch were gathered once, so
            # the step has no id exchange), by a launch of its own otherwise
            epoch_ids = staged and split and self._dp is not None
            if staged and not split:
                kernels.stage_batch(g['epoch_ptrs'], g['cursor'], P, S, g['X'], g['si'], Yg)
            if split:
                # the W operand images are kept current by dccf_adam_touched (checked before every replay)
                stage = (g['epoch_ptrs'], g['cursor'], g['X'], g['si'], g['stage_counter'], Yg) if staged else None
                g['epoch_ids'] = epoch_ids
                pred, loss = self._fused_split_step(call, loss_mode, Yg, opt, hp, True, overlap=True,
                                                    counters=(g['step_dev'], g['offset_dev']), stage=stage,
                                                    epoch_ids=(g['epoch_ptrs'], g['cursor']) if epoch_ids else None)
                g['w_image'] = True     # loss: the step's own output buffer (valid until the next train_step)
            else:
                if self._fused_step_ok(loss_mode):
                    pred, rec = self._launch_fwd_bwd(call, loss_mode, Yg)
                else:
                    pred = self._launch_fwd(call, save=True)
                    rec = self._launch_bwd(call, loss_mode=loss_mode, Y=Yg)
                loss = self._apply_adam(rec, P, opt, hp).clone()
                kernels.state_advance(g['step_dev'], g['offset_dev'], 1)
        # The captured graph holds RAW device pointers: every workspace the capture touched (grow-only buffers that a
        # later, larger call would replace and free), the optimizer state and the exchange buffers stay referenced
        # from the graph entry for as long as the graph can be replayed.
        keep = {'ws': dict(self._ws), 'opt': opt, 'err_flag': self._err_flag,
                'streams': (self.__dict__.get('_side_stream'), self.__dict__.get('_ship_stream'))}
        if self._dp is not None:
            keep['dp'] = (dict(self._dp.get('ex', {})), dict(self._dp.get('ids', {})))
        g.update({'graph': graph, 'pred': pred, 'loss': loss, 'call': call, 'keep_alive': keep,
                  'n_kernels': kernels.LAUNCHES[0] - launches_before})
        kernels.LAUNCHES[0] = launches_before           # capturing launched nothing
        return g

    def _replay(self, g, opt):
        if g.get('w_image') and self.__dict__.get('_wimg_valid_key') != self._wimg_key():
            # W changed outside the fused steps (or this is the first one): rebuild its operand images
            F = self.feature_embedding.shape[1]
            kernels.train_prep_w_image(self.mlp[0].weight.data, F,
                                       self._buf('ws_wimg', (kernels.train_w_image_floats(F),), torch.float32))
        self._rng_offset += 1
        opt.step_count += 1
        self._param_epoch += 1
        if g['synced'] != (opt.step_count, self._rng_offset):
            # device counters out of step with the host mirrors (eager steps or predict calls ran in between)
            g['step_dev'].fill_(opt.step_count)
            g['offset_dev'].fill_(self._rng_offset)
        g['graph'].replay()
        if g.get('w_image'):
            self.__dict__['_wimg_valid_key'] = self._wimg_key()
        kernels.LAUNCHES[0] += g['n_kernels']
        g['synced'] = (opt.step_count + 1, self._rng_offset + 1)
        return {'prediction': g['pred'], 'check': [('prediction', g['pred'])], 'loss': g['loss']}

    def _graph_allowed(self, P):
        if self._dp is not None:
            # graph capture needs the exchange to be plain kernels (peer-memory mode); an NCCL all-gather
            # inside the captured step deadlocked on 2 x B200 with torch 2.11 / NCCL 2.28
            return self._exchange_for(P).mode == 'p2p'
        return True

    def _train_step_graph(self, feed_dict, opt):
        X = feed_dict['X']
        P = X.shape[0]
        if not self._graph_allowed(P):
            return None
        self._check_ready()
        rank_mode = int(feed_dict['rank'])
        p_drop = float(feed_dict.get('dropout', 0.0))
        key = (P, rank_mode, p_drop, opt, False, self._dp is not None)      # (the optimizer OBJECT: its id could be recycled)
        graphs = self.__dict__.setdefault('_graphs', {})
        g = graphs.get(key)
        if g is None:
            # first step of this shape runs eagerly (it also loads every kernel); capture on the second
            graphs[key] = 'warm'
            return None
        S = self.sample_num
        if g == 'warm':
            g = graphs[key] = self._build_step_graph(P, rank_mode, p_drop, opt, staged=False)
        Xs = X if torch.is_tensor(X) else torch.as_tensor(np.asarray(X))
        si = feed_dict.get('sample_item')
        if not Xs.is_cuda and (si is None or not si.is_cuda) and Xs.dtype == torch.int64 and Xs.shape[1] == 2:
            # a batch from the host: ids and confounder draw (DCCF.py:72, the torch CPU generator) are assembled in a
            # pinned staging slot with the layout of the graph's input buffer and uploaded by ONE asynchronous copy;
            # a small ring of slots, each guarded by an event, lets the host run ahead of the device
            ring = g.get('stage')
            if ring is None:
                ring = g['stage'] = {'slots': [[torch.empty(2 * P + P * S, dtype=torch.int64, pin_memory=True), None]
                                                for _ in range(8)], 'next': 0}
            slot = ring['slots'][ring['next'] % len(ring['slots'])]
            ring['next'] += 1
            if slot[1] is not None:
                slot[1].synchronize()           # the upload that last used this slot has completed
            else:
                slot[1] = torch.cuda.Event()
            slot[0][:2 * P].view(P, 2).copy_(Xs)
            if S > 0:
                dst = slot[0][2 * P:].view(P, S)
                if si is None:
                    host_rng.randint(self.item_num, (P, S), out=dst)
                else:
                    dst.copy_(si)
            g['ids'].copy_(slot[0], non_blocking=True)
            slot[1].record()
        else:
            # inputs already on the device (async copies on the current stream into the graph's static buffers)
            g['X'].copy_(Xs[:, :2] if Xs.shape[1] != 2 else Xs, non_blocking=True)
            if si is None:
                si = torch.randint(self.item_num, size=(P, S))          # DCCF.py:72, CPU generator
            g['si'].copy_(si, non_blocking=True)
        if rank_mode != 1:
            g['Y'].copy_(feed_dict['Y'], non_blocking=True)
        return self._replay(g, opt)

    def resident_epoch_available(self, P, opt=None):
        """True when begin_resident_epoch would return a step function for batches of P pairs — lets the runner decide
        BEFORE it consumes the torch CPU generator for the epoch's confounder draws."""
        opt = opt or self.optimizer
        if not isinstance(opt, FusedAdamState) or not self.use_cuda_graph:
            return False
        self._check_ready()
        return bool(self._graph_allowed(P))

    def begin_resident_epoch(self, X_epoch, sample_epoch, dropout, opt=None, Y_epoch=None):
        """Training over a device-resident epoch: X_epoch [n, P, 2] and sample_epoch [n, P, S] int64 CUDA tensors
        (all batches of P pairs; the confounder block is ONE torch.randint(item_num, (n*P, S)) call, which yields
        the same numbers as n per-batch calls on the same generator).  Returns a callable: each call runs the next
        batch as one CUDA-graph launch — the batch is fetched by a kernel through a device-side cursor, so the
        host does nothing per step but launch.  Without Y_epoch the batches are BPR (rank 1) batches; with Y_epoch
        [n, P] (float32 CUDA, the labels) they are rating-prediction (rank 0, MSE) batches, labels fetched beside the
        ids.  Returns None when graphs cannot be used."""
        opt = opt or self.optimizer
        if not isinstance(opt, FusedAdamState) or not self.use_cuda_graph:
            return None
        self._check_ready()
        n, P = X_epoch.shape[0], X_epoch.shape[1]
        rank_mode = 1 if Y_epoch is None else 0
        if Y_epoch is not None:
            if tuple(Y_epoch.shape) != (n, P) or Y_epoch.dtype != torch.float32 or Y_epoch.device != X_epoch.device:
                raise ValueError('Y_epoch must be float32 [%d, %d] on %s, got %s %s on %s'
                                 % (n, P, X_epoch.device, Y_epoch.dtype, tuple(Y_epoch.shape), Y_epoch.device))
            Y_epoch = Y_epoch.contiguous()
        if not self._graph_allowed(P) or n == 0:
            return None
        p_drop = float(dropout)
        key = (P, rank_mode, p_drop, opt, True, self._dp is not None)
        graphs = self.__dict__.setdefault('_graphs', {})
        state = {'next': 0}
        if key not in graphs:
            # the very first step runs kernel by kernel (loads every kernel before capture)
            saved = self.use_cuda_graph
            self.use_cuda_graph = False
            try:
                fd = {'X': X_epoch[0], 'rank': rank_mode, 'train': True, 'dropout': p_drop,
                      'sample_item': sample_epoch[0]}
                if Y_epoch is not None:
                    fd['Y'] = Y_epoch[0]
                first = self.train_step(fd, opt)
            finally:
                self.use_cuda_graph = saved
            state['next'] = 1
            state['first'] = first
            graphs[key] = self._build_step_graph(P, rank_mode, p_drop, opt, staged=True)
        g = graphs[key]
        X_epoch, sample_epoch = X_epoch.contiguous(), sample_epoch.contiguous()
        ptrs = [X_epoch.data_ptr(), sample_epoch.data_ptr(), 0, 0, 0, 0, 0]
        keep = [X_epoch, sample_epoch]
        if Y_epoch is not None:
            # the labels stay on this rank: only its own middle kernel reads them
            ptrs[6] = Y_epoch.data_ptr()
            keep.append(Y_epoch)
        if g.get('epoch_ids'):
            # every rank's batches of this epoch (chunk), gathered ONCE: [world, n, P, 2] / [world, n, P, S]
            import torch.distributed as dist
            world = self._dp['world']
            X_all = torch.empty((world,) + tuple(X_epoch.shape), dtype=torch.int64, device=X_epoch.device)
            si_all = torch.empty((world,) + tuple(sample_epoch.shape), dtype=torch.int64, device=X_epoch.device)
            dist.all_gather_into_tensor(X_all, X_epoch, group=self._dp['group'])
            dist.all_gather_into_tensor(si_all, sample_epoch, group=self._dp['group'])
            ptrs[2:6] = [X_all.data_ptr(), si_all.data_ptr(), X_epoch.numel(), sample_epoch.numel()]
            keep += [X_all, si_all]
        g['epoch_ptrs'].copy_(torch.tensor(ptrs, dtype=torch.int64))
        g['cursor'].fill_(state['next'])
        g['keep'] = tuple(keep)                             # the graph reads these buffers: keep them alive

        def step():
            if state['next'] >= n:
                raise StopIteration('resident epoch exhausted')
            state['next'] += 1
            return self._replay(g, opt)

        step.remaining = lambda: n - state['next']
        step.first = state.get('first')
        return step
