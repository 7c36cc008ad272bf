"""BiasedMF with the reference's model protocol (src/models/BiasedMF.py) on the library's kernels:

    pred = <p_u, q_i> + b_u + b_i + g

Parameters, in creation order (the order in which `apply(init_paras)` consumes the torch CPU generator):
`uid_embeddings` [U, 64], `iid_embeddings` [I, 64], `user_bias` Embedding(U, 1), `item_bias` Embedding(I, 1) and
`global_bias`, a 0-d Parameter that starts at 0.1 (the framework's BiasedMF value; init_paras leaves it alone).  The
state-dict keys are the reference's, so checkpoints interchange.

Training goes through `train_step` only (BaseRunner's fused path): one step is the split optimizer step of the DCCF
tables with no confounder slot (dccf_adam_link_ids / _untouched / _csr_build / _touched) around dccf_mf_step and
dccf_mf_bias_grad; user_bias, item_bias and global_bias are dense tensors of the touched-row launch.  Steps of one batch
shape are captured into a CUDA graph and replayed.  There is no CPU implementation: predict and train_step raise without
CUDA.  IPSBiasedMF (IPSBiasedMF.py) divides the prediction by max(propensity_i, M)."""
import os

import numpy as np
import torch

from .. import kernels
from .DCCF import FusedAdamState
from .RecModel import RecModel


class MFOptimizerState(FusedAdamState):
    """FusedAdamState (same rules, state_dict and resume) over the five parameters of BiasedMF."""

    def __init__(self, model, lr, l2, weight_decay, kind='adam', beta1=0.9, beta2=0.999, eps=None, clip=50.0):
        if kind not in self.RULES:
            raise ValueError('unknown fused optimizer %r (adam, gd, adagrad)' % (kind,))
        self.kind, self.rule = kind, self.RULES[kind]
        self.lr, self.l2, self.weight_decay = lr, l2, weight_decay
        self.beta1, self.beta2, self.clip = beta1, beta2, clip
        self.eps = eps if eps is not None else (1e-10 if kind == 'adagrad' else 1e-8)
        self.step_count = 0
        self.params = {'E_user': model.uid_embeddings.weight, 'E_item': model.iid_embeddings.weight,
                       'user_bias': model.user_bias.weight, 'item_bias': model.item_bias.weight,
                       'global_bias': model.global_bias}
        if kind == 'adam':
            self.exp_avg = {k: torch.zeros_like(p.data) for k, p in self.params.items()}
            self.exp_avg_sq = {k: torch.zeros_like(p.data) for k, p in self.params.items()}
        elif kind == 'adagrad':
            self.state_sum = {k: torch.zeros_like(p.data) for k, p in self.params.items()}
        dev = model.uid_embeddings.weight.device
        self.head_u = torch.full((model.user_num,), -1, dtype=torch.int32, device=dev)
        self.head_i = torch.full((model.item_num,), -1, dtype=torch.int32, device=dev)
        self.csr_pool = torch.zeros(4, dtype=torch.int32, device=dev)
        self.cta_counter = torch.zeros(1, dtype=torch.int32, device=dev)


class BiasedMF(RecModel):
    sample_num = 0          # no confounder items: the runner's per-epoch draw is an empty [n, 0] block
    use_cuda_graph = True

    @staticmethod
    def parse_model_args(parser, model_name='BiasedMF'):
        return RecModel.parse_model_args(parser, model_name)

    def __init__(self, label_min, label_max, feature_num, user_num, item_num, u_vector_size, i_vector_size,
                 random_seed, model_path):
        RecModel.__init__(self, label_min=label_min, label_max=label_max, feature_num=feature_num, user_num=user_num,
                          item_num=item_num, u_vector_size=u_vector_size, i_vector_size=i_vector_size,
                          random_seed=random_seed, model_path=model_path)
        self._ws = {}
        self._err_flag = None
        self._graphs = {}

    def _init_weights(self):
        RecModel._init_weights(self)
        self.user_bias = torch.nn.Embedding(self.user_num, 1)
        self.item_bias = torch.nn.Embedding(self.item_num, 1)
        self.global_bias = torch.nn.Parameter(torch.tensor(0.1))

    # ---- exposure scale: BiasedMF divides by exactly 1 ------------------------------------------------------
    def _scale(self):
        """(propensity [I] on the parameters' device, M): the prediction is divided by max(propensity_i, M)."""
        dev = self.uid_embeddings.weight.device
        ones = self.__dict__.get('_ones')
        if ones is None or ones.device != dev:
            ones = self.__dict__['_ones'] = torch.ones(self.item_num, dtype=torch.float32, device=dev)
        return ones, 1.0

    def factors(self):
        """The parameters as the IPS-MF factor dict of dccf_b200.synth.make_ipsmf_factors (device tensors, the scalars
        as floats): what DCCF(expo_factors=...), full_catalogue.ipsmf_exposure and evaluate_full_catalogue read."""
        return dict(self._factor_tensors(), mf_global_bias=float(self.global_bias.detach()))

    def _factor_tensors(self):
        prop, M = self._scale()
        return {'mf_user': self.uid_embeddings.weight.detach(), 'mf_item': self.iid_embeddings.weight.detach(),
                'mf_user_bias': self.user_bias.weight.detach().view(-1),
                'mf_item_bias': self.item_bias.weight.detach().view(-1), 'propensity': prop,
                'mf_min_propensity': float(M)}

    # ---- kernel plumbing -----------------------------------------------------------------------------------
    def _check_ready(self):
        w = self.uid_embeddings.weight
        if not w.is_cuda:
            raise RuntimeError('%s (dccf_b200) runs on CUDA only: move the model with .cuda(); there is no CPU fallback'
                               % type(self).__name__)
        if w.device.index is not None and w.device.index != torch.cuda.current_device():
            raise RuntimeError('the model lives on %s but the current CUDA device is %d: call torch.cuda.set_device(%d)'
                               % (w.device, torch.cuda.current_device(), w.device.index))
        if self.ui_vector_size != kernels.D:
            raise NotImplementedError('the kernels are compiled for u_vector_size = i_vector_size = %d' % kernels.D)
        if self._err_flag is None or self._err_flag.device != w.device:
            self._err_flag = torch.zeros(1, dtype=torch.int32, device=w.device)

    def _buf(self, name, shape, dtype):
        n = 1
        for s in shape:
            n *= int(s)
        cur = self._ws.get(name)
        if cur is None or cur.numel() < n or cur.dtype != dtype:
            cur = self._ws[name] = torch.empty(max(n, 1), dtype=dtype, device=self.uid_embeddings.weight.device)
        return cur[:n].view(*shape)

    def check_ids(self):
        """Raise if a kernel since the last check met a user / item id outside the tables (they clamp and flag)."""
        if self._err_flag is not None and int(self._err_flag.item()) != 0:
            self._err_flag.zero_()
            raise IndexError("user or item id out of range in feed_dict['X']")

    def _ids(self, X):
        X = X if torch.is_tensor(X) else torch.as_tensor(np.asarray(X))
        X = X.to(self.uid_embeddings.weight.device, torch.int64)
        if X.dim() != 2 or X.shape[1] < 2:
            raise ValueError("feed_dict['X'] must be [P, >=2] with uid in column 0 and iid in column 1")
        return X[:, :2].contiguous()

    # ---- reference protocol ----------------------------------------------------------------------------------
    def predict(self, feed_dict):
        """{'prediction': Tensor[P], 'check': []} — dccf_mf_scores; no autograd (training is train_step)."""
        self._check_ready()
        X = self._ids(feed_dict['X'])
        pred = torch.empty(X.shape[0], dtype=torch.float32, device=X.device)
        kernels.mf_scores(self._factor_tensors(), self.global_bias.data.view(1), X, pred, self._err_flag)
        return {'prediction': pred, 'check': []}

    def draw_confounders(self, n_pairs):
        """The model draws nothing: an empty [n_pairs, 0] block (the torch CPU generator is not touched)."""
        return torch.empty((n_pairs, 0), dtype=torch.int64)

    # ---- fused training step ---------------------------------------------------------------------------------
    def make_fused_optimizer(self, lr, l2, weight_decay=None, kind='adam', **kw):
        """State of the fused step for kind 'adam', 'gd' or 'adagrad' (torch.optim.Adam / SGD / Adagrad with
        weight_decay, as src/runners/BaseRunner.py:83-107 builds them)."""
        self._check_ready()
        return MFOptimizerState(self, lr=lr, l2=l2, weight_decay=l2 if weight_decay is None else weight_decay, kind=kind,
                                **kw)

    def _step(self, X, Y, loss_mode, opt, hp, counters=None, stage=None):
        """One training step on the current stream (every launch capturable).  X [P, 2] (with `stage` the static buffer
        the link kernel stages the batch into), Y [P] for MSE.  counters = step_dev: advanced by the touched-row
        launch's last CTA, with the batch cursor of `stage`.  Returns (prediction, loss) device tensors."""
        P = X.shape[0]
        D = self.ui_vector_size
        U, I = self.user_num, self.item_num
        eu, ei = self.uid_embeddings.weight.data, self.iid_embeddings.weight.data
        ub, ib, g = self.user_bias.weight.data, self.item_bias.weight.data, self.global_bias.data
        gu_rec, gi_rec = self._buf('gu_rec', (P, D), torch.float32), self._buf('gi_rec', (P, D), torch.float32)
        keys_u, keys_i = self._buf('keys_u', (P,), torch.int32), self._buf('keys_i', (P,), torch.int32)
        next_u, next_i = self._buf('next_u', (P,), torch.int32), self._buf('next_i', (P,), torch.int32)
        csr_u = (self._buf('rec_row_u', (P,), torch.int32), self._buf('csr_off_u', (U,), torch.int32),
                 self._buf('csr_u', (2 * P,), torch.int32), opt.csr_pool[0:2])
        csr_i = (self._buf('rec_row_i', (P,), torch.int32), self._buf('csr_off_i', (I,), torch.int32),
                 self._buf('csr_i', (2 * P,), torch.int32), opt.csr_pool[2:4])
        n_cta = kernels.mf_step_ctas(P)
        gb_rec = self._buf('gb_rec', (P,), torch.float32)
        g_user, g_item = self._buf('g_user_bias', (U,), torch.float32), self._buf('g_item_bias', (I,), torch.float32)
        g_part, loss_part = self._buf('g_part', (n_cta,), torch.float32), self._buf('loss_part', (n_cta,), torch.float32)
        pred, loss = self._buf('pred', (P,), torch.float32), self._buf('loss', (1,), torch.float32)
        su, si, sub_, sib, sg = (opt.state_of(k) for k in ('E_user', 'E_item', 'user_bias', 'item_bias', 'global_bias'))
        tables = [kernels.adam_table(eu, *su, keys_u, gu_rec, 1, P, P, P * D, opt.head_u, next_u, csr=csr_u),
                  kernels.adam_table(ei, *si, keys_i, gi_rec, 1, P, P, P * D, opt.head_i, next_i, csr=csr_i)]
        dense = [kernels.adam_tensor(ub, *sub_, g_user, 1, U), kernels.adam_tensor(ib, *sib, g_item, 1, I),
                 kernels.adam_tensor(g, *sg, g_part, n_cta, 1)]
        pf_user = tuple(t for t in (eu,) + su if t is not None)
        pf_item = tuple(t for t in (ei,) + si if t is not None)
        extra = kernels.make_link_extra(stage=stage, prefetch_user=pf_user, prefetch_item=pf_item,
                                        rec_rows=(csr_u[0], csr_i[0]))
        kernels.adam_link_ids(kernels.make_dims(U, I, 0, 0, 1), X, None, opt.head_u, next_u, opt.head_i, next_i,
                              n_seg=1, extra=extra)
        # every row the batch does not touch: the l2 / weight-decay update only, at full occupancy (nothing runs beside)
        kernels.adam_untouched(tables, hp, -1)
        kernels.adam_csr_build(tables)
        prop, M = self._scale()
        kernels.mf_step(eu, ei, ub, ib, g, prop, M, X, Y, loss_mode, pred, gu_rec, gi_rec, gb_rec, keys_u, keys_i, g_part,
                        loss_part, self._err_flag)
        kernels.mf_bias_grad(tables[0], tables[1], gb_rec, g_user, g_item, loss_part, n_cta,
                             1.0 / P if loss_mode == 1 else 1.0, loss)
        kernels.adam_touched(tables, dense, hp, True, None, 0, 0, opt.cta_counter, counters, None,
                             advance_cursor_dev=stage[1] if stage is not None else None)
        return pred, loss

    def train_step(self, feed_dict, opt=None):
        """One iteration of BaseRunner.fit (src/runners/BaseRunner.py:175-188): forward, BPR (rank 1) or MSE (rank 0),
        l2 term, backward, clip, GD / Adagrad / Adam — no autograd, no host sync.  From the second step of a batch shape
        on, the step is one CUDA-graph replay; the returned tensors are then the graph's outputs, valid until the next
        step."""
        opt = opt or self.optimizer
        if not isinstance(opt, MFOptimizerState):
            raise RuntimeError('train_step needs the fused optimizer state (model.make_fused_optimizer)')
        self._check_ready()
        X = self._ids(feed_dict['X'])
        loss_mode = 0 if feed_dict['rank'] == 1 else 1
        Y = feed_dict['Y'].to(X.device, torch.float32).contiguous() if loss_mode == 1 else None
        if X.shape[0] == 0:
            raise ValueError('empty batch')
        if self.use_cuda_graph:
            key = (X.shape[0], loss_mode, opt, False)
            g = self._graphs.get(key)
            if g == 'warm':
                g = self._graphs[key] = self._build_graph(X.shape[0], loss_mode, opt, staged=False)
            if g is not None:
                g['X'].copy_(X, non_blocking=True)
                if Y is not None:
                    g['Y'].copy_(Y, non_blocking=True)
                return self._replay(g, opt)
            self._graphs[key] = 'warm'      # first step of this shape runs eagerly (and loads every kernel)
        opt.step_count += 1
        pred, loss = self._step(X, Y, loss_mode, opt, opt.hp())
        return {'prediction': pred.clone(), 'check': [('prediction', pred.clone())], 'loss': loss[0].clone()}

    def _build_graph(self, P, loss_mode, opt, staged):
        dev = self.uid_embeddings.weight.device
        g = {'X': torch.zeros((P, 2), dtype=torch.int64, device=dev), 'Y': torch.zeros(P, dtype=torch.float32, device=dev),
             'step_dev': torch.zeros(1, dtype=torch.int32, device=dev), 'synced': None}
        stage = None
        if staged:
            # [X_epoch, sample_epoch (unused: S = 0), 4 x unused, Y_epoch (rank 0)]
            g['epoch_ptrs'] = torch.zeros(7, dtype=torch.int64, device=dev)
            g['cursor'] = torch.zeros(1, dtype=torch.int64, device=dev)
            g['stage_counter'] = torch.zeros(1, dtype=torch.int32, device=dev)
            # (the sample-item output of the staging is never written with S = 0: any valid address)
            stage = (g['epoch_ptrs'], g['cursor'], g['X'], g['X'], g['stage_counter'],
                     g['Y'] if loss_mode == 1 else None)
        hp = opt.hp(step=1, step_dev=g['step_dev'])
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        before = kernels.LAUNCHES[0]
        with torch.cuda.graph(graph, capture_error_mode='thread_local'):
            pred, loss = self._step(g['X'], g['Y'] if loss_mode == 1 else None, loss_mode, opt, hp,
                                    counters=g['step_dev'], stage=stage)
        g.update({'graph': graph, 'pred': pred, 'loss': loss, 'n_kernels': kernels.LAUNCHES[0] - before,
                  'keep_alive': (dict(self._ws), opt, self._err_flag)})
        kernels.LAUNCHES[0] = before
        return g

    def _replay(self, g, opt):
        opt.step_count += 1
        if g['synced'] != opt.step_count:
            g['step_dev'].fill_(opt.step_count)      # eager steps ran in between
        g['graph'].replay()
        kernels.LAUNCHES[0] += g['n_kernels']
        g['synced'] = opt.step_count + 1
        return {'prediction': g['pred'], 'check': [('prediction', g['pred'])], 'loss': g['loss'][0]}

    def resident_epoch_available(self, P, opt=None):
        opt = opt or self.optimizer
        return isinstance(opt, MFOptimizerState) and self.use_cuda_graph

    def begin_resident_epoch(self, X_epoch, sample_epoch, dropout, opt=None, Y_epoch=None):
        """Training over a device-resident epoch: X_epoch [n, P, 2] int64 CUDA (rank 1: BPR batches; with Y_epoch [n, P]
        float32 CUDA, rank 0: MSE batches).  sample_epoch (the runner's [n, P, 0] confounder block) and dropout are not
        used.  Returns a callable that runs the next batch as one CUDA-graph replay: the link kernel stages the batch
        from the epoch through a device-side cursor, which the touched-row launch advances."""
        opt = opt or self.optimizer
        if not self.resident_epoch_available(X_epoch.shape[1], opt):
            return None
        self._check_ready()
        n, P = X_epoch.shape[0], X_epoch.shape[1]
        loss_mode = 0 if Y_epoch is None else 1
        if Y_epoch is not None and (tuple(Y_epoch.shape) != (n, P) or Y_epoch.dtype != torch.float32 or
                                    Y_epoch.device != X_epoch.device):
            raise ValueError('Y_epoch must be float32 [%d, %d] on %s' % (n, P, X_epoch.device))
        if n == 0:
            return None
        key = (P, loss_mode, opt, True)
        state = {'next': 0}
        if key not in self._graphs:
            saved = self.use_cuda_graph
            self.use_cuda_graph = False             # the very first step runs launch by launch
            try:
                fd = {'X': X_epoch[0], 'rank': 1 if Y_epoch is None else 0}
                if Y_epoch is not None:
                    fd['Y'] = Y_epoch[0]
                state['first'] = self.train_step(fd, opt)
            finally:
                self.use_cuda_graph = saved
            state['next'] = 1
            self._graphs[key] = self._build_graph(P, loss_mode, opt, staged=True)
        g = self._graphs[key]
        X_epoch = X_epoch.contiguous()
        keep = [X_epoch]
        ptrs = [X_epoch.data_ptr(), 0, 0, 0, 0, 0, 0]
        if Y_epoch is not None:
            Y_epoch = Y_epoch.contiguous()
            ptrs[6] = Y_epoch.data_ptr()
            keep.append(Y_epoch)
        g['epoch_ptrs'].copy_(torch.tensor(ptrs, dtype=torch.int64))
        g['cursor'].fill_(state['next'])
        g['keep'] = tuple(keep)

        def step():
            if state['next'] >= n:
                raise StopIteration('resident epoch exhausted')
            state['next'] += 1
            return self._replay(g, opt)

        step.remaining = lambda: n - state['next']
        step.first = state.get('first')
        return step

    # ---- checkpoints with optimizer state ---------------------------------------------------------------------
    def save_training_state(self, path=None):
        """Weights (the reference's state_dict keys) + fused-optimizer state and step count."""
        path = path or (self.model_path + '.train_state')
        dir_path = os.path.dirname(path)
        if dir_path and not os.path.exists(dir_path):
            os.makedirs(dir_path)
        opt = self.optimizer.state_dict() if isinstance(self.optimizer, MFOptimizerState) else None
        torch.save({'model': self.state_dict(), 'optimizer': opt}, path)
        return path

    def load_training_state(self, path=None):
        path = path or (self.model_path + '.train_state')
        st = torch.load(path, map_location=self.uid_embeddings.weight.device)
        self.load_state_dict(st['model'])
        if st['optimizer'] is not None:
            if not isinstance(self.optimizer, MFOptimizerState):
                o = st['optimizer']
                self.optimizer = self.make_fused_optimizer(lr=o['lr'], l2=o['l2'], weight_decay=o['weight_decay'],
                                                           kind=o.get('kind', 'adam'))
            self.optimizer.load_state_dict(st['optimizer'])
        return self
