"""Train / evaluate driver with the interface of the reference's src/runners/BaseRunner.py:16-355.

Same flags, constructor, `train / fit / predict / evaluate / check / eva_termination`, same log lines and
model-selection rules.  Differences are confined to where the time goes:

  * `fit` — when the model offers `train_step` (dccf_b200's DCCF), each batch is ONE fused step (forward, loss,
    l2 term, backward, clip(+-50), GD / Adagrad / Adam step; BaseRunner.py:175-188) with no autograd and no host
    synchronisation; the loss of the last batch is read back once per epoch.  Any other model goes through the
    reference's autograd sequence and torch optimizer unchanged.
  * `predict` — predictions stay on the device across batches and are re-ordered to data order with one
    vectorised scatter instead of a Python dict with one entry per row (BaseRunner.py:148-156).
  * `evaluate` — ranking metrics come from the dccf_rank_eval kernel on the device-resident predictions.
"""
import logging
import os
from time import time

import numpy as np
import pandas as pd
import torch
from tqdm import tqdm

from ..utils import global_p, utils


class BaseRunner(object):
    @staticmethod
    def parse_runner_args(parser):
        """Flags and defaults of BaseRunner.py:18-48."""
        parser.add_argument('--load', type=int, default=0, help='Whether load model and continue to train')
        parser.add_argument('--epoch', type=int, default=100, help='Number of epochs.')
        parser.add_argument('--check_epoch', type=int, default=1, help='Check every epochs.')
        parser.add_argument('--early_stop', type=int, default=1, help='whether to early-stop.')
        parser.add_argument('--lr', type=float, default=0.01, help='Learning rate.')
        parser.add_argument('--batch_size', type=int, default=128, help='Batch size during training.')
        parser.add_argument('--eval_batch_size', type=int, default=128 * 128, help='Batch size during testing.')
        parser.add_argument('--dropout', type=float, default=0.2, help='Dropout probability for each deep layer')
        parser.add_argument('--l2', type=float, default=1e-4, help='Weight of l2_regularize in loss.')
        parser.add_argument('--optimizer', type=str, default='GD', help='optimizer: GD, Adam, Adagrad')
        parser.add_argument('--metric', type=str, default='RMSE',
                            help='metrics: RMSE, MAE, AUC, F1, Accuracy, Precision, Recall')
        parser.add_argument('--skip_eval', type=int, default=0, help='number of epochs without evaluation')
        return parser

    def __init__(self, optimizer='GD', learning_rate=0.01, epoch=100, batch_size=128, eval_batch_size=128 * 128,
                 dropout=0.2, l2=1e-5, metrics='RMSE', check_epoch=10, early_stop=1):
        self.optimizer_name = optimizer
        self.learning_rate = learning_rate
        self.epoch = epoch
        self.batch_size = batch_size
        self.eval_batch_size = eval_batch_size
        self.dropout = dropout
        self.no_dropout = 0.0
        self.l2_weight = l2
        self.metrics = metrics.lower().split(',')
        self.check_epoch = check_epoch
        self.early_stop = early_stop
        self.time = None
        self.train_results, self.valid_results, self.test_results = [], [], []
        self.show_progress = True
        self._shards = {}          # id(data) -> (data, rows, shard dict, batches): user-sharded evaluation sets

    # ---- optimizer ---------------------------------------------------------------------------
    def _build_optimizer(self, model):
        """SGD / Adagrad / Adam, all with weight_decay = l2 (BaseRunner.py:83-107).  On a model that has the fused
        step, the state of each lives in the fused optimizer state (make_fused_optimizer) instead of a torch optimizer."""
        name = self.optimizer_name.lower()
        if name == 'adam':
            logging.info('Optimizer: Adam')
            if hasattr(model, 'make_fused_optimizer'):
                return model.make_fused_optimizer(lr=self.learning_rate, l2=self.l2_weight, weight_decay=self.l2_weight)
            return torch.optim.Adam(model.parameters(), lr=self.learning_rate, weight_decay=self.l2_weight)
        if name == 'adagrad':
            logging.info('Optimizer: Adagrad')
            if hasattr(model, 'make_fused_optimizer'):
                return model.make_fused_optimizer(lr=self.learning_rate, l2=self.l2_weight, weight_decay=self.l2_weight,
                                                  kind='adagrad')
            return torch.optim.Adagrad(model.parameters(), lr=self.learning_rate, weight_decay=self.l2_weight)
        if name == 'gd':
            logging.info('Optimizer: GD')
            if hasattr(model, 'make_fused_optimizer'):
                return model.make_fused_optimizer(lr=self.learning_rate, l2=self.l2_weight, weight_decay=self.l2_weight,
                                                  kind='gd')
            return torch.optim.SGD(model.parameters(), lr=self.learning_rate, weight_decay=self.l2_weight)
        logging.error('Unknown Optimizer: ' + self.optimizer_name)
        assert self.optimizer_name in ['GD', 'Adagrad', 'Adam']
        return torch.optim.SGD(model.parameters(), lr=self.learning_rate, weight_decay=self.l2_weight)

    def _check_time(self, start=False):
        """[start, last] wall-clock pair; returns seconds since the previous call (BaseRunner.py:109-120)."""
        if self.time is None or start:
            self.time = [time()] * 2
            return self.time[0]
        last = self.time[1]
        self.time[1] = time()
        return self.time[1] - last

    def batches_add_control(self, batches, train):
        """'train' flag and dropout probability per batch: --dropout when training, 0 otherwise
        (BaseRunner.py:122-132)."""
        for batch in batches:
            batch['train'] = train
            batch['dropout'] = self.dropout if train else self.no_dropout
        return batches

    def _bar(self, it, **kw):
        return tqdm(it, leave=False, ncols=100, mininterval=1, disable=not self.show_progress, **kw)

    # ---- inference ---------------------------------------------------------------------------
    def _predict_device(self, model, data, data_processor):
        """Predictions in DATA order as one device tensor (no per-batch device->host copy)."""
        batches = data_processor.prepare_batches(data, self.eval_batch_size, train=False)
        batches = self.batches_add_control(batches, train=False)
        model.eval()
        with torch.no_grad():
            if hasattr(model, 'predict_many'):
                outs = [o.detach() for o in model.predict_many(batches)]
            else:
                outs = [model.predict(batch)['prediction'].detach() for batch in self._bar(batches, desc='Predict')]
        pred = torch.cat(outs) if len(outs) > 1 else outs[0]
        want = np.asarray(data[global_p.K_SAMPLE_ID])
        if self._slices_of(batches, want):
            return pred                         # batches are consecutive slices of `data`: already in data order
        sample_ids = np.concatenate([b[global_p.K_SAMPLE_ID] for b in batches])
        if len(sample_ids) == len(want) and np.array_equal(sample_ids, want):
            return pred
        # general case: position of every requested sample id inside the batch stream
        order = np.argsort(sample_ids, kind='stable')
        pos = order[np.searchsorted(sample_ids[order], want)]
        return pred[torch.from_numpy(pos).to(pred.device)]

    @staticmethod
    def _slices_of(batches, want):
        """True when the batches' sample-id arrays are back-to-back views of `want` itself (what prepare_batches
        hands out for evaluation sets) — decided from addresses, without touching the 4.8e7 ids of a 1000-negative
        test set on every evaluation."""
        if want.ndim != 1 or not want.flags['C_CONTIGUOUS']:
            return False
        at = want.__array_interface__['data'][0]
        for b in batches:
            s = b[global_p.K_SAMPLE_ID]
            if not isinstance(s, np.ndarray) or s.dtype != want.dtype or s.ndim != 1 or \
                    not s.flags['C_CONTIGUOUS'] or s.__array_interface__['data'][0] != at:
                return False
            at += s.nbytes
        return at == want.__array_interface__['data'][0] + want.nbytes

    def predict(self, model, data, data_processor):
        """np.ndarray of predictions aligned with `data` (BaseRunner.py:134-157).  Under data parallelism every
        rank scores its own users and the pieces are gathered, so all ranks return the full array."""
        if self._world(model) > 1:
            import torch.distributed as dist
            rows, pred, _ = self._predict_shard(model, data, data_processor)
            pieces = [None] * dist.get_world_size()
            dist.all_gather_object(pieces, (rows, pred.cpu().numpy()))
            out = np.empty(len(data['Y']), dtype=np.float32)
            for r, p in pieces:
                out[r] = p
            return out
        return self._predict_device(model, data, data_processor).cpu().numpy()

    # ---- user-sharded evaluation (new: the reference is single-process, SURVEY.md §8e) ---------------
    @staticmethod
    def _world(model):
        from ..dist import is_distributed
        if getattr(model, '_dp', None) is None or not is_distributed():
            return 1
        return model._dp['world']

    def _predict_shard(self, model, data, data_processor):
        """(row indices owned by this rank, device predictions for them): contiguous user blocks, all
        candidates of a user on one rank."""
        from ..dist import shard_users
        hit = self._shards.get(id(data))
        if hit is None or hit[0] is not data:
            rows = shard_users(data['uid'], model._dp['rank'], model._dp['world'])
            shard = {k: (np.asarray(v)[rows] if hasattr(v, '__len__') and len(v) == len(data['Y']) else v)
                     for k, v in data.items()}
            shard[global_p.K_SAMPLE_ID] = np.arange(len(rows))
            hit = (data, rows, shard)
            self._shards[id(data)] = hit
        _, rows, shard = hit
        saved = data_processor.vt_batches_buffer
        key = ('shard', id(data), self.eval_batch_size)
        if key not in saved:
            saved[key] = data_processor._prepare_batches_rk(shard, self.eval_batch_size, train=False) \
                if data_processor.rank == 1 else data_processor._prepare_batches_rt(shard, self.eval_batch_size, False)
        batches = self.batches_add_control(saved[key], train=False)
        model.eval()
        with torch.no_grad():
            if hasattr(model, 'predict_many'):
                outs = [o.detach() for o in model.predict_many(batches)]
            else:
                outs = [model.predict(batch)['prediction'].detach() for batch in self._bar(batches, desc='Predict')]
        return rows, (torch.cat(outs) if len(outs) > 1 else outs[0]), shard

    # ---- training ----------------------------------------------------------------------------
    def fit(self, model, data, data_processor, epoch=-1):
        """One epoch over `data`; returns the out_dict of the last batch (BaseRunner.py:159-191)."""
        if model.optimizer is None:
            model.optimizer = self._build_optimizer(model)
        batches = data_processor.prepare_batches(data, self.batch_size, train=True)
        batches = self.batches_add_control(batches, train=True)
        batch_size = self.batch_size if data_processor.rank == 0 else self.batch_size * 2
        model.train()
        fused = hasattr(model, 'train_step') and not isinstance(model.optimizer, torch.optim.Optimizer)
        accumulate_size = 0
        output_dict = None
        world = self._world(model)
        suspended = None
        if world > 1:
            if not (fused and hasattr(model, 'begin_resident_epoch')):
                raise RuntimeError('data-parallel training (torchrun) supports only the fused step of DCCF (GD, '
                                   'Adagrad or Adam): not other models or torch optimizers')
            from ..dist import sync_host_rng
            sync_host_rng(model)            # sharded evaluation left the ranks' generators at different positions
        if fused and hasattr(model, 'begin_resident_epoch') and (len(batches) > 2 or world > 1) \
                and batches[0]['X'].is_cuda:
            # Equal-size batches run from a device-resident epoch: the confounder draws of all of them are ONE
            # torch.randint call (same CPU-generator stream as the reference's per-batch calls, DCCF.py:72) and
            # each step is a single CUDA-graph launch that fetches its batch (with --rank 0 also its labels) through a
            # device-side cursor.
            # Data parallel (world > 1): global step k = batches k*world .. k*world + world - 1, one per rank; every
            # rank draws the confounders of all of them (generators stay in step) and keeps its own slice.
            from ..dist import rank_slice_of_draws, step_partition
            rank = model._dp['rank'] if world > 1 else 0
            P0 = batches[0]['X'].shape[0]
            n_full = 0
            while n_full < len(batches) and batches[n_full]['X'].shape[0] == P0:
                n_full += 1
            mine, _ = step_partition(n_full, world, rank)
            chunk = 1024
            done = 0                                    # global steps run so far
            if hasattr(model, 'resident_epoch_available') and not model.resident_epoch_available(P0):
                # no CUDA-graph step for this configuration: nothing has been drawn from the torch CPU generator yet,
                # so the step-by-step loop below consumes it exactly as the reference does
                if world > 1:
                    raise RuntimeError('data-parallel training needs the CUDA-graph step (peer-memory exchange)')
                mine = []
            while done < len(mine):
                m = min(chunk, len(mine) - done)
                X_epoch = torch.stack([batches[i]['X'] for i in mine[done:done + m]])
                draws = model.draw_confounders(m * world * P0).view(m * world, P0, model.sample_num)
                draws = rank_slice_of_draws(draws, world, rank) if world > 1 else draws
                draws = draws.to(X_epoch.device, non_blocking=True)
                if data_processor.rank == 1:
                    step = model.begin_resident_epoch(X_epoch, draws, self.dropout)
                else:
                    # rating prediction (MSE): this rank's own labels beside its batches
                    Y_epoch = torch.stack([batches[i]['Y'] for i in mine[done:done + m]]).float()
                    step = model.begin_resident_epoch(X_epoch, draws, self.dropout, Y_epoch=Y_epoch)
                if step is None:
                    if world > 1:
                        raise RuntimeError('data-parallel training needs the CUDA-graph step (peer-memory exchange)')
                    break
                if step.first is not None:
                    output_dict = step.first
                while step.remaining() > 0:
                    output_dict = step()
                done += m
            if done > 0:
                output_dict = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in output_dict.items()
                               if k != 'check'}
                output_dict['check'] = [('prediction', output_dict['prediction'])]
            batches = batches[done * world:]
            if world > 1 and batches:
                # what does not fill a global step (< world full batches + the ragged last one): every rank runs these
                # steps itself, un-exchanged, on identical inputs — replicas stay bit-identical, no sample is dropped
                suspended = model.data_parallel_suspended()
                suspended.__enter__()
        try:
            output_dict = self._fit_remaining(model, batches, fused, batch_size, epoch, output_dict)
        finally:
            if suspended is not None:
                suspended.__exit__(None, None, None)
        model.eval()
        if hasattr(model, 'check_ids'):
            model.check_ids()
        return output_dict

    def _fit_remaining(self, model, batches, fused, batch_size, epoch, output_dict):
        """Batches that did not go through the device-resident epoch: step by step."""
        accumulate_size = 0
        if fused and hasattr(model, 'draw_confounders') and batches:
            # forward + (loss + l2) backward + clip + step in one go: the reference steps on every batch
            # (accumulate_size >= batch_size always holds for its batch layout, BaseRunner.py:176,186-188).
            # The confounder draw of batch k+1 (torch CPU generator, DCCF.py:72) is made while batch k runs.
            draw = model.draw_confounders(batches[0]['X'].shape[0])
            for k, batch in enumerate(self._bar(batches, desc='Epoch %5d' % (epoch + 1))):
                fd = dict(batch)
                fd['sample_item'] = draw
                output_dict = model.train_step(fd)
                if k + 1 < len(batches):
                    draw = model.draw_confounders(batches[k + 1]['X'].shape[0])
            batches = []
        for batch in self._bar(batches, desc='Epoch %5d' % (epoch + 1)):
            if fused:
                output_dict = model.train_step(batch)
                continue
            accumulate_size += len(batch['Y'])
            model.optimizer.zero_grad()
            output_dict = model(batch)
            loss = output_dict['loss'] + model.l2() * self.l2_weight
            loss.backward()
            torch.nn.utils.clip_grad_value_(model.parameters(), 50)
            if accumulate_size >= batch_size or batch is batches[-1]:
                model.optimizer.step()
                accumulate_size = 0
        return output_dict

    def eva_termination(self, model):
        """Early-stopping rule on the validation history (BaseRunner.py:193-210)."""
        metric = self.metrics[0]
        valid = self.valid_results
        if len(valid) > 20 and metric in utils.LOWER_METRIC_LIST and utils.strictly_increasing(valid[-5:]):
            return True
        if len(valid) > 20 and metric not in utils.LOWER_METRIC_LIST and utils.strictly_decreasing(valid[-5:]):
            return True
        if len(valid) - valid.index(utils.best_result(metric, valid)) > 20:
            return True
        return False

    def _eval_or_default(self, model, data, data_processor, metrics=None):
        if data is None:
            return [-1.0] * len(self.metrics)
        return self.evaluate(model, data, data_processor, metrics=metrics)

    def train(self, model, data_processor, skip_eval=0):
        """The epoch loop with evaluation, model selection and early stop (BaseRunner.py:212-303)."""
        train_data = data_processor.get_train_data(epoch=-1)
        validation_data = data_processor.get_validation_data()
        test_data = data_processor.get_test_data()
        self._check_time(start=True)
        init_train = self._eval_or_default(model, train_data, data_processor, metrics=['rmse', 'mae'])
        init_valid = self._eval_or_default(model, validation_data, data_processor)
        init_test = self._eval_or_default(model, test_data, data_processor)
        logging.info('Init: \t train= %s validation= %s test= %s [%.1f s] ' % (
            utils.format_metric(init_train), utils.format_metric(init_valid), utils.format_metric(init_test),
            self._check_time()) + ','.join(self.metrics))
        try:
            for epoch in range(self.epoch):
                self._check_time()
                epoch_train_data = data_processor.get_train_data(epoch=epoch)
                last_batch = self.fit(model, epoch_train_data, data_processor, epoch=epoch)
                if self.check_epoch > 0 and (epoch == 1 or epoch % self.check_epoch == 0):
                    self.check(model, last_batch)
                training_time = self._check_time()
                if epoch >= skip_eval:
                    train_result = self._eval_or_default(model, train_data, data_processor, metrics=['rmse', 'mae'])
                    valid_result = self._eval_or_default(model, validation_data, data_processor)
                    test_result = self._eval_or_default(model, test_data, data_processor)
                    testing_time = self._check_time()
                    self.train_results.append(train_result)
                    self.valid_results.append(valid_result)
                    self.test_results.append(test_result)
                    logging.info('Epoch %5d [%.1f s]\t train= %s validation= %s test= %s [%.1f s] '
                                 % (epoch + 1, training_time, utils.format_metric(train_result),
                                    utils.format_metric(valid_result), utils.format_metric(test_result), testing_time)
                                 + ','.join(self.metrics))
                    if utils.best_result(self.metrics[0], self.valid_results) == self.valid_results[-1]:
                        model.save_model()
                    if self.eva_termination(model) and self.early_stop == 1:
                        logging.info('Early stop at %d based on validation result.' % (epoch + 1))
                        break
                if epoch < skip_eval:
                    logging.info('Epoch %5d [%.1f s]' % (epoch + 1, training_time))
        except KeyboardInterrupt:
            logging.info('Early stop manually')
            save_here = input('Save here? (1/0) (default 0):')
            if str(save_here).lower().startswith('1'):
                model.save_model()
        if self.valid_results:
            for name, results in (('validation', self.valid_results), ('test', self.test_results)):
                best = utils.best_result(self.metrics[0], results)
                best_epoch = results.index(best)
                logging.info('Best Iter(%s)= %5d\t train= %s valid= %s test= %s [%.1f s] '
                             % (name, best_epoch + 1, utils.format_metric(self.train_results[best_epoch]),
                                utils.format_metric(self.valid_results[best_epoch]),
                                utils.format_metric(self.test_results[best_epoch]), self.time[1] - self.time[0])
                             + ','.join(self.metrics))
            model.load_model()

    # ---- evaluation --------------------------------------------------------------------------
    def evaluate(self, model, data, data_processor, metrics=None, write_rank=False):
        """Metric values of the model on `data` (BaseRunner.py:305-332); `write_rank` dumps
        uid/iid/score/label sorted by uid to <dataset dir>/rank.csv (tab separated)."""
        if metrics is None:
            metrics = self.metrics
        if self._world(model) > 1 and not write_rank:
            # every rank evaluates its users; sums and user counts are all-reduced (one small collective)
            from ..dist import all_reduce_sum
            rows, pred, shard = self._predict_shard(model, data, data_processor)
            sums, counts = model.evaluate_sums(pred, shard, metrics)
            tot = all_reduce_sum(list(sums) + list(counts))
            n = len(metrics)
            return [float(np.sqrt(tot[i] / tot[n + i])) if metrics[i] == 'rmse' else float(tot[i] / tot[n + i])
                    for i in range(n)]
        pred = self._predict_device(model, data, data_processor)
        if write_rank and (self._world(model) == 1 or model._dp['rank'] == 0):
            df = pd.DataFrame()
            df['uid'] = data['uid']
            df['iid'] = data['iid']
            df['score'] = pred.cpu().numpy()
            df['label'] = data['Y']
            df = df.sort_values(by='uid')
            df.to_csv(os.path.join(data_processor.data_loader.path, global_p.RANK_FILE_NAME), sep='\t', index=False)
        needs_host = any('@' not in m for m in metrics)
        p = pred.cpu().numpy() if needs_host else pred
        return model.evaluate_method(p, data, metrics=metrics)

    def check(self, model, out_dict):
        """Log the 'check' tensors, loss and l2 of a batch; warn when l2 is out of proportion
        (BaseRunner.py:334-355)."""
        logging.info(os.linesep)
        for name, t in out_dict['check']:
            d = t.detach().cpu().numpy()
            logging.info(os.linesep.join([name + '\t' + str(d.shape), np.array2string(d, threshold=20)]) + os.linesep)
        loss = out_dict['loss'].detach()
        with torch.no_grad():
            l2 = model.l2() * self.l2_weight
        logging.info('loss = %.4f, l2 = %.4f' % (loss, l2))
        if not (loss.abs() * 0.005 < l2 < loss.abs() * 0.1):
            logging.warning('l2 inappropriate: loss = %.4f, l2 = %.4f' % (loss, l2))
