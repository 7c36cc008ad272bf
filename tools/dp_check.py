"""Multi-GPU check, run under torchrun (world >= 2): a data-parallel fused step over W ranks equals the
single-GPU step on the concatenated batch, replicas stay bit-identical, user-sharded evaluation equals the
single-GPU evaluation.  Prints 'DP CHECK OK' on rank 0.

    torchrun --nproc-per-node 2 tools/dp_check.py [--optimizer adam|gd|adagrad] [--rank 0|1]

--optimizer: the fused optimizer of both runs (default adam); its state (exp_avg for Adam, state_sum for Adagrad) is
compared as well.  --rank: the task of src/main.py, 1 (default) top-N ranking with the BPR loss, 0 rating prediction
with the MSE loss — there the loss of a global step is the mean over the pairs of all ranks, compared as well."""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from test_gpu_parity import make_model, model_params, random_problem  # noqa: E402


def say(rank, msg):
    print('[dp_check rank %d] %s' % (rank, msg), flush=True)


def rel(a, b):
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max() / np.abs(b).max())


def close(a, b, tol, what):
    """Data-parallel ranks and the single GPU split K / rows differently (different tile counts), so a
    pre-activation within 1e-7 of zero can pass the ReLU on one side only: the derivative of that one element (and
    the row of dW it feeds, 1/64 of W) then differs legitimately.  Hence: 98 % of the entries within `tol` of the
    reference (relative to its largest entry), the rest within 2e-2 — a wrong segment, a missing rank or a
    misplaced record moves most entries by far more."""
    err = np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.abs(b).max()
    q = float(np.quantile(err, 0.98))
    assert q < tol and float(err.max()) < 2e-2, '%s: 98th percentile %.3g, max %.3g' % (what, q, float(err.max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--optimizer', choices=('adam', 'gd', 'adagrad'), default='adam')
    ap.add_argument('--rank', type=int, choices=(0, 1), default=1)
    cli = ap.parse_args()
    kind, task = cli.optimizer, cli.rank
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    U, I, F, S, A, std, drop = 300, 400, 768, 10, 2, 0.1, 0.2
    b_loc = 32
    P = 2 * b_loc * world
    params, X, si, noise, mask = random_problem(17, U, I, F, P, S, A, std, drop)
    R = (S + 1) * A
    b = P // 2
    if task == 1:
        # rank r owns positives [r*b_loc, (r+1)*b_loc) and their negatives
        pos = np.arange(rank * b_loc, (rank + 1) * b_loc)
        pairs = np.concatenate([pos, b + pos])
        labels = np.zeros(P, dtype=np.float32)
    else:
        # rank r owns pairs [r*2*b_loc, (r+1)*2*b_loc) with their ratings
        pairs = np.arange(rank * 2 * b_loc, (rank + 1) * 2 * b_loc)
        labels = np.random.RandomState(3).uniform(1.0, 5.0, P).astype(np.float32)
    rows = (pairs[:, None] * R + np.arange(R)[None, :]).reshape(-1)
    model = make_model(params, S, A, std)
    model.enable_data_parallel(p2p=os.environ.get('DCCF_DP_P2P', '1') == '1')
    model.optimizer = model.make_fused_optimizer(lr=1e-3, l2=1e-4, kind=kind)
    steps = 2
    for t in range(steps):
        fd = {'X': torch.from_numpy(X[pairs]).cuda(), 'rank': task, 'train': True, 'dropout': drop,
              'Y': torch.from_numpy(labels[pairs]).cuda(), 'sample_item': torch.from_numpy(si[pairs]),
              'noise': torch.from_numpy(noise[rows]), 'dropout_mask': torch.from_numpy(mask[rows])}
        out = model.train_step(fd)
    say(rank, 'dp steps done (exchange=%s), loss %.6f' % (model._exchange_for(len(pairs)).mode, float(out['loss'])))
    got = model_params(model)
    # replicas bit-identical
    for k, v in got.items():
        t = torch.from_numpy(v).cuda()
        ref = t.clone()
        dist.broadcast(ref, 0)
        assert torch.equal(t, ref), 'rank %d diverged from rank 0 on %s' % (rank, k)
    # equals the single-GPU step on the whole batch
    single = make_model(params, S, A, std)
    single.optimizer = single.make_fused_optimizer(lr=1e-3, l2=1e-4, kind=kind)
    for t in range(steps):
        fd = {'X': torch.from_numpy(X).cuda(), 'rank': task, 'train': True, 'dropout': drop,
              'Y': torch.from_numpy(labels).cuda(),
              'sample_item': torch.from_numpy(si), 'noise': torch.from_numpy(noise),
              'dropout_mask': torch.from_numpy(mask)}
        out1 = single.train_step(fd)
    say(rank, 'single-GPU steps done')
    want = model_params(single)
    assert abs(float(out['loss']) - float(out1['loss'])) < 1e-5 * abs(float(out1['loss'])), (float(out['loss']), float(out1['loss']))
    for k in ('E_user', 'E_item', 'b'):
        close(got[k], want[k], 1e-5, k)
    close(got['W'], want['W'], 5e-4, 'W')
    state = {'adam': 'exp_avg', 'adagrad': 'state_sum', 'gd': None}[kind]
    for k in (('E_user', 'E_item', 'W', 'b') if state else ()):
        close(getattr(model.optimizer, state)[k].cpu().numpy(), getattr(single.optimizer, state)[k].cpu().numpy(), 1e-5,
              state + ' ' + k)

    say(rank, 'equality with the single-GPU step ok')
    # DP steps on the library's own rng streams keep the replicas identical too
    for t in range(4):
        fd = {'X': torch.from_numpy(X[pairs]).cuda(), 'rank': task, 'train': True, 'dropout': drop,
              'Y': torch.from_numpy(labels[pairs]).cuda(), 'sample_item': torch.from_numpy(si[pairs])}
        model.train_step(fd)
    for k, v in model_params(model).items():
        t = torch.from_numpy(v).cuda()
        ref = t.clone()
        dist.broadcast(ref, 0)
        assert torch.equal(t, ref), 'rank %d diverged from rank 0 on %s after graph replay' % (rank, k)

    say(rank, 'library-rng DP steps ok (exchange=%s, graphs=%d)' % (model._exchange_for(len(pairs)).mode, len(getattr(model, '_graphs', {}))))
    # user-sharded evaluation == single-GPU evaluation (same scores -> same metrics)
    from dccf_b200.dist import all_reduce_sum, shard_users
    from dccf_b200.models.BaseModel import BaseModel
    rs = np.random.RandomState(5)
    n_users, n_c = 40, 101
    uid = np.repeat(rs.choice(U, n_users, replace=False), n_c)
    iid = np.concatenate([rs.choice(I, n_c, replace=False) for _ in range(n_users)])
    Yl = np.zeros(len(uid), dtype=np.float32)
    Yl[::n_c] = 1
    scores = rs.standard_normal(len(uid)).astype(np.float32)
    data = {'uid': uid, 'iid': iid, 'Y': Yl}
    want_m = BaseModel.evaluate_method(scores, data, ['ndcg@5', 'recall@5', 'precision@5'])
    mine = shard_users(uid, rank, world)
    shard = {k: v[mine] for k, v in data.items()}
    sums, counts = BaseModel.evaluate_sums(scores[mine], shard, ['ndcg@5', 'recall@5', 'precision@5'])
    tot = all_reduce_sum(list(sums) + list(counts))
    got_m = [tot[i] / tot[3 + i] for i in range(3)]
    assert np.abs(np.array(got_m) - np.array(want_m)).max() < 1e-9, (got_m, want_m)
    dist.barrier()
    if rank == 0:
        print('DP CHECK OK world=%d optimizer=%s rank=%d' % (world, kind, task))
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
