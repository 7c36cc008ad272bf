"""Evaluate a DCCF checkpoint over the whole catalogue: every item the user has not interacted with is a candidate.

    python tools/full_catalogue_eval.py --path ../datasets/ --dataset yelp --model_path ../model/DCCF/m.pt \\
        --metric ndcg@10,recall@10,precision@10
    python -m torch.distributed.run --nproc-per-node N tools/full_catalogue_eval.py <same flags>

Builds the reference's DataLoader and a DCCF model with the deterministic predictor (sample_num 0, std 0 — a
checkpoint trained with confounders loads into it unchanged), loads the checkpoint and prints one JSON line of metrics
(dccf_b200.full_catalogue.evaluate_full_catalogue).  Under torchrun the evaluated users are split between the ranks.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def main(argv=None):
    from dccf_b200 import dist as dp
    from dccf_b200 import synth
    from dccf_b200.data_loaders.DataLoader import DataLoader
    from dccf_b200.full_catalogue import evaluate_full_catalogue
    from dccf_b200.models.DCCF import DCCF

    ap = argparse.ArgumentParser(description='full-catalogue evaluation of a DCCF checkpoint')
    DataLoader.parse_data_args(ap)
    ap.add_argument('--model_path', type=str, required=True, help='checkpoint written by save_model')
    ap.add_argument('--metric', type=str, default='ndcg@10,recall@10,precision@10',
                    help='comma-separated <name>@k, name in ndcg/hit/precision/recall/f1, k <= 16')
    ap.add_argument('--split', type=str, default='test', choices=('test', 'validation'))
    ap.add_argument('--sentence-model', type=str, default=synth.DEFAULT_SENTENCE_MODEL,
                    help='the name of sentence model (item feature file <dataset>_<name>.npy)')
    a = ap.parse_args(argv)
    rank, local, world = dp.init_from_env()
    torch.cuda.set_device(local)
    if world > 1 and rank != 0:
        torch.distributed.barrier()             # rank 0 writes the files a first load generates
    dl = DataLoader(path=a.path, dataset=a.dataset, label=a.label, sep=a.sep)
    if world > 1 and rank == 0:
        torch.distributed.barrier()
    model = DCCF(path=dl.path, dataset=dl.dataset, sentence_model=a.sentence_model, sample_num=0, attribute_num=2,
                 std=0.0, label_min=dl.label_min, label_max=dl.label_max, feature_num=0, user_num=dl.user_num,
                 item_num=dl.item_num, u_vector_size=64, i_vector_size=64, n_layers=1, random_seed=2018,
                 model_path=a.model_path).cuda()
    model.load_model()
    metrics = [m.strip() for m in a.metric.split(',') if m.strip()]
    values = evaluate_full_catalogue(model, dl, metrics, split=a.split)
    if rank == 0:
        print(json.dumps({'split': a.split, 'n_gpus': world, 'metrics': dict(zip(metrics, values))}))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
