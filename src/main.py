# coding=utf-8
"""Command line of the reference (src/main.py:24-195), unchanged for the user:

    python main.py --rank 1 --model_name DCCF --optimizer Adam --lr 0.001 --dataset Electronics \\
        --metric ndcg@5,recall@5,precision@5 --gpu 0 --epoch 100 --test_neg_n 1000

Two-phase argparse (class names first, then every class adds its own flags), file names derived from
the hyper-parameters, seeding, "Test Before Training" -> train -> "Test After Training" -> result .npy.
The classes come from the dccf_b200 package (B200 kernels behind the reference's plugin protocols).
"""
import argparse
import logging
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _gpu_list_ok(value):
    """Under torchrun (LOCAL_WORLD_SIZE ranks on this node) `--gpu` must name at least one device per local rank to be
    applied as CUDA_VISIBLE_DEVICES; the reference's default `--gpu 0` would pin every rank to the same GPU."""
    local_world = int(os.environ.get('LOCAL_WORLD_SIZE', os.environ.get('WORLD_SIZE', '1')))
    return local_world <= 1 or len([d for d in value.split(',') if d.strip() != '']) >= local_world


def _early_gpu_env(argv):
    """CUDA_VISIBLE_DEVICES must be set before CUDA initialises; the reference sets it after parsing
    (main.py:106), which only works because nothing touched CUDA yet.  Same effect, done first."""
    for i, a in enumerate(argv):
        value = None
        if a == '--gpu' and i + 1 < len(argv):
            value = argv[i + 1]
        elif a.startswith('--gpu='):
            value = a.split('=', 1)[1]
        if value is not None and _gpu_list_ok(value):
            os.environ['CUDA_VISIBLE_DEVICES'] = value


_early_gpu_env(sys.argv[1:])

import numpy as np  # noqa: E402
import torch  # noqa: E402

from dccf_b200.utils import utils  # noqa: E402
from dccf_b200.data_loaders.DataLoader import DataLoader  # noqa: E402,F401
from dccf_b200.models.BaseModel import BaseModel  # noqa: E402,F401
from dccf_b200.models.RecModel import RecModel  # noqa: E402,F401
from dccf_b200.models.DCCF import DCCF  # noqa: E402,F401
from dccf_b200.models.BiasedMF import BiasedMF  # noqa: E402,F401
from dccf_b200.models.IPSBiasedMF import IPSBiasedMF  # noqa: E402,F401
from dccf_b200.runners.BaseRunner import BaseRunner  # noqa: E402,F401
from dccf_b200.data_processor.DataProcessor import DataProcessor  # noqa: E402,F401

_CLASSES = {'DataLoader': DataLoader, 'BaseModel': BaseModel, 'RecModel': RecModel, 'DCCF': DCCF,
            'BiasedMF': BiasedMF, 'IPSBiasedMF': IPSBiasedMF, 'BaseRunner': BaseRunner, 'DataProcessor': DataProcessor}


def _resolve(name):
    if name not in _CLASSES:
        raise SystemExit('Unknown class %r; this build provides %s' % (name, sorted(_CLASSES)))
    return _CLASSES[name]


def main(argv=None):
    # Data parallel (new: the reference is single-process, SURVEY.md §8e): launched with
    #   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 main.py <same flags>
    # every rank runs this same program on its own GPU; --batch_size is then per rank (global step = N batches), rank 0
    # owns the log file, the checkpoint, rank.csv and the result file.
    from dccf_b200 import dist as dp
    rank, local_rank, world = dp.init_from_env() if int(os.environ.get('WORLD_SIZE', '1')) > 1 else (0, 0, 1)
    init_parser = argparse.ArgumentParser(description='Model')
    init_parser.add_argument('--rank', type=int, default=1, help='1=ranking, 0=rating/click')
    init_parser.add_argument('--data_loader', type=str, default='DataLoader', help='Choose data_loader')
    init_parser.add_argument('--model_name', type=str, default='BaseModel', help='Choose model to run.')
    init_parser.add_argument('--runner', type=str, default='BaseRunner', help='Choose runner')
    init_parser.add_argument('--data_processor', type=str, default='DataProcessor', help='Choose runner')
    init_args, _ = init_parser.parse_known_args(argv)

    data_loader_name = _resolve(init_args.data_loader)
    model_name = _resolve(init_args.model_name)
    init_args.runner_name = 'BaseRunner'
    runner_name = _resolve(init_args.runner_name)
    data_processor_name = _resolve(init_args.data_processor)

    parser = argparse.ArgumentParser(description='')
    parser = utils.parse_global_args(parser)
    parser = data_loader_name.parse_data_args(parser)
    parser = model_name.parse_model_args(parser, model_name=init_args.model_name)
    parser = runner_name.parse_runner_args(parser)
    parser = data_processor_name.parse_dp_args(parser)
    args, _ = parser.parse_known_args(argv)

    # file names derived from the hyper-parameters (main.py:63-84)
    name_parts = [str(init_args.rank), init_args.model_name, args.dataset, str(args.random_seed),
                  'embdim' + str(getattr(args, 'i_vector_size', '')), 'optimizer=' + args.optimizer,
                  'epoch=' + str(args.epoch), 'lr=' + str(args.lr), 'l2=' + str(args.l2),
                  'dropout=' + str(args.dropout), 'batch_size=' + str(args.batch_size),
                  'test_num=' + str(args.test_neg_n)]
    if init_args.model_name in ['DCCF']:
        name_parts += ['samnum' + str(args.sample_num), 'feanum' + str(args.attribute_num), 'std' + str(args.std)]
    log_file_name = '__'.join(name_parts).replace(' ', '__')
    if args.log_file == '../log/log.txt':
        args.log_file = '../log/%s/%s/%s.txt' % (init_args.model_name, args.dataset, log_file_name)
    utils.check_dir_and_mkdir(args.log_file)
    if args.result_file == '../result/result.npy':
        args.result_file = '../result/%s.npy' % log_file_name
    utils.check_dir_and_mkdir(args.result_file)   # the reference forgets this directory (SURVEY §8c shim 5)
    if args.model_path == '../model/%s/%s.pt' % (init_args.model_name, init_args.model_name):
        args.model_path = '../model/%s/%s.pt' % (init_args.model_name, log_file_name)
    utils.check_dir_and_mkdir(args.model_path)

    for handler in logging.root.handlers[:]:
        logging.root.removeHandler(handler)
    if rank == 0:
        logging.basicConfig(filename=args.log_file, level=args.verbose)
        logging.getLogger().addHandler(logging.StreamHandler(sys.stdout))
    else:                                       # one log: rank 0's
        logging.basicConfig(handlers=[logging.NullHandler()], level=logging.ERROR)
    logging.info(vars(init_args))
    logging.info(vars(args))
    logging.info('DataLoader: ' + init_args.data_loader)
    logging.info('Model: ' + init_args.model_name)
    logging.info('Runner: ' + init_args.runner_name)
    logging.info('DataProcessor: ' + init_args.data_processor)

    # seeds (main.py:101-103)
    torch.manual_seed(args.random_seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(args.random_seed)
    np.random.seed(args.random_seed)
    if _gpu_list_ok(args.gpu):
        os.environ['CUDA_VISIBLE_DEVICES'] = args.gpu
    logging.info('# cuda devices: %d' % torch.cuda.device_count())
    if world > 1:
        logging.info('data parallel: %d ranks, --batch_size %d per rank' % (world, args.batch_size))

    if world > 1 and rank != 0:
        torch.distributed.barrier()             # rank 0 writes the files a first run generates (.info.json, history csv)
    data_loader = data_loader_name(path=args.path, dataset=args.dataset, label=args.label, sep=args.sep)
    if world > 1 and rank == 0:
        torch.distributed.barrier()
    features, feature_dims, feature_min, feature_max = data_loader.feature_info(
        include_id=model_name.include_id, include_item_features=model_name.include_item_features,
        include_user_features=model_name.include_user_features)

    if init_args.model_name in ['BaseModel']:
        model = model_name(label_min=data_loader.label_min, label_max=data_loader.label_max,
                           feature_num=len(features), random_seed=args.random_seed, model_path=args.model_path)
    elif init_args.model_name in ['RecModel', 'BiasedMF']:
        model = model_name(label_min=data_loader.label_min, label_max=data_loader.label_max, feature_num=0,
                           user_num=data_loader.user_num, item_num=data_loader.item_num,
                           u_vector_size=args.u_vector_size, i_vector_size=args.i_vector_size,
                           random_seed=args.random_seed, model_path=args.model_path)
    elif init_args.model_name in ['IPSBiasedMF']:
        model = model_name(path=data_loader.path, dataset=data_loader.dataset, M=args.M,
                           label_min=data_loader.label_min, label_max=data_loader.label_max, feature_num=0,
                           user_num=data_loader.user_num, item_num=data_loader.item_num,
                           u_vector_size=args.u_vector_size, i_vector_size=args.i_vector_size,
                           random_seed=args.random_seed, model_path=args.model_path)
    elif init_args.model_name in ['DCCF']:
        model = model_name(path=data_loader.path, dataset=data_loader.dataset, sentence_model=args.sentence_model,
                           sample_num=args.sample_num, attribute_num=args.attribute_num, std=args.std,
                           label_min=data_loader.label_min, label_max=data_loader.label_max, feature_num=0,
                           user_num=data_loader.user_num, item_num=data_loader.item_num,
                           u_vector_size=args.u_vector_size, i_vector_size=args.i_vector_size,
                           n_layers=args.n_layers, random_seed=args.random_seed, model_path=args.model_path)
    else:
        logging.error('Unknown Model: ' + init_args.model_name)
        return
    model.apply(model.init_paras)
    if torch.cuda.device_count() > 0:
        model = model.cuda()
    if world > 1:
        if not hasattr(model, 'enable_data_parallel'):
            raise SystemExit('data-parallel runs need --model_name DCCF')
        model.enable_data_parallel()

    if init_args.rank == 1:
        data_loader.drop_neg()
    data_processor = data_processor_name(data_loader, model, rank=init_args.rank, test_neg_n=args.test_neg_n)
    runner = runner_name(optimizer=args.optimizer, learning_rate=args.lr, epoch=args.epoch,
                         batch_size=args.batch_size, eval_batch_size=args.eval_batch_size, dropout=args.dropout,
                         l2=args.l2, metrics=args.metric, check_epoch=args.check_epoch, early_stop=args.early_stop)

    logging.info('Test Before Training = ' + utils.format_metric(
        runner.evaluate(model, data_processor.get_test_data(), data_processor, write_rank=False))
                 + ' ' + ','.join(runner.metrics))
    if args.load > 0:
        model.load_model()
    if args.train > 0:
        runner.train(model, data_processor, skip_eval=args.skip_eval)
    logging.info('Test After Training = ' + utils.format_metric(
        runner.evaluate(model, data_processor.get_test_data(), data_processor, write_rank=True))
                 + ' ' + ','.join(runner.metrics))
    result = runner.predict(model, data_processor.get_test_data(), data_processor)
    if rank == 0:
        np.save(args.result_file, result)
    logging.info('Save Test Results to ' + args.result_file)
    if world > 1:
        # the design invariant of the data-parallel step: replicas stay bit-identical without any parameter broadcast
        sums = torch.stack([p.detach().view(torch.int32).to(torch.int64).sum() for p in model.parameters()])
        every = [torch.empty_like(sums) for _ in range(world)]
        torch.distributed.all_gather(every, sums)
        if not all(torch.equal(every[0], e) for e in every):
            raise SystemExit('data-parallel replicas diverged (parameter checksums differ between ranks)')
        logging.info('data parallel: parameter checksums identical on all %d ranks' % world)
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
