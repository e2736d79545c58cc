"""Command line of the drop-in: same flags and defaults as the reference's
importance_generation.py:8-21, plus opt-in extras (--compress_rate to also emit the kept-channel
sets the prune_* scripts derive, --seed, --out_root, --synthetic, --random_init).

    python importance_generation.py --net resnet_50 --dataset imagenet --data_dir /data/imagenet --pretrain_dir ckpt.pth --batch_size 256
    python importance_generation.py --net resnet_50 --synthetic --random_init --batch_size 256        # no data / checkpoint at hand
    torchrun --nproc-per-node 8 --master-addr 127.0.0.1 importance_generation.py --net resnet_50 ...

Like the reference, the scores are computed on real images (`--dataset`/`--data_dir`, data.load_data) through a real
checkpoint (`--pretrain_dir`): a missing dataset or checkpoint is an error.  Seeded synthetic inputs and seeded random
weights - what the parity tests and the benchmark use, datasets and the Baidu-hosted checkpoints being unavailable offline -
must be asked for with --synthetic / --random_init, so that noise scores never land in importance_score/ by accident.

`prune_main` is the selection side: the first half of the reference's prune_cifar10.py / prune_imagenet.py / prune_u2netp.py
(:83-88 there: get_compress_rate -> pruned net -> load_model) up to the filled pruned net, from score files that already
exist under --imp_score (or regenerated when they do not; --limit is optional here, SURVEY C-8).
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

from . import dist as ddist
from .generate import imp_score
from .sites import score_dir
from .zoo import NETS, get_network


def build_parser():
    p = argparse.ArgumentParser(description='DCT importance-score generation (B200)')
    p.add_argument('--dataset', type=str, default='cifar10', choices=('cifar10', 'imagenet', 'DUTS'), help='dataset')
    p.add_argument('--data_dir', type=str, default='./data', help='path to dataset')
    p.add_argument('--batch_size', type=int, default=128, help='Batch size for scoring.')
    p.add_argument('--pretrain_dir', type=str, default='checkpoints/googlenet.pt', help='load the model from the specified checkpoint')
    p.add_argument('--limit', type=int, default=5, help='The num of batch to get importance score.')
    p.add_argument('--net', type=str, default='googlenet', choices=tuple(NETS), help='net type')
    # opt-in extras
    p.add_argument('--compress_rate', type=str, default=None, help="e.g. '[0.]+[0.18]*29': also write kept_channels.json")
    p.add_argument('--save_pruned', type=str, default=None,
                   help='with --compress_rate: also build the pruned net, fill it from the scored one on the device '
                        '(what load_model does before fine-tuning) and torch.save its state dict here')
    p.add_argument('--synthetic', action='store_true',
                   help='score seeded synthetic images (randn under manual_seed(1000 + batch)) instead of --dataset')
    p.add_argument('--random_init', action='store_true',
                   help='score seeded random-init weights when --pretrain_dir does not exist (otherwise that is an error)')
    p.add_argument('--seed', type=int, default=0, help='seed of --random_init weights and of the data sampling')
    p.add_argument('--out_root', type=str, default='importance_score')
    p.add_argument('--score_op', type=str, default='dct2', choices=('dct2', 'rank', 'rank_sq', 'dct3'),
                   help="per-slice reduction: dct2 (utils/common.py:267, the default) or one of the lines the reference keeps commented out "
                        "beside it: rank (HRank's matrix_rank, :268), rank_sq (the same through the unchanged cnt_score), dct3 (:269)")
    p.add_argument('--input_side', type=int, default=None, help='override the input resolution (e.g. 288 for DUTS crops)')
    p.add_argument('--amp', type=str, default='off', choices=('off', 'bf16', 'fp16'),
                   help='run the forward under torch.autocast in bf16 or fp16 (faster on a B200).  The scores then come from the '
                        'reduced-precision forward\'s activations and differ from the fp32 forward\'s (the reference\'s); files keep '
                        'their names and format.  Default: off (fp32 forward)')
    return p


def load_checkpoint(net, args):
    """Checkpoint handling of importance_generation.py:24-56, net by net.  A missing file is an error (the reference
    raises, :54-56) unless --random_init asks for seeded random weights."""
    if not args.pretrain_dir or not os.path.isfile(args.pretrain_dir):
        if getattr(args, 'random_init', False):
            print('checkpoint %r not found: scoring seeded random-init weights (seed %d)' % (args.pretrain_dir, args.seed))
            return False
        raise FileNotFoundError('please specify a pretrained model: --pretrain_dir %r does not exist '
                                '(pass --random_init to score seeded random weights)' % (args.pretrain_dir,))
    print('==> Resuming from checkpoint..')
    ckpt = torch.load(args.pretrain_dir, map_location='cpu')
    if args.net == 'u2netp':                               # :29-38 keep only the keys the model has, leave the rest as built
        model_dict = net.state_dict()
        model_dict.update({k: v for k, v in ckpt.items() if k in model_dict})
        net.load_state_dict(model_dict)
    elif args.net == 'resnet_50':                          # :44-45 the file is the state dict itself
        net.load_state_dict(ckpt)
    elif args.net in ('densenet_40', 'resnet_110'):        # :46-51 saved from DataParallel
        net.load_state_dict({k.replace('module.', ''): v for k, v in ckpt['state_dict'].items()})
    else:                                                  # :52-53
        net.load_state_dict(ckpt['state_dict'])
    print('Completed! ')
    return True


def build_loader(args):
    """The batches the scoring pass iterates: the reference's training loader (data.load_data), or None for the seeded
    synthetic stream when --synthetic is given."""
    if getattr(args, 'synthetic', False):
        return None
    from .data import load_data
    try:
        return load_data(args, seed=args.seed)[0]
    except FileNotFoundError as e:
        raise SystemExit('%s\n(pass --synthetic to score seeded synthetic images instead)' % e)


def main(argv=None):
    args = build_parser().parse_args(argv)
    if not torch.cuda.is_available():
        sys.exit('importance generation needs a CUDA device (sm_100a); there is no CPU fallback')
    rank, local_rank, world = ddist.init_from_env()
    device = torch.device('cuda', local_rank)
    torch.backends.cudnn.allow_tf32 = False           # activations stay fp32-exact like the reference's
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(args.seed)
    net = get_network(args.net)
    try:
        load_checkpoint(net, args)
    except FileNotFoundError as e:
        raise SystemExit(str(e))
    net = net.to(device).eval()
    files = imp_score(net, args, loader=build_loader(args), out_root=args.out_root)
    if args.compress_rate and rank == 0:
        from .topk import kept_channels
        kept = kept_channels(args.net, args.compress_rate, files, device=device)
        path = os.path.join(score_dir(args.net, args.limit, args.out_root), 'kept_channels.json')
        with open(path, 'w') as f:
            json.dump({'net': args.net, 'compress_rate': args.compress_rate,
                       'selections': [{'file': s.stem, 'conv': s.conv, 'C': s.C, 'k': s.k,
                                       'select_index': [int(i) for i in idx]} for s, idx in kept]}, f)
        print('kept-channel sets ->', path)
        if args.save_pruned:
            from .compress import get_compress_rate
            from .transfer import transfer_weights
            torch.manual_seed(args.seed)
            pruned = get_network(args.net, get_compress_rate(args.compress_rate)).to(device).eval()
            transfer_weights(args.net, pruned, net.state_dict(), kept)
            torch.save({k: v.cpu() for k, v in pruned.state_dict().items()}, args.save_pruned)
            print('pruned %s (%d parameters, was %d) ->' % (args.net, sum(p.numel() for p in pruned.parameters()),
                                                           sum(p.numel() for p in net.parameters())), args.save_pruned)
    if rank == 0:
        print('The importance score of %s has generated completed!' % args.net)
    ddist.shutdown()


def build_prune_parser():
    p = argparse.ArgumentParser(description='Kept-channel selection + pruned-net fill from importance-score files (B200)')
    # the flags prune_cifar10.py:56-78 / prune_imagenet.py:55-77 / prune_u2netp.py:84-106 share, same names and defaults
    p.add_argument('--dataset', type=str, default='cifar10', choices=('cifar10', 'imagenet', 'DUTS'))
    p.add_argument('--data_dir', type=str, default='./data')
    p.add_argument('--batch_size', type=int, default=128)
    p.add_argument('--pretrain_dir', type=str, default='checkpoints/resnet_56.pt', help='the unpruned model')
    p.add_argument('--imp_score', type=str, default='importance_score/resnet_56_limit5', help='importance score file dir')
    p.add_argument('--compress_rate', type=str, default='[0.]+[0.18]*29', help='compress rate of each conv')
    p.add_argument('--net', type=str, default='resnet_56', choices=tuple(NETS))
    p.add_argument('--limit', type=int, default=5, help='only used when --imp_score holds no files and scores are regenerated '
                                                        '(the reference needs it there but its prune_* parsers lack it)')
    p.add_argument('--save_pruned', type=str, default=None, help='torch.save the filled pruned state dict here')
    p.add_argument('--synthetic', action='store_true')
    p.add_argument('--random_init', action='store_true')
    p.add_argument('--seed', type=int, default=0)
    return p


def prune_main(argv=None):
    """get_compress_rate -> kept-channel sets (GPU top-k over the score files) -> pruned net filled from the unpruned one:
    what the reference's prune_* scripts do before their fine-tune loop (prune_cifar10.py:83-88, utils/load_models.py:803-838),
    with the score files taken from --imp_score when they exist."""
    args = build_prune_parser().parse_args(argv)
    if not torch.cuda.is_available():
        sys.exit('selection and weight transfer run on a CUDA device (sm_100a); there is no CPU fallback')
    from .compress import get_compress_rate, selection_plan
    from .prune import pruned_model
    device = torch.device('cuda', int(os.environ.get('LOCAL_RANK', '0')))
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(args.seed)
    rates = get_compress_rate(args.compress_rate)
    origin = get_network(args.net)
    try:
        load_checkpoint(origin, args)
    except FileNotFoundError as e:
        raise SystemExit(str(e))
    origin = origin.to(device).eval()
    stems = [s.stem for s in selection_plan(args.net, rates)]
    have = os.path.isdir(args.imp_score) and all(os.path.isfile(os.path.join(args.imp_score, st + '.npy')) for st in stems)
    if have:
        print('kept-channel selection from the score files in', args.imp_score)
        net, scores, kept = pruned_model(args.net, rates, origin, scores=args.imp_score, seed=args.seed)
    else:
        print('no complete set of score files in %r: scoring %d batches first' % (args.imp_score, args.limit))
        net, scores, kept = pruned_model(args.net, rates, origin, limit=args.limit, batch_size=args.batch_size, loader=build_loader(args),
                                         seed=args.seed, out_root=os.path.dirname(os.path.normpath(args.imp_score)) or '.')
    for sel, idx in kept:
        print('%s: C=%d k=%d' % (sel.stem, sel.C, sel.k))
    n0, n1 = sum(p.numel() for p in origin.parameters()), sum(p.numel() for p in net.parameters())
    print('pruned %s: %d -> %d parameters, %d selections' % (args.net, n0, n1, len(kept)))
    if args.save_pruned:
        torch.save({k: v.cpu() for k, v in net.state_dict().items()}, args.save_pruned)
        print('pruned state dict ->', args.save_pruned)
    return net, kept


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'prune':
        prune_main(sys.argv[2:])
    else:
        main()
