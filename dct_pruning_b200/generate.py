"""Importance generation: the drop-in for `imp_score(net, args)` and its batch drivers.

    imp_score          /root/reference/utils/common.py:367-980  (site enumeration, np.save naming)
    inference          /root/reference/utils/common.py:312-320
    u2netp_inference   /root/reference/utils/common.py:323-332
    CLI                /root/reference/importance_generation.py:8-61

Output is byte-compatible with what the reference's prune_* scripts np.load:
``importance_score/<net>_limit<N>/<stem>.npy``, .npy v1.0, '<f4', shape (C,).

Multi-GPU: launched under torchrun (one process per GPU) every rank scores its own slice of
every batch; the per-layer score sums meet in ONE NCCL all-reduce of the flat fp64 buffer at
the end of the run, rank 0 writes the files.  The result does not depend on the rank count
beyond fp64 summation order.
"""
import os

import numpy as np
import torch

from .hooks import ScoreSession
from .sites import score_dir
from .zoo import NET_INPUT


def synthetic_batches(batch_size, side, limit, seed_base=1000, as_dict=False):
    """Seeded stand-in for the reference loaders (datasets are unavailable offline): batch b is
    randn(B,3,S,S) under manual_seed(seed_base + b) on the CPU generator, so CPU oracle and GPU path
    see identical inputs.  `as_dict` mimics the DUTS loader's {'image': ...} samples."""
    for b in range(limit):
        g = torch.Generator().manual_seed(seed_base + b)
        x = torch.randn(batch_size, 3, side, side, generator=g)
        yield {'image': x} if as_dict else (x, torch.zeros(batch_size, dtype=torch.long))


def _images_of(sample):
    if isinstance(sample, dict):
        return sample['image'].type(torch.FloatTensor)       # common.py:329-330
    if isinstance(sample, (tuple, list)):
        return sample[0]
    return sample


def rank_slice(n, rank, world):
    """Contiguous share of an n-image batch for `rank` (ragged shards allowed, empty ones too)."""
    lo = (n * rank) // world
    hi = (n * (rank + 1)) // world
    return lo, hi


def device_batches(host_batches, device):
    """Yield device copies of host image batches one step ahead of their use: the H2D copy of batch k+1 runs on a
    side stream (from pinned memory) under the forward pass of batch k.  Two device buffers are reused in turn; a
    yielded tensor is valid until the next one is requested."""
    main = torch.cuda.current_stream(device)
    copy_stream = torch.cuda.Stream(device=device)
    bufs, consumed = [None, None], [None, None]

    def put(x, slot):
        x = x if x.is_pinned() else x.pin_memory()
        if bufs[slot] is None or bufs[slot].shape != x.shape or bufs[slot].dtype != x.dtype:
            bufs[slot] = torch.empty(x.shape, dtype=x.dtype, device=device)
            consumed[slot] = None
            # a fresh block may be one the caching allocator just took back from activations of a forward pass that is still
            # running on the main stream (ragged last batch): order the first copy into it behind that work
            copy_stream.wait_stream(main)
        with torch.cuda.stream(copy_stream):
            if consumed[slot] is not None:
                copy_stream.wait_event(consumed[slot])      # the forward pass that read this buffer has finished
            bufs[slot].copy_(x, non_blocking=True)
            done = torch.cuda.Event()
            done.record(copy_stream)
        return x, slot, done                                # (the pinned source stays referenced until its copy is consumed)

    def take(pending):
        _, slot, done = pending
        main.wait_event(done)
        return slot

    pending, k = None, 0
    for x in host_batches:
        ahead = put(x, k & 1)
        k += 1
        if pending is not None:
            slot = take(pending)
            yield bufs[slot]
            consumed[slot] = torch.cuda.Event()
            consumed[slot].record(main)
        pending = ahead
    if pending is not None:
        slot = take(pending)
        yield bufs[slot]


# --amp: the forward's autocast dtype.  The hooks then score the reduced-precision activations the forward produced (bf16 / fp16
# maps are read by the library as they are); those scores are not the reference's, whose forward runs in fp32.
AMP_DTYPES = {'off': None, 'bf16': torch.bfloat16, 'fp16': torch.float16}


def inference(net, loader, limit, device, rank=0, world=1, amp='off'):
    """eval + no_grad forward over the first `limit` batches (common.py:312-320); under
    world > 1 each rank forwards its contiguous slice of every batch.  amp: 'off', or 'bf16' / 'fp16' to run the
    forward under torch.autocast with that dtype."""
    net.eval()
    amp_dtype = AMP_DTYPES[amp]

    def shards():
        for batch_idx, sample in enumerate(loader):
            if batch_idx >= limit:
                break
            x = _images_of(sample)
            if world > 1:
                lo, hi = rank_slice(x.shape[0], rank, world)
                x = x[lo:hi]
            if x.shape[0] > 0:
                yield x

    n = 0
    with torch.no_grad(), torch.autocast(torch.device(device).type, dtype=amp_dtype, enabled=amp_dtype is not None):
        if torch.device(device).type == 'cuda':
            for x in device_batches(shards(), device):
                n += x.shape[0]
                net(x)
        else:                                   # (a CPU net only gets here in tests of the host logic; hooks raise on CPU tensors)
            for x in shards():
                n += x.shape[0]
                net(x.to(device))
    return n


def score_session(net, args, loader=None, path='auto', op=None):
    """Run the scoring pass (all hook sites live, `args.limit` batches, this rank's shard of every batch) and return the
    ScoreSession with its per-site energy sums still on the device, not yet reduced or finalised."""
    import torch.distributed as dist
    device = next(net.parameters()).device
    if device.type != 'cuda':
        raise RuntimeError('imp_score needs the net on a CUDA device (got %s); there is no CPU fallback' % device)
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    if loader is None:
        _, side = NET_INPUT[args.net]
        side = getattr(args, 'input_side', None) or side
        loader = synthetic_batches(args.batch_size, side, args.limit,
                                   seed_base=getattr(args, 'seed_base', 1000), as_dict=(args.net == 'u2netp'))
    session = ScoreSession(net, args.net, path=path, op=op or getattr(args, 'score_op', None) or 'dct2')
    if world > 1:                                       # same flat layout on every rank, also on one whose shards are all empty
        _, side0 = NET_INPUT[args.net]
        side0 = getattr(args, 'input_side', None) or side0
        session.plan_layout(torch.zeros(1, 3, side0, side0, device=device))
    with session:
        inference(net, loader, args.limit, device, rank=rank, world=world, amp=getattr(args, 'amp', None) or 'off')
    return session


def imp_score(net, args, loader=None, out_root='importance_score', write=True, path='auto', op=None):
    """Score every hook site of `net` over `args.limit` batches and write the reference's files.

    args: namespace with .net, .limit, .batch_size (and optionally .seed_base).  Returns
    {file_stem: float32 vector}.  The net must already live on a CUDA device.  `op` (or args.score_op) selects the
    per-slice reduction: 'dct2' (default, common.py:267) or one of the alternatives the reference keeps beside it - 'rank'
    (HRank, :268), 'rank_sq' (:268 through the unchanged cnt_score), 'dct3' (:269, one value per site)."""
    import torch.distributed as dist
    session = score_session(net, args, loader=loader, path=path, op=op)
    files = session.finalize()
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    if write and rank == 0:
        write_score_files(files, score_dir(args.net, args.limit, out_root))
    if world > 1:
        dist.barrier()
    return files


def npy_bytes(vec):
    """The bytes `np.save` writes for a 1-D float32 vector (.npy format 1.0: magic, little-endian header length, the header dict
    padded with spaces to a multiple of 64 bytes and ended by a newline, the data) - what the reference's np.save call (common.py:394)
    produces and its prune_* scripts np.load.  Written out by hand because a run ends with one file per score vector (ResNet-50: 53)
    and np.save's header formatting is most of what such a file costs; tests/test_abi.py compares with np.save and the shipped files."""
    vec = np.ascontiguousarray(vec, dtype='<f4')
    if vec.ndim != 1:
        raise ValueError('score vectors are 1-D, got shape %s' % (vec.shape,))
    head = "{'descr': '<f4', 'fortran_order': False, 'shape': (%d,), }" % vec.shape[0]
    pad = -(10 + len(head) + 1) % 64
    head = (head + ' ' * pad + '\n').encode('latin1')
    return b'\x93NUMPY\x01\x00' + len(head).to_bytes(2, 'little') + head + vec.tobytes()


def write_score_files(files, directory, verbose=True):
    os.makedirs(directory, exist_ok=True)
    for stem, vec in files.items():
        with open(os.path.join(directory, stem + '.npy'), 'wb') as f:
            f.write(npy_bytes(vec))
        if verbose:
            print(os.path.join(directory, stem) + ':done!')   # common.py:395
    return directory
