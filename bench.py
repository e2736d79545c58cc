"""bench.py - DCT importance-score throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--net resnet_50] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (config.workload): ResNet-50 ImageNet 224x224 importance generation, batch 256 per GPU
(BASELINE configs[3], the configuration the metric is quoted on), seeded synthetic images and
random-init weights.  A step is one pass of the hot path over one batch: the 49 hook kernels
(one per hooked layer) accumulating per-channel DCT energies; the run ends with the single
all-reduce, the finalise kernel and the segmented top-k, all inside the timed region.

  value     images/s, whole job over all ranks, activations already resident in HBM (the hooked
            feature maps of one batch, 9.2 GB per GPU: larger than L2, nothing to flush)
  e2e       images/s of complete importance generation through the public API: pinned host batch ->
            H2D -> cuDNN fp32 forward with all hooks live -> D2H of the running score sums, every step
  roofline  dominant kernel (largest share of the step) timed with CUDA events; per launch the bound is the slower of
            4*H*W bytes per scored map at the measured HBM peak and 3 x 2*H*W*(H+W) FLOPs at the measured bf16 peak (DESIGN.md);
            kernel names come from the library (dctp_last_kernel), not from a copy of its dispatch
  strong    the same run with ONE global batch of 256 split over the ranks (rank_slice, what the CLI does)
  u2netp    BASELINE config 5: U^2-Netp at 320 and 288, batch 12 per GPU, in the same line
  cpu_baseline  the oracle port of the reference hooks on this box's host cores, bounded sample

`--impl reference` times the reference's CPU implementation (oracle/reference_port.py: the
reference is pure Python and its DCT dependency torch_dct is absent, so the port is the runnable
form) on a bounded sample per step, rank 0 only.

`--dump-outputs DIR` writes, after the timed steps of the headline net and of the U^2-Netp legs, what the timed run handed
back: DIR/<net>_<side>.score.<file>.npy (float32, one per score file) and DIR/<net>_<side>.kept.<file>.npy (kept channel
ids as float64, one per pruned layer).  Images, weights and the cuDNN forward that makes the scored activations are seeded
and deterministic, so two runs or two builds with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = 'dct_importance_score_images_per_s'
UNIT = 'images/s'

WORKLOADS = {
    'resnet_50': dict(side=224, batch=256, rate='[0.]+[0.1]*3+[0.4]*7+[0.4]*9',
                      name='ResNet-50 ImageNet 224x224 importance generation, batch 256 per GPU, 49 hook sites'),
    'u2netp': dict(side=320, batch=12, rate='[0.40]*40',
                   name='U2-Netp DUTS 320x320 importance generation, batch 12 per GPU, 118 hook sites'),
    'resnet_56': dict(side=32, batch=256, rate='[0.]+[0.18]*29',
                      name='ResNet-56 CIFAR-10 importance generation, batch 256 per GPU, 55 hook sites'),
    'googlenet': dict(side=32, batch=128, rate='[0.4]+[0.85]*2+[0.9]*5+[0.9]*2',
                      name='GoogLeNet CIFAR-10 importance generation, batch 128 per GPU, 10 hook sites'),
    'densenet_40': dict(side=32, batch=256, rate='[0.]+[0.2]*12+[0.]+[0.2]*12+[0.]+[0.2]*12',
                        name='DenseNet-40 CIFAR-10 importance generation, batch 256 per GPU, 39 hook sites'),
    'vgg_16_bn': dict(side=32, batch=128, rate='[0.50]*7+[0.95]*5',
                      name='VGG-16-BN CIFAR-10 importance generation, batch 128 per GPU, 12 hook sites'),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=5)       # = the reference's default --limit
    p.add_argument('--warmup', type=int, default=3)
    p.add_argument('--impl', default='ours', choices=('ours', 'reference'))
    p.add_argument('--net', default='resnet_50', choices=tuple(WORKLOADS))
    p.add_argument('--batch', type=int, default=None)
    p.add_argument('--path', default='auto', choices=('auto', 'umma', 'simt'),
                   help="kernel path of the hook launches (the whole net must fit a forced path, so 'tmem' / 'large' are left to 'auto')")
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--no-e2e', action='store_true')
    p.add_argument('--no-strong', action='store_true', help='skip the strong-scaling leg (global batch split over the ranks)')
    p.add_argument('--no-u2netp', action='store_true', help='skip the U^2-Netp 320/288 summary (BASELINE config 5)')
    p.add_argument('--per-site', action='store_true', help='one launch per hook site in the timed steps too (no multi-site launches): the form the ncu launch list is taken in, so that bytes per launch compare with the per-site algorithmic bytes')
    p.add_argument('--graph', action='store_true', help='replay CUDA graphs (hook launches of a step; forward + hooks in the e2e leg): takes the host out of launch-bound nets')
    p.add_argument('--dump-outputs', metavar='DIR', default=None,
                   help='after the timed steps, write what they computed (per-file scores, kept channel ids) as DIR/<name>.npy, '
                        'for comparing two builds output for output')
    return p.parse_args()


def measured_peaks():
    path = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d['hbm_gbs']), float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1590.0))), 'measured'
    return 6650.0, 1590.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    NAMES = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(self.NAMES, parts[2:6]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm),
                'window': 'warm-up + kernel-only timed region + end-to-end leg (nvidia-smi -lms 100)'}


def dist_setup(args):
    from dct_pruning_b200 import dist as ddist
    rank, local_rank, world = ddist.init_from_env()
    if world != args.gpus and world > 1:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d' % (args.gpus, world))
    return rank, local_rank, world


def max_over_ranks(ms, device, world):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


# ====================================================================== our arm
PASSES = 3            # bf16 split-precision passes the binding roofline charges per contraction (SURVEY 8d: hi*hi + lo*hi + hi*lo)


def site_roofline(shape, scored_channels, hbm_gbs, tflops):
    """Binding roofline of one hook launch (SURVEY 8d): bytes = 4*H*W per scored map read once, FLOPs = 2*H*W*(H+W) per map
    and pass.  Returns (algorithmic bytes, seconds the slower of the two limits allows, 'hbm' | 'tensor')."""
    B, _, H, W = shape
    maps = B * scored_channels
    nbytes = 4 * maps * H * W
    flops = PASSES * 2.0 * maps * H * W * (H + W)
    t_mem, t_mma = nbytes / (hbm_gbs * 1e9), flops / (tflops * 1e12)
    return nbytes, flops, max(t_mem, t_mma), ('hbm' if t_mem >= t_mma else 'tensor')


def dump_outputs(directory, tag, session, plan, scores, kept):
    """The result of the timed run as its caller receives it: every score file's vector (float32, what ScoreSession.finalize
    returns) and every selection's kept channel ids (int64 on the device, stored as float64: exact).  A few hundred kB per net."""
    os.makedirs(directory, exist_ok=True)
    for stem, vec in session.split_files(scores.cpu().numpy()).items():
        np.save(os.path.join(directory, '%s.score.%s.npy' % (tag, stem)), vec)
    for sel, ids in zip(plan, kept):
        np.save(os.path.join(directory, '%s.kept.%s.npy' % (tag, sel.stem)), ids.cpu().numpy().astype(np.float64))


def measure_net(args, net_name, side, B, rank, local_rank, world, device, lib, steps, with_e2e, npy_dir=None, clock_sampler=None,
                dump_dir=None):
    """Kernel-only and end-to-end legs for one net at per-rank batch B.  Returns a dict (all times already max over ranks).
    `dump_dir`: rank 0 writes the kernel-only leg's scores and kept ids there (dump_outputs)."""
    from dct_pruning_b200 import _lib
    from dct_pruning_b200.compress import get_compress_rate, selection_plan
    from dct_pruning_b200.generate import device_batches, write_score_files
    from dct_pruning_b200.hooks import ScoreSession
    from dct_pruning_b200.sites import VARIANT_INPUT, resolve_module
    from dct_pruning_b200.topk import topk_segmented
    from dct_pruning_b200.zoo import get_network

    wl = WORKLOADS[net_name]
    torch.manual_seed(0)
    net = get_network(net_name).to(device).eval()
    g = torch.Generator().manual_seed(1000 + rank)
    host_batch = torch.randn(max(B, 1), 3, side, side, generator=g)[:B].contiguous().pin_memory()
    session = ScoreSession(net, net_name, path=args.path, defer_bytes=0 if getattr(args, 'per_site', False) else None)
    if world > 1:
        session.plan_layout(torch.zeros(1, 3, side, side, device=device))
    out = {'batch_per_gpu': B, 'input_side': side}

    # ---- the hooked feature maps of one batch, resident in HBM for the kernel-only leg
    acts = [None] * len(session.sites)
    if B > 0:
        handles = []
        for idx, site in enumerate(session.sites):
            def cap(module, inputs, output, idx=idx, take_input=(site.variant == VARIANT_INPUT)):
                acts[idx] = (inputs[0] if take_input else output).detach().clone()
            handles.append(resolve_module(net, site.module).register_forward_hook(cap))
        # deterministic cuDNN algorithms (not benchmark's timing-dependent pick): the same activations from run to run, so that
        # --dump-outputs of two runs or two builds compare output for output.  This forward is not timed.
        with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, benchmark=False, deterministic=True, allow_tf32=False):
            net(host_batch.to(device))
        for h in handles:
            h.remove()
    torch.cuda.synchronize()
    live = [i for i, a in enumerate(acts) if a is not None]
    scored = {i: (12 if session.sites[i].variant == 'D' else acts[i].shape[1]) for i in live}
    hbm_peak, tflops, peak_kind = measured_peaks()
    roof = {i: site_roofline(tuple(acts[i].shape), scored[i], hbm_peak, tflops) for i in live}
    act_bytes = sum(acts[i].numel() * 4 for i in live)
    alg_bytes_step = sum(roof[i][0] for i in live)
    plan = selection_plan(net_name, get_compress_rate(wl['rate']))

    def finish_run():
        scores = session.finalize_device(check=False)
        segs = {stem: (off, n) for stem, off, n in session.file_segments()}
        offsets, ks, pieces = [0], [], []
        for sel in plan:
            off, n = segs[sel.stem]
            pieces.append(scores[off:off + n])
            offsets.append(offsets[-1] + n)
            ks.append(sel.k)
        kept = topk_segmented(torch.cat(pieces), offsets, ks) if plan else []
        return scores, kept

    def one_step():
        for i in live:
            session.score(i, acts[i])
        session.flush()                                             # (sites held for a multi-site launch)

    # ---- warm-up (bases uploaded, slots allocated, clocks up), then the kernel the library picked for every site
    for _ in range(max(args.warmup, 3)):
        one_step()
    finish_run()
    _lib.check(lib.dctp_check(None))
    session.reset()
    site_kernel = {}
    defer_bytes, session.defer_bytes = session.defer_bytes, 0      # one launch per site while asking which kernel it runs
    for i in live:
        session.score(i, acts[i])
        site_kernel[i] = lib.dctp_last_kernel().decode()
    torch.cuda.synchronize()
    session.defer_bytes = defer_bytes
    session.reset()

    # ---- the timed region: K steps of back-to-back hook launches + the end-of-run kernels, nothing else on the stream
    step_graph, graph_launches = None, 0
    if args.graph and live:
        warm_stream = torch.cuda.Stream(device=device)
        warm_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(warm_stream):
            one_step()
        torch.cuda.current_stream().wait_stream(warm_stream)
        torch.cuda.synchronize()
        step_graph = torch.cuda.CUDAGraph()
        g0 = lib.dctp_launch_count()
        with torch.cuda.graph(step_graph):
            one_step()
            session.flush()
        graph_launches = lib.dctp_launch_count() - g0
        session.reset()
    barrier(world)
    launches0 = lib.dctp_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for step in range(steps):
        if step_graph is not None:
            step_graph.replay()
            for i in live:
                session.images[i] += B
        else:
            one_step()
    final_scores, final_kept = finish_run()
    t1.record()
    barrier(world)
    launches = lib.dctp_launch_count() - launches0 + (steps * graph_launches if step_graph is not None else 0)
    _lib.check(lib.dctp_check(None))
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, '%s_%d' % (net_name, side), session, plan, final_scores, final_kept)
    ms_total = max_over_ranks(t0.elapsed_time(t1), device, world)
    out.update(ms_per_step=ms_total / steps, gpu_launches=int(launches), hook_sites=len(session.sites),
               activation_bytes_per_step=act_bytes, algorithmic_bytes_per_step=alg_bytes_step,
               hook_path_GBps=alg_bytes_step * steps / (ms_total / 1e3) / 1e9,
               binding_roofline_frac=sum(roof[i][2] for i in live) * steps / (ms_total / 1e3))

    # ---- per-launch durations: the same K steps again with an event pair around every launch (isolated launch durations:
    #      the events keep consecutive launches from overlapping; not part of the timed value)
    session.reset()
    session.defer_bytes = 0                                         # (isolated launches: no multi-site batching in this pass)
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in live] for _ in range(steps)]
    for step in range(steps):
        for j, i in enumerate(live):
            ev[step][j][0].record()
            session.score(i, acts[i])
            ev[step][j][1].record()
    torch.cuda.synchronize()
    session.defer_bytes = defer_bytes
    session.reset()
    per_site_ms = {i: statistics.mean(ev[s][j][0].elapsed_time(ev[s][j][1]) for s in range(steps)) for j, i in enumerate(live)}

    def table(key_of):
        groups = {}
        for i in live:
            d = groups.setdefault(key_of(i), {'launches_per_step': 0, 'ms_per_step': 0.0, 'bytes_per_step': 0, 'flops_per_step': 0.0,
                                              'roofline_s': 0.0, 't_hbm': 0.0})
            d['launches_per_step'] += 1
            d['ms_per_step'] += per_site_ms[i]
            d['bytes_per_step'] += roof[i][0]
            d['flops_per_step'] += roof[i][1]
            d['roofline_s'] += roof[i][2]
            d['t_hbm'] += roof[i][0] / (hbm_peak * 1e9)
        res = {}
        for k, d in groups.items():
            sec = d['ms_per_step'] / 1e3
            bound = 'hbm' if d['t_hbm'] >= d['roofline_s'] * 0.999 else 'tensor'
            res[k] = {'launches_per_step': d['launches_per_step'], 'ms_per_step': round(d['ms_per_step'], 4),
                      'bytes_per_step': d['bytes_per_step'], 'GBps': round(d['bytes_per_step'] / sec / 1e9, 1),
                      'frac_hbm': round(d['bytes_per_step'] / sec / 1e9 / hbm_peak, 3),
                      'TFLOPs': round(d['flops_per_step'] / sec / 1e12, 1),
                      'bound': bound, 'frac': round(d['roofline_s'] / sec, 3)}
        return res

    by_kernel = table(lambda i: site_kernel[i])
    by_shape = table(lambda i: '%dx%dx%d' % (scored[i], acts[i].shape[2], acts[i].shape[3]))
    out.update(by_kernel=by_kernel, by_shape=by_shape)
    # ---- the launches of the timed step as they really are (multi-site launches: all sites of a map side in one or two launches),
    #      an event pair around each, per map side.  by_shape above times one launch per site, where the ~10 us a launch costs beyond
    #      its bytes weighs on the small layers; this table shows what those layers cost inside the step.  Informational: a failure
    #      here must not take the bench line with it.
    try:
        session.reset()
        pairs = []
        raw_single, raw_multi = session._score_accum, session._score_multi

        def timed_launch(fn, side_arg):
            def call(*a):
                e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e_a.record()
                rc = fn(*a)
                e_b.record()
                pairs.append((int(a[side_arg]), e_a, e_b))
                return rc
            return call
        session._score_accum, session._score_multi = timed_launch(raw_single, 2), timed_launch(raw_multi, 2)
        try:
            for _ in range(steps):
                one_step()
            torch.cuda.synchronize()
        finally:
            session._score_accum, session._score_multi = raw_single, raw_multi
        side_tot = {}
        for i in live:
            d = side_tot.setdefault(int(acts[i].shape[2]), {'bytes': 0, 'roofline_s': 0.0, 'sites': 0})
            d['bytes'] += roof[i][0]
            d['roofline_s'] += roof[i][2]
            d['sites'] += 1
        side_ms, side_n = {}, {}
        for side_h, e_a, e_b in pairs:
            side_ms[side_h] = side_ms.get(side_h, 0.0) + e_a.elapsed_time(e_b)
            side_n[side_h] = side_n.get(side_h, 0) + 1
        by_side = {}
        for side_h, d in sorted(side_tot.items(), reverse=True):
            if side_h not in side_ms:
                continue
            sec = side_ms[side_h] / steps / 1e3
            by_side['%dx%d' % (side_h, side_h)] = {'sites': d['sites'], 'launches_per_step': round(side_n[side_h] / steps, 2),
                                                   'ms_per_step': round(sec * 1e3, 4), 'bytes_per_step': d['bytes'],
                                                   'GBps': round(d['bytes'] / sec / 1e9, 1), 'frac_hbm': round(d['bytes'] / sec / 1e9 / hbm_peak, 3),
                                                   'frac': round(d['roofline_s'] / sec, 3)}
        out['by_side_in_step'] = by_side
        session.reset()
    except Exception as exc:                                         # noqa: BLE001
        out['by_side_in_step'] = {'error': repr(exc)}
        session.reset()
    if by_kernel:
        dom_name = max(by_kernel, key=lambda k: by_kernel[k]['ms_per_step'])       # dominant = largest share of the step
        dom = by_kernel[dom_name]
        sec = dom['ms_per_step'] / 1e3
        traffic = None
        tpath = os.path.join(REPO, 'profiles', 'traffic.json')
        if os.path.exists(tpath):
            with open(tpath) as f:
                tab = json.load(f)
            # traffic.json is keyed by the demangled instantiation (score_stack_kernel<64,4,8,1,2>); the library's label names
            # the same first template argument (KP=64 / K2=64): match on kernel + that argument
            import re
            mm = re.match(r'(\w+)(?:<(?:[A-Z0-9]+=)?(\d+))?', dom_name)
            prefix = mm.group(1) + ('<' + mm.group(2) + ',' if mm.group(2) else '')
            hits = [v for k, v in tab.items() if isinstance(v, dict) and k.startswith(prefix)]
            if hits:
                traffic = sum(v['dram_bytes_per_launch'] * v['launches'] for v in hits) / sum(v['launches'] for v in hits)
        if dom['bound'] == 'hbm':
            achieved, peak, unit = dom['bytes_per_step'] / sec / 1e9, hbm_peak, 'GB/s'
        else:
            achieved, peak, unit = dom['TFLOPs'], tflops, 'TFLOP/s'
        out['roofline'] = {'bound': dom['bound'], 'achieved': achieved, 'peak': peak, 'unit': unit, 'frac': dom['frac'],
                           'traffic': traffic, 'peak_kind': peak_kind, 'kernel': dom_name,
                           'share_of_step': dom['ms_per_step'] / sum(per_site_ms.values()),
                           'launches_per_step': dom['launches_per_step'], 'bytes_per_step': dom['bytes_per_step'],
                           'ms_per_step': dom['ms_per_step'], 'passes_charged': PASSES,
                           'timing': 'CUDA event pair around every launch, over a repeat of the K timed steps on the same stream '
                                     '(isolated launch durations; bound = slower of 4*H*W bytes at the measured HBM peak and '
                                     '3 x 2*H*W*(H+W) FLOPs at the measured sustained bf16 peak, per launch)'}

    # ---- end to end: pinned host batch -> H2D -> forward with hooks live -> D2H of the running sums, every step; the run ends
    #      with the all-reduce, finalise, top-k, D2H of the scores and the .npy files (rank 0)
    if with_e2e:
        session.reset()
        pinned_out = torch.empty(session.used + 1, dtype=torch.float64).pin_memory()
        replay = None

        def e2e_steps(n, hooks=True):
            if replay is not None and hooks:
                for _ in range(n):
                    replay(host_batch)
                    pinned_out.copy_(session.flat[:session.used + 1], non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                return
            src = (host_batch for _ in range(n)) if B > 0 else iter(())
            for x in device_batches(src, device):
                with torch.no_grad():
                    net(x)
                pinned_out.copy_(session.flat[:session.used + 1], non_blocking=True)
                torch.cuda.current_stream().synchronize()

        with session:
            if args.graph and B > 0:
                replay = session.capture(host_batch.to(device))
            e2e_steps(2)
            session.reset()
            barrier(world)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            e2e_steps(steps)
            e2e_scores, _ = finish_run()
            host_scores = e2e_scores.cpu()
            if rank == 0 and npy_dir is not None:
                write_score_files(session.split_files(host_scores.numpy()), npy_dir, verbose=False)
            e1.record()
            barrier(world)
            ms_e2e = max_over_ranks(e0.elapsed_time(e1), device, world)
            # the hooks' own share, in line: one more pass with an event pair around every hook launch inside the forward
            session.reset()
            pairs = []
            raw_single, raw_multi = session._score_accum, session._score_multi

            def timed(fn):
                def call(*a):
                    e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e_a.record()
                    rc = fn(*a)
                    e_b.record()
                    pairs.append((e_a, e_b))
                    return rc
                return call
            session._score_accum, session._score_multi = timed(raw_single), timed(raw_multi)      # the two launch points
            e2e_steps(1)
            session._score_accum, session._score_multi = raw_single, raw_multi
            torch.cuda.synchronize()
            hooks_ms = sum(a.elapsed_time(b) for a, b in pairs)
        # the same loop without hooks (accumulator still copied out), for the breakdown
        session.remove()
        e2e_steps(1, hooks=False)
        barrier(world)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        e2e_steps(steps, hooks=False)
        f1.record()
        torch.cuda.synchronize()
        ms_fwd = max_over_ranks(f0.elapsed_time(f1), device, world)
        out['e2e'] = {'ms_per_step': ms_e2e / steps, 'forward_only_ms_per_step': ms_fwd / steps,
                      'hooks_in_line_ms_per_step': hooks_ms,
                      'h2d_bytes_per_step': int(host_batch.numel() * 4), 'd2h_bytes_per_step': int(pinned_out.numel() * 8),
                      'score_checksum': float(host_scores.double().sum()), 'cuda_graph': bool(args.graph),
                      'includes': 'H2D of every batch from pinned memory, fp32 cuDNN forward with all hooks live, D2H of the running sums every '
                                  'step; once per run: all-reduce, finalise, top-k, D2H of the scores, np.save of every score file (rank 0)',
                      'hooks_in_line_how': 'CUDA event pair around every score launch (single-site and multi-site) inside one extra forward pass (not the timed one)'}
    out['_acts_cpu'] = [acts[i][:4].cpu() for i in live] if (rank == 0 and world == 1 and net_name == args.net and not args.no_cpu_baseline) else None
    out['_acts'] = acts if out['_acts_cpu'] is not None else None
    out['_sites'] = session.sites
    return out


def run_ours(args):
    import shutil
    import tempfile
    from dct_pruning_b200 import _lib
    from dct_pruning_b200.generate import rank_slice

    rank, local_rank, world = dist_setup(args)
    device = torch.device('cuda', local_rank)
    torch.cuda.set_device(device)
    wl = WORKLOADS[args.net]
    B = args.batch or wl['batch']
    side = wl['side']
    torch.backends.cudnn.allow_tf32 = False            # activations fp32-exact, like the reference's
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    lib = _lib.load()
    _lib.check(lib.dctp_init())
    steps = args.steps
    tmp = tempfile.mkdtemp(prefix='dctp_bench_') if rank == 0 else None

    # clocks are sampled from here to the end of the last timed leg: every timed region lies inside the window
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---- headline: batch B per GPU (weak scaling: the work per GPU is fixed)
    main = measure_net(args, args.net, side, B, rank, local_rank, world, device, lib, steps, not args.no_e2e,
                       npy_dir=os.path.join(tmp, 'weak') if tmp else None, dump_dir=args.dump_outputs)
    acts_cpu, acts_gpu, sites = main.pop('_acts_cpu'), main.pop('_acts'), main.pop('_sites')
    value = world * B * steps / (main['ms_per_step'] * steps / 1e3)

    # ---- CPU legs (rank 0, single GPU run only) while the activations are still around
    cpu = None
    if acts_cpu is not None:
        cpu = cpu_hooks_baseline(acts_cpu, sites, budget_s=12.0)
        on_gpu = gpu_tensor_reference_baseline(acts_gpu, sites, budget_s=4.0)
        if on_gpu is not None:
            cpu['reference_hook_on_gpu_tensors'] = on_gpu
    del acts_cpu, acts_gpu
    torch.cuda.empty_cache()

    # ---- strong scaling: ONE global batch of B images split over the ranks with rank_slice, exactly what the CLI does
    #      (generate.inference); at one GPU it is the headline run itself
    strong = None
    if not args.no_strong:
        if world == 1:
            strong = {'global_batch': B, 'batch_per_gpu': B, 'value': value, 'ms_per_step': main['ms_per_step'], 'same_as': 'headline (one GPU)'}
            if 'e2e' in main:
                strong['e2e'] = {'value': B / (main['e2e']['ms_per_step'] / 1e3), 'ms_per_step': main['e2e']['ms_per_step']}
        else:
            lo, hi = rank_slice(B, rank, world)
            sres = measure_net(args, args.net, side, hi - lo, rank, local_rank, world, device, lib, steps, not args.no_e2e,
                               npy_dir=os.path.join(tmp, 'strong') if tmp else None)
            for k in ('_acts_cpu', '_acts', '_sites'):
                sres.pop(k)
            strong = {'global_batch': B, 'batch_per_gpu': hi - lo, 'value': B / (sres['ms_per_step'] / 1e3), 'ms_per_step': sres['ms_per_step'],
                      'hook_path_GBps_per_gpu': sres['hook_path_GBps'], 'binding_roofline_frac': sres['binding_roofline_frac'],
                      'by_shape': sres['by_shape']}
            if 'e2e' in sres:
                strong['e2e'] = {'value': B / (sres['e2e']['ms_per_step'] / 1e3), 'ms_per_step': sres['e2e']['ms_per_step'],
                                 'forward_only_ms_per_step': sres['e2e']['forward_only_ms_per_step'],
                                 'hooks_in_line_ms_per_step': sres['e2e']['hooks_in_line_ms_per_step']}
            torch.cuda.empty_cache()

    # ---- BASELINE config 5: U^2-Netp at 320x320 (as BASELINE names it) and 288x288 (what the reference's DUTS loader feeds,
    #      utils/common.py:154-155), batch 12 per GPU (prune_u2netp.py:90)
    u2 = None
    if args.net == 'resnet_50' and not args.no_u2netp:
        u2 = {}
        for s_side in (320, 288):
            r = measure_net(args, 'u2netp', s_side, WORKLOADS['u2netp']['batch'], rank, local_rank, world, device, lib, steps,
                            (not args.no_e2e) and s_side == 320, npy_dir=os.path.join(tmp, 'u2netp%d' % s_side) if tmp else None,
                            dump_dir=args.dump_outputs)
            for k in ('_acts_cpu', '_acts', '_sites'):
                r.pop(k)
            r['value'] = world * r['batch_per_gpu'] / (r['ms_per_step'] / 1e3)
            r['unit'] = UNIT
            if 'e2e' in r:
                r['e2e']['value'] = world * r['batch_per_gpu'] / (r['e2e']['ms_per_step'] / 1e3)
            r.pop('by_kernel')
            u2['side%d' % s_side] = r
            torch.cuda.empty_cache()

    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        hbm_peak, tflops, peak_kind = measured_peaks()
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': main['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16 hi/lo split of fp32 on tcgen05 (fp32 accumulate), fp64 cross-image sums', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'net': args.net, 'batch_per_gpu': B, 'input_side': side, 'limit': steps,
                       'hook_sites': main['hook_sites'], 'activation_bytes_per_step': main['activation_bytes_per_step'],
                       'algorithmic_bytes_per_step': main['algorithmic_bytes_per_step'],
                       'l2': 'inputs (%.1f GB per step) exceed L2; no flush needed' % (main['activation_bytes_per_step'] / 1e9),
                       'compress_rate': wl['rate'], 'path': args.path, 'cuda_graph': bool(args.graph),
                       'parallelism': 'batch-sharded x%d, 1 all-reduce per run' % world,
                       'peaks': {'hbm_gbs': hbm_peak, 'bf16_tflops_sustained': tflops, 'kind': peak_kind}},
            'gpu_launches': main['gpu_launches'],
            'launch_batching': 'activations below 1 GB are held and scored up to 16 sites of a map size per launch (dctp_score_accum_multi); by_kernel / by_shape time one launch per site, by_side_in_step the launches of the timed step themselves (an event pair around each)',
            'roofline': main.get('roofline'),
            'hook_path_GBps': main['hook_path_GBps'],
            'binding_roofline_frac': main['binding_roofline_frac'],
            'by_kernel': main['by_kernel'], 'by_shape': main['by_shape'],
            'by_side_in_step': main.get('by_side_in_step'),
            'clocks': clocks,
        }
        if 'e2e' in main:
            e = dict(main['e2e'])
            e['value'] = world * B / (e['ms_per_step'] / 1e3)
            e['unit'] = UNIT
            line['e2e'] = e
        if strong is not None:
            line['strong'] = strong
        if u2 is not None:
            line['u2netp'] = u2
        if cpu is not None:
            line['cpu_baseline'] = cpu
        print(json.dumps(line))
        shutil.rmtree(tmp, ignore_errors=True)
    from dct_pruning_b200 import dist as ddist
    ddist.shutdown()


# ====================================================================== CPU legs
def cpu_hooks_baseline(acts_cpu, sites, budget_s):
    """The reference's hook (oracle port, op for op) over whole images until the budget is spent."""
    from oracle import reference_port as port
    torch.set_num_threads(os.cpu_count() or 1)
    hooks = {'O': port.hook_output, 'D': port.hook_densenet, 'I': port.hook_u2net_input}
    n_img = acts_cpu[0].shape[0]
    done, slices, t0 = 0, 0, time.perf_counter()
    for i in range(n_img):
        for a, site in zip(acts_cpu, sites):
            st = port.ScoreState()
            x = a[i:i + 1]
            hooks[site.variant](st)(None, (x,), x)
            slices += 12 if site.variant == 'D' else x.shape[1]
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {'value': done / dt, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': '%d image(s) x all %d hook sites (%d slices) through oracle.reference_port hooks, hooks only (no CNN forward), %.1f s'
                      % (done, len(sites), slices, dt),
            'us_per_slice': dt / slices * 1e6}


def gpu_tensor_reference_baseline(acts, sites, budget_s):
    """The reference hook in the mode its authors ran it: activations stay on the GPU, one cuFFT-based DCT and one
    `.item()` sync per (image, channel) slice (oracle port of utils/common.py:262-277).  One image, as many sites as fit."""
    from oracle import reference_port as port
    done_sites, slices, t0 = 0, 0, time.perf_counter()
    total_slices = sum(12 if s.variant == 'D' else a.shape[1] for a, s in zip(acts, sites))
    for a, site in zip(acts, sites):
        if site.variant != 'O':
            continue                               # the other two variants copy every slice to the host for cv2
        x = a[0:1]
        port.hook_output(port.ScoreState())(None, (x,), x)
        torch.cuda.synchronize()
        slices += x.shape[1]
        done_sites += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    if slices == 0:
        return None
    us = dt / slices * 1e6
    return {'us_per_slice': us, 'images_per_s_extrapolated': 1e6 / (us * total_slices),
            'sample': '1 image x %d output-hook site(s) (%d slices) on GPU tensors, per-slice torch.fft DCT + .item() sync, %.1f s; '
                      'extrapolated linearly to all %d slices of an image' % (done_sites, slices, dt, total_slices)}


def run_reference(args):
    """The reference's own CPU implementation (per-site forward sweep + per-slice Python hook),
    restated in oracle/reference_port.py, on a bounded sample: one image per step."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from dct_pruning_b200.sites import hook_sites
    from dct_pruning_b200.zoo import get_network
    from oracle import reference_port as port
    wl = WORKLOADS[args.net]
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    net = get_network(args.net).eval()
    sessions = [(s.module, s.variant, [(f.stem, f.lo, f.hi) for f in s.files]) for s in hook_sites(args.net, net)]
    B = 1

    def batches(seed):
        g = torch.Generator().manual_seed(seed)
        return [torch.randn(B, 3, wl['side'], wl['side'], generator=g)]

    def step(i):
        port.imp_score_port(net, sessions, lambda: batches(1000 + i), 1)

    warm = min(args.warmup, 1)
    for i in range(warm):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(warm + i)
    dt = time.perf_counter() - t0
    value = B * args.steps / dt
    sample = ('%d image per step through the full reference flow (one forward sweep per hook site, %d sites, per-slice Python hook) '
              'on %d host threads' % (B, len(sessions), torch.get_num_threads()))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': warm, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': wl['name'], 'net': args.net, 'batch_per_step': B, 'input_side': wl['side']},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }))


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        if a.dump_outputs:
            raise SystemExit('--dump-outputs writes what the CUDA path computed; it has no meaning with --impl reference')
        run_reference(a)
    else:
        if not torch.cuda.is_available():
            raise SystemExit('bench.py needs a CUDA device; the product path has no CPU fallback')
        run_ours(a)
