"""16-bit activations on a B200: what reading bf16 maps natively buys over widening them first.

ResNet-50@224, batch 256, per map side, the multi-site launches of a step (dctp_score_accum_multi[_ex], 16 sites per launch), an event
pair around each side's launches, three variants alternating in one process:
  (a) native   bf16 maps -> dctp_score_accum_multi_ex(DCTP_DTYPE_BF16)
  (b) widen    the same bf16 maps -> torch .float() -> dctp_score_accum_multi (what ScoreSession did before 16-bit input)
  (c) fp32     fp32 maps of the same shapes -> dctp_score_accum_multi
Every side's maps are hundreds of MB (more than the 126 MB L2), and the variants and sides alternate, so each launch reads HBM.
Rates are reported per element (bytes/s at 2 and at 4 bytes per element) and as the fraction of a measured HBM copy rate, for
the bytes each variant has to move: (a) 2, (b) 2 + 4 + 4, (c) 4 per element.

End to end: images/s of the scoring pass (forward with every hook live, batch resident on the device, TF32 off as in the CLI) with
an fp32 forward and under torch.autocast(bfloat16), ResNet-50@224 and U^2-Netp@320, and the same forward without hooks.

    python tools/bench_half.py --out DIR        (writes DIR/bench_half.json and prints the same JSON line)
"""
import argparse
import ctypes
import json
import os
import struct
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from dct_pruning_b200 import _lib                      # noqa: E402
from dct_pruning_b200.hooks import ScoreSession        # noqa: E402
from dct_pruning_b200.sites import VARIANT_INPUT, resolve_module   # noqa: E402
from dct_pruning_b200.zoo import get_network           # noqa: E402


def device_info():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30)
        info['nvidia_smi'] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info['nvidia_smi'] = None
    return info


def hbm_copy_rate(nbytes=4 << 30, reps=10):
    """Device-to-device copy of 4 GB: bytes read + written per second (the measured HBM peak the fractions refer to)."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device='cuda')
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) / 1e3)


def site_shapes(net_name, side):
    """[(C, H, W)] of every hook site of one forward at batch 1."""
    net = get_network(net_name).cuda().eval()
    session = ScoreSession(net, net_name)
    shapes, hooks = [], []
    for site in session.sites:
        def tap(m, i, o, site=site):
            t = i[0] if site.variant == VARIANT_INPUT else o
            shapes.append(tuple(t.shape[1:]))
        hooks.append(resolve_module(net, site.module).register_forward_hook(tap))
    with torch.no_grad():
        net(torch.zeros(1, 3, side, side, device='cuda'))
    for h in hooks:
        h.remove()
    return shapes


def pack(ptrs):
    buf = bytearray()
    for x_ptr, acc_ptr, B, c in ptrs:
        buf += struct.pack('QQii', x_ptr, acc_ptr, B, c)
    return (ctypes.c_char * len(buf)).from_buffer(buf), buf


def per_side(lib, batch, reps):
    shapes = site_shapes('resnet_50', 224)
    sides = sorted({s[1] for s in shapes}, reverse=True)
    g = torch.Generator(device='cuda').manual_seed(0)
    stream = _lib.current_stream()
    res = {}
    for side in sides:
        group = [s for s in shapes if s[1] == side and s[1] == s[2]]
        x16 = [torch.relu(torch.randn(batch, *s, device='cuda', generator=g)).to(torch.bfloat16) for s in group]
        x32 = [torch.relu(torch.randn(batch, *s, device='cuda', generator=g)) for s in group]
        accs = [torch.zeros(s[0], dtype=torch.float64, device='cuda') for s in group]
        elems = sum(t.numel() for t in x16)

        def multi(tensors, dtype):
            for i in range(0, len(tensors), 16):
                chunk = list(zip(tensors[i:i + 16], accs[i:i + 16]))
                arr, _keep = pack([(t.data_ptr(), a.data_ptr(), t.shape[0], t.shape[1]) for t, a in chunk])
                if dtype is None:
                    _lib.check(lib.dctp_score_accum_multi(arr, len(chunk), side, side, stream))
                else:
                    _lib.check(lib.dctp_score_accum_multi_ex(arr, len(chunk), side, side, dtype, stream))

        variants = {'a_native_bf16': lambda: multi(x16, _lib.DTYPE_BF16),
                    'b_float_then_fp32': lambda: multi([t.float() for t in x16], None),
                    'c_fp32': lambda: multi(x32, None)}
        sums = {}
        for name, fn in variants.items():                          # warm-up, and the channel sums of each variant
            for a in accs:
                a.zero_()
            fn()
            torch.cuda.synchronize()
            sums[name] = torch.cat([a.clone() for a in accs])
        ms = {k: [] for k in variants}
        for _ in range(reps):
            for name, fn in variants.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ms[name].append(e0.elapsed_time(e1))
        rel = ((sums['a_native_bf16'] - sums['b_float_then_fp32']).abs() / sums['b_float_then_fp32'].abs().clamp_min(1e-30)).max().item()
        lib.dctp_score_accum_multi_ex(pack([(x16[0].data_ptr(), accs[0].data_ptr(), batch, group[0][0])])[0], 1, side, side,
                                      _lib.DTYPE_BF16, stream)
        kernel = lib.dctp_last_kernel().decode().split(' ')[0]
        entry = {'sites': len(group), 'elements': elems, 'bytes_bf16': 2 * elems, 'bytes_fp32': 4 * elems, 'native_kernel': kernel,
                 'max_rel_diff_a_vs_b': rel}
        for name, v in ms.items():
            v = sorted(v)
            med = v[len(v) // 2]
            moved = {'a_native_bf16': 2, 'b_float_then_fp32': 10, 'c_fp32': 4}[name] * elems
            entry[name] = {'ms_median': round(med, 4), 'ms_min': round(v[0], 4), 'ms_max': round(v[-1], 4),
                           'GBps_at_2B': round(2 * elems / med / 1e6, 1), 'GBps_at_4B': round(4 * elems / med / 1e6, 1),
                           'bytes_moved': moved, 'GBps_moved': round(moved / med / 1e6, 1)}
        entry['speedup_a_over_b'] = round(entry['b_float_then_fp32']['ms_median'] / entry['a_native_bf16']['ms_median'], 3)
        entry['speedup_a_over_c'] = round(entry['c_fp32']['ms_median'] / entry['a_native_bf16']['ms_median'], 3)
        res['%dx%d' % (side, side)] = entry
        del x16, x32
        torch.cuda.empty_cache()
    return res


def end_to_end(net_name, side, batch, steps):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    out = {}
    for amp in ('off', 'bf16'):
        torch.manual_seed(0)
        net = get_network(net_name).cuda().eval()
        x = torch.randn(batch, 3, side, side, device='cuda')
        session = ScoreSession(net, net_name)
        with session, torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16, enabled=amp == 'bf16'):
            for _ in range(2):
                net(x)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                net(x)
            torch.cuda.synchronize()
            sec = time.perf_counter() - t0
        _lib.check(session.lib.dctp_check(None))
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16, enabled=amp == 'bf16'):    # the same forward, no hooks
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                net(x)
            torch.cuda.synchronize()
            fwd = time.perf_counter() - t0
        out[amp] = {'images_per_s': round(steps * batch / sec, 1), 'ms_per_step': round(sec / steps * 1e3, 3),
                    'forward_only_ms_per_step': round(fwd / steps * 1e3, 3)}
        del net, session, x
        torch.cuda.empty_cache()
    out['speedup'] = round(out['bf16']['images_per_s'] / out['off']['images_per_s'], 3)
    out.update(batch=batch, side=side, steps=steps)
    return out


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--out', required=True, help='directory for bench_half.json')
    p.add_argument('--batch', type=int, default=256)
    p.add_argument('--reps', type=int, default=15)
    p.add_argument('--steps', type=int, default=10)
    args = p.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_half.py measures on a CUDA device (B200); there is none')
    lib = _lib.load()
    _lib.check(lib.dctp_init())
    res = {'device': device_info(), 'hbm_copy_Bps': None}
    res['hbm_copy_Bps'] = hbm_copy_rate()
    res['resnet_50_224_by_side'] = per_side(lib, args.batch, args.reps)
    for entry in res['resnet_50_224_by_side'].values():
        for k in ('a_native_bf16', 'b_float_then_fp32', 'c_fp32'):
            entry[k]['frac_hbm'] = round(entry[k]['GBps_moved'] * 1e9 / res['hbm_copy_Bps'], 3)
    res['e2e_resnet_50_224'] = end_to_end('resnet_50', 224, args.batch, args.steps)
    res['e2e_u2netp_320'] = end_to_end('u2netp', 320, 32, args.steps)
    os.makedirs(args.out, exist_ok=True)
    line = json.dumps(res)
    with open(os.path.join(args.out, 'bench_half.json'), 'w') as f:
        f.write(line + '\n')
    print(line)


if __name__ == '__main__':
    main()
