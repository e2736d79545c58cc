"""Importance generation under torch.autocast: the hooks score the bf16 activations the forward produced, as they are.

The oracle is the float64 energy of those same activations, taken by plain recording hooks on the same forward: scores within
relative 1e-4 (the north_star bar) and exact zeros where the oracle is zero.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

NETS = [('vgg_16_bn', 32), ('resnet_56', 32), ('resnet_110', 32), ('densenet_40', 32), ('googlenet', 32), ('resnet_50', 64),
        ('u2netp', 64)]


def run_session(net_name, side, batch, amp_dtype, device, seed=0):
    """One forward with a ScoreSession and float64 recording hooks on every site; returns (session, oracle sums per site,
    dtypes the sites fired with, launches)."""
    from dct_pruning_b200.hooks import ScoreSession
    from dct_pruning_b200.sites import DENSENET_WINDOW, VARIANT_INPUT, VARIANT_LAST12, resolve_module
    from dct_pruning_b200.zoo import get_network
    torch.manual_seed(seed)
    net = get_network(net_name).to(device).eval()
    session = ScoreSession(net, net_name)
    oracle = [None] * len(session.sites)
    dtypes = [None] * len(session.sites)
    taps = []
    for idx, site in enumerate(session.sites):
        def tap(module, inputs, output, idx=idx, site=site):
            t = inputs[0] if site.variant == VARIANT_INPUT else output
            if site.variant == VARIANT_LAST12:
                t = t[:, t.shape[1] - DENSENET_WINDOW:]
            e = (t.double() ** 2).sum((-2, -1)).sum(0)
            oracle[idx] = e if oracle[idx] is None else oracle[idx] + e
            dtypes[idx] = t.dtype
        taps.append(resolve_module(net, site.module).register_forward_hook(tap))
    g = torch.Generator().manual_seed(1000 + seed)
    x = torch.randn(batch, 3, side, side, generator=g).to(device)
    with session, torch.no_grad(), torch.autocast('cuda', dtype=amp_dtype, enabled=amp_dtype is not None):
        session.launches = 0
        net(x)
    torch.cuda.synchronize()
    for h in taps:
        h.remove()
    return session, oracle, dtypes, session.launches


@pytest.mark.parametrize('net_name,side', NETS)
def test_autocast_scores_match_float64_of_the_same_activations(lib, cuda_device, net_name, side):
    session, oracle, dtypes, _ = run_session(net_name, side, 2, torch.bfloat16, cuda_device)
    assert any(d is torch.bfloat16 for d in dtypes)
    for idx, (site, want) in enumerate(zip(session.sites, oracle)):
        if want is None:
            continue
        off, c = session.slots[idx]
        got = session.flat[off:off + c].cpu().numpy()
        want = want.cpu().numpy()
        live = want > 0
        assert (got[~live] == 0).all(), (site.module, 'dead channels must score exactly 0')
        rel = np.abs(got[live] - want[live]) / want[live]
        assert rel.size == 0 or rel.max() < 1e-4, (site.module, dtypes[idx], rel.max())


@pytest.mark.parametrize('batch', [2, 256])
def test_resnet50_autocast_keeps_the_launch_count(lib, cuda_device, batch):
    """Under bf16 autocast every ResNet-50 site fires in bf16, so the sites group as in fp32 (at batch 256 the halved bytes may
    hold a group back from the held-bytes flush: never more launches than fp32)."""
    _, _, _, launches32 = run_session('resnet_50', 224, batch, None, cuda_device)
    session, _, dtypes16, launches16 = run_session('resnet_50', 224, batch, torch.bfloat16, cuda_device)
    stays_fp32 = [s.module for s, d in zip(session.sites, dtypes16) if d is not torch.bfloat16]
    assert stays_fp32 == [], stays_fp32
    assert launches16 == launches32 if batch == 2 else launches16 <= launches32, (launches16, launches32)


def test_cli_amp_writes_the_usual_files(lib, cuda_device, tmp_path, monkeypatch):
    from dct_pruning_b200 import cli
    from dct_pruning_b200.generate import npy_bytes
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        monkeypatch.delenv(k, raising=False)
    out = tmp_path / 'importance_score'
    cli.main(['--net', 'resnet_56', '--batch_size', '8', '--limit', '2', '--out_root', str(out), '--pretrain_dir',
              str(tmp_path / 'none.pt'), '--synthetic', '--random_init', '--amp', 'bf16'])
    d = out / 'resnet_56_limit2'
    files = sorted(f for f in os.listdir(d) if f.endswith('.npy'))
    assert len(files) == 55
    for f in files:
        raw = open(d / f, 'rb').read()
        v = np.load(d / f)
        assert v.dtype == np.dtype('<f4') and v.ndim == 1 and raw == npy_bytes(v)
        assert np.isfinite(v).all() and (v >= 0).all()
