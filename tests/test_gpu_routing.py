"""Which kernel instantiation each call runs: AUTO's choice per shape, layout and size, forced paths and what they refuse, and
how the multi-site entry splits its sites into launches.  Every launch is also checked against float64 (test_gpu_bounds.score).
"""
import math

import pytest
import torch

from dct_pruning_b200 import _lib
from test_gpu_bounds import ENERGY_TOL, Arena, maps, note, rel_err, score

pytestmark = pytest.mark.gpu

KRON7, KRON8 = 'score_kron_kernel<K2=64,odd>', 'score_kron_kernel<K2=64,even>'
STACK14, STACK56 = 'score_stack_kernel<KP=16,VEC=2,cfg7>', 'score_stack_kernel<KP=64,VEC=4,cfg7>'
STACK56_DEBUG = 'score_stack_kernel<KP=64,VEC=4,cfg6>'
T54, T11 = 'score_t_kernel<64,3,VPE=2>', 'score_t_kernel<32,6,VPE=4>'
T56_PRODUCERS, T60 = 'score_t_kernel<64,3,VPE=1,2 producer warpgroups>', 'score_t_kernel<64,3,VPE=1>'
LARGE, SIMT_SMALL, SIMT_LARGE = 'score_large_kernel', 'score_simt_small_kernel', 'score_simt_large_kernel'

# (what, path, B, C, H, W, keyword arguments of score(), kernel)
CASES = [
    ('7x7', 'auto', 2, 16, 7, 7, {}, KRON7),
    ('8x8', 'auto', 2, 16, 8, 8, {}, KRON8),
    ('14x14', 'auto', 2, 16, 14, 14, {}, STACK14),
    ('56x56', 'auto', 2, 16, 56, 56, {}, STACK56),
    ('56x56 with energy_out and coeff_out', 'auto', 2, 16, 56, 56, {'debug': True}, STACK56_DEBUG),
    ('56x56, one image, window 4+8 (dense)', 'auto', 1, 16, 56, 56, {'c_begin': 4, 'c_count': 8}, STACK56),
    ('54x54', 'auto', 2, 16, 54, 54, {}, T54),
    ('11x11, 33.7 MB', 'auto', 64, 1088, 11, 11, {}, T11),
    ('11x11', 'auto', 2, 16, 11, 11, {}, 'score_umma_kernel<64,2,1>'),
    ('9x9', 'auto', 2, 16, 9, 9, {}, 'score_umma_kernel<64,2,1>'),
    ('13x13', 'auto', 2, 16, 13, 13, {}, 'score_umma_kernel<64,2,1>'),
    ('34x34', 'auto', 2, 16, 34, 34, {}, 'score_umma_kernel<64,1,1>'),
    ('33x33', 'auto', 2, 16, 33, 33, {}, 'score_umma_kernel<64,5,0>'),
    ('72x72', 'auto', 2, 16, 72, 72, {}, 'score_umma_kernel<128,0,1>'),
    ('100x100', 'auto', 2, 16, 100, 100, {}, 'score_umma_kernel<128,0,0>'),
    ('80x80', 'auto', 2, 16, 80, 80, {}, LARGE),
    ('320x320', 'auto', 2, 4, 320, 320, {}, LARGE),
    ('80x80, window 4+12', 'auto', 2, 16, 80, 80, {'c_begin': 4, 'c_count': 12}, 'score_umma_kernel<128,3,0>'),
    ('160x160, window 4+12', 'auto', 2, 16, 160, 160, {'c_begin': 4, 'c_count': 12}, SIMT_LARGE),
    ('56x56, window 36+12', 'auto', 3, 48, 56, 56, {'c_begin': 36, 'c_count': 12}, 'score_umma_kernel<64,3,0>'),
    ('56x56, base 4 mod 16', 'auto', 2, 16, 56, 56, {'x_off': 4}, 'score_umma_kernel<64,5,0>'),
    ('56x56, base 8 mod 16', 'auto', 2, 16, 56, 56, {'x_off': 8}, 'score_umma_kernel<64,4,0>'),
    ('130x130', 'auto', 2, 16, 130, 130, {}, SIMT_LARGE),
    ('32x16', 'auto', 2, 16, 32, 16, {}, SIMT_SMALL),
    ('56x56 in rows of 60', 'auto', 2, 16, 56, 56, {'row': 60}, SIMT_SMALL),
    ('forced tmem, 56x56', 'tmem', 2, 16, 56, 56, {}, T56_PRODUCERS),
    ('forced tmem, 60x60', 'tmem', 2, 16, 60, 60, {}, T60),
]


@pytest.mark.parametrize('what,path,B,C,H,W,kw,kernel', CASES, ids=[c[0] for c in CASES])
def test_kernel_per_call(lib, cuda_device, what, path, B, C, H, W, kw, kernel):
    assert score(lib, path, B, C, H, W, seed=H + C, what=what, **kw) == kernel


# (what, path, B, C, H, W, c_begin, c_count): forced paths that do not take the call
REFUSED = [
    ('stack, 54x54', 'stack', 2, 16, 54, 54, 0, 16),
    ('kron, 9x9', 'kron', 2, 16, 9, 9, 0, 16),
    ('tmem, 15x15', 'tmem', 2, 16, 15, 15, 0, 16),
    ('tmem, 11x11, 363 maps (not a whole number of float4)', 'tmem', 1, 363, 11, 11, 0, 363),
    ('large, 72x72', 'large', 2, 16, 72, 72, 0, 16),
    ('large, 80x80 window 4+12', 'large', 2, 16, 80, 80, 4, 12),
    ('umma, 130x130', 'umma', 2, 16, 130, 130, 0, 16),
    ('umma, 32x16', 'umma', 2, 16, 32, 16, 0, 16),
]


@pytest.mark.parametrize('what,path,B,C,H,W,c_begin,c_count', REFUSED, ids=[r[0] for r in REFUSED])
def test_forced_path_refuses(lib, cuda_device, what, path, B, C, H, W, c_begin, c_count):
    x = torch.zeros(B, C, H, W, device='cuda')
    acc = torch.zeros(c_count, dtype=torch.float64, device='cuda')
    before = lib.dctp_launch_count()
    rc = lib.dctp_score_accum(_lib.ptr(x), B, H, W, x.stride(0), x.stride(1), x.stride(2), c_begin, c_count, _lib.ptr(acc), None,
                              None, _lib.PATHS[path], _lib.current_stream())
    assert rc == _lib.E_UNSUPPORTED, (rc, lib.dctp_last_error())
    assert lib.dctp_launch_count() == before


# (what, side, byte offset mod 128 of each site, launches, kernel of the last launch)
MULTI = [
    ('three aligned 56x56 sites and one 4 bytes off', 56, [0, 16, 64, 4], 2, 'score_umma_kernel<64,5,0>'),
    ('20 sites of 7x7', 7, [(0, 16, 64)[i % 3] for i in range(20)], 2, KRON7),
    ('17 sites of 80x80', 80, [(0, 16, 64)[i % 3] for i in range(17)], 2, LARGE),
    ('3 sites of 72x72', 72, [0, 16, 64], 3, 'score_umma_kernel<128,0,1>'),
]


@pytest.mark.parametrize('what,side,offs,launches,kernel', MULTI, ids=[m[0] for m in MULTI])
def test_multi_site_launches(lib, cuda_device, what, side, offs, launches, kernel):
    B, C, NN = 2, 3, side * side
    xa = Arena([B * C * NN] * len(offs), torch.float32, offs, guard=max(1 << 18, 4 * NN * 4))
    acc = Arena([C] * len(offs), torch.float64, edge=0.0, live=0.0)
    src = [maps(B, C, side, side, seed=side + i) for i in range(len(offs))]
    sites = (_lib.Site * len(offs))()
    for i in range(len(offs)):
        sites[i].B, sites[i].c_count = B, C
        sites[i].x, sites[i].accum = xa.views[i].data_ptr(), acc.views[i].data_ptr()
        xa.views[i].copy_(src[i].reshape(-1))
    stream = _lib.current_stream()
    before = lib.dctp_launch_count()
    _lib.check(lib.dctp_score_accum_multi(sites, len(offs), side, side, stream))
    assert lib.dctp_launch_count() - before == launches
    _lib.check(lib.dctp_check(stream))
    assert note(lib) == kernel
    for i in range(len(offs)):
        want = (src[i].double() ** 2).sum((0, 2, 3))
        live = want > 0
        assert math.isclose(float(acc.views[i][~live].abs().sum()), 0.0)
        assert rel_err(acc.views[i][live], want[live]) < ENERGY_TOL, (what, i)
