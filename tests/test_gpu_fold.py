"""The stacked-basis kernel's folded stage 2 (score_stack.cuh, stack_folded: sides 18..64) on maps with known answers.

With C[u][N-1-h] = (-1)^u C[u][h], stage 2 runs as two chains: even u against the row sums Y[h] + Y[N-1-h] of the stage-1 result,
odd u against the row differences.  The converters' table puts row N-1-h next to its partner in the second half of the map's D1
columns; at sides 18..24, 36, 40, 52 and 56 the middle rows stay unpaired and go to both chains.  A map symmetric in h
(X[N-1-h] = X[h]) has every odd-u coefficient 0, an antisymmetric one every even-u coefficient: a chain handed the wrong half, a
column mapped back to the wrong u, or a row placed at the wrong column puts energy where there must be none.  (Single-mode maps,
each (u, v) on its own coefficient at every side and tile slot: test_gpu_precision.py.)

Every case: B x C maps of a tile count that leaves the last tile ragged (and, where B C N^2 is not a multiple of 32, converted from
global memory), forced and through AUTO, fp32 / bf16 / fp16, the debug instantiation (per-map energies, coefficients) and the
production one (channel sums); and multi-site launches of symmetric and antisymmetric activations.
"""
import pytest
import torch

from dct_pruning_b200 import _lib
from test_gpu_kernels import ENERGY_TOL, STACK_SIDES
from test_gpu_precision import exact

pytestmark = pytest.mark.gpu

FOLD_SIDES = [n for n in STACK_SIDES if n > 16]
DTYPES = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}
COEF_TOL = 3e-5          # of the map's largest coefficient: test_gpu_precision's peak-coefficient bar, far above random maps' errors


def mirrored(B, C, N, sign, dtype, seed):
    """relu(N(0, 1)) rows h < N / 2 (N even) and X[N-1-h] = sign * X[h], rounded to dtype; channels 1 mod 4 dead."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    top = torch.relu(torch.randn(B, C, N // 2, N, generator=g, device='cuda'))
    top[:, 1::4] = 0.0
    return torch.cat([top, sign * top.flip(2)], 2).to(dtype)


def check_coefficients(co, x, sign, label):
    """co: [B, C, N, N] coefficients Z[u][v]; rows u of the parity the symmetry zeroes must hold nothing, the rest float64's values."""
    Z64 = exact(x.double())
    peak = Z64.abs().amax((-2, -1), keepdim=True).clamp_min(1e-30)
    err = (co.double() - Z64).abs() / peak
    quiet = co[:, :, 1::2] if sign > 0 else co[:, :, 0::2]
    assert float((quiet.double().abs() / peak).max()) < COEF_TOL, 'energy in the u the symmetry zeroes: ' + label
    assert float(err.max()) < COEF_TOL, 'coefficients: ' + label


@pytest.mark.parametrize('sign', [1, -1])
@pytest.mark.parametrize('path', ['stack', 'auto'])
@pytest.mark.parametrize('dt', sorted(DTYPES))
@pytest.mark.parametrize('n', FOLD_SIDES)
def test_mirrored_maps(lib, cuda_device, n, dt, path, sign):
    from dct_pruning_b200.ops import dct_energy
    dtype = DTYPES[dt]
    B, C = 3, 37                                  # 111 maps: the last tile (2 or 8 maps) is ragged
    x = mirrored(B, C, n, sign, dtype, seed=31 * n + sign)
    E64 = (x.double() ** 2).sum((2, 3))           # Parseval
    live = E64 > 0
    for debug in (True, False):
        acc, en, co = dct_energy(x, path=path, want_energy=debug, want_coeff=debug)
        name = lib.dctp_last_kernel().decode().split(' (')[0]
        label = '%s %dx%d %s sign %+d %s' % (path, n, n, dt, sign, name)
        assert name.startswith('score_stack_kernel') and ('cfg6' if debug else 'cfg7') in name, label
        if debug:
            assert bool((en[~live] == 0).all()), 'dead map ' + label
            assert float(((en.double() - E64).abs()[live] / E64[live]).max()) < ENERGY_TOL, 'energy_out ' + label
            check_coefficients(co, x, sign, label)
        want = E64.sum(0)
        assert bool((acc[want == 0] == 0).all()), 'dead channel ' + label
        assert float(((acc - want).abs()[want > 0] / want[want > 0]).max()) < ENERGY_TOL, 'accum ' + label


@pytest.mark.parametrize('dt', sorted(DTYPES))
@pytest.mark.parametrize('n', [18, 28, 36, 44, 56, 64])
def test_mirrored_multi_site(lib, cuda_device, n, dt):
    """Five sites of one launch, symmetric and antisymmetric in turn, of sizes that end mid-tile."""
    dtype = DTYPES[dt]
    plan = [(1, 1), (2, 5), (3, 7), (1, 13), (4, 3)]
    xs = [mirrored(B, C, n, 1 if i % 2 == 0 else -1, dtype, seed=7 * n + i) for i, (B, C) in enumerate(plan)]
    accs = [torch.zeros(C, dtype=torch.float64, device='cuda') for _, C in plan]
    sites = (_lib.Site * len(plan))()
    for i, (B, C) in enumerate(plan):
        sites[i].B, sites[i].c_count = B, C
        sites[i].x, sites[i].accum = xs[i].data_ptr(), accs[i].data_ptr()
    _lib.check(lib.dctp_prepare(n, n))
    stream = _lib.current_stream()
    before = lib.dctp_launch_count()
    _lib.check(lib.dctp_score_accum_multi_ex(sites, len(plan), n, n, _lib.dtype_code(dtype), stream))
    _lib.check(lib.dctp_check(stream))
    name = lib.dctp_last_kernel().decode()
    assert lib.dctp_launch_count() - before == 1 and name.startswith('score_stack_kernel'), name
    for i, x in enumerate(xs):
        want = (x.double() ** 2).sum((0, 2, 3))
        got = accs[i]
        assert bool((got[want == 0] == 0).all()), ('dead channel', i, name)
        assert float(((got - want).abs()[want > 0] / want[want > 0]).max()) < ENERGY_TOL, ('site', i, name)
