"""Parity of the CUDA scoring kernels with the CPU oracle, through the C ABI (ctypes).

Bar (BASELINE north_star): per-channel scores within relative 1e-4 of the reference; the
tolerance is written in each assert.  Per-map energies are checked against the float64 oracle
(oracle.reference_port.energy_scipy64 and Parseval), scores against the op-for-op port of the
reference hooks, coefficients against scipy's dctn.  Exact zeros must stay exactly zero (dead
post-ReLU channels are the common case and decide top-k ties).
"""
import numpy as np
import pytest
import torch

from oracle import reference_port as port

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4           # the north_star bar on scores
ENERGY_TOL = 2e-5        # what the bf16x3 / fp32 kernels deliver per map on random maps (relu_maps; the rounding errors cancel),
                         # not a bound: on maps built to line them up they reach 5e-5 (test_gpu_precision.py)


def relu_maps(shape, seed, dead_every=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.relu(torch.randn(*shape, generator=g))
    if dead_every:
        x[:, ::dead_every] = 0.0
    return x


def rel_err(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return np.abs(got - want) / np.maximum(np.abs(want), 1e-30)


UMMA_SIDES = [1, 2, 3, 4, 7, 8, 9, 10, 14, 16, 18, 20, 24, 28, 32, 36, 40, 48, 52, 56, 60, 64, 72, 80, 112, 128]
TMEM_SIDES = [5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 16, 18, 20, 22, 24, 26, 28, 30, 32, 34, 36, 40, 44, 48, 50, 52, 56, 60, 62, 64]


@pytest.mark.parametrize('n', UMMA_SIDES)
@pytest.mark.parametrize('path', ['umma', 'simt'])
def test_energy_matches_float64_oracle(lib, cuda_device, n, path):
    from dct_pruning_b200.ops import dct_energy
    B, C = (3, 37) if n <= 64 else (2, 5)
    x = relu_maps((B, C, n, n), seed=n, dead_every=5)
    acc, en, _ = dct_energy(x.to(cuda_device), path=path, want_energy=True)
    want = port.energy_scipy64(x.numpy())
    pars = port.energy_parseval64(x.numpy())
    en = en.cpu().numpy()
    live = want > 0
    assert (en[~live] == 0).all(), 'dead maps must score exactly 0'
    assert rel_err(en[live], want[live]).max() < ENERGY_TOL
    assert rel_err(en[live], pars[live]).max() < ENERGY_TOL
    got = acc.cpu().numpy()
    assert rel_err(got[want.sum(0) > 0], want.sum(0)[want.sum(0) > 0]).max() < ENERGY_TOL
    # accum is the exact fp64 sum of the per-map fp32 energies
    # (the CUDA-core kernel for maps > 64 adds per-panel partials, so its two outputs agree to fp32 rounding only)
    np.testing.assert_allclose(got, en.astype(np.float64).sum(0), rtol=1e-12 if (path == 'umma' or n <= 64) else 1e-6)


@pytest.mark.parametrize('n', TMEM_SIDES)
def test_tmem_operand_kernel(lib, cuda_device, n):
    """The TMEM-operand formulation (basis resident in TMEM, transposed stage 1) on every side it takes,
    incl. many tiles per slot, a ragged last tile, and the coefficient dump."""
    from scipy.fft import dctn
    from dct_pruning_b200.ops import dct_energy
    # (odd sides: a float4 of the stream may straddle maps, so the call must hold a whole number of float4)
    x = relu_maps((5, 131, n, n) if n % 2 == 0 else (4, 131, n, n), seed=200 + n, dead_every=6)
    acc, en, _ = dct_energy(x.to(cuda_device), path='tmem', want_energy=True)
    want = port.energy_scipy64(x.numpy())
    en = en.cpu().numpy()
    live = want > 0
    assert (en[~live] == 0).all()
    assert rel_err(en[live], want[live]).max() < ENERGY_TOL
    np.testing.assert_allclose(acc.cpu().numpy(), en.astype(np.float64).sum(0), rtol=1e-12)
    small = relu_maps((1, 3, n, n) if n % 2 == 0 else (1, 4, n, n), seed=300 + n)
    _, _, co = dct_energy(small.to(cuda_device), path='tmem', want_coeff=True)
    z = dctn(small.numpy().astype(np.float64), type=2, norm='ortho', axes=(-2, -1))
    assert np.abs(co.cpu().numpy() - z).max() / np.abs(z).max() < 2e-5


@pytest.mark.parametrize('n', [1, 2, 3, 4, 5, 6, 7, 8])
def test_kronecker_kernel(lib, cuda_device, n):
    """Single-stage Kronecker kernel (sides <= 8): several tiles per CTA, ragged last tile, a stream that does not end on a
    128-byte row (odd sides), the coefficient dump, exact zeros."""
    from scipy.fft import dctn
    from dct_pruning_b200.ops import dct_energy
    for shape, seed in (((5, 131, n, n), 610 + n), ((1, 3, n, n), 710 + n), ((64, 2048, n, n), 810 + n)):
        x = relu_maps(shape, seed=seed, dead_every=6)
        acc, en, _ = dct_energy(x.to(cuda_device), path='kron', want_energy=True)
        want = port.energy_parseval64(x.numpy()) if shape[0] == 64 else port.energy_scipy64(x.numpy())
        en = en.cpu().numpy()
        live = want > 0
        assert (en[~live] == 0).all()
        # (a handful of elements per map: the split-precision residuals do not average out, and the maximum is over 131 k maps)
        assert rel_err(en[live], want[live]).max() < (ENERGY_TOL if shape[0] < 64 else 2 * ENERGY_TOL), (shape, rel_err(en[live], want[live]).max())
        np.testing.assert_allclose(acc.cpu().numpy(), en.astype(np.float64).sum(0), rtol=1e-12)
    small = relu_maps((2, 5, n, n), seed=910 + n)
    _, _, co = dct_energy(small.to(cuda_device), path='kron', want_coeff=True)
    z = dctn(small.numpy().astype(np.float64), type=2, norm='ortho', axes=(-2, -1))
    assert np.abs(co.cpu().numpy() - z).max() / np.abs(z).max() < 2e-5


STACK_SIDES = [10, 12, 14, 16, 18, 20, 22, 24, 26, 28, 30, 32, 36, 40, 44, 48, 52, 56, 60, 64]


@pytest.mark.parametrize('n', STACK_SIDES)
def test_stacked_basis_kernel(lib, cuda_device, n):
    """The warp-specialised stacked-basis kernel (TMA-staged tiles, hi/lo basis stacked along the TMEM lanes) on every
    side it takes: many tiles per CTA, a ragged last tile, a stream that does not end on a 128-byte row (the tile that
    is converted straight from global memory), the coefficient dump, exact zeros."""
    from scipy.fft import dctn
    from dct_pruning_b200.ops import dct_energy
    for shape, seed in (((5, 131, n, n), 600 + n), ((1, 3, n, n), 700 + n), ((2, 700, n, n), 800 + n)):
        x = relu_maps(shape, seed=seed, dead_every=6)
        acc, en, _ = dct_energy(x.to(cuda_device), path='stack', want_energy=True)
        want = port.energy_scipy64(x.numpy())
        en = en.cpu().numpy()
        live = want > 0
        assert (en[~live] == 0).all()
        assert rel_err(en[live], want[live]).max() < ENERGY_TOL, shape
        np.testing.assert_allclose(acc.cpu().numpy(), en.astype(np.float64).sum(0), rtol=1e-12)
    small = relu_maps((2, 5, n, n), seed=900 + n)
    _, _, co = dct_energy(small.to(cuda_device), path='stack', want_coeff=True)
    z = dctn(small.numpy().astype(np.float64), type=2, norm='ortho', axes=(-2, -1))
    assert np.abs(co.cpu().numpy() - z).max() / np.abs(z).max() < 2e-5


@pytest.mark.parametrize('n', [1, 3, 7, 8] + STACK_SIDES + [96, 160, 288, 320])
def test_production_instantiations_match_oracle(lib, cuda_device, n):
    """The launches above ask for per-map energies or coefficients, which the stacked-basis and large-map kernels only carry in their
    debug instantiations.  Here nothing but the channel sums is requested - the instantiation every hook launch runs (AUTO's choice) -
    on shapes with many tiles per CTA, a ragged last tile and more maps than one tile holds; per-channel sums vs float64."""
    from dct_pruning_b200 import _lib
    from dct_pruning_b200.ops import dct_energy
    shapes = ((3, 150, n, n), (1, 5, n, n)) if n <= 64 else ((2, 40, n, n), (1, 3, n, n))
    for shape in shapes:
        x = relu_maps(shape, seed=1300 + n, dead_every=5)
        acc, en, co = dct_energy(x.to(cuda_device), path='auto')
        assert en is None and co is None
        name = _lib.load().dctp_last_kernel().decode()
        assert ('cfg6' not in name) and name, name                   # not the debug instantiation
        want = port.energy_scipy64(x.numpy()).sum(0)
        got = acc.cpu().numpy()
        live = want > 0
        assert (got[~live] == 0).all()
        assert rel_err(got[live], want[live]).max() < ENERGY_TOL, (shape, name)


@pytest.mark.parametrize('n', [4, 7, 8, 10, 14, 20, 28, 40, 56, 64, 80, 128])
@pytest.mark.parametrize('path', ['umma', 'simt'])
def test_coefficients_match_scipy(lib, cuda_device, n, path):
    from scipy.fft import dctn
    from dct_pruning_b200.ops import dct_energy
    x = relu_maps((2, 11, n, n), seed=100 + n)
    _, _, co = dct_energy(x.to(cuda_device), path=path, want_coeff=True)
    want = dctn(x.numpy().astype(np.float64), type=2, norm='ortho', axes=(-2, -1))
    err = np.abs(co.cpu().numpy() - want).max() / np.abs(want).max()
    assert err < 2e-5, err


@pytest.mark.parametrize('shape', [(2, 3, 32, 16), (2, 3, 9, 20), (1, 2, 144, 144), (1, 2, 160, 96), (1, 1, 320, 320),
                                   (1, 2, 288, 288), (1, 3, 130, 130)])
def test_general_shapes_on_cuda_cores(lib, cuda_device, shape):
    from dct_pruning_b200.ops import dct_energy
    x = relu_maps(shape, seed=sum(shape))
    _, en, co = dct_energy(x.to(cuda_device), path='auto', want_energy=True, want_coeff=shape[2] <= 160)
    want = port.energy_scipy64(x.numpy())
    assert rel_err(en.cpu().numpy(), want).max() < ENERGY_TOL
    if co is not None:
        from scipy.fft import dctn
        z = dctn(x.numpy().astype(np.float64), type=2, norm='ortho', axes=(-2, -1))
        assert np.abs(co.cpu().numpy() - z).max() / np.abs(z).max() < 2e-5


@pytest.mark.parametrize('n', [80, 96, 112, 128, 144, 160, 176, 256, 288, 320])
def test_large_map_kernel(lib, cuda_device, n):
    """Tiled tensor-core kernel for U^2-Netp's large stages: energies vs the float64 oracle and vs the CUDA-core
    kernel, coefficients vs scipy, several maps per channel and more work items than SMs."""
    from scipy.fft import dctn
    from dct_pruning_b200.ops import dct_energy
    x = relu_maps((2, 3, n, n), seed=400 + n, dead_every=3)
    acc, en, co = dct_energy(x.to(cuda_device), path='large', want_energy=True, want_coeff=True)
    want = port.energy_scipy64(x.numpy())
    en = en.cpu().numpy()
    live = want > 0
    assert (en[~live] == 0).all()
    assert rel_err(en[live], want[live]).max() < ENERGY_TOL
    z = dctn(x.numpy().astype(np.float64), type=2, norm='ortho', axes=(-2, -1))
    assert np.abs(co.cpu().numpy() - z).max() / np.abs(z).max() < 2e-5
    assert rel_err(acc.cpu().numpy()[want.sum(0) > 0], want.sum(0)[want.sum(0) > 0]).max() < ENERGY_TOL
    many = relu_maps((3, 70, n, n), seed=500 + n) if n <= 160 else relu_maps((2, 40, n, n), seed=500 + n)
    _, en_l, _ = dct_energy(many.to(cuda_device), path='large', want_energy=True)
    pars = port.energy_parseval64(many.numpy())
    assert rel_err(en_l.cpu().numpy(), pars).max() < ENERGY_TOL


@pytest.mark.parametrize('path', ['umma', 'simt'])
def test_known_answer_vectors(lib, cuda_device, path):
    from dct_pruning_b200.ops import dct_energy
    n = 8
    k = np.arange(n)[:, None]
    m = np.arange(n)[None, :]
    c = np.cos(np.pi * (2 * m + 1) * k / (2 * n)) * np.sqrt(2.0 / n)
    c[0] *= np.sqrt(0.5)
    x = torch.zeros(1, 4, n, n)
    x[0, 1] = 3.0                                   # constant map: only DC, energy n*n*9
    x[0, 2, 2, 5] = 1.0                             # impulse: coefficients = outer(c[:,2], c[:,5]), energy 1
    x[0, 3] = torch.from_numpy(np.outer(c[3], c[1]).astype(np.float32))   # one cosine mode: Z[3,1] = 1
    _, en, co = dct_energy(x.to(cuda_device), path=path, want_energy=True, want_coeff=True)
    en, co = en.cpu().numpy()[0], co.cpu().numpy()[0]
    assert en[0] == 0.0 and np.abs(co[0]).max() == 0.0
    assert abs(en[1] - n * n * 9.0) < 1e-4 * n * n * 9.0 and abs(co[1, 0, 0] - 3.0 * n) < 1e-4 * 3 * n
    np.testing.assert_allclose(co[2], np.outer(c[:, 2], c[:, 5]), atol=2e-6)
    assert abs(en[2] - 1.0) < 1e-5
    assert abs(co[3, 3, 1] - 1.0) < 1e-5 and abs(en[3] - 1.0) < 1e-5


@pytest.mark.parametrize('path', ['umma', 'simt'])
def test_channel_window_and_strides(lib, cuda_device, path):
    """DenseNet's last-12 window (common.py:285) and non-contiguous batch/channel strides."""
    from dct_pruning_b200.ops import dct_energy
    big = relu_maps((4, 60, 16, 16), seed=7).to(cuda_device)
    view = big[1:4, 6:54]                            # stride_b = 60*256, base offset not a multiple of the map size
    acc, en, _ = dct_energy(view, c_begin=view.shape[1] - 12, c_count=12, path=path, want_energy=True)
    want = port.energy_scipy64(view.cpu().numpy()[:, -12:])
    assert rel_err(en.cpu().numpy(), want).max() < ENERGY_TOL
    odd = relu_maps((2, 9, 14, 14), seed=8).to(cuda_device)[:, 1:8]      # channel offset 1*196 floats: 16-B aligned only by luck
    _, en2, _ = dct_energy(odd, path=path, want_energy=True)
    assert rel_err(en2.cpu().numpy(), port.energy_scipy64(odd.cpu().numpy())).max() < ENERGY_TOL
    shifted = relu_maps((1, 3, 7, 7), seed=9).to(cuda_device).flatten()[1:1 + 2 * 49].view(1, 2, 7, 7)   # 4-B aligned base
    _, en3, _ = dct_energy(shifted, path=path, want_energy=True)
    assert rel_err(en3.cpu().numpy(), port.energy_scipy64(shifted.cpu().numpy())).max() < ENERGY_TOL
    half = relu_maps((1, 3, 8, 8), seed=10).to(cuda_device).flatten()[2:2 + 2 * 64].view(1, 2, 8, 8)       # 8-B aligned base
    _, en4, _ = dct_energy(half, path=path, want_energy=True)
    assert rel_err(en4.cpu().numpy(), port.energy_scipy64(half.cpu().numpy())).max() < ENERGY_TOL


def test_strided_rows_fall_to_cuda_cores(lib, cuda_device):
    from dct_pruning_b200.ops import dct_energy
    from dct_pruning_b200 import _lib
    big = relu_maps((2, 3, 20, 24), seed=11).to(cuda_device)
    crop = big[:, :, :, 2:22]                        # 20x20 maps with stride_h = 24
    _, en, _ = dct_energy(crop, path='auto', want_energy=True)
    assert rel_err(en.cpu().numpy(), port.energy_scipy64(crop.cpu().numpy())).max() < ENERGY_TOL
    with pytest.raises(_lib.DctpError):
        dct_energy(crop, path='umma')


def test_empty_and_ragged_inputs(lib, cuda_device):
    from dct_pruning_b200.ops import dct_energy
    x = torch.zeros(0, 4, 8, 8, device=cuda_device)
    acc, _, _ = dct_energy(x)
    assert float(acc.abs().sum()) == 0.0
    x = relu_maps((5, 7, 8, 8), seed=3).to(cuda_device)        # 35 maps: a ragged last tile of the 128-map tile
    acc, en, _ = dct_energy(x, want_energy=True)
    assert rel_err(en.cpu().numpy(), port.energy_scipy64(x.cpu().numpy())).max() < ENERGY_TOL
    acc0, _, _ = dct_energy(x, c_begin=3, c_count=0)
    assert acc0.numel() == 0


@pytest.mark.parametrize('path', ['umma', 'simt'])
def test_hook_semantics_match_reference_port(lib, cuda_device, path):
    """Three batches through the reference's hook (running fp32 mean) vs accumulate + finalize."""
    from dct_pruning_b200.ops import dct_energy, finalize
    state = port.ScoreState()
    hook = port.hook_output(state)
    acc = None
    n = 0
    for b, bs in enumerate([3, 2, 4]):
        x = relu_maps((bs, 6, 10, 10), seed=40 + b, dead_every=3)
        hook(None, None, x)
        acc, _, _ = dct_energy(x.to(cuda_device), path=path, accum=acc)
        n += bs
    got = finalize(acc, n).cpu().numpy()
    want = state.feature_result.numpy()
    live = want > 0
    assert (got[~live] == 0).all()
    assert rel_err(got[live], want[live]).max() < REL_TOL
    d = port.ScoreState()
    dh = port.hook_densenet(d)
    x = relu_maps((2, 20, 8, 8), seed=50)
    dh(None, None, x)
    acc, _, _ = dct_energy(x.to(cuda_device), c_begin=8, c_count=12, path=path)
    assert rel_err(finalize(acc, 2).cpu().numpy(), d.feature_result.numpy()).max() < REL_TOL


def test_host_buffer_entry(lib, cuda_device):
    import ctypes
    x = relu_maps((3, 5, 14, 14), seed=60).numpy()
    out = np.zeros(4, np.float32)
    rc = lib.dctp_score_host(x.ctypes.data_as(ctypes.c_void_p), 3, 5, 14, 14, 1, 4, out.ctypes.data_as(ctypes.c_void_p), 0)
    assert rc == 0, lib.dctp_last_error()
    want = port.score_scipy64(x, 1, 4)
    assert rel_err(out, want).max() < ENERGY_TOL


def test_bad_arguments_are_refused(lib, cuda_device):
    import ctypes
    x = torch.zeros(1, 1, 8, 8, device=cuda_device)
    acc = torch.zeros(1, dtype=torch.float64, device=cuda_device)
    rc = lib.dctp_score_accum(None, 1, 8, 8, 64, 64, 8, 0, 1, ctypes.c_void_p(acc.data_ptr()), None, None, 0, None)
    assert rc == -1 and b'null' in lib.dctp_last_error()
    rc = lib.dctp_score_accum(ctypes.c_void_p(x.data_ptr()), 1, 8, 8, 64, 64, 4, 0, 1, ctypes.c_void_p(acc.data_ptr()), None, None, 0, None)
    assert rc == -1                                   # stride_h < W
    rc = lib.dctp_score_accum(ctypes.c_void_p(x.data_ptr()), 1, 8, 8, 64, 64, 8, 0, 1, ctypes.c_void_p(acc.data_ptr()), None, None, 9, None)
    assert rc == -1                                   # unknown path
