"""Non-finite maps: a NaN or an Inf in one (image, channel) map changes only its own channel's score, on every score kernel.

The reference scores every (image, channel) slice on its own (one dct_2d and one cnt_score per slice), so a non-finite map makes
only its own channel's score non-finite, and top-k ranks that channel above every finite one.  Several tensor-core kernels put
more than one map into one MMA and keep them apart with zero blocks in an operand; 0 * NaN and 0 * Inf are NaN, so there a
non-finite map also reaches the other maps of its tile.  The kernels test each contribution they add to `accum` / `energy_out`
for finiteness and recompute a non-finite one from the map in global memory (NaN for a map that holds a non-finite element, the
float64 value otherwise).  What this module pins, for dctp_score_accum, dctp_score_accum_multi and dctp_score_op(DCT2 / DCT3):

  1. culprit     a channel with a non-finite scored map gets a non-finite accum entry, the map a non-finite energy_out entry
                 (NaN or Inf: not pinned).  FLT_MAX is finite but overflows inside the kernel: non-finite, or within ENERGY_TOL
                 of float64.
  2. the others  every other channel and map within ENERGY_TOL of float64 Parseval on the same tensor; dead maps (all +0.0 or
                 all -0.0) exactly 0, also next to a culprit.
  3. DCT3        values_out[b] is non-finite exactly for the images with a non-finite map inside the window.
  4. no fault    dctp_check returns DCTP_OK, also when every map or every other map is non-finite.

Culprits sit at the first and the last map of the stream (a ragged last tile), at maps P - 1 and P for P = 2 .. 128 (the first
or last map of a tile for every kernel's maps per tile) and at a few seeded random maps; at (0, 0), (N-1, N-1), (0, N-1) and
the middle of their map; in distinct channels, at most one in eight.  The oracle is float64 on the host with the culprits left
out, and for small cases the finite / non-finite pattern of the op-for-op port of the reference hook.  test_gpu_half_bounds.py runs
the same matrix on bf16 and fp16 maps (dctp_score_accum_ex, dctp_score_accum_multi_ex) through the helpers here, with the bit
patterns of those types (KINDS16).
"""
import numpy as np
import pytest
import torch

from dct_pruning_b200 import _lib
from oracle import reference_port as port
from test_gpu_bounds import LARGE_SIDES, geometry, maps
from test_gpu_kernels import ENERGY_TOL, STACK_SIDES, TMEM_SIDES

pytestmark = pytest.mark.gpu

# culprit kinds: float32 bit patterns; 'all_nan' fills the whole map; 'flt_max' is the largest finite value of the type
KINDS = {'nan': 0x7fc00000, 'neg_nan': 0xffc00000, 'snan': 0x7f800001, 'inf': 0x7f800000, 'neg_inf': 0xff800000,
         'all_nan': 0x7fc00000, 'flt_max': 0x7f7fffff}
KINDS16 = {torch.bfloat16: {'nan': 0x7fc0, 'neg_nan': 0xffc0, 'snan': 0x7f81, 'inf': 0x7f80, 'neg_inf': 0xff80, 'all_nan': 0x7fc0,
                            'flt_max': 0x7f7f},
           torch.float16: {'nan': 0x7e00, 'neg_nan': 0xfe00, 'snan': 0x7c01, 'inf': 0x7c00, 'neg_inf': 0xfc00, 'all_nan': 0x7e00,
                           'flt_max': 0x7bff}}
TILE_EDGES = (2, 4, 8, 16, 32, 64, 128)

AUTO_SIDES = sorted(set(range(1, 9)) | set(STACK_SIDES) | {9, 11, 13, 34, 50, 54, 62, 72, 80, 96, 144, 160, 288, 320, 100, 130})
PATH_SIDES = ([('auto', n) for n in AUTO_SIDES] + [('kron', n) for n in range(1, 9)] + [('stack', n) for n in STACK_SIDES]
              + [('tmem', n) for n in TMEM_SIDES] + [('umma', n) for n in (1, 4, 7, 8, 14, 16, 28, 32, 40, 56, 64, 72, 128)]
              + [('large', n) for n in (80, 96, 160, 256, 320)] + [('simt', n) for n in (7, 14, 33)])

FAMILY = {'kron': 'score_kron_kernel', 'stack': 'score_stack_kernel', 'tmem': 'score_t_kernel', 'umma': 'score_umma_kernel',
          'large': 'score_large_kernel', 'simt': 'score_simt_'}


def family(path, N):
    """Name prefix of the kernel `path` runs on dense N x N maps."""
    if path == 'auto':
        path = ('kron' if N <= 8 else 'stack' if N in STACK_SIDES else 'large' if N in LARGE_SIDES else
                'tmem' if N in (54, 58, 62) else 'umma' if N <= 128 else 'simt')
    return FAMILY[path]


def bits(kind, dtype=torch.float32):
    """The bit pattern of culprit `kind` in `dtype` (float32, bfloat16 or float16) as a signed integer of its width."""
    if dtype == torch.float32:
        return int(np.array([KINDS[kind]], np.uint32).view(np.int32)[0])
    return int(np.array([KINDS16[dtype][kind]], np.uint16).view(np.int16)[0])


def plant(x, b, c, kind, pos):
    """Culprit `kind` into map x[b, c] at position `pos` (0: (0, 0), 1: (H-1, W-1), 2: (0, W-1), 3: the middle)."""
    H, W = x.shape[2:]
    xi = x.view(torch.int32 if x.element_size() == 4 else torch.int16)
    if kind == 'all_nan':
        xi[b, c] = bits(kind, x.dtype)
    else:
        i, j = ((0, 0), (H - 1, W - 1), (0, W - 1), (H // 2, W // 2))[pos]
        xi[b, c, i, j] = bits(kind, x.dtype)


def culprit_maps(B, cc, seed):
    """Flat map indices (b * cc + c) of the culprits of a [B, cc] window: the first and the last map, maps P - 1 and P, a few
    random ones; distinct channels, at most one in eight channels (at least one)."""
    n = B * cc
    rng = np.random.default_rng(seed)
    cand = [0, n - 1] + [m for P in TILE_EDGES for m in (P - 1, P) if m < n] + [int(m) for m in rng.choice(n, min(n, 4), replace=False)]
    chosen, chans = [], set()
    for m in cand:
        if m % cc not in chans and len(chosen) < max(1, cc // 8):
            chosen.append(m)
            chans.add(m % cc)
    return chosen


def launch(lib, path, x, cb, cc, debug):
    """dctp_score_accum (dctp_score_accum_ex for 16-bit x) of x[:, cb:cb + cc] into a zeroed accumulator (and energy_out set to -1
    when `debug`)."""
    B, _, H, W = x.shape
    acc = torch.zeros(cc, dtype=torch.float64, device='cuda')
    en = torch.full((B, cc), -1.0, device='cuda') if debug else None
    stream = _lib.current_stream()
    args = (B, H, W, x.stride(0), x.stride(1), x.stride(2), cb, cc, _lib.ptr(acc), _lib.ptr(en), None, _lib.PATHS[path], stream)
    code = _lib.dtype_code(x.dtype)
    _lib.check(lib.dctp_score_accum(_lib.ptr(x), *args) if code == _lib.DTYPE_F32 else lib.dctp_score_accum_ex(_lib.ptr(x), code, *args))
    _lib.check(lib.dctp_check(stream))
    return acc.cpu().numpy(), (en.cpu().numpy() if debug else None), lib.dctp_last_kernel().decode()


def rel(got, want):
    return np.abs(got - want) / np.maximum(np.abs(want), 1e-30)


def culprit_ok(got, want, kind, may_overflow):
    """Rule 1: non-finite; the largest finite value: within ENERGY_TOL of float64, or non-finite where its energy may overflow."""
    if kind != 'flt_max':
        return not np.isfinite(got)
    return rel(got, want) < ENERGY_TOL if np.isfinite(got) else may_overflow


def check(acc, en, want, bad, kind, tol, label, may_overflow=True):
    """Rules 1 and 2.  want: float64 [B, cc] energies of the maps as scored; bad: [B, cc] culprit mask; may_overflow: False where
    the square of the largest finite value of the input type is far from the fp32 range (fp16), so that culprit must stay finite."""
    bad_ch = bad.any(0)
    chan = want.sum(0)
    for c in np.flatnonzero(bad_ch):
        assert culprit_ok(acc[c], chan[c], kind, may_overflow), 'culprit channel %d scored %r: %s' % (c, acc[c], label)
    ok = ~bad_ch
    assert np.isfinite(acc[ok]).all(), 'non-finite score in clean channels %s: %s' % (np.flatnonzero(ok & ~np.isfinite(acc)), label)
    dead = ok & (chan == 0)
    assert (acc[dead] == 0).all(), 'a dead channel scored %s: %s' % (acc[dead][acc[dead] != 0], label)
    live = ok & (chan > 0)
    err = rel(acc[live], chan[live]).max(initial=0)
    assert err < tol, (err, label)
    if en is None:
        return
    for b, c in zip(*np.nonzero(bad)):
        e = float(en[b, c])
        assert culprit_ok(e, want[b, c], kind, may_overflow), 'culprit map (%d, %d) energy %r: %s' % (b, c, e, label)
    assert np.isfinite(en[~bad]).all(), 'non-finite energy_out of a clean map: %s' % label
    dead = ~bad & (want == 0)
    assert (en[dead] == 0).all(), 'dead maps must score exactly 0: %s' % label
    live = ~bad & (want > 0)
    err = rel(en[live].astype(np.float64), want[live]).max(initial=0)
    assert err < tol, (err, label)


def port_pattern(window):
    """Finite / non-finite per channel of the op-for-op port of the reference hook (CPU, fp32)."""
    st = port.ScoreState()
    port.hook_output(st)(None, None, window)
    return np.isfinite(st.feature_result.numpy())


def culprits_everywhere(lib, path, x, cb, cc, kernel, seed, what, tol=ENERGY_TOL, port_check=False):
    """Every culprit kind at the culprit maps of the window x[:, cb:cb + cc] (fp32, bf16 or fp16), with and without energy_out.
    Returns the kernels that ran."""
    B = x.shape[0]
    names = set()
    win = x[:, cb:cb + cc]
    clean = win.clone()
    picks = culprit_maps(B, cc, seed)
    bad = np.zeros((B, cc), bool)
    for m in picks:
        bad[m // cc, m % cc] = True
    for kind in KINDS:
        for i, m in enumerate(picks):
            plant(win, m // cc, m % cc, kind, i % 4)
        host = win.cpu()
        want = port.energy_parseval64(host.double().numpy())
        for debug in (True, False):
            acc, en, name = launch(lib, path, x, cb, cc, debug)
            names.add(name.split(' (')[0])
            label = '%s %s %s, culprit %s at maps %s%s: %s' % (path, str(x.dtype).split('.')[-1], what, kind, picks,
                                                              ' [energy_out]' if debug else '', name)
            assert name.startswith(kernel), label
            check(acc, en, want, bad, kind, tol, label, may_overflow=x.dtype != torch.float16)
            if port_check and kind != 'flt_max' and not debug:
                np.testing.assert_array_equal(np.isfinite(acc), port_pattern(host.float()), err_msg=label)
        win.copy_(clean)
    return names


def dense_shape(lib, path, N, dtype=torch.float32):
    """(B, C) of a dense call on N x N maps of `dtype`: a ragged last tile, and a whole number of float4 where the TMEM-operand
    kernel needs it.  Maps of 72 x 72 and more: 32 maps (the kernels there take one map, or one 128-row slab of one, per work
    item)."""
    if N >= 72:
        return 2, 16
    mt, _ = geometry(lib, path, N, dtype)
    tmem = path == 'tmem' or (path == 'auto' and family('auto', N) == 'score_t_kernel')
    for B, C in ((3, 139), (3, 140), (3, 141), (2, 139), (2, 140)):
        if (mt == 1 or (B * C) % mt) and not (tmem and N % 2 and (B * C * N * N) % 4):
            return B, C
    raise AssertionError((path, N, mt))


# ---------------------------------------------------------------------------------------------------------- every kernel path
@pytest.mark.parametrize('path,n', PATH_SIDES)
def test_non_finite_map_stays_in_its_channel(lib, cuda_device, path, n):
    B, C = dense_shape(lib, path, n)
    x = maps(B, C, n, n, seed=17 * n + len(path))
    tol = 2 * ENERGY_TOL if n <= 2 else ENERGY_TOL       # (2 x 2 maps: the split-precision residuals do not average out)
    culprits_everywhere(lib, path, x, 0, C, family(path, n), seed=n, what='%dx%dx%dx%d' % (B, C, n, n), tol=tol,
                        port_check=B * C * n * n <= 1 << 16)


def test_umma_generic_loads(lib, cuda_device):
    """The smem-operand kernel's per-map pointer loads: a DenseNet last-12 window on a strided batch, a channel offset that is
    16-byte aligned by luck only, 4- and 8-byte aligned bases (the views of test_gpu_kernels.test_channel_window_and_strides)."""
    big = maps(4, 60, 16, 16, seed=7)
    view = big[1:4, 6:54]
    culprits_everywhere(lib, 'umma', view, view.shape[1] - 12, 12, 'score_umma_kernel', seed=1, what='last 12 of a strided batch')
    odd = maps(2, 9, 14, 14, seed=8)[:, 1:8]
    culprits_everywhere(lib, 'umma', odd, 0, 7, 'score_umma_kernel', seed=2, what='channel offset 1')
    shifted = maps(1, 3, 7, 7, seed=9).flatten()[1:1 + 2 * 49].view(1, 2, 7, 7)
    culprits_everywhere(lib, 'umma', shifted, 0, 2, 'score_umma_kernel', seed=3, what='base 4 mod 16')
    half = maps(1, 3, 8, 8, seed=10).flatten()[2:2 + 2 * 64].view(1, 2, 8, 8)
    culprits_everywhere(lib, 'umma', half, 0, 2, 'score_umma_kernel', seed=4, what='base 8 mod 16')


def test_simt_non_square_and_cropped(lib, cuda_device):
    culprits_everywhere(lib, 'simt', maps(3, 40, 9, 20, seed=11), 0, 40, 'score_simt_', seed=5, what='9x20')
    crop = maps(3, 40, 20, 24, seed=12)[:, :, :, 2:22]
    culprits_everywhere(lib, 'simt', crop, 0, 40, 'score_simt_', seed=6, what='20x20 crops of 20x24 rows')


# ------------------------------------------------------------------------------------------------------ the multi-site entry
def multi_site_culprit(lib, side, k, kinds, dtype=torch.float32):
    """dctp_score_accum_multi (_ex for 16-bit `dtype`) over 16 dense sites with a culprit of each of `kinds` in site k: the culprit
    follows the rules of check() and every other site matches float64 and a clean call per site.  Returns the kernel that ran."""
    n_sites = 16
    code = _lib.dtype_code(dtype)
    shapes = [(1 + i % 3, (9, 16, 11)[i % 3]) for i in range(n_sites)]
    xs = [maps(B, c, side, side, seed=100 * side + i, dtype=dtype) for i, (B, c) in enumerate(shapes)]
    Bk, ck = shapes[k]
    bc = (Bk - 1, ck - 1 - k % 3)
    clean = xs[k].clone()
    for kind in kinds:
        xs[k].copy_(clean)
        plant(xs[k], bc[0], bc[1], kind, k % 4)
        accs = [torch.zeros(c, dtype=torch.float64, device='cuda') for _, c in shapes]
        sites = (_lib.Site * n_sites)()
        for i, (B, c) in enumerate(shapes):
            sites[i].B, sites[i].c_count = B, c
            sites[i].x, sites[i].accum = xs[i].data_ptr(), accs[i].data_ptr()
        stream = _lib.current_stream()
        _lib.check(lib.dctp_prepare(side, side))
        if code == _lib.DTYPE_F32:
            _lib.check(lib.dctp_score_accum_multi(sites, n_sites, side, side, stream))
        else:
            _lib.check(lib.dctp_score_accum_multi_ex(sites, n_sites, side, side, code, stream))
        _lib.check(lib.dctp_check(stream))
        name = lib.dctp_last_kernel().decode()
        assert name.startswith(family('auto', side)), name
        for i, (B, c) in enumerate(shapes):
            want = port.energy_parseval64(xs[i].double().cpu().numpy())
            bad = np.zeros((B, c), bool)
            if i == k:
                bad[bc] = True
            check(accs[i].cpu().numpy(), None, want, bad, kind, ENERGY_TOL, 'site %d of 16, side %d, %s culprit %s in site %d: %s'
                  % (i, side, str(dtype).split('.')[-1], kind, k, name), may_overflow=dtype != torch.float16)
            if i != k:
                ref = torch.zeros(c, dtype=torch.float64, device='cuda')
                args = (B, side, side, c * side * side, side * side, side, 0, c, _lib.ptr(ref), None, None, _lib.PATH_AUTO, stream)
                _lib.check(lib.dctp_score_accum(xs[i].data_ptr(), *args) if code == _lib.DTYPE_F32
                           else lib.dctp_score_accum_ex(xs[i].data_ptr(), code, *args))
                np.testing.assert_allclose(accs[i].cpu().numpy(), ref.cpu().numpy(), rtol=1e-12, err_msg='site %d' % i)
        _lib.check(lib.dctp_check(stream))
    return name


@pytest.mark.parametrize('k', [0, 7, 15])
@pytest.mark.parametrize('side', [7, 14, 28, 56, 160])
def test_multi_site_culprit_stays_in_its_site(lib, cuda_device, side, k):
    """dctp_score_accum_multi over 16 dense sites with a culprit in site k: every other site matches float64 and a clean call
    per site (tiles and work items never span two sites)."""
    multi_site_culprit(lib, side, k, ('nan', 'neg_inf'))


# ---------------------------------------------------------------------------------------------------------------- density
@pytest.mark.parametrize('every', [1, 2])
@pytest.mark.parametrize('shape', [(64, 512, 28, 28), (64, 1024, 14, 14), (4, 64, 320, 320)])
def test_every_map_or_every_other_map_non_finite(lib, cuda_device, shape, every):
    """Every map (every = 1) or every other map (every = 2: the odd channels) holds one NaN, at a place that moves from map to
    map.  The call returns with dctp_check clean, in the production and the debug instantiation."""
    B, C, H, W = shape
    x = maps(B, C, H, W, seed=sum(shape) + every)
    flat = x.view(B * C, H * W)
    m = torch.arange(every - 1, B * C, every, device='cuda')
    flat[m, (m * 7919) % (H * W)] = float('nan')
    bad = np.zeros((B, C), bool)
    bad.reshape(-1)[m.cpu().numpy()] = True
    want = port.energy_parseval64(x.cpu().numpy())
    for debug in (True, False):
        acc, en, name = launch(lib, 'auto', x, 0, C, debug)
        assert name.startswith(family('auto', H)), name
        check(acc, en, want, bad, 'nan', ENERGY_TOL, '%s, every %d maps non-finite%s: %s' % (shape, every, ' [energy_out]' if debug else '', name))


# ---------------------------------------------------------------------------------------------------------------------- dct3
@pytest.mark.parametrize('window', [False, True])
@pytest.mark.parametrize('shape', [(3, 64, 14, 14), (2, 24, 32, 32), (2, 12, 56, 56)])
def test_dct3_culprit_image(lib, cuda_device, shape, window):
    """One value per image: non-finite exactly for the image with a non-finite map inside the channel window; a non-finite map
    outside the window changes nothing.  With the window (an odd channel count) the culprit is the first scored map of the last
    image, so the tile that holds it also holds maps of the image before."""
    from dct_pruning_b200.ops import score_op
    from oracle import alt_ops_port as ao
    B, C, H, W = shape
    cb, cc = (C // 4, C // 2 - 1) if window else (0, C)
    for kind in ('nan', 'inf'):
        x = maps(B, C, H, W, seed=sum(shape) + window)
        plant(x, B - 1, cb if window else cb + cc - 2, kind, 3)
        if window:
            plant(x, 0, cb + cc, kind, 0)                     # outside the window
        acc, values = score_op(x, 'dct3', c_begin=cb, c_count=cc, want_values=True)
        _lib.check(_lib.load().dctp_check(_lib.current_stream()))
        v = values.cpu().numpy().astype(np.float64)
        assert not np.isfinite(v[B - 1]) and not np.isfinite(float(acc[0])), (shape, window, kind, v)
        want = ao.dct3_energy64(x.cpu().numpy()[:B - 1, cb:cb + cc])
        assert np.isfinite(v[:B - 1]).all(), (shape, window, kind, v)
        np.testing.assert_allclose(v[:B - 1], want, rtol=1e-4)


# -------------------------------------------------------------------------------------------------------------- end to end
def test_resnet56_nan_in_last_site(lib, cuda_device):
    """ScoreSession over ResNet-56 (batch 16, 32 x 32, small sites held and scored in multi-site launches).  A hook registered
    before the session's sets one element of one (image, channel) of the last hooked site's output to NaN; nothing scored later
    sees it.  That file has exactly one non-finite entry, every other score equals a clean run, and top-k keeps the NaN channel
    with the rest of its selection unchanged.  (imp_conv55 is a block output, which ResNet-56's loader never prunes, so its
    selection is taken with the device top-k the loader uses, at the k a 0.18 rate gives.)"""
    from dct_pruning_b200.generate import synthetic_batches
    from dct_pruning_b200.hooks import ScoreSession
    from dct_pruning_b200.sites import resolve_module
    from dct_pruning_b200.topk import kept_channels, select_index
    from dct_pruning_b200.zoo import get_network
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    torch.manual_seed(0)
    net = get_network('resnet_56').to(cuda_device).eval()
    x = next(iter(synthetic_batches(16, 32, 1)))[0].to(cuda_device)
    image, channel = 5, 37

    def poison(module, inputs, output):
        output[image, channel, 3, 4] = float('nan')

    runs = {}
    for mode in ('clean', 'nan'):
        session = ScoreSession(net, 'resnet_56')
        last = session.sites[-1]
        handle = resolve_module(net, last.module).register_forward_hook(poison) if mode == 'nan' else None
        with session, torch.no_grad():
            net(x)
        if handle is not None:
            handle.remove()
        runs[mode] = session.finalize()
    stem = last.files[0].stem
    clean, bad = runs['clean'], runs['nan']
    assert sorted(clean) == sorted(bad)
    for s in clean:
        c, g = clean[s], bad[s].copy()
        if s == stem:
            assert np.flatnonzero(~np.isfinite(g)).tolist() == [channel], (s, g)
            g[channel], c = 0.0, c.copy()
            c[channel] = 0.0
        assert np.isfinite(g).all(), s
        np.testing.assert_allclose(g, c, rtol=1e-6, atol=0, err_msg=s)
        assert ((g == 0) == (c == 0)).all(), s
    k = int(clean[stem].size * (1 - 0.18))
    kept = select_index(bad[stem], k, device=cuda_device)
    assert channel in kept
    forced = clean[stem].astype(np.float64)
    forced[channel] = np.inf                              # NaN ranks above every score
    np.testing.assert_array_equal(kept, port.select_index_stable(forced, k))
    rate = '[0.]+[0.18]*29'
    for (sel, a), (_, b) in zip(kept_channels('resnet_56', rate, clean, device=cuda_device),
                                kept_channels('resnet_56', rate, bad, device=cuda_device)):
        np.testing.assert_array_equal(a, b, err_msg=sel.stem)
