"""bf16 / fp16 input under the rules of the fp32 guard-band and non-finite suites (test_gpu_bounds.py, test_gpu_nonfinite.py),
through their helpers: dctp_score_accum_ex and dctp_score_accum_multi_ex.

The stacked-basis (K1s, even sides 10..64) and Kronecker (K1k, sides 1..8) kernels read 16-bit maps themselves.  They view a
stream as rows of 32 elements (64 bytes in 16-bit); a segment whose element count is not a multiple of 32 has its last tile read
element by element from global memory, with bounds checks of their own.  In 16-bit, K1k's row layout (sides 4 and 8) has a TMA box
wider than a map row, and sides 2 and 6 take the flat layout (side 6: 128 maps per tile, not 256).  Every other route widens the
scored window into a dense fp32 copy (widen_window_kernel, which follows the caller's strides) and runs the fp32 kernels on it.

  A  native kernels   every native side, forced and through AUTO, debug (energy_out, coeff_out) and production instantiations:
                      one map, one tile, ragged last tiles (the stream ending on a 32-element row, inside one, and half-way
                      through one), and enough tiles that every CTA's mbarrier ring wraps more than twice; inputs in a 16-bit NaN
                      arena, outputs between -0.0 guards (test_gpu_bounds.score).  Oracles: float64 Parseval, exact zeros for dead
                      maps and channels, scipy's dctn for the coefficients of small cases.
  B  widened windows  channel windows, a batch stride that skips images, bases at every 2-byte offset mod 16, cropped and
                      non-square maps: float64, and bit-identical to the fp32 entry on the window widened on the host.  Forced
                      native paths refuse a base that is not 16-byte aligned, and launch nothing.
  C  multi-site       every native side and one widened side; segments that end inside a 32-element row, empty and 2-byte
                      misaligned sites, two sites sharing an accumulator: guards, float64, one call per site, launch counts.
  D  non-finite maps  the culprit matrix of test_gpu_nonfinite.py with bf16 / fp16 bit patterns (KINDS16), inputs in a NaN arena
                      whose guards are larger than the stream.  The fp16 maximum (65504) squares far inside the fp32 range, so a
                      map holding it must score finite and within ENERGY_TOL; bf16's maximum may overflow the fp32 energy.
  E  session          a ScoreSession whose sites of one map side fire in bf16 and fp32 in one forward: one multi-site launch per
                      dtype, and every site equal to a call per activation.
The last test checks that the module launched every 16-bit instantiation of K1s and K1k.
"""
import math

import numpy as np
import pytest
import torch

from dct_pruning_b200 import _lib
from test_gpu_bounds import GUARD, NEG0, Arena, acc_err, geometry, map_counts, maps, rel_err, score, site_plan
from test_gpu_kernels import ENERGY_TOL, STACK_SIDES
from test_gpu_nonfinite import KINDS16, culprits_everywhere, dense_shape, family, multi_site_culprit

pytestmark = pytest.mark.gpu

DTYPES = {'bf16': torch.bfloat16, 'fp16': torch.float16}
NATIVE_SIDES = list(range(1, 9)) + STACK_SIDES
SEEN = set()                         # kernel instantiations the score launches of this module ran


def seen(name):
    name = name.split(' (')[0]
    SEEN.add(name)
    return name


def native(n):
    return 'kron' if n <= 8 else 'stack'


def in_tag(dtype):
    return 'IN=' + ('bf16' if dtype == torch.bfloat16 else 'f16')


# ---------------------------------------------------------------------------------------------------- A: the native kernels
@pytest.mark.parametrize('how', ['forced', 'auto'])
@pytest.mark.parametrize('n', NATIVE_SIDES)
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_native_kernels_stay_inside_their_buffers(lib, cuda_device, dt, n, how):
    dtype = DTYPES[dt]
    path = native(n) if how == 'forced' else 'auto'
    mt, wrap = geometry(lib, native(n), n, dtype)
    counts = map_counts(native(n), n, mt, wrap)
    # 16 elements are 32 bytes: a tail rule taken in bytes rather than elements would miss this stream's last row
    half = next((m for m in range(mt + 1, 65 * mt) if m % mt and (m * n * n) % 32 == 16), None)
    if half:
        counts['ragged last tile, stream ends half-way through a 32-element row'] = half
    for i, (what, count) in enumerate(counts.items()):
        B = 3 if count % 3 == 0 and count >= 6 else 2 if count % 2 == 0 and count >= 4 else 1
        tol = 2 * ENERGY_TOL if count >= 100000 or n <= 2 else ENERGY_TOL        # (as in test_gpu_bounds.py)
        for debug in (True, False):
            name = score(lib, path, B, count // B, n, n, x_off=(0, 16, 64)[i % 3], acc_off=(0, 8, 64)[i % 3], debug=debug,
                         seed=1000 * n + 10 * i + debug, tol=tol, what=what, dtype=dtype)
            assert name.startswith(family(native(n), n)) and in_tag(dtype) in name, (path, n, what, name)
            assert n <= 8 or ('cfg6' if debug else 'cfg7') in name, name
            seen(name)


# ------------------------------------------------------------------------------------------ B: widened windows and refusals
def widened(lib, path, B, C, H, W, *, dtype, debug, **kw):
    """score() of a 16-bit window that no native kernel takes, then the fp32 entry with the same path on that window widened on the
    host: the same kernel, bit-identical accum (both start at 0.5), energy_out and coeff_out."""
    got = {}
    name = score(lib, path, B, C, H, W, dtype=dtype, debug=debug, out=got, **kw)
    src, acc, en, co = got['src'], got['acc'], got['en'], got['co']
    assert 'IN=' not in name, name
    ref_in = src.float().contiguous()
    cc = ref_in.shape[1]
    acc32 = torch.full((cc,), 0.5, dtype=torch.float64, device='cuda')
    en32 = torch.full((B, cc), float('nan'), device='cuda') if debug else None
    co32 = torch.full((B, cc, H, W), float('nan'), device='cuda') if debug else None
    stream = _lib.current_stream()
    _lib.check(lib.dctp_score_accum(_lib.ptr(ref_in), B, H, W, ref_in.stride(0), ref_in.stride(1), ref_in.stride(2), 0, cc,
                                    _lib.ptr(acc32), _lib.ptr(en32), _lib.ptr(co32), _lib.PATHS[path], stream))
    _lib.check(lib.dctp_check(stream))
    label = '%s %s %dx%dx%dx%d %s: %s' % (path, dtype, B, C, H, W, kw.get('what', ''), name)
    assert lib.dctp_last_kernel().decode().split(' (')[0] == name, label
    assert torch.equal(acc, acc32), label
    if debug:
        assert torch.equal(en.view(B, cc), en32), label
        assert torch.equal(co.view(B, cc, H, W), co32), label
    seen(name)


@pytest.mark.parametrize('n', [7, 14, 32, 96])
@pytest.mark.parametrize('path', ['auto', 'umma', 'simt'])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_widened_windows_read_nothing_outside(lib, cuda_device, dt, path, n):
    """Windows the widening kernel copies through the caller's strides; everything the call does not score is NaN."""
    dtype = DTYPES[dt]
    for debug in (True, False):
        kw = dict(dtype=dtype, debug=debug)
        widened(lib, path, 3, 48, n, n, c_begin=36, c_count=12, seed=n + debug, what='last 12 channels', **kw)
        widened(lib, path, 2, 40, n, n, c_begin=10, c_count=17, x_off=16, seed=2 * n + debug, what='middle window', **kw)
        widened(lib, path, 3, 9, n, n, batch_step=2, x_off=64, seed=3 * n + debug, what='every other image', **kw)
        for off in (2, 4, 6, 8, 10, 12, 14):
            widened(lib, path, 2, 5, n, n, x_off=off, acc_off=8, seed=4 * n + off + debug, what='base %d mod 16' % off, **kw)


@pytest.mark.parametrize('path', ['auto', 'simt'])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_widened_cropped_and_non_square_maps(lib, cuda_device, dt, path):
    dtype = DTYPES[dt]
    for debug in (True, False):
        kw = dict(dtype=dtype, debug=debug)
        widened(lib, path, 2, 3, 20, 20, row=24, seed=20 + debug, what='20x20 crops of 20x24 rows', **kw)
        widened(lib, path, 2, 3, 20, 20, row=24, x_off=6, seed=22 + debug, what='20x20 crops, base 6 mod 16', **kw)
        widened(lib, path, 3, 5, 12, 20, seed=24 + debug, what='non-square', **kw)
        widened(lib, path, 2, 4, 9, 33, row=40, x_off=10, seed=26 + debug, what='9x33 crops of 9x40 rows, base 10 mod 16', **kw)


def refused(lib, path, n, dtype, off):
    """A forced path on dense n x n maps of `dtype` at a base `off` bytes past a 128-byte boundary: DCTP_E_UNSUPPORTED, an error
    text that names the alignment, nothing launched and the accumulator untouched."""
    B, C = 2, 3
    xa = Arena([B * C * n * n], dtype, [off])
    xa.live.copy_(maps(B, C, n, n, seed=off, dtype=dtype).reshape(-1))
    acc = Arena([C], torch.float64, [8], edge=NEG0, live=0.5)
    before = lib.dctp_launch_count()
    rc = lib.dctp_score_accum_ex(_lib.ptr(xa.live), _lib.dtype_code(dtype), B, n, n, C * n * n, n * n, n, 0, C, _lib.ptr(acc.live),
                                 None, None, _lib.PATHS[path], _lib.current_stream())
    label = '%s %s %dx%d, base %d mod 16' % (path, dtype, n, n, off)
    assert rc == _lib.E_UNSUPPORTED, (rc, label)
    assert '16-B aligned' in lib.dctp_last_error().decode(), (lib.dctp_last_error(), label)
    assert lib.dctp_launch_count() == before, label
    _lib.check(lib.dctp_check(_lib.current_stream()))
    assert acc.guards_intact() and bool((acc.live == 0.5).all()), label


@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_forced_native_paths_refuse_unaligned_bases(lib, cuda_device, dt):
    """The Kronecker and stacked-basis kernels read through a TMA descriptor, which needs a 16-byte aligned base: a 16-bit base
    at 2..14 mod 16 is refused rather than encoded (AUTO widens it: test_widened_windows_read_nothing_outside)."""
    for n in NATIVE_SIDES:
        for off in (2, 4, 6, 8, 10, 12, 14):
            refused(lib, native(n), n, DTYPES[dt], off)


@pytest.mark.parametrize('path,n', [('tmem', 56), ('large', 96)])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_widened_dense_maps_on_forced_fp32_kernels(lib, cuda_device, dt, path, n):
    """The TMEM-operand and large-map kernels take dense 16-byte aligned streams only: 16-bit ones are widened and scored there;
    an unaligned base is refused."""
    dtype = DTYPES[dt]
    for debug in (True, False):
        kw = dict(dtype=dtype, debug=debug)
        for i, off in enumerate((0, 16, 64)):
            widened(lib, path, 2, 3 + i, n, n, x_off=off, acc_off=8 * i, seed=n + i + debug, what='dense, base %d mod 128' % off, **kw)
        widened(lib, path, 1, 40, n, n, c_begin=10, c_count=17, x_off=16, seed=n + 5 + debug, what='channel window of one image', **kw)
    for off in (2, 8, 14):
        refused(lib, path, n, dtype, off)


# -------------------------------------------------------------------------------------------------- C: the multi-site entry
@pytest.mark.parametrize('n_sites', [1, 15, 16, 17, 33, 40])
@pytest.mark.parametrize('side', NATIVE_SIDES + [9])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_multi_site_entry(lib, cuda_device, dt, side, n_sites):
    """dctp_score_accum_multi_ex against float64 and one dctp_score_accum_ex per site, the plan of test_gpu_bounds.site_plan
    with 2-byte misaligned sites; channel counts are bumped until the segment ends inside a 32-element row (where B * N * N is not
    a multiple of 32 itself)."""
    dtype = DTYPES[dt]
    NN = side * side
    plan = site_plan(n_sites)
    for p in plan:
        while p[0] * p[1] > 0 and (p[0] * NN) % 32 and (p[0] * p[1] * NN) % 32 == 0:
            p[1] += 1
    slot = list(range(n_sites))
    if n_sites >= 15:
        plan[2][1] = plan[1][1]
        slot[2] = 1
    nmaps = [B * c for B, c, _ in plan]
    unaligned = [i for i in range(n_sites) if plan[i][2] == 'unaligned']
    offs = [(2, 6, 10)[unaligned.index(i) % 3] if i in unaligned else (0, 16, 64)[i % 3] for i in range(n_sites)]
    xa = Arena([m * NN for m in nmaps], dtype, offs, guard=max(GUARD, 4 * NN * 4))
    acc = Arena([c for _, c, _ in plan], torch.float64, [(0, 8, 64)[i % 3] for i in range(n_sites)], edge=NEG0, live=0.5)
    live = [i for i in range(n_sites) if nmaps[i] > 0]
    src = {i: maps(plan[i][0], plan[i][1], side, side, seed=100 * side + i, dtype=dtype) for i in live}
    sites = (_lib.Site * n_sites)()
    for i, (B, c, _) in enumerate(plan):
        sites[i].B, sites[i].c_count = B, c
        sites[i].x = xa.views[i].data_ptr() if i in src else None
        sites[i].accum = acc.views[slot[i]].data_ptr() if i in src else None
    code = _lib.dtype_code(dtype)
    _lib.check(lib.dctp_prepare(side, side))
    stream = _lib.current_stream()
    before = lib.dctp_launch_count()
    for i in live:
        xa.views[i].copy_(src[i].reshape(-1))
    _lib.check(lib.dctp_score_accum_multi_ex(sites, n_sites, side, side, code, stream))
    launches = lib.dctp_launch_count() - before
    _lib.check(lib.dctp_check(stream))
    name = lib.dctp_last_kernel().decode()

    aligned = [i for i in live if plan[i][2] == 'dense']
    # native sides: one launch per 16 aligned sites, and widen + fp32 kernel for each unaligned one; side 9: widen + fp32 kernel per site
    want_launches = -(-len(aligned) // 16) + 2 * (len(live) - len(aligned)) if side != 9 else 2 * len(live)
    assert launches == want_launches, (launches, want_launches, name)
    assert acc.guards_intact(), 'accumulator guard written'
    energy = [torch.zeros(c, dtype=torch.float64, device='cuda') for _, c, _ in plan]
    images = [0] * n_sites                      # maps each channel of an accumulator receives
    for i in live:
        energy[slot[i]] += (src[i].double() ** 2).sum((2, 3)).sum(0)
        images[slot[i]] += plan[i][0]
    for j, e in enumerate(energy):
        got = acc.views[j]
        assert not bool(torch.isnan(got).any()), ('NaN in the accumulator of site', j, name)
        assert bool((got[e == 0] == 0.5).all()), ('a dead channel (or an unused accumulator) changed', j, name)
        assert acc_err(got[e > 0], e[e > 0], images[j]) < ENERGY_TOL, (j, name)

    ref = [torch.full((c,), 0.5, dtype=torch.float64, device='cuda') for _, c, _ in plan]
    for i in live:
        B, c, _ = plan[i]
        _lib.check(lib.dctp_score_accum_ex(_lib.ptr(xa.views[i]), code, B, side, side, c * NN, NN, side, 0, c, _lib.ptr(ref[slot[i]]),
                                           None, None, _lib.PATH_AUTO, stream))
        name = seen(lib.dctp_last_kernel().decode())
        assert (in_tag(dtype) in name) == (side != 9 and i in aligned), (i, name)
    _lib.check(lib.dctp_check(stream))
    for j in range(n_sites):
        np.testing.assert_allclose(acc.views[j].cpu().numpy(), ref[j].cpu().numpy(), rtol=1e-10, err_msg='site %d' % j)


# ------------------------------------------------------------------------------------------------------ D: non-finite maps
def guarded(x):
    """x copied into a NaN arena whose guards are larger than x (a read of the stream at twice its element size stays inside)."""
    xa = Arena([x.numel()], x.dtype, [0], guard=max(GUARD, 2 * x.numel() * x.element_size() + 4096))
    xa.live.copy_(x.reshape(-1))
    return xa.live.view(x.shape)


@pytest.mark.parametrize('how', ['forced', 'auto'])
@pytest.mark.parametrize('n', NATIVE_SIDES)
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_non_finite_map_stays_in_its_channel(lib, cuda_device, dt, n, how):
    """Culprits at the first and last map (the last in a tile read from global memory wherever N * N is not a multiple of 32), at
    maps P - 1 and P for P = 2..128, at seeded random maps, at four places in their maps; both instantiations."""
    dtype = DTYPES[dt]
    path = native(n) if how == 'forced' else 'auto'
    B, C = dense_shape(lib, native(n), n, dtype)
    x = guarded(maps(B, C, n, n, seed=17 * n + len(how), dtype=dtype))
    tol = 2 * ENERGY_TOL if n <= 2 else ENERGY_TOL
    names = culprits_everywhere(lib, path, x, 0, C, family(native(n), n), seed=n, what='%dx%dx%dx%d' % (B, C, n, n), tol=tol,
                                port_check=B * C * n * n <= 1 << 16)
    assert all(in_tag(dtype) in s for s in names), names
    SEEN.update(names)


@pytest.mark.parametrize('k', [0, 7, 15])
@pytest.mark.parametrize('side', [14, 28, 56])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_multi_site_culprit_stays_in_its_site(lib, cuda_device, dt, side, k):
    dtype = DTYPES[dt]
    name = multi_site_culprit(lib, side, k, list(KINDS16[dtype]), dtype)
    assert in_tag(dtype) in name, name
    seen(name)


@pytest.mark.parametrize('case', ['9x9', '80x80', 'channel window 28'])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_non_finite_map_on_widened_routes(lib, cuda_device, dt, case):
    dtype = DTYPES[dt]
    if case == 'channel window 28':
        B, C, n, cb, cc = 3, 60, 28, 20, 33
    else:
        n = int(case.split('x')[0])
        (B, C), cb = dense_shape(lib, 'auto', n, dtype), 0
        cc = C
    x = guarded(maps(B, C, n, n, seed=n + C, dtype=dtype))
    names = culprits_everywhere(lib, 'auto', x, cb, cc, family('auto', n), seed=n, what='%s (%dx%dx%dx%d)' % (case, B, C, n, n))
    assert not any('IN=' in s for s in names), names


# ---------------------------------------------------------------------------------------------- E: a session of mixed dtypes
class MixedDtypes(torch.nn.Module):
    """Four hook sites of 14 x 14 maps (8, 16, 24, 32 channels); the first and third fire in bf16 (autocast), the others in fp32."""

    def __init__(self):
        super().__init__()
        self.c1, self.c2 = torch.nn.Conv2d(3, 8, 3, padding=1), torch.nn.Conv2d(8, 16, 3, padding=1)
        self.c3, self.c4 = torch.nn.Conv2d(16, 24, 3, padding=1), torch.nn.Conv2d(24, 32, 3, padding=1)
        self.r1, self.r2, self.r3, self.r4 = (torch.nn.ReLU() for _ in range(4))

    def forward(self, x):
        with torch.autocast('cuda', dtype=torch.bfloat16):
            x = self.r1(self.c1(x))
        x = self.r2(self.c2(x.float()))
        with torch.autocast('cuda', dtype=torch.bfloat16):
            x = self.r3(self.c3(x))
        return self.r4(self.c4(x.float()))


def test_session_launches_one_group_per_dtype(lib, cuda_device):
    """Two forwards (the first takes every site's full path, the second the geometry it remembered): the held sites of each
    forward are scored in one multi-site launch per dtype, and every site equals one dctp_score_accum_ex per activation."""
    from dct_pruning_b200.hooks import ScoreSession
    from dct_pruning_b200.sites import ScoreFile, Site, VARIANT_OUTPUT
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(0)
    net = MixedDtypes().to(cuda_device).eval()
    names = ['r1', 'r2', 'r3', 'r4']
    session = ScoreSession(net, 'mixed', sites=[Site(m, VARIANT_OUTPUT, (ScoreFile(m),)) for m in names])
    acts = {m: [] for m in names}
    taps = [getattr(net, m).register_forward_hook(lambda mod, i, out, m=m: acts[m].append(out.detach().clone())) for m in names]
    g = torch.Generator().manual_seed(1)
    per_forward = []
    with session, torch.no_grad():
        for _ in range(2):
            x = torch.randn(4, 3, 14, 14, generator=g).to(cuda_device)
            l0, n0 = session.launches, lib.dctp_launch_count()
            net(x)
            per_forward.append((session.launches - l0, lib.dctp_launch_count() - n0, seen(lib.dctp_last_kernel().decode())))
    for t in taps:
        t.remove()
    assert [acts[m][0].dtype for m in names] == [torch.bfloat16, torch.float32, torch.bfloat16, torch.float32]
    assert all(p[:2] == (2, 2) for p in per_forward), per_forward
    stream = _lib.current_stream()
    for idx, m in enumerate(names):
        off, c = session.slots[idx]
        ref = torch.zeros(c, dtype=torch.float64, device=cuda_device)
        for a in acts[m]:
            B, C, H, W = a.shape
            _lib.check(lib.dctp_score_accum_ex(_lib.ptr(a), _lib.dtype_code(a.dtype), B, H, W, a.stride(0), a.stride(1), a.stride(2), 0,
                                               C, _lib.ptr(ref), None, None, _lib.PATH_AUTO, stream))
            seen(lib.dctp_last_kernel().decode())
        _lib.check(lib.dctp_check(stream))
        got = session.flat[off:off + c]
        torch.testing.assert_close(got, ref, rtol=1e-12, atol=0, msg=m)
        want = sum((a.double() ** 2).sum((2, 3)).sum(0) for a in acts[m])
        assert bool((got[want == 0] == 0).all()), m
        assert rel_err(got[want > 0], want[want > 0]) < ENERGY_TOL, m


# ---------------------------------------------------------------------------------------------------- instantiation coverage
REQUIRED = (['score_stack_kernel<KP=%d,VEC=%d,cfg%d,IN=%s>' % (kp, vec, cfg, t)
             for t in ('bf16', 'f16') for kp, vec in ((16, 2), (16, 4), (32, 2), (32, 4), (48, 4), (64, 4)) for cfg in (6, 7)]
            + ['score_kron_kernel<K2=%d,%s,IN=%s>' % (k2, lay, t)
               for t in ('bf16', 'f16') for k2, lay in ((16, 'even'), (64, 'even'), (16, 'odd'), (32, 'odd'), (48, 'odd'), (64, 'odd'))])


def test_every_16bit_instantiation_was_launched(request, cuda_device):
    """Last test of the module: the cases above ran every 16-bit instantiation of the stacked-basis and Kronecker kernels."""
    if request.config.getoption('keyword') or any('::' in a for a in request.config.args):
        pytest.skip('only part of the module ran')
    missing = [k for k in REQUIRED if k not in SEEN]
    assert not missing, 'never launched: %s (launched: %s)' % (', '.join(missing), ', '.join(sorted(SEEN)))
