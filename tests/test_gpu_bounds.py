"""Guard-band tests: every kernel stays inside the buffers it is given, and reads its input only after the kernel before it on
the stream has written it.

Every buffer the library reads or writes here is a view inside a larger allocation, with a guard on each side of at least 256 KiB
and at least four maps (more than any kernel's tile, TMA box or map slab), at a chosen byte offset (0, 16 or 64 mod 128; 4, 8 or 12
mod 16 for the unaligned fallbacks):

  inputs         the whole allocation - guards, channels outside the scored window, images a batch stride skips, columns a
                 cropped row skips - is NaN.  The scored maps are copied in from a prepared tensor on the current stream directly
                 before the launch, with no host synchronisation in between.  A read of memory the caller did not hand over, or a
                 read before the copy has landed, turns a score NaN.
  accum (fp64)   guards hold -0.0 and are compared bitwise: a store, or an atomic add of +0.0, turns -0.0 into +0.0.  Live entries
                 start at 0.5, so a store where an add was meant shows, and a dead channel must read exactly 0.5.
  energy_out, coeff_out (fp32)   guards -0.0, compared bitwise; the live region starts as NaN, so every element must be written.

Oracle: float64 sums of squares (Parseval) per map and per channel, scipy's dctn for the coefficients of small cases, exactly 0
for dead maps (all +0.0 or all -0.0).  NaN never sits inside the caller's tensors here; what a non-finite map does to its own and
to the other channels is pinned by test_gpu_nonfinite.py.

The module records which kernel instantiation every score launch ran (dctp_last_kernel); its last test checks that the cases
reached each one in REQUIRED.  bf16 / fp16 input (dctp_score_accum_ex, dctp_score_accum_multi_ex) is held to the same rules by
test_gpu_half_bounds.py, through the helpers here (Arena, maps, score, geometry, map_counts take a dtype).
"""
import math

import numpy as np
import pytest
import torch

from dct_pruning_b200 import _lib
from test_gpu_kernels import ENERGY_TOL, STACK_SIDES, TMEM_SIDES

pytestmark = pytest.mark.gpu

COEFF_TOL = 2e-5                     # coefficients vs scipy, relative to the largest coefficient (as in test_gpu_kernels.py)
GUARD = 256 << 10                    # bytes on each side of every view, at the least
NEG0 = 'neg0'                        # edge value: -0.0, written and compared as a bit pattern
_INT = {torch.float32: (torch.int32, -2 ** 31), torch.float64: (torch.int64, -2 ** 63), torch.bfloat16: (torch.int16, -2 ** 15),
        torch.float16: (torch.int16, -2 ** 15)}

LARGE_SIDES = list(range(80, 321, 16))
AUTO_ELSEWHERE = [9, 11, 13, 34, 50, 54, 62, 72, 100, 130]     # sides AUTO sends to neither the Kronecker nor the stacked-basis kernel
SIDES = sorted(set(range(1, 9)) | set(STACK_SIDES) | set(TMEM_SIDES) | set(LARGE_SIDES) | set(AUTO_ELSEWHERE)
               | {29})                                        # 29: the odd-side dense load of the smem-operand kernel without prefetch


class Arena:
    """Views of sizes[i] elements of `dtype` inside ONE allocation.  View i starts `guard` bytes plus offs[i] (mod 128) after the
    end of view i - 1 (or the start of the allocation); `guard` bytes follow the last one.  Everything outside the views holds
    `edge` (NEG0: -0.0 bit patterns), the views `live` (or `edge` when None)."""

    def __init__(self, sizes, dtype, offs=None, edge=float('nan'), live=None, guard=GUARD):
        es = torch.empty(0, dtype=dtype).element_size()
        offs = offs or [0] * len(sizes)
        guard = -(-guard // 128) * 128
        starts, cur = [], 0
        for n, off in zip(sizes, offs):
            assert off % es == 0 and 0 <= off < 128
            cur = -(-cur // 128) * 128 + guard + off
            starts.append(cur // es)
            cur += n * es
        total = (-(-cur // 128) * 128 + guard) // es
        self.dtype, self.edge = dtype, edge
        self.buf = torch.empty(total, dtype=dtype, device='cuda')
        if edge == NEG0:
            itype, bits = _INT[dtype]
            self.buf.view(itype).fill_(bits)
        else:
            self.buf.fill_(edge)
        self.mask = torch.zeros(total, dtype=torch.bool, device='cuda')
        self.views = []
        for s, n in zip(starts, sizes):
            self.mask[s:s + n] = True
            self.views.append(self.buf[s:s + n])
            if live is not None:
                self.views[-1].fill_(live)
        self.live = self.views[0]

    def guards_intact(self):
        outside = self.buf[~self.mask]
        if self.edge == NEG0:
            itype, bits = _INT[self.dtype]
            return bool((outside.view(itype) == bits).all())
        if isinstance(self.edge, float) and math.isnan(self.edge):
            return bool(torch.isnan(outside).all())
        return bool((outside == self.edge).all())


SEEN = set()                         # kernel instantiations the score launches of this module ran


def note(lib):
    name = lib.dctp_last_kernel().decode().split(' (')[0]
    SEEN.add(name)
    return name


def maps(B, C, H, W, seed, dtype=torch.float32):
    """relu(N(0, 1)) maps on the device, rounded to `dtype`.  Channels c % 7 == 1 are all +0.0 and c % 7 == 4 all -0.0 in every
    image (dead channels); image 1 of channel 2 is a dead map of a live channel."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.relu(torch.randn(B, C, H, W, generator=g, device='cuda')).to(dtype)
    x[:, 1::7] = 0.0
    x[:, 4::7] = -0.0
    if B > 1 and C > 2:
        x[1, 2] = 0.0
    return x


def rel_err(got, want):
    if got.numel() == 0:
        return 0.0
    return float(((got.double() - want).abs() / want.abs().clamp_min(1e-30)).max())


SHARES = 8                           # fp64 adds one map makes into its channel's accumulator, at the most (score kernels: 1 to 5)


def acc_err(acc, want, maps_per_channel):
    """rel_err of acc - 0.5 against `want`, for accumulators that started at 0.5, less the rounding that start costs: the sum is
    held at 0.5 and above, so each of the SHARES * maps_per_channel fp64 adds (and the subtraction of 0.5) may round by half an
    ulp of the final value.  (That is 5.6e-17 absolute: more than ENERGY_TOL of a channel whose only live map is a value near 1e-6.)"""
    if acc.numel() == 0:
        return 0.0
    got = acc.double()
    ulp = torch.nextafter(got, torch.full_like(got, math.inf)) - got
    diff = ((got - 0.5 - want).abs() - (SHARES * maps_per_channel + 1) * 0.5 * ulp).clamp_min(0)
    return float((diff / want.abs().clamp_min(1e-30)).max())


def score(lib, path, B, C, H, W, *, c_begin=0, c_count=None, batch_step=1, row=None, x_off=0, acc_off=0, debug=False, seed=0,
          tol=ENERGY_TOL, what='', dtype=torch.float32, out=None):
    """dctp_score_accum (dctp_score_accum_ex for bf16 / fp16 `dtype`) on x[::batch_step, c_begin:c_begin + c_count, :, :W] of a NaN
    arena [B * batch_step, C, H, row], into guarded outputs (energy_out and coeff_out when `debug`); checks every output and guard.
    Returns the kernel that ran; `out` (a dict), when given, receives the scored maps and the live views of the outputs (src, acc,
    en, co; None where not asked for)."""
    row = row or W
    cc = C - c_begin if c_count is None else c_count
    n = B * cc
    full = (B * batch_step, C, H, row)
    guard = max(GUARD, 4 * H * row * 4)
    xa = Arena([math.prod(full)], dtype, [x_off], guard=guard)
    x = xa.live.view(full)[::batch_step, :, :, :W]
    src = maps(B, cc, H, W, seed, dtype)
    acc = Arena([cc], torch.float64, [acc_off], edge=NEG0, live=0.5)
    en = Arena([n], torch.float32, [4 * (seed % 2)], edge=NEG0, live=float('nan')) if debug else None
    co = Arena([n * H * W], torch.float32, [64], edge=NEG0, live=float('nan'), guard=guard) if debug else None
    _lib.check(lib.dctp_prepare(H, W))                       # (bases are uploaded synchronously on first use of a size)
    stream = _lib.current_stream()
    x[:, c_begin:c_begin + cc].copy_(src)                   # the launch below must wait for this copy
    args = (B, H, W, x.stride(0), x.stride(1), x.stride(2), c_begin, cc, _lib.ptr(acc.live), _lib.ptr(en.live) if en else None,
            _lib.ptr(co.live) if co else None, _lib.PATHS[path], stream)
    code = _lib.dtype_code(dtype)
    rc = lib.dctp_score_accum(_lib.ptr(x), *args) if code == _lib.DTYPE_F32 else lib.dctp_score_accum_ex(_lib.ptr(x), code, *args)
    _lib.check(rc)
    _lib.check(lib.dctp_check(stream))
    name = note(lib)
    label = '%s %s %dx%dx%dx%d (window %d+%d, batch step %d, row %d, offset %d) %s: %s%s' % (
        path, str(dtype).split('.')[-1], B, C, H, W, c_begin, cc, batch_step, row, x_off, what, name,
        ' [energy_out, coeff_out]' if debug else '')

    want = (src.double() ** 2).sum((2, 3))                  # [B, cc]
    chan = want.sum(0)
    live = chan > 0
    assert acc.guards_intact(), 'accum guard written: ' + label
    assert not bool(torch.isnan(acc.live).any()), 'NaN in accum: ' + label
    assert bool((acc.live[~live] == 0.5).all()), 'a dead channel changed (it must read exactly 0.5): ' + label
    err = acc_err(acc.live[live], chan[live], B)
    assert err < tol, (err, label)
    if out is not None:
        out.update(src=src, acc=acc.live, en=en.live if en else None, co=co.live if co else None)
    if not debug:
        return name
    e = en.live.view(B, cc)
    assert en.guards_intact(), 'energy_out guard written: ' + label
    assert not bool(torch.isnan(e).any()), 'energy_out not written everywhere: ' + label
    dead = want == 0
    assert bool((e[dead] == 0).all()), 'dead maps must score exactly 0: ' + label
    err = rel_err(e[~dead], want[~dead])
    assert err < tol, (err, label)
    assert co.guards_intact(), 'coeff_out guard written: ' + label
    assert not bool(torch.isnan(co.live).any()), 'coeff_out not written everywhere: ' + label
    if n * H * W <= 1 << 18:
        from scipy.fft import dctn
        z = dctn(src.double().cpu().numpy(), type=2, norm='ortho', axes=(-2, -1))
        got = co.live.view(B, cc, H, W).cpu().numpy()
        assert np.abs(got - z).max() <= COEFF_TOL * np.abs(z).max(), label
    return name


# ---------------------------------------------------------------------------------------------------------- every kernel path
def takes(path, n):
    return {'auto': True, 'simt': True, 'umma': n <= 128, 'kron': n <= 8, 'stack': n in STACK_SIDES,
            'tmem': 5 <= n <= 64 and (n % 2 == 0 or n <= 13), 'large': n in LARGE_SIDES}[path]


PATH_SIDES = [(p, n) for p in ('auto', 'kron', 'stack', 'tmem', 'umma', 'large', 'simt') for n in SIDES if takes(p, n)]


def geometry(lib, path, N, dtype=torch.float32):
    """(maps per tile, tiles at which every CTA loops over its ring of stages more than twice) of the kernel that `path` runs on
    N x N maps of `dtype`; (maps per CTA tile, None) for the CUDA-core kernels, which have no ring."""
    sm = lib.dctp_sm_count()
    kern = path
    if path == 'auto':
        kern = ('kron' if N <= 8 else 'stack' if N in STACK_SIDES else 'large' if N in LARGE_SIDES else
                'tmem' if 52 <= N <= 64 else 'umma' if N <= 128 else 'simt')
    ms = -(-N // 8) * 8
    if kern == 'kron':                                       # 128-map sub-tiles, 1, 2 or 4 per TMA tile; a ring of 3
        if N % 2 == 0 and (N * N * dtype.itemsize) % 16 == 0:  # row layout: every even side in fp32, sides 4 and 8 in 16-bit
            return 128 * (1 if N == 8 else 2), sm * 7
        return 128 * (1 if N in (6, 7) else 2 if N in (2, 5) else 4), sm * 7
    if kern == 'stack':                                      # G * J maps per tile; a ring of 3
        kp = -(-N // 16) * 16
        return (32 if kp == 16 else 8 if kp == 32 else 2), sm * 7
    if kern == 'tmem':                                       # G * J maps per tile; 6 slots per CTA up to side 32, 3 above
        return (128 // ms) * (4 if N <= 8 else 2 if N <= 16 else 1), sm * (13 if N <= 32 else 7)
    if kern == 'umma':                                       # several resident CTAs per SM
        kp = 64 if N <= 64 else 128
        occ = max(lib.dctp_occupancy(kp, mode) for mode in (0, 3))
        return (128 // ms) * (kp // ms), sm * occ * 7
    if kern == 'large':                                      # one work item per 128 coefficient rows of a map; slab rings of 2 and 3
        return 1, -(-sm * 7 // -(-N // 128))
    return (64 // N if N <= 64 else 1), None


def map_counts(path, N, mt, wrap):
    """{case: number of maps} for the tile size mt of the kernel."""
    NN = N * N

    def ok(n):                  # the TMEM-operand kernel takes odd sides only as a whole number of float4
        return not (path == 'tmem' and N % 2 and (n * NN) % 4)

    def first(lo, pred):
        return next((n for n in range(lo, lo + 64 * mt + 64) if ok(n) and pred(n)), None)

    cases = {'one map': first(1, lambda n: n == 1)}
    if mt > 1:
        cases['one tile'] = first(mt, lambda n: n == mt)
        cases['ragged last tile, stream ends on a 32-element row'] = first(mt + 1, lambda n: n % mt and (n * NN) % 32 == 0)
        cases['ragged last tile, stream ends inside a 32-element row'] = first(mt + 1, lambda n: n % mt and (n * NN) % 32)
    else:
        cases['several maps'] = 5
    if wrap:
        cases['more than two passes over the ring per CTA'] = first(wrap * mt + 1, lambda n: mt == 1 or n % mt)
    return {k: v for k, v in cases.items() if v}


@pytest.mark.parametrize('path,n', PATH_SIDES)
def test_score_stays_inside_its_buffers(lib, cuda_device, path, n):
    """Each kernel path on each side: one map, one tile, ragged last tiles (the stream ending on a 32-element row and inside one), and
    enough tiles that every CTA's mbarrier phases wrap - with per-map energies and coefficients (the debug instantiations) and
    without (the production ones)."""
    mt, wrap = geometry(lib, path, n)
    for i, (what, count) in enumerate(map_counts(path, n, mt, wrap).items()):
        B = 3 if count % 3 == 0 and count >= 6 else 2 if count % 2 == 0 and count >= 4 else 1
        # (maps of a handful of elements: the split-precision residuals do not average out, and with 2x2 maps or a maximum over
        # a hundred thousand maps the largest per-map error reaches 2e-5)
        tol = 2 * ENERGY_TOL if count >= 100000 or n <= 2 else ENERGY_TOL
        for debug in (True, False):
            score(lib, path, B, count // B, n, n, x_off=(0, 16, 64)[i % 3], acc_off=(0, 8, 64)[i % 3], debug=debug,
                  seed=1000 * n + 10 * i + debug, tol=tol, what=what)


@pytest.mark.parametrize('n', [7, 14, 32, 96])
@pytest.mark.parametrize('path', ['auto', 'umma', 'simt'])
def test_windows_and_strides_read_nothing_outside(lib, cuda_device, path, n):
    """Per-map pointers: channel windows, a batch stride that skips images, and bases that are not 16-byte aligned.  Everything
    the call does not score is NaN."""
    for debug in (True, False):
        score(lib, path, 3, 48, n, n, c_begin=36, c_count=12, debug=debug, seed=n + debug, what='last 12 channels')
        score(lib, path, 2, 40, n, n, c_begin=10, c_count=17, x_off=16, debug=debug, seed=2 * n + debug, what='middle window')
        score(lib, path, 3, 9, n, n, batch_step=2, x_off=64, debug=debug, seed=3 * n + debug, what='every other image')
        for off in (4, 8, 12):
            score(lib, path, 2, 5, n, n, x_off=off, acc_off=8, debug=debug, seed=4 * n + off + debug, what='base %d mod 16' % off)


@pytest.mark.parametrize('path', ['auto', 'simt'])
def test_cropped_and_non_square_maps(lib, cuda_device, path):
    for debug in (True, False):
        score(lib, path, 2, 3, 20, 20, row=24, debug=debug, seed=20 + debug, what='20x20 crops of 20x24 rows')
        score(lib, path, 2, 3, 20, 20, row=24, x_off=8, debug=debug, seed=22 + debug, what='20x20 crops, base 8 mod 16')
        score(lib, path, 3, 5, 12, 20, debug=debug, seed=24 + debug, what='non-square')
        score(lib, path, 2, 4, 9, 33, row=40, x_off=4, debug=debug, seed=26 + debug, what='non-square crops')


# ------------------------------------------------------------------------------------------------------ the multi-site entry
MULTI_SIDES = [7, 14, 56, 96, 34]          # Kronecker, stacked-basis (two tile sizes), large-map, and a side they do not take
MULTI_COUNTS = [1, 15, 16, 17, 32, 33, 40]


def site_plan(n_sites):
    """[B, c_count, kind] per site; kind 'dense' (16-byte aligned), 'unaligned' or 'empty'.  15 and 40 sites have empty and
    unaligned sites in the middle of the list and end on one (15: empty, 40: unaligned); the other counts are all dense, so that
    16 and 32 fill whole launches and 17 and 33 leave one site over.  Site 0 is a single map."""
    plan = []
    for i in range(n_sites):
        B, c = (1, 1) if i == 0 else (1 + i % 3, (5, 3, 12, 2, 7, 1)[i % 6])
        kind = 'dense'
        if n_sites in (15, 40):
            kind = 'empty' if i % 7 == 3 else 'unaligned' if i % 9 == 5 else 'dense'
            if i == n_sites - 1:
                kind = 'empty' if n_sites == 15 else 'unaligned'
        if kind == 'empty':
            B, c = (0, c) if i % 2 else (B, 0)
        plan.append([B, c, kind])
    return plan


@pytest.mark.parametrize('n_sites', MULTI_COUNTS)
@pytest.mark.parametrize('side', MULTI_SIDES)
def test_multi_site_entry(lib, cuda_device, side, n_sites):
    """dctp_score_accum_multi against float64 and against one dctp_score_accum call per site; per-site guarded accumulators,
    sites 1 and 2 sharing one; the number of launches its batching issues."""
    NN = side * side
    plan = site_plan(n_sites)
    slot = list(range(n_sites))                 # the accumulator slice each site adds into
    if n_sites >= 15:
        plan[2][1] = plan[1][1]
        slot[2] = 1
    nmaps = [B * c for B, c, _ in plan]
    unaligned = [i for i in range(n_sites) if plan[i][2] == 'unaligned']
    offs = [(4, 8, 12)[unaligned.index(i) % 3] if i in unaligned else (0, 16, 64)[i % 3] for i in range(n_sites)]
    xa = Arena([m * NN for m in nmaps], torch.float32, offs, guard=max(GUARD, 4 * NN * 4))
    acc = Arena([c for _, c, _ in plan], torch.float64, [(0, 8, 64)[i % 3] for i in range(n_sites)], edge=NEG0, live=0.5)
    live = [i for i in range(n_sites) if nmaps[i] > 0]
    src = {i: maps(plan[i][0], plan[i][1], side, side, seed=100 * side + i) for i in live}
    sites = (_lib.Site * n_sites)()
    for i, (B, c, _) in enumerate(plan):
        sites[i].B, sites[i].c_count = B, c
        sites[i].x = xa.views[i].data_ptr() if i in src else None
        sites[i].accum = acc.views[slot[i]].data_ptr() if i in src else None
    _lib.check(lib.dctp_prepare(side, side))
    stream = _lib.current_stream()
    before = lib.dctp_launch_count()
    for i in live:
        xa.views[i].copy_(src[i].reshape(-1))
    _lib.check(lib.dctp_score_accum_multi(sites, n_sites, side, side, stream))
    launches = lib.dctp_launch_count() - before
    _lib.check(lib.dctp_check(stream))
    name = note(lib)

    aligned = [i for i in live if plan[i][2] == 'dense']
    batched = side <= 8 or side in STACK_SIDES or side in LARGE_SIDES
    want_launches = -(-len(aligned) // 16) + len(live) - len(aligned) if batched else len(live)
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
        _lib.check(lib.dctp_score_accum(_lib.ptr(xa.views[i]), B, side, side, c * NN, NN, side, 0, c, _lib.ptr(ref[slot[i]]),
                                        None, None, _lib.PATH_AUTO, stream))
        note(lib)
    _lib.check(lib.dctp_check(stream))
    for j in range(n_sites):
        np.testing.assert_allclose(acc.views[j].cpu().numpy(), ref[j].cpu().numpy(), rtol=1e-12, err_msg='site %d' % j)


# ------------------------------------------------------------------------------------------------------------- other kernels
@pytest.mark.parametrize('H,W', [(14, 14), (12, 7)])
def test_rank_ops_read_only_their_window(lib, cuda_device, H, W):
    from test_gpu_alt_ops import check_ranks, feature_like
    B, C, cb, cc = 3, 20, 8, 12
    src = feature_like(B, cc, H, W, seed=31 * H + W)
    values = {}
    for op in ('rank', 'rank_sq'):
        xa = Arena([B * C * H * W], torch.float32, [4])
        x = xa.live.view(B, C, H, W)
        acc = Arena([cc], torch.float64, [8], edge=NEG0, live=0.5)
        vals = Arena([B * cc], torch.float32, [12], edge=NEG0, live=float('nan'))
        stream = _lib.current_stream()
        x[:, cb:cb + cc].copy_(src.to('cuda'))
        _lib.check(lib.dctp_score_op(_lib.OPS[op], _lib.ptr(x), B, H, W, x.stride(0), x.stride(1), x.stride(2), cb, cc,
                                     _lib.ptr(acc.live), _lib.ptr(vals.live), stream))
        _lib.check(lib.dctp_check(stream))
        assert note(lib) == 'rank_jacobi_kernel'
        assert acc.guards_intact() and vals.guards_intact(), op
        v = vals.live.view(B, cc)
        assert not bool(torch.isnan(v).any()), op
        assert torch.equal(acc.live - 0.5, v.double().sum(0)), op
        values[op] = v.cpu()
    check_ranks(values['rank'], src)
    assert torch.equal(values['rank_sq'], values['rank'] ** 2)


def test_dct3_reads_only_its_window(lib, cuda_device):
    from oracle import alt_ops_port as ao
    B, C, cb, cc, n = 3, 20, 5, 9, 16
    src = maps(B, cc, n, n, seed=33)
    want = ao.dct3_energy64(src.cpu().numpy())
    for with_values in (True, False):
        xa = Arena([B * C * n * n], torch.float32, [16])
        x = xa.live.view(B, C, n, n)
        acc = Arena([1], torch.float64, [8], edge=NEG0, live=0.5)
        vals = Arena([B], torch.float32, [4], edge=NEG0, live=float('nan')) if with_values else None
        stream = _lib.current_stream()
        x[:, cb:cb + cc].copy_(src)
        _lib.check(lib.dctp_score_op(_lib.OP_DCT3, _lib.ptr(x), B, n, n, x.stride(0), x.stride(1), x.stride(2), cb, cc,
                                     _lib.ptr(acc.live), _lib.ptr(vals.live) if vals else None, stream))
        _lib.check(lib.dctp_check(stream))
        note(lib)
        assert acc.guards_intact()
        np.testing.assert_allclose(float(acc.live[0]) - 0.5, want.sum(), rtol=1e-4)
        if vals:
            assert vals.guards_intact()
            np.testing.assert_allclose(vals.live.cpu().numpy().astype(np.float64), want, rtol=1e-4)


def test_finalize_writes_only_its_output(lib, cuda_device):
    n = 1000                                                   # not a multiple of the 256-thread block
    g = torch.Generator(device='cuda').manual_seed(5)
    src = torch.rand(n, dtype=torch.float64, generator=g, device='cuda') * 100
    acc = Arena([n], torch.float64, [8])
    out = Arena([n], torch.float32, [4], edge=NEG0, live=float('nan'))
    acc.live.copy_(src)
    _lib.check(lib.dctp_finalize(_lib.ptr(acc.live), 7.0, _lib.ptr(out.live), n, _lib.current_stream()))
    _lib.check(lib.dctp_check(_lib.current_stream()))
    assert out.guards_intact()
    assert torch.equal(out.live, (src / 7.0).float())


def test_topk_writes_only_its_segments_ranges(lib, cuda_device):
    """Output ranges with gaps between some of them (and none between others); int64 guards and gaps hold -1.  The scores sit in a
    NaN arena: NaN ranks above every score, so a read past the last segment changes its selection."""
    from oracle import reference_port as port
    rng = np.random.default_rng(3)
    lens = [1, 100, 1000, 9000, 0, 257, 33]                   # 9000: more than the kernel's shared-memory key buffer
    ks = [1, 10, 500, 3000, 0, 256, 17]
    gaps = [3, 0, 5, 1, 2, 0, 4]
    vecs = [(rng.integers(0, 40, L) if i % 2 else rng.standard_normal(L)).astype(np.float32) for i, L in enumerate(lens)]
    seg_off = np.cumsum([0] + lens)
    out_off, cur = [], 0
    for k, gap in zip(ks, gaps):
        out_off.append(cur)
        cur += k + gap
    out_off.append(cur)
    scores = Arena([int(seg_off[-1])], torch.float32, [4])
    scores.live.copy_(torch.from_numpy(np.concatenate(vecs)).to('cuda'))
    out = Arena([cur], torch.int64, [8], edge=-1, live=-1)
    dev_i32 = lambda v: torch.tensor(np.asarray(v), dtype=torch.int32, device='cuda')
    so, sk, oo = dev_i32(seg_off), dev_i32(ks), dev_i32(out_off)
    _lib.check(lib.dctp_topk_segmented(_lib.ptr(scores.live), _lib.ptr(so), _lib.ptr(sk), len(lens), _lib.ptr(out.live),
                                       _lib.ptr(oo), _lib.current_stream()))
    _lib.check(lib.dctp_check(_lib.current_stream()))
    want = np.full(cur, -1, np.int64)
    for s, (v, k) in enumerate(zip(vecs, ks)):
        want[out_off[s]:out_off[s] + k] = port.select_index_stable(v, k)
    np.testing.assert_array_equal(out.live.cpu().numpy(), want)
    assert out.guards_intact()


def test_gather_weight_stays_inside_its_buffers(lib, cuda_device):
    c_out, c_in, inner = 37, 19, 9
    g = torch.Generator(device='cuda').manual_seed(6)
    w = torch.randn(c_out, c_in, inner, generator=g, device='cuda')
    sel_o = torch.tensor([0, 5, 36, 12, 7], dtype=torch.int64, device='cuda')
    sel_i = torch.tensor([18, 0, 3], dtype=torch.int64, device='cuda')
    for so, si in ((sel_o, sel_i), (sel_o, None), (None, None)):
        k_out = c_out if so is None else so.numel()
        k_in = c_in if si is None else si.numel()
        wa = Arena([w.numel()], torch.float32, [4])
        out = Arena([k_out * k_in * inner], torch.float32, [12], edge=NEG0, live=float('nan'))
        wa.live.copy_(w.reshape(-1))
        _lib.check(lib.dctp_gather_weight(_lib.ptr(wa.live), c_out, c_in, inner, _lib.ptr(so), k_out, _lib.ptr(si), k_in,
                                          _lib.ptr(out.live), _lib.current_stream()))
        _lib.check(lib.dctp_check(_lib.current_stream()))
        want = w if so is None else w[so]
        want = want if si is None else want[:, si]
        assert torch.equal(out.live.view(k_out, k_in, inner), want)
        assert out.guards_intact()


# --------------------------------------------------------------------------------------------------- instantiation coverage
REQUIRED = (
    # Kronecker kernel: sides 1..8 reach six of its eight compiled instantiations (K2 follows from the side: no even side has
    # K2 = 32, no odd side K2 = 48)
    ['score_kron_kernel<K2=16,even>', 'score_kron_kernel<K2=16,odd>', 'score_kron_kernel<K2=32,odd>',
     'score_kron_kernel<K2=48,even>', 'score_kron_kernel<K2=64,even>', 'score_kron_kernel<K2=64,odd>']
    # stacked-basis kernel: every (KP, VEC) of its sides, debug (cfg6) and production (cfg7) instantiations
    + ['score_stack_kernel<KP=%d,VEC=%d,cfg%d>' % (kp, vec, cfg)
       for kp, vec in ((16, 2), (16, 4), (32, 2), (32, 4), (48, 4), (64, 4)) for cfg in (6, 7)]
    # TMEM-operand kernel
    + ['score_t_kernel<32,6,VPE=1>', 'score_t_kernel<32,6,VPE=2>', 'score_t_kernel<32,6,VPE=4>',
       'score_t_kernel<64,3,VPE=1>', 'score_t_kernel<64,3,VPE=2>', 'score_t_kernel<64,3,VPE=1,2 producer warpgroups>']
    # smem-operand kernel <KP, load mode, prefetch>: dense 8/4/2-byte scatter (0/1/2), generic 128/64/32-bit loads (3/4/5)
    + ['score_umma_kernel<64,%d,%d>' % mp for mp in ((0, 0), (0, 1), (1, 0), (1, 1), (2, 0), (2, 1), (3, 0), (4, 0), (5, 0))]
    + ['score_umma_kernel<128,%d,%d>' % mp for mp in ((0, 0), (0, 1), (3, 0), (4, 0), (5, 0))]
    + ['score_large_kernel', 'score_simt_small_kernel', 'score_simt_large_kernel', 'rank_jacobi_kernel'])


def test_every_instantiation_was_launched(request, cuda_device):
    """Last test of the module: the cases above ran every kernel instantiation in REQUIRED."""
    if request.config.getoption('keyword') or any('::' in a for a in request.config.args):
        pytest.skip('only part of the module ran')
    missing = [k for k in REQUIRED if k not in SEEN]
    assert not missing, 'never launched: %s (launched: %s)' % (', '.join(missing), ', '.join(sorted(SEEN)))
