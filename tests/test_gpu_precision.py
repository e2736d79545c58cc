"""Precision of the split-bf16 arithmetic of every score kernel, on maps built to defeat it.

Every tensor-core score kernel splits each operand into bf16 hi + lo (hi = rn_bf16(x), lo = rn_bf16(x - hi)), issues three MMAs per
product (hi.hi + lo.hi + hi.lo; lo.lo is dropped, except in the stacked-basis kernel's stage 1) and accumulates in fp32 (DESIGN
section 3).  The Kronecker kernel (sides 1..8) does
this once, against the split C_N (x) C_N; the others twice, with the stage-1 result D1 held in fp32 and split again.  On random ReLU
maps the rounding errors of that arithmetic take both signs and cancel in a map's energy, so the suite's random-map bars
(ENERGY_TOL) cannot tell it from something cheaper.  The maps here keep the errors from cancelling:

  1  single-mode maps   a * outer(c_u, c_v) of the float64 orthonormal DCT-II basis, rounded to the input dtype: the energy sits
                        in one coefficient, and the dropped lo.lo products of a basis row and a map built from that row share a
                        sign.  Every basis row u is the first and the second index of a mode (sides <= 32: all N * N modes), and
                        every mode sits in every map slot of a tile.  The channels of the stream are the modes (images: the
                        slots), so the production instantiation, which returns channel sums only, puts a defect of one row or
                        one slot into few channels instead of averaging it over the stream.
  2  worst residuals    fp32 values whose rounding error under rn_bf16, the hi + lo split, tf32 rounding and tf32 truncation is
                        the largest possible and of one sign (found by search over [1, 2)): constant maps, maps of those values
                        times random powers of two, and post-ReLU-shaped maps.
  3  scale by 2^k       score(2^k x) == 4^k score(x), bitwise, in energy_out, coeff_out (2^k) and accum, over a range of k
                        derived below in which no intermediate of the arithmetic leaves the normal fp32 range.

Every case runs the debug instantiation (energy_out, coeff_out: per-map energy, the peak coefficient and the largest leakage into
the others) and the production one (channel sums only, the instantiation every hook launch runs), through the forced paths and
AUTO, and is held to float64: the maps exactly as handed to the kernel (fp32, or 16-bit widened exactly), their energies by
Parseval and their coefficients through the float64 basis (scipy), computed on the device.  The bars (BARS) follow from the split's
error model and the B200 measurement.

emulate() is the split arithmetic in float64 (the same hi / lo rules, three products, fp32 between the stages) with the
degradations a cheaper kernel would make: the map read as tf32 or as bf16, one basis row or the whole basis without its lo part,
D1 without its lo part.  test_bars_separate_the_degradations (no GPU) runs the families and judge() against it: the correct
arithmetic passes, each degradation fails.  The kernels are not compared with emulate() itself: the order and rounding of their
fp32 accumulation, and the stacked-basis kernel's stage 1 (which keeps lo.lo: its lanes hold C_hi and C_lo times X_hi + X_lo), put
them up to 2.4e-5 away from it on these maps, as far as the arithmetic is from float64.
"""
import functools

import numpy as np
import pytest
import torch
from scipy.fft import dct

from test_gpu_bounds import PATH_SIDES, geometry
from test_gpu_half_bounds import DTYPES, NATIVE_SIDES, native
from test_gpu_kernels import REL_TOL

# ------------------------------------------------------------------------------------------------------------------------ bars
# Error model of one split product a * b: hi_a hi_b + lo_a hi_b + hi_a lo_b misses lo_a lo_b (|lo| <= 2^-8 |x|: <= 2^-16 |a b|) and
# the split residuals (<= 2^-17 |x| each), 3.1e-5 of |a b| when every error has the same sign, and the fp32 accumulation adds up
# to 2^-24 of the sum per add.  A two-stage coefficient collects the split's share twice and its square doubles it: 1.2e-4 of the
# energy in the worst case.  The maps here line up most of those signs.  Every bar below is relative to float64 (energies: to the
# map's or channel's energy; coefficients: to the map's largest coefficient) and sits >= 2x above the worst of every kernel, side
# and input dtype measured on a B200 at its 1000 W power limit, and >= 3x below each emulated degradation the family is meant to
# catch (test_bars_separate_the_degradations):
#
#   single / energy            measured 2.6e-5 (stacked-basis, fp16 input at 16x16); emulated correct arithmetic 1.9e-5.  A row
#                              without lo: >= 7.7e-4 up to side 96; no lo in the basis or in D1: >= 9.4e-4.
#   single / peak coefficient  half the energy's: measured 1.3e-5.
#   single / leakage           any other coefficient, relative to the peak: measured 8.6e-6, emulated 4.5e-6.  A row without lo
#                              leaks 2^-9 / sqrt(N) of every mode into itself: 3.9e-4 at side 320, where the energy moves by
#                              7.5e-5 only (3x the measured 2.6e-5: no energy bar can hold both); maps read as bf16 3.5e-4.
#   worst / energy             measured 5.0e-5 (large-map kernel at 176, smem-operand at 11x11); the emulated arithmetic 4.9e-5 at
#                              11x11.  Maps read as tf32: 9.7e-4, as bf16: 7.8e-3; basis hi only: 4.6e-4; D1 without lo: 3.5e-3.
#                              (Above the product's 1e-4 on channel scores, which run() holds the channel sums to as well.)
#   worst / coefficients       measured 2.7e-5; the degradations >= 2.3e-4.
BARS = {'single': {'energy': 6e-5, 'peak coefficient': 3e-5, 'leakage': 2e-5},
        'worst': {'energy': 1.1e-4, 'coefficients': 6e-5}}


# ------------------------------------------------------------------------------------------------------- float64 emulation
def bf16(t):
    """rn_bf16 of a float64 tensor that holds fp32 values (or of float64 values, through fp32, as the host tables do)."""
    return t.float().bfloat16().double()


def split(t):
    """hi, lo of split2 (device, fp32 operands: x - hi is exact) and of split_bf16 (host, the float64 basis: lo = rn_bf16(c - hi))."""
    hi = bf16(t)
    return hi, bf16(t - hi)


def f32(t):
    return t.float().double()


def tf32_rn(x):
    """x (float64 holding fp32) rounded to tf32 (10 mantissa bits), ties to even."""
    u = x.cpu().numpy().astype(np.float32).view(np.uint32).astype(np.uint64)
    u = ((u + 0xFFF + ((u >> 13) & 1)) >> 13) << 13
    return torch.from_numpy(u.astype(np.uint32).view(np.float32).astype(np.float64)).to(x.device)


def tf32_rz(x):
    u = x.cpu().numpy().astype(np.float32).view(np.uint32) & np.uint32(0xFFFFE000)
    return torch.from_numpy(u.view(np.float32).astype(np.float64)).to(x.device)


@functools.lru_cache(maxsize=None)
def _basis(N, device):
    return torch.from_numpy(dct(np.eye(N), type=2, norm='ortho', axis=0)).to(device)      # C[k, n]


def basis(N, device='cpu'):
    return _basis(N, str(device))


CORRECT = {}
DEGRADED = {                          # the arithmetic each precision family must tell from the correct one
    'maps read as tf32': {'x': 'tf32'},
    'maps read as bf16': {'x': 'bf16'},
    'one basis row without lo': {'row': None},       # row chosen per side: degraded_row()
    'basis hi only': {'hi_only': True},
    'D1 without lo': {'d1_lo': False},
}


def degraded_row(N):
    return N // 2 + 1 if N > 2 else N - 1


def emulate(X, kind, arith=CORRECT):
    """Coefficients (float64 holding fp32) of the maps X [..., N, N] (float64, the values the kernel reads) under split-bf16
    arithmetic: kind 'rows' (stage 1 contracts the columns, D1 = X C^T, then Z = C D1), 'cols' (D1 = C X, Z = D1 C^T), or 'kron'
    (one stage against the split C_N (x) C_N).  `arith` degrades it: x 'tf32' / 'bf16' (the map read as tf32, or without its lo
    part), row (that basis row without its lo part), hi_only (no basis lo parts), d1_lo False (D1 without its lo part)."""
    N = X.shape[-1]
    C = basis(N, X.device)
    if arith.get('x') == 'tf32':
        X = tf32_rn(X)
    xh, xl = split(X)
    if arith.get('x') == 'bf16':
        xl = torch.zeros_like(xl)

    def degrade(lo):
        if arith.get('hi_only'):
            return torch.zeros_like(lo)
        if 'row' in arith:
            lo = lo.clone()
            lo[degraded_row(N) if arith['row'] is None else arith['row']] = 0
        return lo

    if kind == 'kron':
        ch, cl = split(torch.kron(C, C))
        cl = degrade(cl)
        x2h, x2l = xh.reshape(*X.shape[:-2], N * N), xl.reshape(*X.shape[:-2], N * N)
        z = x2h @ ch.T + x2l @ ch.T + x2h @ cl.T
        return f32(z).reshape(X.shape)
    ch, cl = split(C)
    cl = degrade(cl)
    if kind == 'rows':
        d1 = f32(xh @ ch.T + xl @ ch.T + xh @ cl.T)
    else:
        d1 = f32(ch @ xh + ch @ xl + cl @ xh)
    dh, dl = split(d1)
    if arith.get('d1_lo') is False:
        dl = torch.zeros_like(dl)
    if kind == 'rows':
        return f32(ch @ dh + ch @ dl + cl @ dh)
    return f32(dh @ ch.T + dl @ ch.T + dh @ cl.T)


def exact(X):
    C = basis(X.shape[-1], X.device)
    return C @ X @ C.T


# ---------------------------------------------------------------------------------------------------------------- map families
def round_to(X, dtype):
    return X.to(dtype).double()


def single_modes(N, dtype=torch.float32, device='cpu', only=None):
    """[D, N, N] maps N * outer(c_u, c_v) rounded to dtype: every (u, v) for N <= 32, else (u, (7u + 3) mod N) and its transpose
    for every u - every basis row is the first and the second index of a mode.  `only`: the modes that hold these rows."""
    if N <= 32:
        pairs = [(u, v) for u in range(N) for v in range(N)]
    else:
        pairs = [(u, (7 * u + 3) % N) for u in range(N)]
        pairs += [(v, u) for u, v in pairs]
    if only is not None:
        pairs = [p for p in pairs if p[0] in only or p[1] in only]
    C = basis(N, device)
    u = torch.tensor([p[0] for p in pairs], device=device)
    v = torch.tensor([p[1] for p in pairs], device=device)
    return round_to(N * C[u][:, :, None] * C[v][:, None, :], dtype)


def _search(err):
    """The 16 fp32 values of [1, 2) with the largest err(x) / x > 0 (a rounding error of the largest size, all of one sign)."""
    x = torch.arange(1 << 23, dtype=torch.int32).add_(0x3F800000).view(torch.float32).double()
    e = err(x) / x
    top = torch.topk(e, 16).indices
    assert bool((e[top] > 0).all())
    return x[top]


@functools.lru_cache(maxsize=None)
def worst_values():
    """{criterion: 16 fp32 values in [1, 2)} for (a) rn_bf16, (b) the split residual x - hi - lo, (c) tf32 rounding, (d) tf32
    truncation.  (b)'s largest is 1.0020065307617188 (residual 2^-17.4 of x); (a) and (c) reach just under half an ulp of their
    format (2^-9, 2^-12 of x), (d) just under one (2^-11)."""
    def residual(x):
        hi, lo = split(x)
        return x - hi - lo
    return {'bf16': _search(lambda x: x - bf16(x)), 'split': _search(residual),
            'tf32 rn': _search(lambda x: x - tf32_rn(x)), 'tf32 rz': _search(lambda x: x - tf32_rz(x))}


def worst_maps(N, device='cpu', seed=0):
    """[D, N, N] fp32 maps of the worst_values: per criterion two constant maps, two maps of the values times 2^e (e in -4..3:
    the size of the error varies, its sign does not), and two post-ReLU-shaped maps (1 in 8 elements 0, the rest the values)."""
    g = torch.Generator().manual_seed(seed + N)
    out = []
    for vals in worst_values().values():
        out += [torch.full((N, N), float(vals[0])), torch.full((N, N), float(vals[1]))]
        for _ in range(2):
            pick = vals[torch.randint(16, (N, N), generator=g)]
            out.append(pick * torch.pow(2.0, torch.randint(-4, 4, (N, N), generator=g).double()))
        for _ in range(2):
            pick = vals[torch.randint(16, (N, N), generator=g)]
            out.append(torch.where(torch.rand(N, N, generator=g) < 0.125, torch.zeros(()).double(), pick))
    return torch.stack(out).to(device)


# ------------------------------------------------------------------------------------------------------------------ the checks
def peak_and_leak(Z, Z64):
    """Per map of [..., N, N] coefficients: the error of the largest float64 coefficient relative to it, and the largest error
    of every other coefficient relative to it (the leakage the arithmetic adds)."""
    z, z64 = Z.flatten(-2), Z64.flatten(-2)
    idx = z64.abs().argmax(-1, keepdim=True)
    peak = z64.gather(-1, idx).abs().clamp_min(1e-30)
    err = (z - z64).abs()
    peak_err = err.gather(-1, idx) / peak
    leak = err.scatter(-1, idx, 0.0).amax(-1, keepdim=True) / peak
    return peak_err.max().item(), leak.max().item()


def judge(family, E, E64, Z=None, Z64=None):
    """Errors of energies E (any shape) and coefficients Z ([..., N, N]) against float64 and the bars of `family` they break:
    {'worst': {metric: error}, 'broken': [text]}.  Dead entries (E64 == 0) must be exactly 0."""
    live = E64 > 0
    worst = {}
    broken = [] if bool((E[~live] == 0).all()) else ['a dead map or channel did not score exactly 0']
    worst['energy'] = ((E[live] - E64[live]).abs() / E64[live]).max().item() if bool(live.any()) else 0.0
    if Z is not None:
        if family == 'single':
            worst['peak coefficient'], worst['leakage'] = peak_and_leak(Z, Z64)
        else:
            peak = Z64.abs().amax((-2, -1)).clamp_min(1e-30)
            worst['coefficients'] = ((Z - Z64).abs().amax((-2, -1)) / peak).max().item()
    for metric, err in worst.items():
        if err >= BARS[family][metric]:
            broken.append('%s %.3g from float64 (bar %.3g)' % (metric, err, BARS[family][metric]))
    return {'worst': worst, 'broken': broken}


def layout(maps, mt):
    """[B, C, N, N] stream in which channel c < D holds map c in every image and the other channels are dead (0): C = 1 mod mt
    and B = mt, so map (b, c) sits in slot (b + c) mod mt of its tile and every map is seen in every slot."""
    D, N = maps.shape[0], maps.shape[-1]
    C = D if mt == 1 else D + (1 - D) % mt
    x = torch.zeros(mt, C, N, N, dtype=maps.dtype, device=maps.device)
    x[:, :D] = maps
    return x


def run(lib, path, N, maps, family, dtype=torch.float32, debug=True):
    """Score `maps` (float64 holding dtype values, [D, N, N]) laid out by layout() through dct_energy on `path`; judge the per-map
    energies and coefficients (debug) or the channel sums (production).  Returns (kernel name, judge()'s result)."""
    from dct_pruning_b200.ops import dct_energy
    mt, _ = geometry(lib, path, N, dtype)
    x = layout(maps.to('cuda'), mt)
    acc, en, co = dct_energy(x.to(dtype), path=path, want_energy=debug, want_coeff=debug)
    name = lib.dctp_last_kernel().decode().split(' (')[0]
    assert 'cfg' not in name or debug == ('cfg6' in name), name     # (the stacked-basis kernel names its debug instantiation)
    D = maps.shape[0]
    Z64 = exact(x[0, :D])
    E64 = torch.zeros(x.shape[1], dtype=torch.float64, device='cuda')
    E64[:D] = (Z64 ** 2).sum((-2, -1))
    if debug:
        res = judge(family, en.double(), E64.expand(mt, -1), co[:, :D].double(), Z64.expand(mt, -1, -1, -1))
    else:
        res = judge(family, acc, E64 * mt)
        if res['worst']['energy'] >= REL_TOL:                          # the product's bar on channel scores holds on every family
            res['broken'].append('channel sum %.3g from float64 (bar %.3g)' % (res['worst']['energy'], REL_TOL))
    return name, res


def check(lib, path, N, maps, family, dtype=torch.float32, what=''):
    for debug in (True, False):
        name, res = run(lib, path, N, maps, family, dtype, debug)
        assert not res['broken'], '%s %dx%d %s %s%s: %s; %s' % (
            path, N, N, str(dtype).split('.')[-1], what, ' [energy_out, coeff_out]' if debug else '', name, '; '.join(res['broken']))


# -------------------------------------------------------------------------------------------------------------------- family 1
@pytest.mark.gpu
@pytest.mark.parametrize('path,n', PATH_SIDES)
def test_single_mode_maps(lib, cuda_device, path, n):
    """Every basis row in both stages and in every tile slot, fp32 input, debug and production instantiations."""
    check(lib, path, n, single_modes(n, device='cuda'), 'single', what='single-mode maps')


@pytest.mark.gpu
@pytest.mark.parametrize('how', ['forced', 'auto'])
@pytest.mark.parametrize('n', NATIVE_SIDES)
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_single_mode_maps_16bit(lib, cuda_device, dt, n, how):
    """The same on the kernels that read bf16 / fp16 themselves.  A bf16 map is exact in hi, so here nothing but the basis split
    stands between the kernel and float64."""
    dtype = DTYPES[dt]
    path = native(n) if how == 'forced' else 'auto'
    check(lib, path, n, single_modes(n, dtype, device='cuda'), 'single', dtype, what='single-mode maps')


# -------------------------------------------------------------------------------------------------------------------- family 2
@pytest.mark.gpu
@pytest.mark.parametrize('path,n', PATH_SIDES)
def test_worst_residual_maps(lib, cuda_device, path, n):
    check(lib, path, n, worst_maps(n, device='cuda'), 'worst', what='worst-residual maps')


# -------------------------------------------------------------------------------------------------------------------- family 3
# Maps: relu(N(0, 1)) rounded to the input dtype, with every |x| < 2^-8 set to 0, so the nonzero |x| lie in [2^-8, 8); sides up to
# 320 < 2^9.  Scaled by 2^k:
#   top     |D1|, |Z| <= ||X||_F < 2^12 * 2^k, and a map's energy (or the share of it one fp32 sum holds before it is added to the fp64
#           accumulator) < 2^24 * 4^k: finite for k <= 51; k <= 50 here.  fp16 input must hold 8 * 2^k exactly: k <= 12.
#   bottom  stage 1: a value's lo part is 0 or at least its last bit (2^-31 * 2^k); a basis entry (of C_N, or of C_N (x) C_N for the
#           Kronecker kernel) is 0 or >= 2^-24 (sqrt(2/N) sin(pi/2N) >= 2^-12 at N <= 320) and its lo part 0 or >= 2^-77 (the float64
#           residual): every product the MMAs keep is 0 or >= 2^-85 * 2^k, normal for k >= -41.  (The basis's exact zeros must be
#           held as 0: test_basis_zeros_are_exact.)  The energy: a live map's is >= 2^-16 * 4^k, and squares below 2^-43 of it
#           cannot reach a bit of it even all 2^17 of them together (half an ulp is 2^-25): the rest is normal for k >= -33.  fp16
#           input must stay normal: 2^-8 * 2^k >= 2^-14, k >= -6.
SCALE_K = {torch.float32: (-33, 50), torch.bfloat16: (-33, 50), torch.float16: (-6, 12)}


def scale_maps(B, C, N, dtype, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.relu(torch.randn(B, C, N, N, generator=g, device='cuda')).to(dtype)
    x[x.abs() < 2 ** -8] = 0
    x[:, 1::5] = 0
    return x


def scale_case(lib, path, n, dtype):
    """Both instantiations of `path` on 2 images of more channels than a tile holds, at 2^k x for the k of SCALE_K: accum,
    energy_out and coeff_out must be 4^k, 4^k and 2^k times those at k = 0, bit for bit.  (The CUDA-core kernel for maps above 64
    adds the energies of a map's 64-column panels into energy_out with fp32 atomics, in whatever order its CTAs finish: there the
    bar is that order's rounding, and accum, the exact fp64 sum of the same partials, is held bitwise.)"""
    from dct_pruning_b200.ops import dct_energy
    mt, _ = geometry(lib, path, n, dtype)
    B, C = 2, min(mt, 512) + 3 if mt > 1 else 5
    while (B * C * n * n) % 4:                                  # (the TMEM-operand kernel takes whole float4 at odd sides)
        C += 1
    x = scale_maps(B, C, n, dtype, seed=7 * n + len(path))
    lo, hi = SCALE_K[dtype]
    ref = {}
    for debug in (True, False):
        acc, en, co = dct_energy(x, path=path, want_energy=debug, want_coeff=debug)
        ref[debug] = (acc, en, co, lib.dctp_last_kernel().decode())
    for k in sorted({lo, lo + 1, (lo - 1) // 2, -1, 1, 2, hi // 2, hi - 1, hi}):
        xs = x * 2.0 ** k                                          # exact: stays normal in dtype over SCALE_K
        assert torch.equal(xs.double(), x.double() * 2.0 ** k)
        for debug in (True, False):
            acc0, en0, co0, name = ref[debug]
            acc, en, co = dct_energy(xs, path=path, want_energy=debug, want_coeff=debug)
            label = '%s %dx%d %s k=%d: %s' % (path, n, n, str(dtype).split('.')[-1], k, name)
            assert lib.dctp_last_kernel().decode() == name, label
            assert torch.equal(acc, acc0 * 4.0 ** k), 'accum ' + label
            if not debug:
                continue
            assert torch.equal(co, co0 * 2.0 ** k), 'coeff_out ' + label
            if name.startswith('score_simt_large_kernel'):
                panels = -(-n // 64)
                err = ((en.double() - en0.double() * 4.0 ** k).abs() - panels * 2.0 ** -24 * en.double().abs()).max().item()
                assert err <= 0, 'energy_out ' + label
            else:
                assert torch.equal(en, en0 * 4.0 ** k), 'energy_out ' + label
    return ref[True][3]


@pytest.mark.gpu
@pytest.mark.parametrize('path,n', PATH_SIDES)
def test_power_of_two_scaling_is_exact(lib, cuda_device, path, n):
    scale_case(lib, path, n, torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize('how', ['forced', 'auto'])
@pytest.mark.parametrize('n', NATIVE_SIDES)
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_power_of_two_scaling_is_exact_16bit(lib, cuda_device, dt, n, how):
    name = scale_case(lib, native(n) if how == 'forced' else 'auto', n, DTYPES[dt])
    assert 'IN=' in name, name


def basis_zeros(N):
    """(k, n) with C_N[k][n] = 0 in exact arithmetic: cos(pi (2n + 1) k / 2N) at an odd multiple of pi / 2."""
    return [(k, n) for k in range(N) for n in range(N) if ((2 * n + 1) * k) % (2 * N) == N]


def impulse_at_a_zero(lib, path, n, dtype):
    """An impulse at (n0, n0), C_N[k0][n0] = 0, in every slot of a tile: its coefficients C_N[u][n0] C_N[v][n0] are exactly 0 in row
    and column k0, so coeff_out must hold exact zeros there (and energy_out the float64 energy)."""
    from dct_pruning_b200.ops import dct_energy
    k0, n0 = basis_zeros(n)[0]
    mt, _ = geometry(lib, path, n, dtype)
    maps = torch.zeros(1, n, n, dtype=torch.float64, device='cuda')
    maps[0, n0, n0] = 1.0
    _, en, co = dct_energy(layout(maps, mt).to(dtype), path=path, want_energy=True, want_coeff=True)
    name = lib.dctp_last_kernel().decode()
    label = '%s %dx%d %s, impulse at (%d, %d), C[%d][%d] = 0: %s' % (path, n, n, str(dtype).split('.')[-1], n0, n0, k0, n0, name)
    co = co.view(mt, n, n)
    assert int((co[:, k0] != 0).sum()) == 0 and int((co[:, :, k0] != 0).sum()) == 0, label
    assert float((en.double() - 1).abs().max()) < BARS['single']['energy'], label
    return name


@pytest.mark.gpu
@pytest.mark.parametrize('path,n', [(p, n) for p, n in PATH_SIDES if basis_zeros(n)])
def test_basis_zeros_are_exact(lib, cuda_device, path, n):
    """The host tables hold the zeros of the DCT-II basis as 0, not as the rounding noise of cos(pi / 2) (down to 1e-33 in the
    Kronecker image, with lo parts down to 2^-117, which a map of small values turns into underflowing products)."""
    impulse_at_a_zero(lib, path, n, torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize('how', ['forced', 'auto'])
@pytest.mark.parametrize('n', [n for n in NATIVE_SIDES if basis_zeros(n)])
@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_basis_zeros_are_exact_16bit(lib, cuda_device, dt, n, how):
    assert 'IN=' in impulse_at_a_zero(lib, native(n) if how == 'forced' else 'auto', n, DTYPES[dt])


# -------------------------------------------------------------------------------------------------------- CPU self-check
SELF_CHECK_SIDES = {8: 'kron', 14: 'rows', 56: 'cols', 320: 'rows'}


def emulated_verdicts(N, kind):
    """{arithmetic: {(family, instantiation): bars broken}} of the emulated correct and degraded arithmetic on the two families at
    side N (side 320: the single-mode maps that hold the degraded row, and a sample of the others).  'production' judges the
    energies alone, which is what a channel holding one map in every image sums."""
    only = {degraded_row(N), 0, 1, N // 3, N - 1} if N > 64 else None
    families = {'single': single_modes(N, only=only), 'worst': worst_maps(N)[::3 if N > 64 else 1]}
    out = {}
    for label, arith in [('correct', CORRECT)] + list(DEGRADED.items()):
        out[label] = {}
        for fam, X in families.items():
            Z64, Z = exact(X), emulate(X, kind, arith)
            E64, E = (Z64 ** 2).sum((-2, -1)), (Z ** 2).sum((-2, -1))
            out[label][fam, 'debug'] = judge(fam, E, E64, Z, Z64)
            out[label][fam, 'production'] = judge(fam, E, E64)
    return out


# the degradations each family is built to catch, in the debug instantiation (energies and coefficients) and in the production
# one (channel sums); a row without its lo part at side 320 moves the energy of its modes by 7e-5 only, too close to the correct
# arithmetic's 2e-5 for a channel-sum bar, and is caught by the leakage it adds (3.9e-4 of the peak, against 3e-6)
CATCHES = {'maps read as tf32': {'worst': ('debug', 'production')},
           'maps read as bf16': {'worst': ('debug', 'production'), 'single': ('debug',)},
           'one basis row without lo': {'single': ('debug', 'production')},
           'basis hi only': {'single': ('debug', 'production'), 'worst': ('debug', 'production')},
           'D1 without lo': {'single': ('debug', 'production'), 'worst': ('debug', 'production')}}


@pytest.mark.parametrize('N', sorted(SELF_CHECK_SIDES))
def test_bars_separate_the_degradations(N):
    """The families and judge() on the CPU: the emulated correct arithmetic passes every bar, and every emulated degradation breaks
    one on each family and instantiation of CATCHES."""
    kind = SELF_CHECK_SIDES[N]
    verdicts = emulated_verdicts(N, kind)
    assert not any(v['broken'] for v in verdicts['correct'].values()), verdicts['correct']
    for label, fams in CATCHES.items():
        if label == 'D1 without lo' and kind == 'kron':
            continue                                           # one stage: there is no D1
        for fam, insts in fams.items():
            for inst in insts:
                if (label, inst, N) == ('one basis row without lo', 'production', 320):
                    continue
                assert verdicts[label][fam, inst]['broken'], '%s passes family %s (%s) at side %d: %s' % (
                    label, fam, inst, N, verdicts[label][fam, inst]['worst'])
