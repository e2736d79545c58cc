"""bf16 / fp16 activations (the maps of a forward pass under torch.autocast) through the C ABI: dctp_score_accum_ex and
dctp_score_accum_multi_ex.

The stacked-basis (even sides 10..64) and Kronecker (sides <= 8) kernels read 16-bit maps themselves; their per-map energies are
held to the float64 energy of the widened maps at the bar tests/test_gpu_kernels.py applies to those kernels in fp32.  Every other
shape and path widens the scored window to fp32 and runs the fp32 kernels: bit-identical to the fp32 entry on that copy.
The guard-band and non-finite rules of test_gpu_bounds.py and test_gpu_nonfinite.py are applied to 16-bit input in
test_gpu_half_bounds.py.
"""
import ctypes
import struct

import pytest
import torch

from dct_pruning_b200 import _lib

pytestmark = pytest.mark.gpu

ENERGY_TOL = 2e-5                     # tests/test_gpu_kernels.py: what the bf16x3 kernels deliver per map
DTYPES = {'bf16': (torch.bfloat16, _lib.DTYPE_BF16), 'fp16': (torch.float16, _lib.DTYPE_F16)}
KRON_SIDES = [1, 2, 3, 4, 5, 6, 7, 8]
STACK_SIDES = [10, 12, 14, 16, 18, 20, 22, 24, 26, 28, 30, 32, 36, 40, 44, 48, 52, 56, 60, 64]
SEEN = set()                          # dctp_last_kernel() of every call of this module


def maps_per_tile(n):
    if n <= 8:
        return 128 if n in (6, 7, 8) else 256 if n in (2, 4, 5) else 512
    return 32 if n <= 16 else 8 if n <= 32 else 2


def relu_maps(shape, seed, dtype, dead_every=0, device='cuda'):
    g = torch.Generator(device='cpu').manual_seed(seed)
    x = torch.relu(torch.randn(*shape, generator=g)).to(dtype)
    if dead_every:
        x[:, ::dead_every] = 0
    return x.to(device)


def energy64(x):
    """float64 Parseval energy per (image, channel) of the maps as they are (widened exactly)."""
    return (x.double() ** 2).sum((-2, -1))


def score(lib, x, dtype_code, path='auto', c_begin=0, c_count=None, energy=False, stream=None):
    B, C, H, W = x.shape
    c_count = C - c_begin if c_count is None else c_count
    acc = torch.zeros(c_count, dtype=torch.float64, device=x.device)
    en = torch.full((B, c_count), -1.0, dtype=torch.float32, device=x.device) if energy else None
    s = ctypes.c_void_p(stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.dctp_score_accum_ex(_lib.ptr(x), dtype_code, B, H, W, x.stride(0), x.stride(1), x.stride(2), c_begin, c_count,
                                       _lib.ptr(acc), _lib.ptr(en), None, _lib.PATHS[path], s))
    SEEN.add(lib.dctp_last_kernel().decode())
    return acc, en


def fp32_score(lib, x, path='auto', energy=False):
    B, C, H, W = x.shape
    acc = torch.zeros(C, dtype=torch.float64, device=x.device)
    en = torch.full((B, C), -1.0, dtype=torch.float32, device=x.device) if energy else None
    _lib.check(lib.dctp_score_accum(_lib.ptr(x), B, H, W, x.stride(0), x.stride(1), x.stride(2), 0, C, _lib.ptr(acc), _lib.ptr(en),
                                    None, _lib.PATHS[path], _lib.current_stream()))
    return acc, en


def check_energies(en, acc, x):
    want = energy64(x)
    en64 = en.double()
    live = want > 0
    assert (en[~live] == 0).all(), 'dead maps must score exactly 0'
    rel = ((en64 - want).abs() / want.clamp_min(1e-30))[live]
    assert rel.numel() == 0 or rel.max().item() < ENERGY_TOL, rel.max().item()
    torch.testing.assert_close(acc, en64.sum(0), rtol=1e-12, atol=0)


def cases(n):
    """(B, C): one map, one tile, a ragged last tile whose stream ends inside a 32-element row, and more tiles than SMs with
    several turns of every mbarrier ring per CTA."""
    mt = maps_per_tile(n)
    return [(1, 1), (1, mt), (3, (mt * 7) // 3 + 1), (4, (148 * 6 * mt) // 4 + 3)]


@pytest.mark.parametrize('dt', sorted(DTYPES))
@pytest.mark.parametrize('n', KRON_SIDES + STACK_SIDES)
def test_native_energies_match_float64(lib, cuda_device, dt, n):
    torch_dtype, code = DTYPES[dt]
    path = 'kron' if n <= 8 else 'stack'
    for i, (B, C) in enumerate(cases(n)):
        x = relu_maps((B, C, n, n), seed=1000 * n + i, dtype=torch_dtype, dead_every=5)
        acc, en = score(lib, x, code, path=path, energy=True)
        assert ('IN=%s' % ('bf16' if dt == 'bf16' else 'f16')) in lib.dctp_last_kernel().decode()
        check_energies(en, acc, x)
        # the production instantiation (no per-map output; a map's shares reach accum in fp64, not summed in fp32 first) and AUTO
        acc_p, _ = score(lib, x, code, path=path)
        acc_a, _ = score(lib, x, code, path='auto')
        torch.testing.assert_close(acc_p, acc, rtol=1e-6, atol=0)
        torch.testing.assert_close(acc_a, acc_p, rtol=1e-12, atol=0)
        torch.testing.assert_close(acc_p, energy64(x).sum(0), rtol=ENERGY_TOL, atol=0)
        assert (acc_p[energy64(x).sum(0) == 0] == 0).all()


@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_native_matches_fp32_kernel_on_widened_maps(lib, cuda_device, dt):
    """bf16 input drops the X_lo pass, which only adds zeros: the same kernel in fp32 on the widened maps gives the same energies
    (fp16: the same split of the same values)."""
    torch_dtype, code = DTYPES[dt]
    for n in (7, 14, 28, 56):
        x = relu_maps((8, 64, n, n), seed=n, dtype=torch_dtype, dead_every=7)
        acc, en = score(lib, x, code, energy=True)
        acc32, en32 = fp32_score(lib, x.float().contiguous(), energy=True)
        torch.testing.assert_close(en, en32, rtol=2e-6, atol=0)


WIDENED = [
    # (name, shape, path, c_window, row pad)
    ('9x9', (3, 21, 9, 9), 'auto', None, 0),
    ('72x72', (2, 9, 72, 72), 'auto', None, 0),
    ('80x80', (2, 6, 80, 80), 'auto', None, 0),
    ('160x160', (2, 5, 160, 160), 'auto', None, 0),
    ('320x320', (1, 4, 320, 320), 'auto', None, 0),
    ('channel window 28', (4, 24, 28, 28), 'auto', (3, 12), 0),
    ('channel window 7', (4, 30, 7, 7), 'auto', (18, 12), 0),
    ('strided rows 28', (3, 10, 28, 28), 'auto', None, 4),
    ('non-square 12x20', (3, 11, 12, 20), 'auto', None, 0),
    ('forced simt 28', (3, 10, 28, 28), 'simt', None, 0),
    ('forced umma 28', (3, 10, 28, 28), 'umma', None, 0),
    ('forced tmem 56', (3, 10, 56, 56), 'tmem', None, 0),
    ('forced large 96', (2, 5, 96, 96), 'large', None, 0),
]


def widened_input(shape, dtype, pad, seed):
    B, C, H, W = shape
    base = relu_maps((B, C, H, W + pad), seed=seed, dtype=dtype, dead_every=4)
    return base[..., :W] if pad else base


@pytest.mark.parametrize('dt', sorted(DTYPES))
@pytest.mark.parametrize('case', WIDENED, ids=[c[0] for c in WIDENED])
def test_widened_routes_are_bit_identical_to_fp32_entry(lib, cuda_device, dt, case):
    name, shape, path, window, pad = case
    torch_dtype, code = DTYPES[dt]
    x = widened_input(shape, torch_dtype, pad, seed=len(name))
    cb, cc = window if window else (0, shape[1])
    ref_in = x[:, cb:cb + cc].float().contiguous()
    for energy in (False, True):
        acc, en = score(lib, x, code, path=path, c_begin=cb, c_count=cc, energy=energy)
        acc32, en32 = fp32_score(lib, ref_in, path=path, energy=energy)
        assert torch.equal(acc, acc32), name
        if energy:
            assert torch.equal(en, en32), name


@pytest.mark.parametrize('dt', sorted(DTYPES))
def test_two_streams_and_cuda_graph(lib, cuda_device, dt):
    """Widened and native calls on two streams at once, and both inside one captured CUDA graph (the widening scratch is
    allocated on the call's stream)."""
    torch_dtype, code = DTYPES[dt]
    xs = [widened_input((3, 10, 28, 28), torch_dtype, 4, seed=1), relu_maps((2, 6, 80, 80), seed=2, dtype=torch_dtype),
          relu_maps((8, 40, 14, 14), seed=3, dtype=torch_dtype), relu_maps((8, 40, 7, 7), seed=4, dtype=torch_dtype)]
    want = [score(lib, x, code)[0] for x in xs]
    for x in xs:
        _lib.check(lib.dctp_prepare(x.shape[2], x.shape[3]))
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    accs = [torch.zeros(x.shape[1], dtype=torch.float64, device=cuda_device) for x in xs]
    torch.cuda.synchronize()

    def launch(x, acc, stream):
        B, C, H, W = x.shape
        _lib.check(lib.dctp_score_accum_ex(_lib.ptr(x), code, B, H, W, x.stride(0), x.stride(1), x.stride(2), 0, C, _lib.ptr(acc), None,
                                           None, _lib.PATH_AUTO, ctypes.c_void_p(stream.cuda_stream)))
    for rep in range(3):
        for a in accs:
            a.zero_()
        torch.cuda.synchronize()
        for i, (x, a) in enumerate(zip(xs, accs)):
            launch(x, a, s1 if i % 2 == 0 else s2)
        torch.cuda.synchronize()
        for a, w in zip(accs, want):
            torch.testing.assert_close(a, w, rtol=1e-12, atol=0)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for a in accs:
            a.zero_()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            for x, a in zip(xs, accs):
                launch(x, a, s)
    for _ in range(2):
        for a in accs:
            a.zero_()
        g.replay()
        torch.cuda.synchronize()
        for a, w in zip(accs, want):
            torch.testing.assert_close(a, w, rtol=1e-12, atol=0)
    assert lib.dctp_check(None) == 0


def pack_sites(ptrs):
    buf = bytearray()
    for x_ptr, acc_ptr, B, c in ptrs:
        buf += struct.pack('QQii', x_ptr, acc_ptr, B, c)
    return (ctypes.c_char * len(buf)).from_buffer(buf), buf


@pytest.mark.parametrize('dt', sorted(DTYPES))
@pytest.mark.parametrize('side', [7, 14, 28, 56, 9, 80])
@pytest.mark.parametrize('n_sites', [1, 15, 16, 17, 33])
def test_multi_site_matches_one_call_per_site(lib, cuda_device, dt, side, n_sites):
    """Sites in NaN-filled guards, an empty site, one site at an address that is not 16-byte aligned (scored alone); accumulators
    between -0.0 guards.  Native sides take ceil(n / 16) launches as in fp32."""
    torch_dtype, code = DTYPES[dt]
    NN = side * side
    g = torch.Generator().manual_seed(side * 100 + n_sites)
    shapes = [(1 + int(torch.randint(0, 3, (1,), generator=g)), 1 + int(torch.randint(0, 20, (1,), generator=g))) for _ in range(n_sites)]
    if n_sites > 2:
        shapes[1] = (0, 5)                                               # empty site
    unaligned = n_sites - 1 if n_sites > 3 else -1
    GAP = 40                                                             # NaN elements between sites (keeps 16-byte alignment: 80 bytes)
    sizes = [B * c * NN for B, c in shapes]
    offs, o = [], GAP
    for i, sz in enumerate(sizes):
        if i == unaligned:
            o += 1
        offs.append(o)
        o += sz + GAP + (-(sz + GAP)) % 8
    arena = torch.full((o + GAP,), float('nan'), dtype=torch_dtype, device=cuda_device)
    src = [relu_maps((B, c, side, side), seed=i, dtype=torch_dtype, dead_every=3) for i, (B, c) in enumerate(shapes)]
    acc_arena = torch.full((sum(c for _, c in shapes) + 8 * n_sites + 8,), -0.0, dtype=torch.float64, device=cuda_device)
    acc_offs, a = [], 4
    for _, c in shapes:
        acc_offs.append(a)
        a += c + 8
    accs = [acc_arena[ao:ao + c] for ao, (_, c) in zip(acc_offs, shapes)]
    views = [arena[of:of + sz].view(B, c, side, side) for of, sz, (B, c) in zip(offs, sizes, shapes)]
    for acc in accs:
        acc.zero_()
    for v, x in zip(views, src):                                        # filled on the stream right before the launch
        v.copy_(x)
    arr, _keep = pack_sites([(v.data_ptr(), acc.data_ptr(), B, c) for v, acc, (B, c) in zip(views, accs, shapes)])
    n0 = lib.dctp_launch_count()
    _lib.check(lib.dctp_score_accum_multi_ex(arr, n_sites, side, side, code, _lib.current_stream()))
    launches = lib.dctp_launch_count() - n0
    torch.cuda.synchronize()
    assert lib.dctp_check(None) == 0
    guard = torch.ones_like(acc_arena, dtype=torch.bool)
    for ao, (_, c) in zip(acc_offs, shapes):
        guard[ao:ao + c] = False
    assert (torch.signbit(acc_arena[guard]) & (acc_arena[guard] == 0)).all(), 'accumulator guards touched'
    for i, (x, acc) in enumerate(zip(src, accs)):
        if x.numel() == 0:
            assert (acc == 0).all()
            continue
        ref, _ = score(lib, x.contiguous(), code)
        torch.testing.assert_close(acc, ref, rtol=1e-10, atol=0)
        torch.testing.assert_close(acc, energy64(x).sum(0), rtol=ENERGY_TOL, atol=0)
    if side <= 8 or side in STACK_SIDES:
        live = [i for i, (B, c) in enumerate(shapes) if B * c > 0]
        batched = [i for i in live if i != unaligned]
        assert launches == -(-len(batched) // 16) + 2 * (unaligned in live)      # (the unaligned site: widen + fp32 kernel)


@pytest.mark.parametrize('dt', sorted(DTYPES))
@pytest.mark.parametrize('n', [3, 7, 8, 14, 28, 56])
@pytest.mark.parametrize('bad', ['nan', 'inf'])
def test_non_finite_map_changes_only_its_channel(lib, cuda_device, dt, n, bad):
    torch_dtype, code = DTYPES[dt]
    B, C = 4, 48
    x = relu_maps((B, C, n, n), seed=n, dtype=torch_dtype, dead_every=5)
    x[:, 10] = 0
    clean_acc, clean_en = score(lib, x, code, energy=True)
    clean_prod, _ = score(lib, x, code)
    y = x.clone()
    y[2, 11, n // 2, n // 3] = float(bad)
    y[1, 10, 0, 0] = float(bad)                                         # an otherwise dead channel
    for energy in (True, False):
        acc, en = score(lib, y, code, energy=energy)
        ref = clean_acc if energy else clean_prod
        others = torch.ones(C, dtype=torch.bool, device=cuda_device)
        others[10] = others[11] = False
        assert not torch.isfinite(acc[10]) and not torch.isfinite(acc[11])
        # (maps that share MMA lanes with a culprit are recomputed in fp64: equal to the clean run within the energy bar)
        torch.testing.assert_close(acc[others], ref[others], rtol=ENERGY_TOL, atol=0)
        assert (acc[others][ref[others] == 0] == 0).all()
        if energy:
            mask = torch.ones_like(en, dtype=torch.bool)
            mask[2, 11] = mask[1, 10] = False
            assert not torch.isfinite(en[2, 11]) and not torch.isfinite(en[1, 10])
            torch.testing.assert_close(en[mask], clean_en[mask], rtol=ENERGY_TOL, atol=0)
            assert (en[mask][clean_en[mask] == 0] == 0).all()
    assert lib.dctp_check(None) == 0


def test_unknown_dtype_is_invalid(lib, cuda_device):
    x = torch.zeros(1, 1, 8, 8, device=cuda_device)
    acc = torch.zeros(1, dtype=torch.float64, device=cuda_device)
    assert lib.dctp_score_accum_ex(_lib.ptr(x), 3, 1, 8, 8, 64, 64, 8, 0, 1, _lib.ptr(acc), None, None, 0, None) == _lib.E_INVALID
    assert lib.dctp_score_accum_multi_ex(None, 0, 8, 8, -1, None) == _lib.E_INVALID


def test_dct_energy_takes_16bit_tensors(lib, cuda_device):
    from dct_pruning_b200.ops import dct_energy
    for dtype in (torch.bfloat16, torch.float16):
        x = relu_maps((2, 5, 28, 28), seed=9, dtype=dtype)
        acc, en, _ = dct_energy(x, want_energy=True)
        acc32, en32, _ = dct_energy(x.float())
        torch.testing.assert_close(acc, acc32, rtol=2e-6, atol=0)
    with pytest.raises(ValueError):
        dct_energy(torch.zeros(1, 1, 4, 4, dtype=torch.float64, device=cuda_device))


def test_every_16bit_instantiation_ran(lib, cuda_device):
    """Runs last in the module: every stacked-basis (KP, VEC, production / debug) and Kronecker (K2, layout) instantiation of
    both 16-bit types was launched by the tests above."""
    want = set()
    for t in ('bf16', 'f16'):
        for kp, vec in ((16, 4), (16, 2), (32, 4), (32, 2), (48, 4), (64, 4)):
            for cfg in (6, 7):
                want.add('score_stack_kernel<KP=%d,VEC=%d,cfg%d,IN=%s>' % (kp, vec, cfg, t))
        for k2, lay in ((16, 'even'), (64, 'even'), (16, 'odd'), (32, 'odd'), (48, 'odd'), (64, 'odd')):
            want.add('score_kron_kernel<K2=%d,%s,IN=%s>' % (k2, lay, t))
    seen = {s.split(' ')[0] for s in SEEN}
    assert want <= seen, sorted(want - seen)
