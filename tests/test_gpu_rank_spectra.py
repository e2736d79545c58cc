"""rank / rank_sq (rank_jacobi_kernel behind dctp_score_op) against float64 SVDs of maps with constructed spectra.

Every map is built in float64 as U diag(s) V^T (U, V from the QR of a seeded Gaussian) and rounded to fp32.  The reference is
the rank rule applied to the float64 singular values of that exact fp32 matrix, which is what the kernel is given:
cut = s0 * max(H, W) * 2^-23.  A map is well defined when no singular value lies in (cut / 4, 4 * cut); there every
backward-stable SVD gives the same count, so torch's fp32 matrix_rank (the reference hook's rule) must agree with it and the
kernel's value must be identical to it.  Every constructed case is asserted to be well defined: a construction that is not
fails here instead of being skipped.

The families aim at what the kernel's fp32 arithmetic and its stopping rules find hard: large maps whose null vectors are
rounding noise, graded spectra (the skip rule for a vector negligible against its partner), singular values just outside the
factor-4 gap on both sides of the cut, equal clusters, rows and columns scaled over 12 decades, magnitudes from 2^-120 to
2^100, and ReLU-like structure.  The shapes cross every launch threshold of the kernel: lanes per pair, threads per CTA, odd
and even vector counts, several maps per CTA with a ragged last group, and more maps than the grid covers in one pass.
"""
import numpy as np
import pytest
import torch

EPS32 = 2.0 ** -23
GAP = 4.0
NEAR = 4.5            # 'tight' singular values sit this factor from the cut, just outside the factor-4 gap
FAR = 32.0            # ... and the rest of their spectrum at least this factor away

SQUARES = [1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 17, 31, 32, 33, 64, 65, 127, 128, 129, 200, 224, 225]
NON_SQUARE = [(256, 1), (1, 256), (256, 198), (198, 256), (129, 256), (256, 64), (65, 3)]
SHAPES = [(s, s) for s in SQUARES] + NON_SQUARE


# ------------------------------------------------------------------ host side: constructors and the float64 reference

def cut_of(s, H, W):
    """The rank rule's threshold for singular values s (descending) of an H x W map."""
    return s[..., 0] * max(H, W) * EPS32


def ref_rank(a32):
    """Ranks and well-definedness of fp32 maps [..., H, W]: the rule on the float64 singular values of the exact fp32 values."""
    a32 = np.asarray(a32, dtype=np.float32)
    H, W = a32.shape[-2:]
    s = np.linalg.svd(a32.astype(np.float64), compute_uv=False)
    cut = cut_of(s, H, W)[..., None]
    rank = (s > cut).sum(-1)
    defined = ~((s > cut / GAP) & (s < cut * GAP)).any(-1)
    return rank, defined, s


def torch_rank(a32):
    """torch.linalg.matrix_rank in fp32: the rule of the reference hook (oracle/alt_ops_port.py), batched."""
    return torch.linalg.matrix_rank(torch.from_numpy(np.ascontiguousarray(a32, dtype=np.float32))).numpy()


def orthonormal(rng, k, rows, cols):
    """k matrices [rows, cols] with orthonormal columns (cols <= rows), from the QR of a Gaussian."""
    q, r = np.linalg.qr(rng.standard_normal((k, rows, cols)))
    return q * np.sign(np.diagonal(r, axis1=-2, axis2=-1))[..., None, :]


def signed_permutation(rng, k, rows, cols):
    """k matrices [rows, cols] whose columns are distinct signed unit vectors: orthonormal, with one non-zero per column."""
    q = np.zeros((k, rows, cols))
    for i in range(k):
        q[i, rng.permutation(rows)[:cols], np.arange(cols)] = rng.choice([-1.0, 1.0], cols)
    return q


def from_spectrum(rng, sig, H, W, u_perm=False):
    """fp32 maps U diag(sig) V^T for sig [k, min(H, W)] (float64 product, one rounding).  u_perm: U a signed permutation,
    so that every row is one singular value times a row of V^T and fp32 rounds each row relative to its own norm."""
    sig = np.atleast_2d(np.asarray(sig, dtype=np.float64))
    k, n = sig.shape
    u = (signed_permutation if u_perm else orthonormal)(rng, k, H, n)
    v = orthonormal(rng, k, W, n)
    return ((u * sig[:, None, :]) @ v.transpose(0, 2, 1)).astype(np.float32)


def cut_guess(H, W):
    """The cut of a map whose largest singular value is 1 (the fp32 rounding moves it by O(eps), far inside the margins)."""
    return max(H, W) * EPS32


def family_low_rank(rng, H, W):
    n = min(H, W)
    maps = []
    for r in sorted({r for r in (0, 1, 2, n // 2, n - 1, n) if r <= n}):
        sig = np.zeros(n)
        sig[:r] = np.sort(rng.uniform(1.0, 10.0, r))[::-1]
        maps.append(from_spectrum(rng, sig, H, W))
    return np.concatenate(maps)


def family_graded(rng, H, W):
    """s_i = 10^(-i d) from 1 down to 1e-12, with the cut mid-spectrum: the values within NEAR of the cut are moved out to
    NEAR * cut or cut / NEAR (keeping their side), so the spectrum stays graded and the count well defined.  With a
    Gaussian U the fp32 rounding turns the values below ~eps into noise; with a permutation U (rows graded themselves)
    they survive, and the vectors many decades below their partners are the ones the kernel's skip rule leaves alone."""
    n = min(H, W)
    if n < 2:
        return np.zeros((0, H, W), np.float32)
    c = cut_guess(H, W)
    sig = 10.0 ** (-12.0 * np.arange(n) / (n - 1))
    near = (sig > c / NEAR) & (sig < c * NEAR)
    sig[near & (sig >= c)] = c * NEAR
    sig[near & (sig < c)] = c / NEAR
    return np.concatenate([from_spectrum(rng, sig, H, W), from_spectrum(rng, sig, H, W, u_perm=True)])


def family_tight(rng, H, W):
    """One or two singular values at NEAR * cut and cut / NEAR, the rest at >= FAR * cut or zero."""
    n = min(H, W)
    if n < 3:
        return np.zeros((0, H, W), np.float32)
    c = cut_guess(H, W)
    out = []
    for above in (1, n // 3):
        sig = np.zeros(n)
        sig[0] = 1.0
        k = 1
        top = max(1, n // 4)
        sig[k:k + top - 1] = rng.uniform(FAR * c * 4, 1.0, top - 1)
        k = top
        sig[k:k + above] = c * NEAR
        k += above
        if k < n:
            sig[k] = c / NEAR
        out.append(sig)
    return from_spectrum(rng, np.sort(np.array(out), axis=1)[:, ::-1], H, W)


def family_clusters(rng, H, W):
    """All n singular values equal (a scaled orthogonal matrix), and a cluster at 8 * cut under a cluster at 1."""
    n = min(H, W)
    c = cut_guess(H, W)
    sig = [np.full(n, 3.0)]
    if n >= 2:
        s = np.zeros(n)
        s[:max(1, n // 3)] = 1.0
        s[max(1, n // 3):max(2, 2 * n // 3)] = 8.0 * c
        sig.append(s)
    return from_spectrum(rng, np.array(sig), H, W)


def family_scaled(rng, H, W):
    """D1 B D2 with B of spectrum in [1, 2] and the diagonals drawn from three decades-apart levels in 1e-6 .. 1e6: the
    singular values are the level products to within a small factor, all far from the cut, and rows or columns many
    decades below their partners are what the kernel's skip rule leaves alone."""
    n = min(H, W)
    b = from_spectrum(rng, np.sort(rng.uniform(1.0, 2.0, (2, n)), axis=1)[:, ::-1], H, W).astype(np.float64)
    d1 = rng.choice([1e6, 1e4, 1e-6], size=(2, H, 1), p=[0.4, 0.3, 0.3])
    d2 = rng.choice([1e6, 1e-6], size=(2, 1, W), p=[0.6, 0.4])
    d1[:, 0] = 1e6
    d2[:, :, 0] = 1e6
    return (d1 * b * d2 / 1e12).astype(np.float32)


def quantized(a32):
    """The same maps with every entry a multiple of 2^-29: scaling them by 2^k, k >= -120, stays exact (no subnormal rounding)."""
    return (np.round(a32.astype(np.float64) * 2.0 ** 29) * 2.0 ** -29).astype(np.float32)


MAGNITUDES = [-120, -60, 60, 100]


def family_magnitude_base(rng, H, W):
    n = min(H, W)
    sig = np.zeros((2, n))
    sig[0] = rng.uniform(1.0, 10.0, n)
    sig[1, :max(1, n // 2)] = rng.uniform(1.0, 10.0, max(1, n // 2))
    return quantized(from_spectrum(rng, -np.sort(-sig, axis=1), H, W))


def family_relu(rng, H, W):
    """Dead rows and columns in a low-rank map, a single non-zero entry, all entries equal."""
    n = min(H, W)
    out = []
    a = from_spectrum(rng, np.r_[rng.uniform(1.0, 10.0, max(1, n // 2)), np.zeros(n - max(1, n // 2))], H, W)[0]
    a[rng.random(H) < 0.3] = 0.0
    a[:, rng.random(W) < 0.3] = 0.0
    out.append(np.maximum(a, 0.0))
    one = np.zeros((H, W), np.float32)
    one[H // 3, W // 2] = 2.5
    out.append(one)
    out.append(np.full((H, W), 0.75, np.float32))
    return np.stack(out).astype(np.float32)


FAMILIES = {'low_rank': family_low_rank, 'graded': family_graded, 'tight': family_tight, 'clusters': family_clusters,
            'scaled': family_scaled, 'relu': family_relu}


def build_case(H, W, seed=0):
    """Every family for one shape as the channels of one [B, C, H, W] tensor (B = 2 draws), with the family of each channel.
    The magnitude family follows as its own block: base maps, then the base maps scaled by 2^k and by 1e+-30."""
    maps, names = [], []
    for b in range(2):
        rng = np.random.default_rng([H, W, seed, b])
        per = []
        for name, make in FAMILIES.items():
            m = make(rng, H, W)
            per.append(m)
            if b == 0:
                names += [name] * len(m)
        base = family_magnitude_base(rng, H, W)
        per.append(base)
        for k in MAGNITUDES:
            per.append((base.astype(np.float64) * 2.0 ** k).astype(np.float32))
        per.append((base.astype(np.float64) * 1e30).astype(np.float32))
        per.append((base.astype(np.float64) * 1e-30).astype(np.float32))
        if b == 0:
            names += ['mag_base'] * len(base) + ['mag_2^%d' % k for k in MAGNITUDES for _ in base] + \
                     ['mag_1e30'] * len(base) + ['mag_1e-30'] * len(base)
        maps.append(np.concatenate(per))
    return np.stack(maps), names


def rank_launch(H, W, n_maps, sm_count):
    """The launch geometry dctp_score_op picks for the rank op: (lanes per pair L, maps per CTA G, CTAs)."""
    n, m = min(H, W), max(H, W)
    per_map = (n * (m | 1) + n + 1) * 4
    log2L = 0
    while (8 << log2L) < m:
        log2L += 1
    L = 1 << log2L
    workers = (256 if m <= 64 else 512 if m <= 128 else 1024) // L
    wpm = min((n + 1) // 2, workers)
    G = max(1, min(workers // wpm, 64 * 1024 // per_map))
    G = min(G, n_maps)
    return L, G, min(-(-n_maps // G), sm_count * 32)


def test_constructions_are_well_defined_and_torch_agrees():
    """Host only: every constructed spectrum is well defined against float64, the placed singular values are where they were
    put, and torch's fp32 matrix_rank gives the float64 rank.  (Sizes up to 65; the GPU test checks the same at every shape.)"""
    for H, W in [(1, 1), (2, 2), (3, 3), (8, 8), (9, 9), (17, 17), (65, 65), (65, 3), (3, 65), (1, 40)]:
        x, names = build_case(H, W)
        rank, defined, s = ref_rank(x)
        assert defined.all(), (H, W, [names[c] for c in np.nonzero(~defined.all(0))[0]])
        np.testing.assert_array_equal(torch_rank(x), rank)
        names = np.array(names)
        n = min(H, W)
        low = rank[:, names == 'low_rank']
        want = sorted({r for r in (0, 1, 2, n // 2, n - 1, n) if r <= n})
        assert (low == np.array(want)).all(), (H, W, low, want)
        for k in MAGNITUDES:                                          # power-of-two scaling is exact on the quantised maps
            base = x[:, names == 'mag_base'].astype(np.float64)
            np.testing.assert_array_equal(x[:, names == 'mag_2^%d' % k].astype(np.float64) * 2.0 ** -k, base)
        assert (rank[:, names == 'relu'][:, 1:] == 1).all()           # one non-zero entry, all entries equal
        if n >= 3:                                                    # the tight pair brackets the cut at NEAR
            t = s[:, names == 'tight']
            cut = cut_of(t, H, W)[..., None]
            r = t / cut
            assert (np.abs(r - NEAR) < 0.1).any(-1).all() and (np.abs(r - 1 / NEAR) < 0.02).any(-1).all(), r
    L, G, blocks = rank_launch(8, 8, 10 ** 6, 148)
    assert (L, G, blocks) == (1, 64, 148 * 32)


# ------------------------------------------------------------------ the kernel

def rank_call(lib, x, op='rank', c_begin=0, c_count=None, check=True):
    """dctp_score_op(RANK / RANK_SQ) on an fp32 CUDA view [B, C, H, W] with unit column stride.  Values start NaN so a map
    the kernel never reaches shows; returns (accum fp64 [c_count], values fp32 [B, c_count], return code)."""
    from dct_pruning_b200 import _lib
    B, C, H, W = x.shape
    c_count = C - c_begin if c_count is None else c_count
    accum = torch.zeros(c_count, dtype=torch.float64, device=x.device)
    values = torch.full((B, c_count), float('nan'), dtype=torch.float32, device=x.device)
    assert x.stride(3) == 1 or W == 1
    rc = lib.dctp_score_op(_lib.OPS[op], _lib.ptr(x), B, H, W, x.stride(0), x.stride(1), x.stride(2), c_begin, c_count,
                           _lib.ptr(accum), _lib.ptr(values), _lib.current_stream())
    if check:
        _lib.check(rc)
        _lib.check(lib.dctp_check(_lib.current_stream()))
    return accum, values, rc


def launched(lib):
    """(lanes per pair, maps per CTA) of the last rank launch, from the library's own note."""
    text = lib.dctp_last_kernel().decode()
    assert text.startswith('rank_jacobi_kernel'), text
    words = text.split('(')[1].split()
    return int(words[words.index('lanes') - 1]), int(words[words.index('maps') - 1])


def assert_ranks(lib, dev, x, want, what):
    """The kernel's rank and rank_sq of every map of x equal `want` exactly; accum is the batch sum of the values exactly."""
    xd = torch.from_numpy(x).to(dev) if isinstance(x, np.ndarray) else x
    acc, val, _ = rank_call(lib, xd)
    got = val.cpu().numpy()
    bad = np.argwhere(got != want)
    assert bad.size == 0, '%s: %d of %d maps wrong, first (b, c, kernel, float64): %s' % (
        what, len(bad), want.size, [(int(b), int(c), float(got[b, c]), int(want[b, c])) for b, c in bad[:6]])
    np.testing.assert_array_equal(acc.cpu().numpy(), want.sum(0).astype(np.float64))
    acc2, val2, _ = rank_call(lib, xd, op='rank_sq')
    np.testing.assert_array_equal(val2.cpu().numpy(), (want * want).astype(np.float32))
    np.testing.assert_array_equal(acc2.cpu().numpy(), (want.astype(np.float64) ** 2).sum(0))


@pytest.mark.gpu
@pytest.mark.parametrize('H,W', SHAPES, ids=['%dx%d' % s for s in SHAPES])
def test_rank_matches_float64_on_constructed_spectra(lib, cuda_device, H, W):
    x, names = build_case(H, W)
    rank, defined, _ = ref_rank(x)
    assert defined.all(), [names[c] for c in np.nonzero(~defined.all(0))[0]]
    np.testing.assert_array_equal(torch_rank(x), rank)
    names = np.array(names)
    for tag in ['mag_2^%d' % k for k in MAGNITUDES] + ['mag_1e30', 'mag_1e-30']:
        np.testing.assert_array_equal(rank[:, names == tag], rank[:, names == 'mag_base'])
    assert_ranks(lib, cuda_device, x, rank, '%dx%d' % (H, W))
    assert launched(lib)[0] == rank_launch(H, W, 1, 1)[0]               # the shape lists cross every lanes-per-pair step
    xt = x.transpose(0, 1, 3, 2).copy()                            # the other orientation: rows <-> columns as vectors
    assert_ranks(lib, cuda_device, xt, rank, '%dx%d transposed' % (H, W))


@pytest.mark.gpu
@pytest.mark.parametrize('side', [1, 8, 16])
def test_rank_grid_stride_wrap_and_ragged_last_group(lib, cuda_device, side):
    """More maps than G * sm_count * 32 (the grid), and a count that is not a multiple of G: every map is scored once.
    The maps are 512 distinct well-defined ones (ranks 0..side) in a seeded order, so a map scored twice, skipped or
    written to the wrong slot shows."""
    rng = np.random.default_rng(side)
    sm = lib.dctp_sm_count()
    _, G, _ = rank_launch(side, side, 10 ** 9, sm)
    n_maps = G * sm * 32 + 3 * G + G // 2 + 1
    if side == 1:
        pool = np.array([0.0, 1.0, -3.5, 1e-40, -1e-45, 3e38, 2.0 ** -126, 7e-3], np.float32)
        idx = rng.integers(0, len(pool), n_maps)
        x = pool[idx].reshape(-1, 1, 1, 1)
        want = (x != 0).reshape(-1).astype(np.int64)
        x = x.reshape(1, n_maps, 1, 1)
    else:
        sig = np.zeros((512, side))
        r = rng.integers(0, side + 1, 512)
        for i in range(512):
            sig[i, :r[i]] = np.sort(rng.uniform(1.0, 10.0, r[i]))[::-1]
        pool = from_spectrum(rng, sig, side, side)
        prank, defined, _ = ref_rank(pool)
        assert defined.all()
        np.testing.assert_array_equal(prank, r)
        idx = rng.integers(0, 512, n_maps)
        x = pool[idx][None]
        want = prank[idx]
    assert_ranks(lib, cuda_device, x, want.reshape(1, -1), 'side %d, %d maps' % (side, n_maps))
    G = launched(lib)[1]                                            # the case wraps the grid, and has a ragged last group when G > 1
    assert n_maps > G * sm * 32 and (G == 1 or n_maps % G), (n_maps, G)


@pytest.mark.gpu
def test_rank_channel_window_strided_batch_and_cropped_rows(lib, cuda_device):
    x, _ = build_case(129, 256)
    rank, defined, _ = ref_rank(x)
    assert defined.all()
    B, C = rank.shape
    big = torch.full((2 * B, C + 4, 129, 256), float('nan'), device=cuda_device)
    big[::2, 2:C + 2] = torch.from_numpy(x).to(cuda_device)
    acc, val, _ = rank_call(lib, big[::2], c_begin=5, c_count=C - 4)          # batch stride 2 images, maps 3 .. C - 2 of x
    np.testing.assert_array_equal(val.cpu().numpy(), rank[:, 3:C - 1])
    np.testing.assert_array_equal(acc.cpu().numpy(), rank[:, 3:C - 1].sum(0).astype(np.float64))
    for H, W in [(200, 200), (65, 3)]:
        x, _ = build_case(H, W)
        rank, defined, _ = ref_rank(x)
        assert defined.all()
        wide = torch.full(x.shape[:3] + (W + 13,), float('nan'), device=cuda_device)
        wide[..., 7:W + 7] = torch.from_numpy(x).to(cuda_device)
        crop = wide[..., 7:W + 7]                                              # stride_h = W + 13, NaN beside every row
        assert crop.stride(2) > W
        assert_ranks(lib, cuda_device, crop, rank, 'cropped %dx%d' % (H, W))


@pytest.mark.gpu
@pytest.mark.parametrize('side', [8, 16])
def test_rank_non_finite_maps_leave_their_neighbours_alone(lib, cuda_device, side):
    """A map with a NaN and one with an Inf among finite maps of the same CTA: the call returns, dctp_check is clean and the
    finite maps' ranks are those of the float64 reference.  (The non-finite maps' values are not pinned: torch raises on them.)"""
    rng = np.random.default_rng(side + 100)
    sig = np.zeros((40, side))
    for i in range(40):
        sig[i, :i % (side + 1)] = rng.uniform(1.0, 10.0, i % (side + 1))
    x = from_spectrum(rng, -np.sort(-sig, axis=1), side, side)
    rank, defined, _ = ref_rank(x)
    assert defined.all()
    x[5, 2, 3] = np.nan
    x[9, 0, side - 1] = np.inf
    x[17] = np.inf
    finite = np.isfinite(x).all((1, 2))
    _, G, _ = rank_launch(side, side, 40, lib.dctp_sm_count())
    assert G >= 16                                                  # every bad map shares a CTA with finite ones
    _, val, _ = rank_call(lib, torch.from_numpy(x[None]).to(cuda_device))
    got = val.cpu().numpy()[0]
    np.testing.assert_array_equal(got[finite], rank[finite])


@pytest.mark.gpu
def test_rank_shared_memory_acceptance_boundary(lib, cuda_device):
    """A map has to fit in 200 KiB: (n * (m | 1) + n + 1) * 4 bytes for n vectors of length m <= 256."""
    from dct_pruning_b200 import _lib
    for H, W in [(225, 225), (256, 198), (198, 256), (256, 1), (1, 256)]:
        _, _, rc = rank_call(lib, torch.zeros(1, 1, H, W, device=cuda_device))
        assert rc == _lib.OK, (H, W, lib.dctp_last_error())
    for H, W in [(226, 226), (256, 199), (199, 256), (257, 1), (1, 257)]:
        _, _, rc = rank_call(lib, torch.zeros(1, 1, H, W, device=cuda_device), check=False)
        assert rc == _lib.E_UNSUPPORTED, (H, W, rc)
    _lib.check(lib.dctp_check(_lib.current_stream()))
