"""The alternative per-slice scoring ops behind dctp_score_op (SURVEY §8f-3) against their CPU oracle.

    rank / rank_sq   /root/reference/utils/common.py:268  torch.matrix_rank per (image, channel) slice (HRank)
    dct3             /root/reference/utils/common.py:269  dct_3d over [C, H, W] -> cnt_score: one value per image

Bars: ranks are integers - bit-exact wherever the rank is well defined (no singular value within a factor 4 of the cut
`S.max() * max(H, W) * eps`; there every backward-stable SVD gives the same count) and never more than 1 off elsewhere
(LAPACK's divide-and-conquer and a Jacobi SVD may put a singular value that sits ON the cut on different sides of it);
dct3 energies within 1e-4 relative (the north_star tolerance) of the double-precision 3-D transform.
"""
import numpy as np
import pytest
import torch

from dct_pruning_b200 import _lib
from oracle import alt_ops_port as ao

pytestmark = pytest.mark.gpu


def feature_like(B, C, H, W, seed):
    """ReLU conv outputs: rank-deficient in the way real activations are (dead rows/columns, smooth regions)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 3, 2 * H, 2 * W, generator=g)
    w1 = torch.randn(8, 3, 3, 3, generator=g) * 0.3
    w2 = torch.randn(C, 8, 3, 3, generator=g) * 0.2
    y = torch.relu(torch.nn.functional.conv2d(x, w1, padding=1))
    y = torch.relu(torch.nn.functional.conv2d(y, w2, padding=1, stride=2) - 0.5)
    return y.contiguous()


def check_ranks(got, x):
    from oracle import alt_ops_port as ao
    B, C = x.shape[:2]
    want = ao.rank_values(x)
    got = got.cpu().to(torch.int64)
    assert got.shape == want.shape
    exact = off = 0
    for b in range(B):
        for c in range(C):
            if ao.rank_gap(x[b, c]):
                assert int(got[b, c]) == int(want[b, c]), (b, c, int(got[b, c]), int(want[b, c]))
                exact += 1
            else:
                assert abs(int(got[b, c]) - int(want[b, c])) <= 1, (b, c, int(got[b, c]), int(want[b, c]))
                off += int(got[b, c]) != int(want[b, c])
    return exact, off


SIDES = [(1, 1), (2, 2), (3, 3), (4, 4), (7, 7), (8, 8), (14, 14), (16, 16), (28, 28), (32, 32), (56, 56), (64, 64),
         (5, 9), (12, 7), (9, 33)]


@pytest.mark.parametrize('H,W', SIDES)
def test_rank_matches_matrix_rank_on_feature_maps(lib, cuda_device, H, W):
    from dct_pruning_b200.ops import score_op
    x = feature_like(3, 10, H, W, seed=H * 100 + W)
    accum, values = score_op(x.to(cuda_device), 'rank', want_values=True)
    exact, off = check_ranks(values, x)
    assert exact >= 0.5 * x.shape[0] * x.shape[1] or H * W <= 16
    np.testing.assert_array_equal(accum.cpu().numpy(), values.double().sum(0).cpu().numpy())


@pytest.mark.parametrize('side', [112, 144, 224])
def test_rank_large_maps(lib, cuda_device, side):
    from dct_pruning_b200.ops import score_op
    x = feature_like(1, 3, side, side, seed=side)
    _, values = score_op(x.to(cuda_device), 'rank', want_values=True)
    check_ranks(values, x)


def test_rank_constructed_cases(lib, cuda_device):
    """Known answers: zero map, rank-1 outer product, identity, low-rank products, duplicated rows, tiny and huge scales."""
    from dct_pruning_b200.ops import score_op
    g = torch.Generator().manual_seed(5)
    N = 24
    maps, want = [], []
    maps.append(torch.zeros(N, N)); want.append(0)
    maps.append(torch.outer(torch.rand(N, generator=g) + 0.1, torch.rand(N, generator=g) + 0.1)); want.append(1)
    maps.append(torch.eye(N)); want.append(N)
    for r in (2, 5, 11, 23):
        maps.append(torch.randn(N, r, generator=g) @ torch.randn(r, N, generator=g)); want.append(r)
    dup = torch.randn(N, N, generator=g); dup[1::2] = dup[0::2]
    maps.append(dup); want.append(N // 2)
    full = torch.randn(N, N, generator=g)
    maps.append(full * 1e-30); want.append(N)
    maps.append(full * 1e30); want.append(N)
    one = torch.zeros(N, N); one[3, 7] = 2.5
    maps.append(one); want.append(1)
    x = torch.stack(maps)[None].contiguous()                         # [1, C, N, N]
    accum, values = score_op(x.to(cuda_device), 'rank', want_values=True)
    assert [int(v) for v in values[0].cpu()] == want
    from oracle import alt_ops_port as ao
    assert [ao.matrix_rank(m) for m in maps] == want                   # the oracle agrees with the construction
    _, sq = score_op(x.to(cuda_device), 'rank_sq', want_values=True)
    assert [int(v) for v in sq[0].cpu()] == [w * w for w in want]


def test_rank_channel_window_strides_and_accumulation(lib, cuda_device):
    from dct_pruning_b200.ops import score_op
    from oracle import alt_ops_port as ao
    x = feature_like(4, 20, 14, 14, seed=77)
    xd = x.to(cuda_device)
    want = ao.rank_values(x).double()
    gaps = torch.tensor([[ao.rank_gap(x[b, c]) for c in range(20)] for b in range(4)])
    # DenseNet-style window of the last 12 channels
    acc, vals = score_op(xd, 'rank', c_begin=8, c_count=12, want_values=True)
    assert bool(((vals.cpu().double() - want[:, 8:]).abs() <= (~gaps[:, 8:]).double()).all())
    # two batches into one accumulator == one call
    acc2, _ = score_op(xd[:2], 'rank')
    acc2, _ = score_op(xd[2:], 'rank', accum=acc2)
    acc1, _ = score_op(xd, 'rank')
    np.testing.assert_array_equal(acc1.cpu().numpy(), acc2.cpu().numpy())
    # a channel-strided view (every second channel) scores like its contiguous copy
    view = xd[:, ::2]
    a_view, _ = score_op(view, 'rank')
    a_copy, _ = score_op(view.contiguous(), 'rank')
    np.testing.assert_array_equal(a_view.cpu().numpy(), a_copy.cpu().numpy())


@pytest.mark.parametrize('shape', [(2, 16, 8, 8), (3, 64, 14, 14), (2, 24, 32, 32), (2, 12, 56, 56), (1, 6, 160, 160), (2, 5, 9, 13)])
def test_dct3_energy_matches_3d_transform(lib, cuda_device, shape):
    """One value per image: the energy of dct_3d(x[b]) - double-precision scipy dctn, and the fp32 op-for-op hook."""
    from dct_pruning_b200.ops import score_op
    from oracle import alt_ops_port as ao
    from oracle.reference_port import ScoreState
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.relu(torch.randn(*shape, generator=g))
    accum, values = score_op(x.to(cuda_device), 'dct3', want_values=True)
    want = ao.dct3_energy64(x.numpy())
    np.testing.assert_allclose(values.cpu().numpy().astype(np.float64), want, rtol=1e-4)
    assert accum.shape == (1,)
    np.testing.assert_allclose(float(accum[0]), want.sum(), rtol=1e-4)
    accum2, _ = score_op(x.to(cuda_device), 'dct3')                 # without per-image values: the per-channel-sum route
    np.testing.assert_allclose(float(accum2[0]), want.sum(), rtol=1e-4)
    st = ScoreState()
    ao.hook_dct3(st)(None, None, x)
    np.testing.assert_allclose(float(accum[0]) / shape[0], float(st.feature_result[0]), rtol=1e-4)


def test_dct3_calls_on_two_streams_keep_their_own_scratch(lib, cuda_device):
    """A long dct3 call on one stream and a short one on a second stream, issued back to back with no synchronisation: both
    equal float64.  The 24x20 maps take the CUDA-core kernel, which leaves room on the SMs for the short call to run while
    the long one is still accumulating; with scratch shared between calls, the short call's memset and sums land in the
    long call's partial sums.  Both routes: per-channel sums (no per-image values) and per-image energies."""
    from dct_pruning_b200.ops import score_op
    g = torch.Generator().manual_seed(11)
    big = torch.rand(128, 816, 24, 20, generator=g)                  # 200 MB
    small = torch.rand(2, 4, 24, 20, generator=g)
    want_big = big.double().square().sum((1, 2, 3)).numpy()            # Parseval: the orthonormal 3-D DCT keeps the sum of squares
    want_small = ao.dct3_energy64(small.numpy())
    xb, xs = big.to(cuda_device), small.to(cuda_device)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for want_values in (False, True):
        acc1 = torch.zeros(1, dtype=torch.float64, device=cuda_device)
        acc2 = torch.zeros(1, dtype=torch.float64, device=cuda_device)
        torch.cuda.synchronize()
        with torch.cuda.stream(s1):
            _, v1 = score_op(xb, 'dct3', accum=acc1, want_values=want_values, check=False)
        with torch.cuda.stream(s2):
            _, v2 = score_op(xs, 'dct3', accum=acc2, want_values=want_values, check=False)
        torch.cuda.synchronize()
        _lib.check(lib.dctp_check(None))
        np.testing.assert_allclose(float(acc1[0]), want_big.sum(), rtol=1e-4, err_msg='long call, values=%s' % want_values)
        np.testing.assert_allclose(float(acc2[0]), want_small.sum(), rtol=1e-4, err_msg='short call, values=%s' % want_values)
        if want_values:
            np.testing.assert_allclose(v1.cpu().numpy(), want_big, rtol=1e-4)
            np.testing.assert_allclose(v2.cpu().numpy(), want_small, rtol=1e-4)


def test_dct3_captured_in_a_cuda_graph(lib, cuda_device):
    """Both dct3 routes captured into one CUDA graph (the scratch is allocated and freed inside it) and replayed with two
    different inputs: each replay equals float64."""
    g = torch.Generator().manual_seed(12)
    x = torch.rand(4, 16, 14, 14, generator=g).to(cuda_device)
    acc_sum = torch.zeros(1, dtype=torch.float64, device=cuda_device)
    acc_val = torch.zeros(1, dtype=torch.float64, device=cuda_device)
    vals = torch.zeros(4, dtype=torch.float32, device=cuda_device)

    def both():
        for acc, out in ((acc_sum, None), (acc_val, vals)):
            _lib.check(lib.dctp_score_op(_lib.OP_DCT3, _lib.ptr(x), 4, 14, 14, x.stride(0), x.stride(1), x.stride(2), 0, 16,
                                         _lib.ptr(acc), _lib.ptr(out), _lib.current_stream()))

    both()                                                           # bases uploaded and kernels loaded outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        both()
    for seed in (1, 2):
        new = torch.relu(torch.randn(4, 16, 14, 14, generator=torch.Generator().manual_seed(seed)))
        x.copy_(new)
        acc_sum.zero_()
        acc_val.zero_()
        vals.fill_(float('nan'))
        graph.replay()
        torch.cuda.synchronize()
        _lib.check(lib.dctp_check(None))
        want = ao.dct3_energy64(new.numpy())
        np.testing.assert_allclose(vals.cpu().numpy(), want, rtol=1e-4)
        np.testing.assert_allclose(float(acc_sum[0]), want.sum(), rtol=1e-4)
        np.testing.assert_allclose(float(acc_val[0]), want.sum(), rtol=1e-4)


@pytest.mark.parametrize('op', ['rank', 'rank_sq', 'dct3'])
def test_session_with_alternative_op_matches_oracle_hooks(lib, cuda_device, op):
    """ScoreSession(op=...) on ResNet-56: the same hooked activations through the oracle hook and through the kernels."""
    from dct_pruning_b200.generate import synthetic_batches
    from dct_pruning_b200.hooks import ScoreSession
    from dct_pruning_b200.sites import resolve_module
    from dct_pruning_b200.zoo import get_network
    from oracle import alt_ops_port as ao
    from oracle.reference_port import ScoreState
    torch.manual_seed(0)
    net = get_network('resnet_56').eval()
    all_sites = ScoreSession(net, 'resnet_56').sites
    sites = all_sites[:3] + all_sites[20:22] + all_sites[-3:]       # 32x32, 16x16 and 8x8 stages (the oracle's SVDs are slow)
    session = ScoreSession(net, 'resnet_56', op=op, sites=sites)
    states = [ScoreState() for _ in sites]
    make = {'rank': lambda st: ao.hook_rank(st), 'rank_sq': lambda st: ao.hook_rank(st, through_cnt_score=True), 'dct3': ao.hook_dct3}[op]
    oracle_hooks = [make(st) for st in states]
    gap_ok = []
    handles = []
    for idx, site in enumerate(sites):
        def both(module, inputs, output, idx=idx):
            oracle_hooks[idx](module, inputs, output)
            if op != 'dct3':
                gap_ok.append((idx, torch.tensor([all(ao.rank_gap(output[b, c]) for b in range(output.shape[0]))
                                                  for c in range(output.shape[1])])))
            session.score(idx, output.to(cuda_device))
        handles.append(resolve_module(net, site.module).register_forward_hook(both))
    with torch.no_grad():
        for x, _ in synthetic_batches(2, 32, 1):
            net(x)
    for h in handles:
        h.remove()
    got = session.finalize()
    ok_of = dict(gap_ok)
    for idx, (site, st) in enumerate(zip(sites, states)):
        w = st.feature_result.numpy().astype(np.float64)
        g = got[site.files[0].stem].astype(np.float64)
        assert g.shape == w.shape, (site.module, g.shape, w.shape)
        if op == 'dct3':
            assert g.shape == (1,)
            np.testing.assert_allclose(g, w, rtol=1e-4)
        else:
            ok = ok_of[idx].numpy()
            np.testing.assert_array_equal(g[ok], w[ok])              # well-defined ranks: identical means
            assert ok.sum() >= 0.5 * ok.size
            slack = (2 * 32 + 1) / 2.0 if op == 'rank_sq' else 0.5   # one slice of the batch of 2 one rank off
            assert np.abs(g - w).max() <= slack * 2


def test_rank_op_refuses_maps_that_do_not_fit(lib, cuda_device):
    from dct_pruning_b200 import _lib
    from dct_pruning_b200.ops import score_op
    x = torch.zeros(1, 1, 320, 320, device=cuda_device)
    with pytest.raises(_lib.DctpError) as e:
        score_op(x, 'rank')
    assert e.value.code == _lib.E_UNSUPPORTED
