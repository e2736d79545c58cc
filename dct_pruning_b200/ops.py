"""Functional face of the C ABI for callers that hold a CUDA tensor rather than a hooked net."""
import torch

from . import _lib


def dct_energy(x, c_begin=0, c_count=None, path='auto', accum=None, want_energy=False, want_coeff=False, check=True):
    """Per-channel sum over the batch of the orthonormal 2-D DCT-II energy of x[b, c] (what
    get_feature_hook computes before its running mean, /root/reference/utils/common.py:262-274).

    x: CUDA fp32, bf16 or fp16 [B, C, H, W] (16-bit: an autocast forward's activations; the energies are those of the values x
    holds, computed as for fp32).  Returns (accum fp64 [c_count], energies fp32 [B, c_count] or None, coefficients fp32
    [B, c_count, H, W] or None)."""
    if not x.is_cuda:
        raise RuntimeError('dct_energy runs on CUDA only; there is no CPU fallback')
    dtype = _lib.dtype_code(x.dtype)
    if dtype is None or x.dim() != 4:
        raise ValueError('expected an fp32, bf16 or fp16 NCHW tensor')
    if x.stride(3) != 1 or x.stride(2) < x.shape[3]:
        x = x.contiguous()
    lib = _lib.load()
    B, C, H, W = x.shape
    c_count = C - c_begin if c_count is None else c_count
    if c_begin < 0 or c_count < 0 or c_begin + c_count > C:
        raise ValueError('channel window [%d, %d) outside 0..%d' % (c_begin, c_begin + c_count, C))
    with torch.cuda.device(x.device):
        _lib.check(lib.dctp_init())
        if accum is None:
            accum = torch.zeros(c_count, dtype=torch.float64, device=x.device)
        energy = torch.empty(B, c_count, dtype=torch.float32, device=x.device) if want_energy else None
        coeff = torch.empty(B, c_count, H, W, dtype=torch.float32, device=x.device) if want_coeff else None
        code = _lib.PATHS[path] if isinstance(path, str) else int(path)
        _lib.check(lib.dctp_score_accum_ex(_lib.ptr(x), dtype, B, H, W, x.stride(0), x.stride(1), x.stride(2), c_begin, c_count,
                                           _lib.ptr(accum), _lib.ptr(energy), _lib.ptr(coeff), code, _lib.current_stream()))
        if check:
            _lib.check(lib.dctp_check(_lib.current_stream()))
    return accum, energy, coeff


def finalize(accum, n_images):
    lib = _lib.load()
    out = torch.empty(accum.numel(), dtype=torch.float32, device=accum.device)
    with torch.cuda.device(accum.device):
        _lib.check(lib.dctp_finalize(_lib.ptr(accum), float(n_images), _lib.ptr(out), accum.numel(), _lib.current_stream()))
    return out


def score_op(x, op, c_begin=0, c_count=None, accum=None, want_values=False, check=True):
    """The alternative per-slice reductions of get_feature_hook behind the same boundary (dctp_score_op):
    op = 'dct2' (/root/reference/utils/common.py:267), 'rank' (:268, torch.matrix_rank per slice: HRank), 'rank_sq' (:268
    followed by the unchanged cnt_score, which squares), 'dct3' (:269, dct_3d over [C,H,W]: ONE value per image).

    x: CUDA fp32 [B, C, H, W].  Returns (accum fp64 [c_count] - [1] for 'dct3' -, values fp32 [B, c_count] - [B] for 'dct3' -
    or None): sums over the batch, and the per-slice (per-image) values."""
    if not x.is_cuda:
        raise RuntimeError('score_op runs on CUDA only; there is no CPU fallback')
    if x.dtype != torch.float32 or x.dim() != 4:
        raise ValueError('expected an fp32 NCHW tensor')
    if op not in _lib.OPS:
        raise ValueError('unknown scoring op %r' % (op,))
    if x.stride(3) != 1 or x.stride(2) < x.shape[3]:
        x = x.contiguous()
    lib = _lib.load()
    B, C, H, W = x.shape
    c_count = C - c_begin if c_count is None else c_count
    if c_begin < 0 or c_count < 0 or c_begin + c_count > C:
        raise ValueError('channel window [%d, %d) outside 0..%d' % (c_begin, c_begin + c_count, C))
    with torch.cuda.device(x.device):
        _lib.check(lib.dctp_init())
        if accum is None:
            accum = torch.zeros(1 if op == 'dct3' else c_count, dtype=torch.float64, device=x.device)
        values = None
        if want_values:
            values = torch.empty((B,) if op == 'dct3' else (B, c_count), dtype=torch.float32, device=x.device)
        _lib.check(lib.dctp_score_op(_lib.OPS[op], _lib.ptr(x), B, H, W, x.stride(0), x.stride(1), x.stride(2), c_begin, c_count,
                                     _lib.ptr(accum), _lib.ptr(values), _lib.current_stream()))
        if check:
            _lib.check(lib.dctp_check(_lib.current_stream()))
    return accum, values
