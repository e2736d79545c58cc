"""--amp of the importance-generation parser (no GPU needed): default off, the two autocast dtypes, nothing else."""
import pytest
import torch


def test_amp_flag_and_default():
    from dct_pruning_b200.cli import build_parser
    from dct_pruning_b200.generate import AMP_DTYPES
    p = build_parser()
    assert p.parse_args([]).amp == 'off'
    assert p.parse_args(['--amp', 'bf16']).amp == 'bf16'
    assert p.parse_args(['--amp', 'fp16']).amp == 'fp16'
    with pytest.raises(SystemExit):
        p.parse_args(['--amp', 'fp8'])
    assert AMP_DTYPES == {'off': None, 'bf16': torch.bfloat16, 'fp16': torch.float16}
    assert 'reduced-precision' in p.format_help()
