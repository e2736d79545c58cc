"""The kernel headers stand on their own: each compiles as the only include of a translation unit, and no kernel header
reaches into another kernel's file (what they share lives in score_common.cuh)."""
import glob
import os
import re
import shutil
import subprocess

import pytest

from conftest import REPO

CSRC = os.path.join(REPO, 'dct_pruning_b200', 'csrc')
HEADERS = sorted(os.path.basename(p) for p in glob.glob(os.path.join(CSRC, '*.cuh')))


def nvcc():
    from dct_pruning_b200.build import find_nvcc
    cand = find_nvcc()
    return cand if os.path.exists(cand) or shutil.which(cand) else None


@pytest.mark.parametrize('header', HEADERS)
def test_header_compiles_alone(header, tmp_path):
    exe = nvcc()
    if exe is None:
        pytest.skip('nvcc not found')
    tu = tmp_path / 'only.cu'
    tu.write_text('#include "%s"\n' % os.path.join(CSRC, header))
    proc = subprocess.run([exe, '-gencode', 'arch=compute_100a,code=sm_100a', '-std=c++17', '-c', str(tu), '-o', str(tmp_path / 'only.o')],
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert proc.returncode == 0, proc.stdout


def test_no_kernel_header_includes_another():
    assert 'score_common.cuh' in HEADERS
    for header in HEADERS:
        text = open(os.path.join(CSRC, header)).read()
        included = re.findall(r'#include\s+"(score_\w+\.cuh)"', text)
        assert all(inc == 'score_common.cuh' for inc in included), (header, included)
