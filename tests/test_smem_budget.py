"""Shared-memory budget of the packed family kernel: at 150 bp reads, 8 single-warp CTAs of classify_kernel<true> must
fit one B200 SM (DESIGN.md §4.1: persistent_ctas caps the kernel at the 8 resident warps per SM it was tuned for).  An
addition to the kernel's static shared memory that silently drops the eighth CTA fails here, without a GPU: the static
bytes come from cuobjdump -res-usage of the built library (which includes the 1 KB the system reserves per block), the
dynamic bytes from the host's formula."""
import os
import re
import shutil
import subprocess

import pytest

from tredparse_b200 import build

SM_SHARED_BYTES = 233472           # shared memory of one sm_100 SM (228 KB)
CTAS_PER_SM = 8


def _cuobjdump():
    for cand in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if cand and os.path.exists(cand):
            return cand
    return None


def dynamic_smem(max_read_len):
    # tredsw_internal_classify: boundary column [rows][32] u32 + codes [rows][32] u8 + 64, rows = max_read_len + 2
    rows_alloc = max_read_len + 2
    return rows_alloc * 32 * 4 + rows_alloc * 32 + 64


def test_eight_packed_ctas_fit_an_sm_at_150bp():
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump not available")
    if not os.path.exists(build.OUT):
        pytest.skip("libtredsw.so not built")
    out = subprocess.run([tool, "-res-usage", build.OUT], capture_output=True, text=True, check=True).stdout
    m = re.search(r"Function \S*classify_kernelILb1E\S*:\s*\n\s*REG:\d+.*?SHARED:(\d+)", out)
    assert m, "classify_kernel<true> not found in cuobjdump -res-usage output"
    static = int(m.group(1))
    per_cta = static + dynamic_smem(150)
    assert CTAS_PER_SM * per_cta <= SM_SHARED_BYTES, (
        "classify_kernel<true> needs {} B per CTA at 150 bp ({} B static incl. the 1 KB reserve): {} CTAs need {} B of "
        "the SM's {} B".format(per_cta, static, CTAS_PER_SM, CTAS_PER_SM * per_cta, SM_SHARED_BYTES))
