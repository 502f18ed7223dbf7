"""The opt-in kernel forms kept in the tree as measured alternatives (profiles/r02_experiments.md) must keep compiling for sm_100a
against the current shared pieces (FactorDesc, DoneSignal, accumulate_point_f ...): B2_VGICP_IMPL = 2 (TMA / mbarrier / cp.async
staged), 3 (two launches), 4 (single role).  nvcc cross-compiles without a GPU.  The TMA form's SASS must contain the bulk-copy and
mbarrier instructions its description claims (profiles/r02_v2_sass_excerpt.txt is an excerpt of exactly this object)."""
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

import pytest

from gtsam_points_b200 import build as b2build

CSRC = b2build.CSRC


def _compile(impl, out):
    cmd = [b2build.NVCC] + b2build.NVCC_FLAGS + [f"-DB2_VGICP_IMPL={impl}", "-c", os.path.join(CSRC, "b2_factors.cu"), "-o", out]
    return subprocess.run(cmd, capture_output=True, text=True)


@pytest.mark.skipif(shutil.which(b2build.NVCC) is None and not os.path.exists(b2build.NVCC), reason="nvcc not available")
def test_alternative_kernel_forms_compile_and_the_tma_form_contains_tma(tmp_path):
    impls = (2, 3, 4)
    with ThreadPoolExecutor(len(impls)) as ex:
        results = list(ex.map(lambda i: _compile(i, str(tmp_path / f"factors_impl{i}.o")), impls))
    for impl, r in zip(impls, results):
        assert r.returncode == 0, f"B2_VGICP_IMPL={impl} no longer compiles:\n{r.stderr[-2000:]}"
    cuobjdump = os.path.join(os.path.dirname(b2build.NVCC), "cuobjdump")  # the toolkit's bin/ need not be on PATH
    sass = subprocess.run([cuobjdump, "-sass", str(tmp_path / "factors_impl2.o")], capture_output=True, text=True).stdout
    for mnemonic in ("UBLKCP", "SYNCS.ARRIVE.TRANS64", "SYNCS.PHASECHK.TRANS64.TRYWAIT", "LDGSTS", "USETMAXREG"):
        assert mnemonic in sass, f"{mnemonic} missing from the TMA-staged kernel's SASS"
