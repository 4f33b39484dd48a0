"""CPU: the built library's hot path really is tcgen05 + TMEM + TMA code (static SASS, cuobjdump), and the
round-2 packed fp32 pairs are in the unmasked cosine sweeps.  Mirrors tools/sass_opcodes.py / profiles/r02_sass_opcodes.txt."""
import collections
import re
import shutil
import subprocess

import pytest


@pytest.fixture(scope="module")
def sass_per_kernel(lib_built):
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    out = subprocess.run(["cuobjdump", "-sass", lib_built], capture_output=True, text=True, check=True).stdout
    per, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = per.setdefault(m.group(1), collections.Counter())
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", line)
        if m and cur is not None:
            cur[m.group(1)] += 1
    return per


def _kernels(per, fragment):
    return {k: v for k, v in per.items() if fragment in k}


def test_sweeps_are_tcgen05_tmem_tma(sass_per_kernel):
    fwd, bwd = _kernels(sass_per_kernel, "tc_fwd_kernel"), _kernels(sass_per_kernel, "tc_bwd_kernel")
    assert len(fwd) >= 8 and len(bwd) >= 8
    for name, ops in {**fwd, **bwd}.items():
        assert ops["UTCHMMA"] >= 16, name          # tcgen05.mma
        assert ops["LDTM"] >= 1 and ops["STTM"] >= 1, name     # tcgen05.ld / st (TMEM)
        assert ops["UTMALDG"] >= 1, name           # cp.async.bulk.tensor (TMA)
        assert ops["SYNCS"] >= 8, name             # mbarrier pipeline
        assert ops["HMMA"] == 0, name              # no legacy mma.sync
    assert sum(sum(o.values()) for o in sass_per_kernel.values()) > 100000
    assert all(o["HMMA"] == 0 for o in sass_per_kernel.values())


def test_unmasked_cosine_sweeps_use_packed_fp32_pairs(sass_per_kernel):
    # mangled template arguments: tc_fwd_kernel<SIM, UNI, MINE, NCH, PLIN>, tc_bwd_kernel<SIM, UNI, MINE, NCH, PLIN>
    fwd_plin = [v for k, v in sass_per_kernel.items() if "tc_fwd_kernelILi0ELb0ELb0ELi2ELb1EE" in k]
    bwd_plin = [v for k, v in sass_per_kernel.items() if "tc_bwd_kernelILi0ELb0ELb0ELi1ELb1EE" in k]
    assert len(fwd_plin) == 1 and len(bwd_plin) == 1
    assert fwd_plin[0]["FFMA2"] >= 32 and fwd_plin[0]["FADD2"] >= 32
    assert bwd_plin[0]["FFMA2"] >= 32 and bwd_plin[0]["FADD2"] >= 32 and bwd_plin[0]["FMUL2"] >= 32
    # the geodesic sweeps keep scalar arithmetic (the acos chain is per element)
    geo = [v for k, v in sass_per_kernel.items() if "tc_fwd_kernelILi1E" in k]
    assert geo and all(v["FFMA2"] == 0 for v in geo)
