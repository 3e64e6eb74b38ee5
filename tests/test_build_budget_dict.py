"""CPU: budgets of the dictionary-encoded kernels (cg_persist<..., DICT = true>, spmv_tma_kernel<..., DICT = true>),
read from the build artefacts like test_build_budget.py: 3 CTAs of 288 threads per SM (<= 72 registers, no spills),
the gathers of a row issued together, and no Float64 vector read through the non-coherent path in the persistent
kernel (its vectors change between the phases of one launch)."""
import re

import pytest

from test_build_budget import _demangle, _entries, _sass_of


def _longest_gather_run(body):
    best = cur = 0
    for line in body:
        if "LDG.E.64" in line and "STRONG" not in line:
            cur += 1
            best = max(best, cur)
        elif "DMUL" in line or "DADD" in line or "DFMA" in line:
            cur = 0
    return best


@pytest.mark.parametrize("obj,pat,count", [
    ("cg_fused", r"cg_persist<(double|float), [02], 3, 8, true>", 4),
    ("spmv", r"spmv_tma_kernel<(double|float), false, kb::XPlain<(double|float)>, true>", 2),
])
def test_encoded_kernels_fit_three_ctas_per_sm(obj, pat, count):
    ents = _entries(obj)
    dm = _demangle([e[0] for e in ents])
    hit = [(dm[n], r, s) for n, r, s in ents if re.search(pat, dm[n])]
    assert len(hit) == count, hit
    for name, regs, spill in hit:
        assert regs <= 72 and spill == 0, (name, regs, spill)


@pytest.mark.parametrize("obj,mangled", [
    ("cg_fused", "cg_persistIdLi0ELi3ELi8ELb1E"),
    ("cg_fused", "cg_persistIdLi2ELi3ELi8ELb1E"),
    ("spmv", "spmv_tma_kernelIdLb0ENS_6XPlainIdEELb1E"),
])
def test_encoded_gather_batches_keep_loads_in_flight(obj, mangled):
    assert _longest_gather_run(_sass_of(obj, mangled)) >= 6


def test_encoded_persistent_cg_reads_vectors_coherently():
    body = _sass_of("cg_fused", "cg_persistIdLi0ELi3ELi8ELb1E")
    assert not any("LDG.E.64.CONSTANT" in line for line in body), "a Float64 vector is read through the read-only path"


@pytest.mark.parametrize("obj,mangled", [
    ("cg_fused", "cg_persistIdLi0ELi3ELi8E"),
    ("cg_fused", "cg_persistIdLi1ELi3ELi8E"),
    ("cg_fused", "cg_k1_tmaIdLi0ELi3ELb1"),
    ("spmv", "spmv_tma_kernelIdLb0ENS_6XPlain"),
])
def test_existing_patterns_still_name_csr_instantiations(obj, mangled):
    """test_build_budget.py selects kernels by these mangled prefixes: each must still cover a CSR instantiation."""
    from test_build_budget import BUILD
    import os
    import shutil
    import subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not available")
    path = os.path.join(BUILD, obj + ".o")
    if not os.path.exists(path):
        pytest.skip("objects absent: run __graft_entry__.build()")
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    names = [l.split("Function :")[1].strip() for l in sass.splitlines() if "Function :" in l]
    hits = [n for n in names if mangled in n]
    assert hits, mangled
    csr = [n for n in hits if "cg_k1_tma" in n or "ELb0E" in n[n.index(mangled) + len(mangled) - 1:]]
    assert csr, (mangled, hits)
