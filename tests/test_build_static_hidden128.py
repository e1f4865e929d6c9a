"""Static facts about the hidden-size-128 recurrence kernels (no GPU): they use the same Blackwell instructions as the 64 ones,
none of them spills, and their register counts allow the one 256-thread CTA per SM that gru.cu's header comment budgets.
Reads cuobjdump's SASS and ptxas' log through tools/sass_evidence.py; skipped where the CUDA toolkit is absent."""
import shutil
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tools"))

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or shutil.which("c++filt") is None,
                                reason="cuobjdump / c++filt not on PATH")

KERNELS = ("gru_fwd_v2_kernel<128>", "gru_bwd_ring_kernel<128, 4>", "gru_bwd_ring_kernel<128, 8>")
MANGLED = ("gru_fwd_v2_kernelILi128E", "gru_bwd_ring_kernelILi128ELi4E", "gru_bwd_ring_kernelILi128ELi8E")


@pytest.fixture(scope="module")
def facts():
    from multimodalsignal_b200.build import build
    build()
    import sass_evidence
    return sass_evidence.kernel_facts(), sass_evidence.ptxas_facts()


def test_h128_recurrence_kernels_use_packed_fma_and_async_copies(facts):
    k, _ = facts
    for name in KERNELS:
        f = k[name]
        assert f.get("FFMA2 (fma.rn.f32x2)", 0) >= 4 * 96, name        # 96 packed FMAs per step at H = 128, >= 4 unrolled steps
        assert f.get("LDGSTS (cp.async)", 0) >= 8, name


def test_h128_kernels_do_not_spill_and_fit_one_cta_per_sm(facts):
    _, px = facts
    for frag in MANGLED:
        found = [v for n, v in px.items() if frag in n]
        assert len(found) == 1, frag
        v = found[0]
        assert not v.get("spill_stores") and not v.get("spill_loads"), (frag, v)
        assert v["registers"] * 256 <= 65536, (frag, v)            # 2H = 256 threads per CTA, one CTA per SM
    # the multi-row and register-ring kernels are not built at this size
    assert not [n for n in px if "gru_fwd_kernelILi128E" in n or "gru_bwd_kernelILi128E" in n]
