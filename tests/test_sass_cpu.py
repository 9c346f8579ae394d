"""The hardware claims of DESIGN.md, checked on the built library itself (cuobjdump works without a GPU): sm_100a only,
TMA tensor loads AND stores in the headline GAE kernels, bulk copies where the docs say so, packed fp32 in the pairwise
quantile sweep -- and no floating-point atomic anywhere (every reduction has a fixed order)."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


@pytest.fixture(scope="module")
def sass():
    from di_hpc_b200 import build
    from tools import sass_opcodes
    if sass_opcodes.cuobjdump() is None:
        pytest.skip("cuobjdump not found (neither on PATH nor in the CUDA toolkit)")
    lib = build.build()
    kernels, atomics, arch = sass_opcodes.parse(lib)
    assert len(kernels) > 100
    return kernels, atomics, arch


def pick(kernels, fragment):
    hit = {k: c for k, c in kernels.items() if fragment in k}
    assert hit, "no kernel matching %r in the library" % fragment
    return hit


def test_only_sm_100a_cubins(sass):
    _, _, arch = sass
    assert arch == {"sm_100a"}, arch


def test_headline_gae_kernels_use_tma_loads_and_tma_stores(sass):
    kernels, _, _ = sass
    for frag in ("gae_fwd_tma_st", "gae_bwd_tma_st"):
        for name, c in pick(kernels, frag).items():
            assert c["UTMALDG"] > 0 and c["UTMASTG"] > 0 and c["SYNCS"] > 0, (name, c["UTMALDG"], c["UTMASTG"])


def test_scan_kernels_of_the_other_ops_use_tma_loads(sass):
    kernels, _, _ = sass
    for frag in ("td_lambda_fwd_tma", "vtrace_scan_tma", "upgo_scan_tma"):
        for name, c in pick(kernels, frag).items():
            assert c["UTMALDG"] > 0, name


def test_c51_lane_kernel_gathers_with_tma_and_stores_in_bulk(sass):
    kernels, _, _ = sass
    for name, c in pick(kernels, "dist_nstep_fwd_lane_kernel").items():
        assert c["UTMALDG"] > 0 and c["UBLKCP"] > 0, (name, dict(c))


def test_backward_scatter_writes_with_bulk_copies(sass):
    kernels, _, _ = sass
    for name, c in pick(kernels, "scatter_rows_bulk_kernel").items():
        assert c["UBLKCP"] > 0 and c["STG"] <= 8, (name, c["UBLKCP"], c["STG"])  # (STG: the tail rows only)


def test_pairwise_quantile_sweep_uses_packed_fp32(sass):
    kernels, _, _ = sass
    assert any(c["FFMA2"] > 0 for c in pick(kernels, "qrdqn_fwd_kernel").values())


def test_no_floating_point_atomics(sass):
    _, atomics, _ = sass
    for name, ops in atomics.items():
        for op in ops:
            assert ".F32" not in op and ".F64" not in op and ".F16" not in op, (name, op)
        # the only kernels with atomics at all are the ticket / done counters of the look-back scans
        assert "lookback" in name, (name, sorted(ops))
