"""Static check of the built libapgp.so (cuobjdump, no GPU): the cluster log-likelihood kernel with gradients runs its
products on the FP64 tensor pipe (DMMA), feeds them by bulk TMA (UBLKCP) behind mbarriers (SYNCS), meets at cluster
barriers between its phases (CGABAR) and keeps everything in registers (no local memory)."""
import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_loglik_grad_group_kernel_has_dmma_bulk_tma_and_no_spills():
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    lib = os.path.join(ROOT, "approxposterior_b200", "libapgp.so")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_summary
    finally:
        sys.path.pop(0)
    rows = {r["kernel"]: r for r in sass_summary.collect(lib)}
    r = rows["loglik_grad_group_kernel"]
    assert r["local"] == 0, r
    # the factorisation's own DMMA / UBLKCP come with chol_group_loglik: the gradient phases add to them
    base = rows["loglik_group_kernel"]
    assert r["DMMA"] > base["DMMA"] and r["UBLKCP"] > base["UBLKCP"] and r["SYNCS"] > base["SYNCS"], (r, base)
    assert r["CGABAR"] > 0, r
