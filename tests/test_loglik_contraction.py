"""The log-likelihood evaluators of csrc/loglik.cuh are compiled into factor.cu (multiply-add contraction on) and into
optimize.cu (-fmad=false), and the batched log-likelihood must return the optimiser objective's bits.  So they spell out
every multiply-add.  A probe that calls the small evaluator and chol_group_loglik is compiled both ways (no GPU needed):
the FP64 arithmetic must be the same instruction for instruction class."""
import os
import shutil
import subprocess
import sys

import pytest

from conftest import ROOT

PROBE = os.path.join(ROOT, "tests", "probes", "loglik_contraction_probe.cu")


def _counts(tmp_path, flags):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_summary
    finally:
        sys.path.pop(0)
    cubin = str(tmp_path / ("probe%s.cubin" % "".join(flags).replace("=", "_")))
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-DOPAQUE_LOG", "-cubin",
                    "-o", cubin, PROBE] + flags, check=True)
    return {r["kernel"]: (r["DFMA"], r["DMUL"], r["DADD"]) for r in sass_summary.collect(cubin)}


def test_loglik_evaluators_round_the_same_with_and_without_fmad(tmp_path):
    if shutil.which("nvcc") is None or shutil.which("cuobjdump") is None:
        pytest.skip("nvcc / cuobjdump not on PATH")
    fused = _counts(tmp_path, [])
    plain = _counts(tmp_path, ["-fmad=false"])
    assert set(fused) == {"probe_small", "probe_group"}
    for k in fused:
        assert min(fused[k]) > 0, (k, fused[k])
        assert fused[k] == plain[k], (k, "DFMA/DMUL/DADD with contraction", fused[k], "without", plain[k])
