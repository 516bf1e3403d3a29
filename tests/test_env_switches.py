"""The environment variables the library reads are a fixed, documented set.  A faster kernel form is measured against the
old one behind an `LTX_*` switch; once it wins, the switch and the old form go, so the hot path keeps one form to maintain.
A new switch has to be named here, with the reason it stays."""
import glob
import os
import re

from helpers import ROOT

CSRC = os.path.join(ROOT, "ltx-video-swift-mlx_b200", "csrc")

ALLOWED = {
    "LTX_CONV_PAIR": "tests run the convolution with one CTA per tile as the reference for the CTA-pair form",
    "LTX_CONV_SLAB": "tests run the convolution with per-tap stages as the reference for the slab form",
    "LTX_ATT_PAIR": "tests run attention with one CTA per query tile as the reference for the CTA-pair form",
    "LTX_P2P": "tests/dist_check.py runs the multi-GPU paths with and without peer memory",
    "LTX_GRAPH": "eager steps instead of CUDA-graph replay, for per-launch profiles",
    "LTX_BATCHED_CFG": "mirrors the disable_batched_cfg option of the denoise loops",
    "LTX_PDL": "launches without programmatic dependent launch, to diagnose kernel ordering",
    "LTX_PDL_MASK": "PDL per kernel class, to diagnose kernel ordering",
    "LTX_GEMM_FORCE_BN": "tile width / kernel of ltx_op_gemm_resid, for tools/gemm_bench.py's sweeps",
}


def sources():
    paths = []
    for ext in ("cu", "cuh", "h"):
        paths += glob.glob(os.path.join(CSRC, f"*.{ext}"))
    assert paths, CSRC
    return {os.path.basename(p): open(p).read() for p in sorted(paths)}


def test_env_reads_are_the_allowed_set():
    found = {}
    for name, src in sources().items():
        assert len(re.findall(r"getenv\s*\(", src)) == len(re.findall(r'getenv\s*\(\s*"LTX_[A-Z0-9_]+"\s*\)', src)), \
            f"{name}: getenv with an argument other than a literal LTX_* name"
        for var in re.findall(r'getenv\s*\(\s*"(LTX_[A-Z0-9_]+)"\s*\)', src):
            found.setdefault(var, []).append(name)
    assert set(found) == set(ALLOWED), (f"not allowed: {sorted(set(found) - set(ALLOWED))}; "
                                        f"no longer read: {sorted(set(ALLOWED) - set(found))}")


def test_gemm_dispatch_reads_no_switch():
    # launch_gemm runs hundreds of times per step on the un-graphed path; the width override is read by the diagnostic op
    src = sources()
    assert "LTX_GEMM_FORCE_BN" not in src["gemm.cu"]
    assert re.search(r'getenv\s*\(\s*"LTX_GEMM_FORCE_BN"', src["api.cu"])
