"""Static SASS guard on the tracker's control flow (CPU only; skips without the built library or the CUDA binary tools).

The tracker kernels and the refine kernel keep every branch around a shuffle, vote or __syncwarp visibly warp-uniform (DESIGN.md §3,
"Warp-uniform control"), so ptxas emits their collectives bare: no BRA.DIV test and no WARPSYNC.COLLECTIVE fallback.  The elimination
step forms its update predicate without a divergent region.  Both properties hang on source details that a small edit can undo
without changing any result, so they are checked on the built library.
"""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import sass_counts  # noqa: E402

PKG = os.path.join(ROOT, "trifocal_pose_estimation_using_improved_gpuhc_b200")
LIB = os.path.join(PKG, "lib", "libhcb200.so")
SRC = os.path.join(PKG, "csrc", "hc_tracker.cu")
HOT_KERNELS = ("hc_track_kernel<false,false,false>", "hc_track_kernel<false,true,false>", "hc_track_kernel<true,false,false>",
               "hc_track_kernel<true,false,true>", "hc_refine_kernel")


def _tool(name):
    for d in (None, os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")):
        p = shutil.which(name, path=d)
        if p:
            return p
    return None


CUOBJDUMP, NVDISASM = _tool("cuobjdump"), _tool("nvdisasm")
pytestmark = pytest.mark.skipif(not os.path.exists(LIB) or CUOBJDUMP is None, reason="needs the built libhcb200.so and cuobjdump")


@pytest.fixture(scope="module")
def counts():
    return sass_counts.sass_counts(LIB, cuobjdump=CUOBJDUMP)


def test_hot_kernels_issue_collectives_without_divergence_fallbacks(counts):
    for k in HOT_KERNELS:
        assert k in counts, "kernel %s not found in %s" % (k, LIB)
        c = counts[k]
        assert c["WARPSYNC.COLLECTIVE"] == 0 and c["BRA.DIV"] == 0, "%s: %s" % (k, c)
        assert c["SHFL"] > 0 and c["CREDUX"] > 0, "%s: the solve's shuffles and REDUX are expected in the kernel: %s" % (k, c)


@pytest.mark.skipif(NVDISASM is None, reason="needs nvdisasm")
def test_elimination_step_has_no_divergent_region(tmp_path):
    """No BSSY of the hot kernels is attributed to the line that forms the elimination step's update predicate (the trifocal build
    uses the branch-free form, HCG_BRANCH_FREE_UPDATE in csrc/hc_problem_gen.h)."""
    with open(SRC) as f:
        lines = [i + 1 for i, l in enumerate(f) if re.search(r"const bool update = active &(?!&)", l)]
    assert len(lines) == 1, lines
    upd_line = lines[0]
    subprocess.run([CUOBJDUMP, "-xelf", "all", LIB], cwd=tmp_path, check=True, capture_output=True)
    cubins = [os.path.join(tmp_path, f) for f in os.listdir(tmp_path) if f.endswith(".cubin")]
    assert cubins
    with_lines = set()
    for cub in cubins:
        dis = subprocess.run([NVDISASM, "-g", "-c", cub], check=True, capture_output=True, text=True).stdout
        kernel, line = None, None
        for l in dis.splitlines():
            m = re.match(r"\s*\.text\.(\S+):", l)
            if m:
                kernel, line = sass_counts.kernel_name(m.group(1)), None
                continue
            m = re.search(r'//## File ".*hc_tracker\.cu", line (\d+)', l)
            if m:
                line = int(m.group(1))
                if kernel in HOT_KERNELS:
                    with_lines.add(kernel)
                continue
            if kernel in HOT_KERNELS and re.search(r"\bBSSY\b", l):
                assert line != upd_line, "%s: BSSY at hc_tracker.cu:%d (elimination-step update predicate)" % (kernel, upd_line)
    assert with_lines == set(HOT_KERNELS), "no hc_tracker.cu line info (-lineinfo) for %s" % (set(HOT_KERNELS) - with_lines)
