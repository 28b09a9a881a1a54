"""bench.py reports `roofline.traffic` from profiles/k2_traffic.json (DRAM bytes of the C2 votes launch from a committed
`ncu --set full` capture) while s2d_version() equals the capture's lib_version. This test backs that rule: as long as the
version is unchanged, the benchmarked kernel in the built library must compile to the same SASS as the kernel the capture
was taken on. tests/golden/k2_traffic_kernel.sass.gz holds that SASS (instructions without their encodings), made with
tools/sass_same.sh's compile of the capture commit's point_votes.cu by nvcc 12.9 for sm_100a. Needs cuobjdump and the built
library."""
import gzip
import json
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _instructions(sass_text):
    """the instruction lines of `cuobjdump -sass` output, encodings dropped and blanks collapsed"""
    return [" ".join(re.sub(r"/\* 0x[0-9a-f]* \*/", "", ln).split())
            for ln in sass_text.splitlines() if re.match(r"^\s+/\*[0-9a-f]{4}\*/", ln)]


def test_traffic_capture_matches_the_built_kernel():
    tj = json.load(open(os.path.join(ROOT, "profiles", "k2_traffic.json")))
    src = open(os.path.join(ROOT, "s2d_b200", "csrc", "capi.cu")).read()
    version = int(re.search(r"s2d_version\(void\)\s*\{\s*return\s+(\d+)\s*;", src).group(1))
    if version != int(tj["lib_version"]):
        pytest.skip("library version differs from the capture's: bench.py reports no traffic figure")
    lib = os.path.join(ROOT, "s2d_b200", "libs2d_b200.so")
    if not (shutil.which("cuobjdump") and os.path.exists(lib)):
        pytest.skip("needs cuobjdump and the built library")
    with gzip.open(os.path.join(ROOT, "tests", "golden", "k2_traffic_kernel.sass.gz"), "rt") as f:
        want = f.read().splitlines()
    r = subprocess.run(["cuobjdump", "-sass", "-fun", tj["kernel_symbol"], lib], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    got = _instructions(r.stdout)
    assert len(want) > 1000 and got, (len(want), len(got))
    first = next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), min(len(got), len(want)))
    assert got == want, (f"{tj['kernel_symbol']}: {len(got)} instructions built, {len(want)} captured; first difference at "
                         f"line {first}: {got[first:first + 1]} vs {want[first:first + 1]}")
