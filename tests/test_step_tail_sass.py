"""CPU test (no GPU): adding the learned-table payload to the step tail (k_step_tail_embed) leaves the machine code of the
existing tail kernels k_step_tail<false> / k_step_tail<true> (grapes_step_tail, grapes_allreduce_adam_peer) unchanged.
tests/golden/step_tail_sass.json holds the sha256 of their SASS (instructions and encodings, addresses stripped) as the
recorded nvcc release compiles them with the library's flags; another nvcc release may schedule differently, so the
test skips there."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "step_tail_sass.json")


def _tool(name):
    return shutil.which(name) or (f"/usr/local/cuda/bin/{name}" if os.path.isfile(f"/usr/local/cuda/bin/{name}") else None)


def sass_digests(sass: str) -> dict:
    out = {}
    for m in re.finditer(r"Function : (\S+)\n(.*?)(?=\n\s*Function :|\Z)", sass, re.S):
        lines = [re.sub(r"/\*[0-9a-f]{4,}\*/", "", ln).strip() for ln in m.group(2).splitlines()]
        out[m.group(1)] = hashlib.sha256("\n".join(ln for ln in lines if ln).encode()).hexdigest()
    return out


def test_existing_step_tail_kernels_keep_their_sass(tmp_path):
    nvcc, cuobjdump = _tool("nvcc"), _tool("cuobjdump")
    if not nvcc or not cuobjdump:
        pytest.skip("nvcc / cuobjdump not available")
    golden = json.load(open(GOLDEN))
    ver = subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout
    if golden["nvcc"] not in ver:
        pytest.skip(f"SASS recorded with nvcc {golden['nvcc']}")
    from grapes_b200.build import NVCC_FLAGS
    cubin = str(tmp_path / "peer_comm.cubin")
    subprocess.run([nvcc] + NVCC_FLAGS + ["-cubin", "-o", cubin, os.path.join(ROOT, "grapes_b200", "csrc", "peer_comm.cu")],
                   check=True, capture_output=True)
    got = sass_digests(subprocess.run([cuobjdump, "-sass", cubin], check=True, capture_output=True, text=True).stdout)
    for name, digest in golden["functions"].items():
        assert got.get(name) == digest, f"SASS of {name} changed"
    assert "_Z17k_step_tail_embed8TailArgs9EmbedPush" in got
