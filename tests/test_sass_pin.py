"""The default-schedule column-major search kernels of rows of up to 64 slots (the default full evaluator of the
headline layouts, the kernel bench.py times) are pinned by their SASS (profiles/column_major_sass_pin.json).  Work on
the engine, the host emulation hooks or the build must not perturb them silently — a deliberate change re-pins
them together with new measurements."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_column_major_kernels_are_the_measured_ones():
    pin = json.load(open(os.path.join(ROOT, "profiles", "column_major_sass_pin.json")))
    obj = os.path.join(ROOT, pin["object"])
    if not os.path.exists(obj) or not shutil.which("cuobjdump"):
        pytest.skip("object files of the in-tree build or cuobjdump not available")
    nvcc = subprocess.run(["nvcc", "--version"], capture_output=True, text=True).stdout if shutil.which("nvcc") else ""
    if "12.9" not in nvcc:
        pytest.skip("pinned for nvcc 12.9")
    assert len(pin["kernels"]) == 2
    for k in pin["kernels"]:
        out = subprocess.run(["cuobjdump", "-sass", "-fun", k["mangled"], obj], capture_output=True, text=True, check=True).stdout
        ins = [m.group(1).strip() for m in (re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", l) for l in out.splitlines()) if m]
        assert len(ins) == k["instructions"], k["kernel"]
        assert hashlib.sha256("\n".join(ins).encode()).hexdigest() == k["sha256_of_sass_text"], k["kernel"]
