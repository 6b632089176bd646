"""compute-sanitizer over a small run of every kernel (scripts/sanitize.py): no
out-of-bounds or misaligned accesses, no shared-memory hazards, no barrier misuse.
The reference has no sanitizer story (single-threaded Python, SURVEY.md section 5)."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("tool", ["memcheck", "racecheck", "synccheck"])
def test_compute_sanitizer_clean(tool):
    exe = shutil.which("compute-sanitizer") or "/usr/local/cuda/bin/compute-sanitizer"
    if not os.access(exe, os.X_OK):
        pytest.skip("compute-sanitizer not installed or not executable")
    res = subprocess.run([exe, "--tool", tool, "--print-limit", "5", sys.executable,
                          os.path.join(ROOT, "scripts", "sanitize.py")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    tail = (res.stdout + res.stderr)[-3000:]
    assert "sanitize run ok" in res.stdout, tail
    assert ("ERROR SUMMARY: 0 errors" in tail) or ("0 hazards displayed (0 errors" in tail), tail
