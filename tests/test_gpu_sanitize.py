"""compute-sanitizer memcheck over the C-ABI entry points (tools/sanitize_smoke.py, reduced shape set).  Skipped where
compute-sanitizer is not installed or this user may not run it.  racecheck and the full shape set are a manual run
(profiles/README.md, "Sanitizers")."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_memcheck_clean():
    tool = shutil.which("compute-sanitizer") or "/usr/local/cuda/bin/compute-sanitizer"
    if not os.access(tool, os.X_OK):
        pytest.skip("compute-sanitizer not installed or not executable")
    env = dict(os.environ, SANITIZE_ONLY="new")
    out = subprocess.run([tool, "--tool", "memcheck", "--error-exitcode", "17", sys.executable,
                          os.path.join(ROOT, "tools", "sanitize_smoke.py")], capture_output=True, text=True, env=env, timeout=850)
    tail = (out.stdout + out.stderr)[-3000:]
    assert out.returncode == 0, tail
    assert "sanitize smoke ok" in out.stdout, tail
    assert "ERROR SUMMARY: 0 errors" in out.stdout + out.stderr, tail
