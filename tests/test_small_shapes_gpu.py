"""GPU: every kernel on tiny / ragged grids (V not a multiple of 32 or 4, odd channel counts,
heavy collisions, generic fallback, both tail paths) against the CPU oracle.  This is the
bounds-check substitute for compute-sanitizer, which is closed on the build pool."""
import os
import runpy

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_small_and_ragged_shapes(capsys):
    runpy.run_path(os.path.join(ROOT, "tools", "sanitize_small.py"), run_name="__main__")
    assert "ALL OK" in capsys.readouterr().out


def test_streaming_forward_kernel_is_bit_exact_at_every_ring_size():
    """tools/fwd_check.py runs 64-channel volumes of several geometries and batches through the
    two-role streaming kernel with rings of 2, 4, 8 and 16 slots per SM (slots are reused across
    generations) and compares them with the general kernel's bit for bit, three calls each (the
    ring and its barriers are reused)."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fwd_check.py"), "check"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("check ")]
    assert len(lines) >= 7 and all("equal=True" in ln for ln in lines), r.stdout
