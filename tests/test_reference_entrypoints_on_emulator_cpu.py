"""CPU: tests/test_gpu_reference_entrypoints.py -- the drop-in packages reproduce what the reference's unmodified
render() / render_post() returned on them (tests/golden/reference_render*.npz) -- executed against the emulation build
of the kernels (H3DGS_EMULATE=1, tests/conftest.py)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_render_and_render_post_run_unmodified_on_the_emulator():
    env = dict(os.environ, H3DGS_EMULATE="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "tests/test_gpu_reference_entrypoints.py", "-q", "-p", "no:cacheprovider"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    tail = r.stdout[-1500:]
    assert r.returncode == 0, tail + r.stderr[-1500:]
    m = re.search(r"(\d+) passed", tail)
    assert m and int(m.group(1)) == 2 and "skipped" not in tail, tail
