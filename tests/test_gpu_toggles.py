"""The pipeline's result must not depend on the host-side hand-over of the clouds nor on where the library's device
blocks come from (the process-wide cache or fresh allocations).  One digest over every exported table, several ways to
get there."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _digest_in_subprocess(env_extra, mode="numpy"):
    env = dict(os.environ)
    env.update(env_extra)
    out = subprocess.run([sys.executable, os.path.join(HERE, "toggle_digest.py"), mode], env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("DIGEST ")][-1]
    return line.split()[1]


def test_handover_modes_agree():
    from toggle_digest import digest

    ref = digest("numpy")
    assert digest("cuda_batches") == ref  # deferred CUDA-tensor inserts handed over two poses at a time
    assert digest("pinned") == ref        # page-locked host arrays through the two upload streams
    assert digest("numpy") == ref         # and again: blocks now come from the process-wide cache


def test_internal_switches_do_not_change_results():
    from toggle_digest import digest

    ref = digest("numpy")
    assert _digest_in_subprocess({"OL_CACHE_BYTES": "0"}) == ref  # no block cache: every device block freshly allocated


def test_release_cached_memory():
    import torch

    import octreelib_b200
    from toggle_digest import digest

    digest("numpy", n_poses=3)
    torch.cuda.synchronize()
    held = octreelib_b200.release_cached_memory()
    assert held > 0                      # the forest's blocks had been parked for the next one
    assert octreelib_b200.release_cached_memory() == 0
    digest("numpy", n_poses=3)           # and everything still works with a cold cache
