"""The reference's own pytest suite (tests/python/load_spz_test.py, 26 tests) run UNCHANGED against this
repo's `spz` Python module on the GPU.  The file under tests/golden/ref_suite/ is a byte-identical copy
(the GPU box has no /root/reference); nothing in it is edited, skipped or re-stated here."""
from __future__ import annotations

import hashlib
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUITE = os.path.join(ROOT, "tests", "golden", "ref_suite", "load_spz_test.py")
ORIGINAL = "/root/reference/tests/python/load_spz_test.py"
SHA256 = "31b60e3b58e6b6bd82ef25ba5b342208babc0dd951a0fb93340a89a7715bcdab"


def test_fixture_is_the_unmodified_reference_suite():
    data = open(SUITE, "rb").read()
    assert hashlib.sha256(data).hexdigest() == SHA256
    if os.path.exists(ORIGINAL):
        assert data == open(ORIGINAL, "rb").read()
    assert len(re.findall(rb"^def test_", data, flags=re.M)) == 25  # 26 cases: one is parametrised


def _run_suite(extra_env=None):
    from spz_b200 import build
    build.build_python_module()
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "spz_b200", "pyspz") + os.pathsep + os.environ.get("PYTHONPATH", ""),
               SPZB200_NO_REBUILD="1")
    env.update(extra_env or {})
    # -c /dev/null + --rootdir: the reference's file runs under no conftest / ini of this repo.  --confcutdir: without
    # it pytest takes the ini file's directory (/dev) as the limit and collects down from /, which fails wherever a
    # directory above the checkout cannot be listed
    return subprocess.run([sys.executable, "-m", "pytest", SUITE, "-q", "-p", "no:cacheprovider", "-c", os.devnull,
                           "--rootdir", os.path.dirname(SUITE), "--confcutdir", os.path.dirname(SUITE)],
                          capture_output=True, text=True, env=env, timeout=900, cwd=os.path.dirname(SUITE))


@pytest.mark.gpu
def test_reference_python_suite_passes_unchanged_on_the_gpu():
    r = _run_suite()
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert re.search(r"\b26 passed\b", r.stdout), tail


def test_reference_python_suite_fails_loudly_without_a_gpu():
    """On a box without a CUDA device the suite imports and every codec-independent test passes; the ones
    that need packGaussians / unpackGaussians FAIL (there is no CPU codec to fall back to)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = _run_suite()
    m = re.search(r"(\d+) failed, (\d+) passed", r.stdout)
    assert m, (r.stdout + r.stderr)[-2000:]
    failed, passed = int(m.group(1)), int(m.group(2))
    assert failed + passed == 26 and failed >= 5 and passed >= 10
