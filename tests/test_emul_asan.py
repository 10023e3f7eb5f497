"""
CPU tier: the kernel sources, compiled for the CPU emulator with AddressSanitizer and -fsanitize=alignment, run every
kernel family once (tests/emul/asan_check.sh + asan_driver.py).  compute-sanitizer is closed on the GPU pool; an
out-of-bounds access to a global buffer or to shared memory, or a misaligned vector access, shows up here instead.  Test infrastructure only -- the package never loads the emulator.
"""
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def test_kernels_under_address_sanitizer(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not installed")
    env = dict(os.environ, TMPDIR=str(tmp_path))
    run = subprocess.run(["bash", os.path.join(HERE, "emul", "asan_check.sh")], capture_output=True, text=True, env=env,
                         timeout=900)
    tail = (run.stdout + run.stderr)[-3000:]
    assert run.returncode == 0, tail
    assert "AddressSanitizer" not in run.stdout + run.stderr, tail
    assert "runtime error:" not in run.stdout + run.stderr, tail        # -fsanitize=alignment: misaligned vector access
    assert "asan run done" in run.stdout, tail
