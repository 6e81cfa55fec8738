"""The drop-in as a C++ user sees it: a program written against upstream's documented API
(README usage: `avir::CImageResizer<> ImageResizer( 8 ); ImageResizer.resizeImage( ... )`,
`avir::CLancIR`), with only the include changed, in TWO translation units (the front-end is
header-only: it must link from many), against libavirb200.so.  Without a GPU the call throws
(no CPU fallback); on a GPU its output equals upstream's bits."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import avir_b200 as ab
import cases as cs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "dropin")


@pytest.fixture(scope="module")
def program():
    ab.lib()  # (builds libavirb200.so when stale)
    exe = os.path.join(tempfile.mkdtemp(prefix="avirb200_dropin_"), "user")
    libdir = os.path.join(ROOT, "avir_b200")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
           os.path.join(SRC, "user_a.cpp"), os.path.join(SRC, "user_b.cpp"),
           "-L" + libdir, "-lavirb200", "-Wl,-rpath," + libdir, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return exe


@pytest.mark.skipif(ab.device_count() > 0, reason="checks the no-GPU behaviour")
def test_user_program_links_and_fails_loudly_without_gpu(program):
    r = subprocess.run([program], capture_output=True, text=True, timeout=120)
    assert r.returncode == 3, (r.returncode, r.stdout, r.stderr)
    assert "threw:" in r.stdout and "CUDA" in r.stdout


@pytest.mark.gpu
def test_user_program_reproduces_upstream_bits(program, tmp_path):
    case = (0, 640, 480, 1024, 768, 3, np.uint8, np.uint8, 8, {})  # upstream's README example
    src = cs.make_input(case)
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    src.tofile(fin)
    r = subprocess.run([program, fout, fin], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    got = np.fromfile(fout, np.uint8).reshape(768, 1024, 3)
    assert cs.matches_upstream(case, src, got)
