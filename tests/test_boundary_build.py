"""CPU: the reference's own callers (example.c, main.c, mappy) build and link against libminimap2_b200.so -- every symbol they need is
exported (the run itself needs a GPU: tests/test_gpu_boundary.py). The binaries are the ones build() leaves in oracle/_ref/boundary."""
import os
import subprocess
import sys
import pytest
import oracle_lib as O

sys.path.insert(0, os.path.join(O.ROOT, "tests", "boundary"))
import build_boundary  # noqa: E402


@pytest.mark.skipif(not os.path.exists(os.path.join(build_boundary.OUT, "example")), reason="oracle/_ref/boundary not built")
def test_reference_callers_link_against_this_library():
    d = build_boundary.OUT
    for f in ("example", "minimap2-refmain"):
        out = subprocess.run(["ldd", os.path.join(d, f)], stdout=subprocess.PIPE).stdout.decode()
        assert "libminimap2_b200.so" in out and "not found" not in out, out
    exts = [f for f in os.listdir(d) if f.startswith("mappy") and f.endswith(".so")]
    assert exts
    undefined = subprocess.run(["ldd", "-r", os.path.join(d, exts[0])], stdout=subprocess.PIPE, stderr=subprocess.STDOUT).stdout.decode()
    assert "libminimap2_b200.so" in undefined
    assert not [l for l in undefined.splitlines() if "undefined symbol" in l and ("mm_" in l or "kseq" in l or "seq_comp" in l)], undefined
    # without a GPU the library refuses loudly instead of falling back to anything
    p = subprocess.run([os.path.join(d, "example"), "MT-human.fa", "MT-orang.fa"], cwd=os.path.join(O.ROOT, "tests", "golden", "data"), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    import ctypes
    try:
        has_gpu = ctypes.CDLL("libcuda.so.1").cuInit(0) == 0
    except OSError:
        has_gpu = False
    if not has_gpu:
        assert p.returncode != 0 and b"no CPU" in p.stderr
