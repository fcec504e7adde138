"""TEST INFRASTRUCTURE: builds the reference's OWN callers of the minimap.h API -- example.c, main.c and the Cython binding mappy
(python/mappy.pyx + cmappy.h) -- UNMODIFIED from /root/reference, against this repository's library (libminimap2_b200.so). Nothing of the
reference is copied into the repository: the sources are compiled where they lie and only the binaries land in oracle/_ref/boundary/
(git-ignored, next to the other reference builds; they find the library through an $ORIGIN-relative rpath, so the built tree can be moved).
The same three callers can be linked against the reference library (oracle/_ref) with --ref, into oracle/_ref/boundary_ref/: that is how
the expected outputs under tests/golden/expected/ were produced (make_boundary_golden.py).

  example          <- example.c        + include/minimap.h (this repo's header)   + libminimap2_b200.so
  minimap2-refmain <- main.c           + the reference's private headers (ketopt.h, mmpriv.h, bseq.h) + libminimap2_b200.so
  mappy*.so        <- python/mappy.pyx (cythonized) + cmappy.h + kseq.h (mappy's FASTX helper, compiled from the reference's header exactly
                      as its setup.py does)                                           + libminimap2_b200.so
"""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
OUT = os.path.join(ROOT, "oracle", "_ref", "boundary")


def build(ref=False):
    if not os.path.exists(os.path.join(REF, "minimap.h")):
        return None
    out = OUT + "_ref" if ref else OUT
    os.makedirs(out, exist_ok=True)
    if ref:
        libdir, lib, inc = os.path.join(ROOT, "oracle", "_ref"), "minimap2_ref", REF
    else:
        libdir, lib, inc = os.path.join(ROOT, "minimap2_b200"), "minimap2_b200", os.path.join(ROOT, "include")
    link = ["-L" + libdir, "-l" + lib, "-Wl,-rpath,$ORIGIN/" + os.path.relpath(libdir, out), "-lz", "-lm", "-lpthread"]
    subprocess.check_call(["gcc", "-O2", "-w", "-I" + inc, "-o", os.path.join(out, "example"), os.path.join(REF, "example.c")] + link)
    subprocess.check_call(["gcc", "-O2", "-w", "-I" + REF, "-o", os.path.join(out, "minimap2-refmain"), os.path.join(REF, "main.c")] + link)
    c = os.path.join(out, "mappy.c")
    subprocess.check_call([sys.executable, "-m", "cython", "-3", "-I" + os.path.join(REF, "python"), os.path.join(REF, "python", "mappy.pyx"), "-o", c])
    shim = os.path.join(out, "kseq_shim.c")
    open(shim, "w").write('#include <zlib.h>\n#include "kseq.h"\nKSEQ_INIT2(, gzFile, gzread)\n')
    ext = sysconfig.get_config_var("EXT_SUFFIX")
    srcs = [c] if ref else [c, shim]  # the reference library already carries its kseq functions (bseq.c)
    subprocess.check_call(["gcc", "-O2", "-w", "-shared", "-fPIC", "-I" + (REF if ref else inc), "-I" + REF, "-I" + os.path.join(REF, "python"),
                           "-I" + sysconfig.get_paths()["include"]] + srcs + ["-o", os.path.join(out, "mappy" + ext)] + link)
    return out


if __name__ == "__main__":
    print(build("--ref" in sys.argv))
