"""CPU tests of the drop-in boundary: libminimap2_b200.so loads without a GPU, exports every symbol that include/minimap.h
and include/mm_b200.h declare, and the public structs have the reference's layout (sizes/offsets checked against the
reference build through oracle/_ref when it is present, and against pinned numbers otherwise)."""
import ctypes as C
import os
import re
import pytest
import oracle_lib as O

ROOT = O.ROOT
LIB = os.path.join(ROOT, "minimap2_b200", "libminimap2_b200.so")


def declared_functions(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    txt = re.sub(r"//[^\n]*", "", txt)
    names = set()
    for m in re.finditer(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\([^;{]*\)\s*;", txt):
        n = m.group(1)
        if n.startswith("mm_") or n.startswith("mmb_"):
            names.add(n)
    return names


@pytest.mark.skipif(not os.path.exists(LIB), reason="library not built")
def test_library_exports_every_declared_symbol():
    L = C.CDLL(LIB)  # must load on a machine without a GPU (no CUDA call at load time)
    missing = []
    for hdr in ("minimap.h", "mm_b200.h"):
        for fn in sorted(declared_functions(hdr)):
            if not hasattr(L, fn):
                missing.append("%s:%s" % (hdr, fn))
    assert not missing, missing
    for g in ("mm_verbose", "mm_dbg_flag", "mm_realtime0"):
        C.c_int.in_dll(L, g)


@pytest.mark.skipif(not os.path.exists(LIB), reason="library not built")
def test_options_match_reference_presets():
    """mm_set_opt / mm_check_opt: same values as the reference for every preset (byte comparison of the option structs)"""
    from minimap2_b200 import api
    L = C.CDLL(LIB)
    L.mm_set_opt.argtypes = [C.c_char_p, C.POINTER(api.IdxOpt), C.POINTER(api.MapOpt)]
    presets = [None, "map-ont", "lr", "ava-ont", "map-pb", "map10k", "ava-pb", "map-hifi", "map-ccs", "lr:hq", "lr:hqae", "map-iclr",
               "map-iclr-prerender", "asm5", "asm10", "asm20", "sr", "short", "splice", "splice:hq", "splice:sr", "cdna"]

    def set_opt(lib_, p):
        io, mo = api.IdxOpt(), api.MapOpt()
        lib_.mm_set_opt(None, C.byref(io), C.byref(mo))
        if p is not None:
            assert lib_.mm_set_opt(p.encode(), C.byref(io), C.byref(mo)) == 0
        return [bytes(io).hex(), bytes(mo).hex()]

    def produce():
        R = O.ref()
        R.mm_set_opt.argtypes = [C.c_char_p, C.POINTER(api.IdxOpt), C.POINTER(api.MapOpt)]
        return [set_opt(R, p) for p in presets]
    ref = O.recorded(["mm_set_opt"] + [str(p) for p in presets], produce)
    for p, r in zip(presets, ref):
        io, mo = set_opt(L, p)
        assert io == r[0], p
        assert mo == r[1], p
    io, mo = api.IdxOpt(), api.MapOpt()
    assert L.mm_set_opt(b"no-such-preset", C.byref(io), C.byref(mo)) == -1
    assert L.mm_set_opt(b"asm7", C.byref(io), C.byref(mo)) == -1


def test_struct_layouts():
    from minimap2_b200 import api
    assert C.sizeof(api.Reg1) == 80 and C.sizeof(api.Extra) == 28 and C.sizeof(api.IdxOpt) == 24
    assert C.sizeof(api.Idx) == 96 and C.sizeof(api.MapOpt) == 264 and C.sizeof(api.IdxSeq) == 24
    if O.have_ref():
        R = O.ref()
        assert R.refshim_sizeof_reg1() == C.sizeof(api.Reg1)
        assert R.refshim_sizeof_extra() == C.sizeof(api.Extra)
        assert R.refshim_sizeof_idxopt() == C.sizeof(api.IdxOpt)
        assert R.refshim_sizeof_idx() == C.sizeof(api.Idx)
        assert R.refshim_sizeof_mapopt() == C.sizeof(api.MapOpt)


@pytest.mark.skipif(not os.path.exists(LIB), reason="library not built")
def test_no_gpu_fails_loudly():
    """Without a CUDA device the product must refuse to run (no CPU fallback): mmb_ctx_create returns NULL."""
    import subprocess, sys
    code = ("import ctypes as C; L=C.CDLL(%r); L.mmb_ctx_create.restype=C.c_void_p; "
            "n=L.mmb_device_count(); import sys; sys.exit(0 if (n > 0 or not L.mmb_ctx_create(0)) else 1)" % LIB)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()
