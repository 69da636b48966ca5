"""CPU: the C-ABI library loads without a GPU, exports every symbol that include/avdsp_b200.h declares, the
ctypes binding lists the same set, the header compiles as plain C, and the table structs are layout-identical
to the reference's (sizes/offsets from oracle/_ref when it is built).  No compute entry point is called."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "include", "avdsp_b200.h")


def _declared():
    src = open(HDR).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b((?:avb200|ff|sws)_[A-Za-z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_every_declared_symbol_is_exported_and_bound(built):
    import libav_b200._lib as L
    decl = _declared()
    assert len(decl) > 30
    for name in decl:
        assert hasattr(L.lib, name), "not exported: " + name
    assert sorted(L.PROTOTYPES) == decl


def test_header_is_plain_c_and_layout_matches_reference(built, tmp_path):
    exe = str(tmp_path / "abi_probe")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "abi_probe.c"), "-o", exe])
    mine = [int(x) for x in subprocess.check_output([exe]).split()]
    from libav_b200 import tables
    assert C.sizeof(tables.IDCTDSPContext) == mine[0] and C.sizeof(tables.MECmpContext) == mine[7]
    assert C.sizeof(tables.H264DSPContext) == mine[11] and C.sizeof(tables.H264QpelContext) == mine[17]
    assert C.sizeof(tables.H264ChromaContext) == mine[19] and C.sizeof(tables.HpelDSPContext) == mine[20]
    assert tables.IDCTDSPContext.idct_permutation.offset == mine[2] and tables.MECmpContext.pix_abs.offset == mine[10]
    assert tables.H264DSPContext.h264_idct_add16.offset == mine[14] and tables.HpelDSPContext.avg_no_rnd_pixels_tab.offset == mine[22]
    assert C.sizeof(tables.H264PredContext) == mine[23] and tables.H264PredContext.pred16x16_add.offset == mine[27]
    assert C.sizeof(tables.PixblockDSPContext) == mine[28] and tables.PixblockDSPContext.diff_pixels.offset == mine[29]
    assert C.sizeof(tables.QpelDSPContext) == mine[30] and tables.QpelDSPContext.put_no_rnd_qpel_pixels_tab.offset == mine[31]
    from oracle import loader
    r = loader.ref()
    if r is None:       # the reference's sizes and offsets (ref_abi_info), recorded where oracle/_ref was built
        ref_abi = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_abi.json")))
    else:
        out = np.zeros(64, np.int32)
        r.lib.ref_abi_info.restype = C.c_int
        ref_abi = out[:r.lib.ref_abi_info(out.ctypes.data_as(C.c_void_p), 64)].tolist()
    assert ref_abi == mine


def test_no_gpu_means_loud_failure(built):
    import libav_b200._lib as L
    if L.lib.avb200_device_count() > 0:
        pytest.skip("a GPU is visible")
    assert L.lib.avb200_init(0) == -1
    assert "no CUDA device" in L.last_error()
    L.lib.avb200_clear_error()
    with pytest.raises(L.AVB200Error):
        L.check(L.lib.avb200_init(0), "avb200_init")


def test_product_does_not_link_or_import_the_oracle():
    """The product library and package must not reference anything under oracle/."""
    for root, _, files in os.walk(os.path.join(ROOT, "libav_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")) :
                txt = open(os.path.join(root, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "oracle_api.h" not in txt and "liboracle" not in txt and "libavref" not in txt or f == "build.py", f
    out = subprocess.check_output(["ldd", os.path.join(ROOT, "libav_b200", "libavdsp_b200.so")]).decode()
    assert "oracle" not in out and "avref" not in out


def test_null_and_zero_arguments_fail_loudly_not_fatally(built):
    """every batched / scaler entry point called with NULL pointers and zero (then small non-zero) counts, without a GPU: an error return
    or an empty success, never a crash (run in a child process so that a crash would be a test failure, not the end of the suite)"""
    import subprocess
    import sys
    code = r'''
import ctypes as C, sys
sys.path.insert(0, %r)
import libav_b200._lib as L
names = [n for n in L.PROTOTYPES if n.startswith("ff_") and n.endswith("_cuda") and "init" not in n] + \
        ["sws_scale_cuda", "sws_scale_frames_cuda", "sws_setColorspaceDetails_cuda", "sws_is_fused_cuda", "sws_freeContext_cuda"]
for name in names:
    res, args = L.PROTOTYPES[name]
    for variant in (0, 4):
        vals = [None if a in (C.c_void_p, C.c_char_p) else 1.0 if a == C.c_double else variant for a in args]
        r = getattr(L.lib, name)(*vals)
        assert r in (None, 0, -1), (name, variant, r)
        L.lib.avb200_clear_error()
print("ok", len(names))
''' % ROOT
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and p.stdout.startswith("ok"), (p.returncode, p.stdout[-300:], p.stderr[-300:])


def test_reference_side_binding_compiles(built):
    """examples/reference_binding/dsp_init_cuda.c -- the glue INTEGRATION.md describes -- against the reference's OWN headers: every hook
    prototype and every slot assignment is type-checked with the reference's struct definitions (needs /root/reference; skipped on the GPU box)"""
    ref, cfg = "/root/reference", os.path.join(ROOT, "oracle", "_ref", "cfg")
    if not os.path.isdir(ref) or not os.path.exists(os.path.join(cfg, "config.h")):
        pytest.skip("no reference tree here")
    src = os.path.join(ROOT, "examples", "reference_binding", "dsp_init_cuda.c")
    r = subprocess.run(["gcc", "-std=c99", "-c", "-Wall", "-Werror", "-Wno-unused-function", "-Wno-attributes", "-I", cfg, "-I", ref, src, "-o", os.devnull],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    # the slot table declared there with the reference's typedefs has the layout of the one in include/avdsp_b200.h
    from libav_b200 import tables
    assert C.sizeof(tables.SwsLineSlotsCUDA) == 12 * C.sizeof(C.c_void_p)
