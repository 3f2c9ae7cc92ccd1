"""CPU tests of the drop-in boundary: the C-ABI library builds, loads, exports every symbol that
include/yolob200.h declares, and refuses to run without a GPU (no CPU fallback anywhere)."""
import ctypes
import os
import re
import struct
import subprocess
import sys
import tempfile

import pytest

from tests.util import ROOT, shipped_bin


def header_functions():
    src = open(os.path.join(ROOT, "include", "yolob200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(yb_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(built_lib):
    lib = ctypes.CDLL(built_lib)
    names = header_functions()
    assert len(names) >= 19
    for n in names:
        assert hasattr(lib, n), f"{n} declared in yolob200.h but not exported"
    from yolosharp_b200 import _lib
    assert sorted(_lib.SIGNATURES) == names, "ctypes table and header disagree"


def test_integration_md_mentions_every_entry_point():
    """INTEGRATION.md shows the reference-side binding of the boundary: every function of the header must appear in it, and
    the generated P/Invoke listing (tools/gen_pinvoke.py) must cover the whole header."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    missing = [n for n in header_functions() if n not in text]
    assert not missing, f"INTEGRATION.md lacks {missing}"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_pinvoke.py")], capture_output=True, text=True, check=True).stdout
    declared = sorted(set(re.findall(r"\b(yb_[a-z0-9_]+)\(", out)))
    assert declared == header_functions()


def test_header_compiles_as_c(built_lib):
    """The boundary is plain C: the header must compile with gcc -std=c99 and link against the .so."""
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write('#include "yolob200.h"\nint main(void){ return yb_abi_version() == YB_ABI_VERSION ? 0 : 1; }\n')
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), c, "-o", exe,
                               built_lib, "-Wl,-rpath," + os.path.dirname(built_lib)])
        assert subprocess.call([exe]) == 0


def test_sass_is_blackwell_native(built_lib):
    """tcgen05.mma / TMA / TMEM loads must be in the shipped SASS (B200_PROFILING.md table)."""
    sass = subprocess.run(["cuobjdump", "-sass", built_lib], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic


def test_no_cpu_fallback(built_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import yolosharp_b200 as y
    with pytest.raises(y.YbError) as ei:
        y.Engine()
    assert "no CPU fallback" in str(ei.value)
    with pytest.raises(Exception):
        y.Yolov8().forward(torch.zeros(1, 3, 64, 64))


def test_argument_errors_without_gpu(built_lib):
    from yolosharp_b200 import _lib as L
    lib = L.lib()
    assert lib.yb_abi_version() == 1
    h = ctypes.c_void_p()
    cfg = L.yb_config(arch=7, size=0, task=0, nc=80, reg_max=16, precision=0, device=0, max_batch=1, height=640,
                      width=640, flags=0)
    assert lib.yb_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    assert b"arch" in lib.yb_last_error()
    cfg.arch, cfg.height = 8, 100
    assert lib.yb_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    assert b"multiples of 32" in lib.yb_last_error()
    assert lib.yb_nms(None, 1, 84, 10, 80, 0.25, 0.45, 300, 30000, 7680, None, None, None, None) == -1


def test_bin_roundtrip(tmp_path):
    from yolosharp_b200 import binfmt
    t = [("model.0.conv.weight", 5, (2, 3), struct.pack("<6e", *range(6))),
         ("model.22.anchors", 5, (0,), b""),
         ("a.long.name." + "x" * 200, 6, (1,), struct.pack("<f", 1.5))]
    p = str(tmp_path / "w.bin")
    binfmt.write_bin(p, t)
    assert binfmt.read_bin(p) == t
    ref = shipped_bin(tmp_path, "Yolov8n.bin")
    r = binfmt.read_bin(ref)
    assert len(r) == 357
    binfmt.write_bin(p, r)
    assert open(p, "rb").read() == open(ref, "rb").read()


@pytest.mark.parametrize("arch,task,size", [("v8", "detect", "n"), ("v8", "detect", "s"), ("v8", "detect", "m"),
                                           ("v8", "detect", "l"), ("v8", "detect", "x"), ("v11", "detect", "n"),
                                           ("v11", "detect", "s"), ("v11", "detect", "m"), ("v11", "detect", "x"),
                                           ("v8", "segment", "n"), ("v8", "segment", "s"), ("v11", "segment", "n")])
def test_graph_tensor_names_match_reference_state_dict(built_lib, arch, task, size):
    """The engine's op graph (dry run, no GPU) asks for exactly the reference's state_dict entries:
    every oracle key is expected except the bookkeeping ones the reference never reads on this path."""
    import yolosharp_b200 as y
    from yolosharp_b200 import _lib as L
    from oracle import yolo as oyolo
    e = y.Engine(arch, size, task, 80, "f32", 0, 1, 64, 64, flags=L.YB_FLAG_DRY_RUN)
    want = e.expected_tensors()
    e.close()
    assert len(want) == len(set(want))
    keys = [k for k in oyolo.build(arch, task, size).state_dict()
            if not k.endswith(("num_batches_tracked", ".anchors", ".strides", "dfl.conv.weight"))]
    assert sorted(want) == sorted(keys)
