"""Native checkpoint reader / writer (csrc/ckpt.cu) against the independent Python reader (yolosharp_b200/binfmt.py),
the committed copy of the reference's shipped Yolov8n.bin (tests/golden/yolov8n_f16.npz) and the shipped file itself, rebuilt
from that copy and checked against its SHA-256 (byte-exact round trip)."""
import json
import os
import struct

import numpy as np
import pytest
import torch

from tests.util import GOLDEN, shipped_bin
from yolosharp_b200 import binfmt
from yolosharp_b200 import engine as E
from yolosharp_b200._lib import YbError

CODE = {torch.float16: 5, torch.float32: 6, torch.int64: 4, torch.int32: 3}


def golden_sd():
    z = np.load(os.path.join(GOLDEN, "yolov8n_f16.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def test_bin_native_reader_equals_python_reader(tmp_path):
    sd = golden_sd()
    p = str(tmp_path / "a.bin")
    binfmt.write_bin(p, [(k, CODE[v.dtype], list(v.shape), v.numpy().tobytes()) for k, v in sd.items()])
    got = E.read_checkpoint(p)
    assert list(got) == list(sd) and len(got) == 357
    for k, v in sd.items():
        assert got[k].dtype == v.dtype and tuple(got[k].shape) == tuple(v.shape) and torch.equal(got[k], v), k


def test_bin_native_writer_equals_python_writer_and_reference_file(tmp_path):
    sd = golden_sd()
    a, b = str(tmp_path / "a.bin"), str(tmp_path / "b.bin")
    binfmt.write_bin(a, [(k, CODE[v.dtype], list(v.shape), v.numpy().tobytes()) for k, v in sd.items()])
    E.write_checkpoint_bin(b, sd)
    assert open(a, "rb").read() == open(b, "rb").read()
    ref = shipped_bin(tmp_path, "Yolov8n.bin")  # the shipped file round-trips byte for byte
    c = str(tmp_path / "c.bin")
    E.write_checkpoint_bin(c, E.read_checkpoint(ref))
    assert open(c, "rb").read() == open(ref, "rb").read()


def test_safetensors_reader(tmp_path):
    sd = {k: v for k, v in list(golden_sd().items())[:20] if v.numel()}
    sd["extra.bf16"] = torch.randn(3, 5).to(torch.bfloat16)
    hdr, blob = {"__metadata__": {"format": "pt"}}, b""
    names = {torch.float16: "F16", torch.float32: "F32", torch.int64: "I64", torch.bfloat16: "BF16"}
    for k, v in sd.items():
        raw = v.view(torch.int16).numpy().tobytes() if v.dtype == torch.bfloat16 else v.numpy().tobytes()
        hdr[k] = {"dtype": names[v.dtype], "shape": list(v.shape), "data_offsets": [len(blob), len(blob) + len(raw)]}
        blob += raw
    hj = json.dumps(hdr).encode()
    p = str(tmp_path / "m.safetensors")
    open(p, "wb").write(struct.pack("<Q", len(hj)) + hj + blob)
    got = E.read_checkpoint(p)
    assert set(got) == set(sd)
    for k, v in sd.items():
        assert got[k].dtype == v.dtype and torch.equal(got[k], v), k


def test_checkpoint_errors(tmp_path):
    with pytest.raises(YbError):
        E.read_checkpoint(str(tmp_path / "missing.bin"))
    bad = str(tmp_path / "bad.safetensors")
    open(bad, "wb").write(b"\x05\x00\x00\x00\x00\x00\x00\x00{\"a\"")
    with pytest.raises(YbError):
        E.read_checkpoint(bad)
    trunc = str(tmp_path / "t.bin")
    sd = golden_sd()
    full = str(tmp_path / "f.bin")
    E.write_checkpoint_bin(full, sd)
    open(trunc, "wb").write(open(full, "rb").read()[:-7])
    with pytest.raises(YbError):
        E.read_checkpoint(trunc)
    with pytest.raises(YbError) as ei:
        E.read_checkpoint(str(tmp_path / "model.pt"))
    assert "cannot read" in str(ei.value)
    notzip = str(tmp_path / "x.pt")
    open(notzip, "wb").write(b"\x80\x02}q\x00." * 8)  # a bare pickle, not a torch.save archive
    with pytest.raises(YbError):
        E.read_checkpoint(notzip)


def test_engine_load_checkpoint_dry_run(tmp_path):
    """yb_load_checkpoint on a dry-run engine (no GPU): every expected tensor of Yolov8n is found in the file."""
    import yolosharp_b200 as y
    from yolosharp_b200 import _lib as L
    p = str(tmp_path / "n.bin")
    E.write_checkpoint_bin(p, golden_sd())
    e = y.Engine("v8", "n", "detect", 80, "f16", 0, 1, 64, 64, flags=L.YB_FLAG_DRY_RUN)
    loaded, missing = e.load_checkpoint(p)
    assert missing == 0 and loaded >= len(e.expected_tensors())
    e2 = y.Engine("v8", "s", "detect", 80, "f16", 0, 1, 64, 64, flags=L.YB_FLAG_DRY_RUN)
    with pytest.raises(YbError):  # n-size file into an s-size graph: shapes are checked at finalize; here names match, so
        e2.load_checkpoint(p)     # loading succeeds and ...
        e2.finalize()             # ... finalize refuses (dry-run engine / shape mismatch)
    e.close()
    e2.close()


def test_train_state_dict_roundtrip(tmp_path):
    """ADVICE r1: trained weights go back to the reference checkpoint format (SaveWeight) and load again."""
    from tests.torch_train_ops import TorchOps
    from tests.util import oracle_model
    from yolosharp_b200.train import TrainStepV8
    m = oracle_model("v8", "detect", "n")
    sd0 = {k: v.detach().clone() for k, v in m.state_dict().items()}
    st = TrainStepV8(sd0, "n", 80, device="cpu", ops=TorchOps(), lr=1e-3)
    st.step_count = 3
    p = str(tmp_path / "last.bin")
    st.save(p)
    back = E.read_checkpoint(p)
    assert set(back) == set(sd0), (set(sd0) ^ set(back))
    for k, v in sd0.items():
        if k.endswith("num_batches_tracked"):
            assert int(back[k]) == 3
        elif v.numel():
            assert torch.equal(back[k].float(), v.float()), k


# ---- torch.save archives (.pt): zip + pickle, read natively (replaces ModelLoader/PickleLoader.cs) ----
def _same(got, want):
    assert list(got) == list(want), (list(got)[:5], list(want)[:5])
    for k, v in want.items():
        assert got[k].dtype == v.dtype and tuple(got[k].shape) == tuple(v.shape) and torch.equal(got[k], v), k


@pytest.mark.parametrize("proto", [2, 4])
def test_pt_state_dict(tmp_path, proto):
    from tests.util import oracle_model
    sd = oracle_model("v8", "detect", "n").state_dict()  # OrderedDict with _metadata, fp32 + int64 num_batches_tracked
    sd["extra.half"] = torch.randn(4, 3).half()
    sd["extra.bf16"] = torch.randn(2, 5).bfloat16()
    sd["extra.bool"] = torch.tensor([True, False, True])
    sd["extra.u8"] = torch.arange(7, dtype=torch.uint8)
    sd["extra.f64"] = torch.randn(3, dtype=torch.float64)
    sd["extra.i32"] = torch.arange(5, dtype=torch.int32).view(5, 1)
    sd["extra.scalar"] = torch.tensor(3.5)
    sd["extra.empty"] = torch.zeros(0, 4)
    p = str(tmp_path / "sd.pt")
    torch.save(sd, p, pickle_protocol=proto)
    _same(E.read_checkpoint(p), sd)


def test_pt_nested_checkpoint_and_shared_storage(tmp_path):
    """An Ultralytics-style dict {'epoch', 'model': state_dict, ...}: names are dotted paths (ExtractTensors, PickleLoader.cs:49-88);
    views that share one storage keep their storage offsets."""
    base = torch.arange(24, dtype=torch.float32)
    ck = {"epoch": 7, "best_fitness": 0.25, "names": {0: "person", 1: "car"}, "date": "2024", "model": {"a.weight": base[4:16].view(3, 4),
                                                                                                 "a.bias": base[16:20]},
          "lst": [torch.ones(2), None, torch.zeros(1, 3)], "train_args": {"imgsz": 640, "rect": False}}
    p = str(tmp_path / "ck.pth")
    torch.save(ck, p)
    got = E.read_checkpoint(p)
    want = {"model.a.weight": ck["model"]["a.weight"], "model.a.bias": ck["model"]["a.bias"], "lst.0": ck["lst"][0], "lst.2": ck["lst"][2]}
    _same(got, want)


def test_pt_pickled_module_gives_state_dict_names(tmp_path):
    """torch.save(module): the object tree of nn.Module instances (BUILD states with _parameters / _buffers / _modules) yields
    the names module.state_dict() has; non-persistent extras (num_batches_tracked is a buffer, so it is included)."""
    torch.manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, bias=False), torch.nn.BatchNorm2d(8), torch.nn.SiLU(),
                            torch.nn.Sequential(torch.nn.Conv2d(8, 4, 1), torch.nn.Identity()))
    p = str(tmp_path / "m.pt")
    torch.save({"model": m, "epoch": 1}, p)
    got = E.read_checkpoint(p)
    want = {"model." + k: v for k, v in m.state_dict().items()}
    assert set(got) == set(want)
    for k, v in want.items():
        assert torch.equal(got[k], v), k


def test_pt_rejects_non_contiguous(tmp_path):
    p = str(tmp_path / "t.pt")
    torch.save({"w": torch.arange(12.).view(3, 4).t()}, p)
    with pytest.raises(YbError) as ei:
        E.read_checkpoint(p)
    assert "contiguous" in str(ei.value)


def test_engine_load_checkpoint_from_pt(tmp_path):
    import yolosharp_b200 as y
    from yolosharp_b200 import _lib as L
    p = str(tmp_path / "n.pt")
    torch.save(golden_sd(), p)
    e = y.Engine("v8", "n", "detect", 80, "f16", 0, 1, 64, 64, flags=L.YB_FLAG_DRY_RUN)
    loaded, missing = e.load_checkpoint(p)
    assert missing == 0 and loaded >= len(e.expected_tensors())
    e.close()


def test_pt_whole_yolo_model_object(tmp_path):
    """The way Ultralytics checkpoints are written: {'model': <model object in half precision>, ...}: every state_dict() entry
    of a YOLOv11n object tree comes back under 'model.', bit for bit."""
    from tests.util import oracle_model
    m = oracle_model("v11", "detect", "n").half()
    p = str(tmp_path / "full.pt")
    torch.save({"model": m, "ema": None, "epoch": -1, "train_args": {"imgsz": 640}}, p)
    got = E.read_checkpoint(p)
    want = {"model." + k: v for k, v in m.state_dict().items()}
    assert set(got) == set(want) and len(got) == 501
    for k, v in want.items():
        assert got[k].dtype == v.dtype and torch.equal(got[k], v), k


@pytest.mark.parametrize("kind", ["bin", "pt", "pt_module"])
def test_checkpoint_readers_survive_corruption(tmp_path, kind):
    """Truncated or bit-flipped files must come back as an error (or as a successfully parsed file), never as a crash: the
    readers bounds-check every length they take from the file."""
    import random
    sd = {"a.weight": torch.randn(4, 3, 3, 3), "a.bias": torch.randn(4).half(), "n": torch.tensor([5])}
    if kind == "bin":
        p = str(tmp_path / "x.bin")
        E.write_checkpoint_bin(p, sd)
    elif kind == "pt":
        p = str(tmp_path / "x.pt")
        torch.save({"model": sd, "epoch": 3}, p)
    else:
        p = str(tmp_path / "x.pt")
        torch.save({"model": torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.BatchNorm2d(8))}, p, pickle_protocol=4)
    raw = open(p, "rb").read()
    rng = random.Random(0)
    q = str(tmp_path / ("f" + os.path.splitext(p)[1]))
    outcomes = {"ok": 0, "err": 0}
    for it in range(200):
        b = bytearray(raw)
        if it % 2:
            b = b[: rng.randrange(0, len(b))]
        else:
            for _ in range(rng.randrange(1, 8)):
                b[rng.randrange(len(b))] = rng.randrange(256)
        open(q, "wb").write(bytes(b))
        try:
            E.read_checkpoint(q)
            outcomes["ok"] += 1
        except (YbError, KeyError):  # KeyError: a corrupted dtype code the Python table does not know
            outcomes["err"] += 1
    assert outcomes["err"] >= 90  # every truncation is an error


def test_engine_load_checkpoint_from_ultralytics_style_pt(tmp_path):
    """{'model': <model object>} checkpoints name their tensors "model.<state_dict key>": yb_load_checkpoint drops that level
    when nothing matches as it stands."""
    import yolosharp_b200 as y
    from tests.util import oracle_model
    from yolosharp_b200 import _lib as L
    p = str(tmp_path / "u.pt")
    torch.save({"model": oracle_model("v8", "detect", "n").half(), "epoch": -1}, p)
    e = y.Engine("v8", "n", "detect", 80, "f16", 0, 1, 64, 64, flags=L.YB_FLAG_DRY_RUN)
    loaded, missing = e.load_checkpoint(p)
    assert missing == 0 and loaded >= len(e.expected_tensors())
    e.close()


def test_convert_checkpoint_tool(tmp_path):
    """tools/convert_checkpoint.py: an Ultralytics-style .pt becomes a .bin that loads into the engine (dry run)."""
    import subprocess
    import sys

    import yolosharp_b200 as y
    from tests.util import oracle_model
    from yolosharp_b200 import _lib as L
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, dst = str(tmp_path / "u.pt"), str(tmp_path / "u.bin")
    m = oracle_model("v8", "detect", "n")
    torch.save({"model": m, "epoch": 3}, src)
    subprocess.check_call([sys.executable, os.path.join(root, "tools", "convert_checkpoint.py"), src, dst, "--strip", "model.", "--half"])
    got = E.read_checkpoint(dst)
    want = m.state_dict()
    assert list(got) == list(want)
    for k, v in want.items():
        ref = v.half() if v.dtype == torch.float32 else v
        assert got[k].dtype == ref.dtype and torch.equal(got[k], ref), k
    e = y.Engine("v8", "n", "detect", 80, "f16", 0, 1, 64, 64, flags=L.YB_FLAG_DRY_RUN)
    loaded, missing = e.load_checkpoint(dst)
    assert missing == 0
    e.close()
