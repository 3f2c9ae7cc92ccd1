"""Shared helpers for the parity tests (the oracle is the checker, never the thing measured)."""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle import modules as om  # noqa: E402
from oracle import yolo as oyolo  # noqa: E402


def nms_case(seed, B, nc, A, extra=0, score_scale=1.0, quant=None, frac=1.0):
    """Same generator as tests/golden/make_golden.py (kept in sync by test_oracle.py)."""
    g = torch.Generator().manual_seed(seed)
    cxy = torch.rand(B, 2, A, generator=g) * 640
    wh = torch.exp(torch.randn(B, 2, A, generator=g) * 0.8 + np.log(60.0)).clamp(2, 600)
    cls = torch.rand(B, nc, A, generator=g) ** 4 * score_scale
    cls = cls * (torch.rand(B, 1, A, generator=g) < frac)
    if quant:
        cls = (cls * quant).round() / quant
        cxy = (cxy / 16).round() * 16
        wh = (wh / 16).round().clamp(min=1) * 16
    parts = [cxy, wh, cls]
    if extra:
        parts.append(torch.randn(B, extra, A, generator=g))
    return torch.cat(parts, 1).contiguous()


def golden_nms_cases():
    z = np.load(os.path.join(GOLDEN, "nms_cases.npz"))
    names = sorted(k[:-5] for k in z.files if k.endswith("_spec"))
    for name in names:
        seed, B, nc, A, extra, quant, ss, frac = [int(v) for v in z[name + "_spec"]]
        pred = nms_case(seed, B, nc, A, extra, ss / 1000.0, quant or None, frac / 1000.0)
        if name == "basic":
            pred[1, 4:] = 0.0
        for conf, iou in ((0.25, 0.45), (0.3, 0.7)):
            tag = f"{name}_{conf}_{iou}"
            yield tag, pred, nc, conf, iou, z[tag + "_counts"], z[tag + "_rows"], z[tag + "_keep"]


def synth_image(B, H=640, W=640, seed=0, dtype=torch.float32):
    """SURVEY.md §8(d): randint(0,256) uint8 -> /255."""
    g = torch.Generator().manual_seed(seed)
    u8 = torch.randint(0, 256, (B, 3, H, W), dtype=torch.uint8, generator=g)
    if dtype == torch.uint8:
        return u8
    return (u8.float() / 255.0).to(dtype)


def oracle_model(arch="v8", task="detect", size="n", nc=80, seed=0, cls_bias=-4.5, head_gain=10.0):
    """Seeded synthetic weights; the head gain/bias give ~2k conf>0.25 candidates and a few hundred NMS
    survivors per 640x640 image, so decode + NMS are exercised (SURVEY.md §8(d))."""
    m = oyolo.build(arch, task, size, nc).eval()
    oyolo.synth_weights(m, seed=seed, cls_bias=cls_bias, head_gain=head_gain)
    return m


def oracle_real_v8n():
    """Oracle v8n with the shipped checkpoint (golden fixture copy)."""
    z = np.load(os.path.join(GOLDEN, "yolov8n_f16.npz"))
    m = oyolo.build("v8", "detect", "n").eval()
    own = m.state_dict()
    new = {k: torch.from_numpy(z[k].astype(np.float32)).reshape(own[k].shape) for k in z.files if k in own}
    m.load_state_dict(new, strict=False)
    return m, {k: torch.from_numpy(z[k]) for k in z.files}


def shipped_bin(directory, name):
    """The reference's shipped checkpoint `name` (Yolov8n.bin, yolov11n.bin or yolov8n-seg.bin), written into `directory`
    from the golden copy of its tensors and checked byte for byte (size and SHA-256) against the shipped file.  -> path."""
    from yolosharp_b200 import binfmt
    spec = json.load(open(os.path.join(GOLDEN, "shipped_bins.json")))[name]
    z = np.load(os.path.join(GOLDEN, spec["npz"]))
    code = {np.dtype(np.float16): 5, np.dtype(np.float32): 6}
    path = os.path.join(str(directory), name)
    binfmt.write_bin(path, [(k, code[z[k].dtype], z[k].shape, z[k].tobytes()) for k in z.files])
    raw = open(path, "rb").read()
    assert len(raw) == spec["bytes"] and hashlib.sha256(raw).hexdigest() == spec["sha256"], f"{name} differs from the shipped file"
    return path


def oracle_activations(model, x):
    """Run the oracle and capture every submodule's output by reference name."""
    acts, hooks = {}, []
    for name, mod in model.named_modules():
        if name:
            hooks.append(mod.register_forward_hook(lambda m, i, o, n=name: acts.__setitem__(n, o)))
    with torch.no_grad():
        out = model(x)
    for h in hooks:
        h.remove()
    return out, acts


def expected_for_op(model, acts, op_name):
    """Oracle tensor that the engine op `op_name` should reproduce (or None if not comparable).
    A Bottleneck's cv2 op includes the shortcut add, so it maps to the Bottleneck output."""
    if op_name.endswith(".m") and op_name[:-2] in acts:
        sppf = model.get_submodule(op_name[:-2])
        if isinstance(sppf, om.SPPF):  # SPPF pool op: the engine view is the first pooled map
            return sppf.m(acts[op_name[:-2] + ".cv1"])
    if op_name.endswith((".attn.pe", ".attn.proj", ".proto.upsample")):
        return None  # engine op = module output + fused residual / pre-shuffle layout: no oracle twin
    if op_name.endswith(".ffn.1"):  # PSABlock output: b1 + ffn(b1)
        return acts.get(op_name[:-len(".ffn.1")])
    if op_name.endswith(".upsample.shuffle"):
        return acts.get(op_name[:-len(".shuffle")])
    if "+" in op_name:  # merged first convs of the Detect branches: outputs concatenated along channels
        first = op_name.split("+")[0]
        prefix = first[:first.rfind(".cv")]
        names = [first] + [prefix + "." + p for p in op_name.split("+")[1:]]
        if all(n in acts for n in names):
            return torch.cat([acts[n] for n in names], 1)
        return None
    if op_name not in acts:
        return None
    t = acts[op_name]
    if not torch.is_tensor(t):
        return None
    parent_name = op_name.rsplit(".", 1)[0]
    try:
        parent = model.get_submodule(parent_name)
    except AttributeError:
        parent = None
    if isinstance(parent, om.Bottleneck) and op_name.endswith(".cv2") and parent.add:
        return acts[parent_name]
    return t


def rel_err(a, b):
    """max |a-b| / max(|b|) - scale-aware error used for activation tensors."""
    a, b = a.float(), b.float()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-12))
