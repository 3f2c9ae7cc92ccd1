"""Generates the committed golden fixtures from the ORACLE (run in the authoring container, where
/root/reference is mounted).  The reference itself is C#/TorchSharp and cannot be executed here
(no .NET), so these vectors pin the oracle + the reference's shipped assets, not the reference
binary:  python tests/golden/make_golden.py

  yolov8n_f16.npz   the reference's shipped YoloSharpDemo/Assets/PreTrainedModels/Yolov8n.bin
                    (fp16 payload, re-encoded as npz; data fixture, not source code)
  bus_u8.npy        YoloSharpDemo/Assets/TestImage/bus.jpg decoded to uint8 CHW RGB (torchvision)
  v8n_bus.npz       oracle outputs for that image: post-NMS rows, kept anchors, a strided sample of
                    the (1,84,6300) prediction tensor
  nms_cases.npz     synthetic NMS inputs + oracle outputs (ties, empty image, >max_det, class offsets)
  shipped_bins.json size and SHA-256 of the shipped Yolov8n.bin, yolov11n.bin and yolov8n-seg.bin; their tensors,
                    in file order, are the *_f16.npz fixtures, so tests rebuild each file from its npz and check it
                    against these (tests/util.py shipped_bin)
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torchvision

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import binfmt, ops, yolo  # noqa: E402

REF = "/root/reference/YoloSharpDemo/Assets/"
SHIPPED_BINS = (("Yolov8n.bin", "yolov8n_f16.npz"), ("yolov11n.bin", "yolov11n_f16.npz"),
                ("yolov8n-seg.bin", "yolov8n-seg_f16.npz"))


def nms_case(seed, B, nc, A, extra=0, score_scale=1.0, quant=None, frac=1.0):
    g = torch.Generator().manual_seed(seed)
    cxy = torch.rand(B, 2, A, generator=g) * 640
    wh = torch.exp(torch.randn(B, 2, A, generator=g) * 0.8 + np.log(60.0)).clamp(2, 600)
    cls = torch.rand(B, nc, A, generator=g) ** 4 * score_scale
    cls = cls * (torch.rand(B, 1, A, generator=g) < frac)  # only a fraction of anchors carry objects
    if quant:  # force score ties and identical boxes
        cls = (cls * quant).round() / quant
        cxy = (cxy / 16).round() * 16
        wh = (wh / 16).round().clamp(min=1) * 16
    parts = [cxy, wh, cls]
    if extra:
        parts.append(torch.randn(B, extra, A, generator=g))
    return torch.cat(parts, 1).contiguous()


def main():
    torch.manual_seed(0)
    sd, trailing = binfmt.load_bin(REF + "PreTrainedModels/Yolov8n.bin")
    assert trailing == 0 and len(sd) == 357
    np.savez_compressed(os.path.join(HERE, "yolov8n_f16.npz"), **{k: v.numpy() for k, v in sd.items()})
    img = torchvision.io.read_image(REF + "TestImage/bus.jpg", torchvision.io.ImageReadMode.RGB)
    np.save(os.path.join(HERE, "bus_u8.npy"), img.numpy())
    m = yolo.build("v8", "detect", "n").eval()
    binfmt.load_into(m, REF + "PreTrainedModels/Yolov8n.bin")
    with torch.no_grad():
        pred = m(ops.preprocess(img))[0]["boxes"]
    out, keep = ops.non_max_suppression(pred, 0.3, 0.7)
    np.savez(os.path.join(HERE, "v8n_bus.npz"), rows=out[0].numpy(), keep=keep[0].numpy(),
             pred_sample=pred[0, :, ::37].numpy(), pred_shape=np.array(pred.shape))
    print("bus rows:\n", out[0])

    cases = {}
    specs = {
        "basic": dict(seed=1, B=2, nc=8, A=700, frac=0.15),
        "ties": dict(seed=2, B=2, nc=4, A=900, quant=8, frac=0.3),
        "dense": dict(seed=3, B=1, nc=3, A=3000, score_scale=1.0),       # > max_det survivors
        "extra": dict(seed=4, B=2, nc=5, A=500, extra=32),
        "sparse": dict(seed=5, B=3, nc=80, A=8400, score_scale=0.6, frac=0.02),
    }
    for name, sp in specs.items():
        p = nms_case(**sp)
        if name == "basic":
            p[1, 4:] = 0.0  # image with no candidates
        for (conf, iou) in ((0.25, 0.45), (0.3, 0.7)):
            out, keep = ops.non_max_suppression(p, conf, iou, nc=sp["nc"])
            tag = f"{name}_{conf}_{iou}"
            cases[tag + "_counts"] = np.array([o.shape[0] for o in out])
            cases[tag + "_rows"] = np.concatenate([o.numpy() for o in out], 0)
            cases[tag + "_keep"] = np.concatenate([k.numpy() for k in keep], 0)
        cases[name + "_spec"] = np.array([sp["seed"], sp["B"], sp["nc"], sp["A"], sp.get("extra", 0),
                                          int(sp.get("quant") or 0), int(sp.get("score_scale", 1.0) * 1000),
                                          int(sp.get("frac", 1.0) * 1000)])
    np.savez_compressed(os.path.join(HERE, "nms_cases.npz"), **cases)
    print({k: v.tolist() for k, v in cases.items() if k.endswith("_counts")})
    write_shipped_digests()


def write_shipped_digests():
    digests = {}
    for f, npz in SHIPPED_BINS:
        raw = open(REF + "PreTrainedModels/" + f, "rb").read()
        digests[f] = {"npz": npz, "bytes": len(raw), "sha256": hashlib.sha256(raw).hexdigest()}
    with open(os.path.join(HERE, "shipped_bins.json"), "w") as fh:
        json.dump(digests, fh, indent=1)
        fh.write("\n")


if __name__ == "__main__":
    main()
