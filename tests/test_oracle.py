"""CPU tests: the oracle against its golden vectors, the reference's shipped checkpoints (rebuilt from their golden
copies and checked against the shipped files' SHA-256), and an independent NMS restatement.  No GPU, and no product
code except the pure-Python .bin writer that rebuilds those checkpoints."""
import os

import numpy as np
import pytest
import torch

from oracle import binfmt, ops, yolo
from tests.util import GOLDEN, golden_nms_cases, oracle_real_v8n, shipped_bin


def test_nms_golden_and_independent_restatement():
    """ops.non_max_suppression reproduces the committed vectors; its torchvision core agrees with
    the scalar numpy restatement of the same contract (ties, class offsets)."""
    n = 0
    for tag, pred, nc, conf, iou, counts, rows, keep in golden_nms_cases():
        out, keepi = ops.non_max_suppression(pred, conf, iou, nc=nc)
        assert [o.shape[0] for o in out] == counts.tolist(), tag
        np.testing.assert_array_equal(np.concatenate([o.numpy() for o in out], 0), rows, err_msg=tag)
        np.testing.assert_array_equal(np.concatenate([k.numpy() for k in keepi], 0), keep, err_msg=tag)
        n += 1
    assert n == 10
    g = torch.Generator().manual_seed(7)
    boxes = torch.rand(400, 4, generator=g) * 300
    boxes[:, 2:] += boxes[:, :2]
    boxes = (boxes / 8).round() * 8  # many exact overlaps / IoU ties
    scores = (torch.rand(400, generator=g) * 16).round() / 16
    import torchvision
    for thr in (0.3, 0.45, 0.7):
        a = torchvision.ops.nms(boxes, scores, thr).numpy()
        b = ops.greedy_nms_numpy(boxes.numpy(), scores.numpy(), thr)
        np.testing.assert_array_equal(a, b)


def test_nms_argument_checks():
    p = torch.zeros(1, 84, 10)
    with pytest.raises(ValueError):
        ops.non_max_suppression(p, conf_thres=1.5)
    with pytest.raises(ValueError):
        ops.non_max_suppression(p, iou_thres=-0.1)
    out, keep = ops.non_max_suppression(p)
    assert out[0].shape == (0, 6) and keep[0].numel() == 0


def test_v8n_bus_golden():
    """Oracle + shipped Yolov8n weights on bus.jpg: bus 0.896 + 3 persons (SURVEY.md §4)."""
    m, _ = oracle_real_v8n()
    img = torch.from_numpy(np.load(os.path.join(GOLDEN, "bus_u8.npy")))
    with torch.no_grad():
        pred = m(ops.preprocess(img))[0]["boxes"]
    z = np.load(os.path.join(GOLDEN, "v8n_bus.npz"))
    assert tuple(pred.shape) == tuple(z["pred_shape"]) == (1, 84, 6300)
    np.testing.assert_allclose(pred[0, :, ::37].numpy(), z["pred_sample"], rtol=1e-4, atol=1e-4)
    out, keep = ops.non_max_suppression(pred, 0.3, 0.7)
    np.testing.assert_allclose(out[0].numpy(), z["rows"], rtol=1e-4, atol=1e-3)
    np.testing.assert_array_equal(keep[0].numpy(), z["keep"])
    res = ops.to_yolo_results(out[0])
    assert [r["ClassID"] for r in res[:4]] == [5, 0, 0, 0]
    assert abs(res[0]["Score"] - 0.896) < 2e-3


def test_model_sizes_match_survey():
    """Parameter counts of the restated graphs (SURVEY.md §6: 3.157 M / 11.17 M / 68.23 M / 9.46 M)."""
    def nparams(m):
        return sum(p.numel() for n, p in m.named_parameters() if "dfl" not in n)
    assert abs(nparams(yolo.build("v8", "detect", "n")) / 1e6 - 3.157) < 0.01
    assert abs(nparams(yolo.build("v8", "detect", "s")) / 1e6 - 11.167) < 0.01
    assert abs(nparams(yolo.build("v11", "detect", "s")) / 1e6 - 9.459) < 0.01


def test_bin_reader_on_shipped_checkpoints(tmp_path):
    for arch, task, f, cnt in (("v8", "detect", "Yolov8n.bin", 357), ("v11", "detect", "yolov11n.bin", 501),
                               ("v8", "segment", "yolov8n-seg.bin", 419)):
        path = shipped_bin(tmp_path, f)
        sd, trailing = binfmt.load_bin(path)
        assert trailing == 0 and len(sd) == cnt
        m = yolo.build(arch, task, "n")
        missing, unexpected = binfmt.load_into(m, path)
        assert missing == [] and unexpected == []


def test_golden_weights_equal_shipped_checkpoint(tmp_path):
    sd, _ = binfmt.load_bin(shipped_bin(tmp_path, "Yolov8n.bin"))
    z = np.load(os.path.join(GOLDEN, "yolov8n_f16.npz"))
    assert sorted(z.files) == sorted(sd.keys())
    for k in z.files:
        np.testing.assert_array_equal(z[k], sd[k].numpy())
