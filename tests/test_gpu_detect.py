"""Device-side detection decode + NMS of the whole batch (yb_network_detect, SURVEY 8f row 1) against
(a) the host restatement yb_get_network_boxes, image by image, on the very tensors the device produced, and
(b) the unmodified reference's get_network_boxes + do_nms_sort run on each image separately (its rows are stored in
tests/golden/reference_arrays.npz, "detect_*")."""
import os

import numpy as np
import pytest

import ybtest_util as util
from yolo2_light_b200 import cfgs

pytestmark = pytest.mark.gpu


def _sorted(rows):
    if rows.shape[0] == 0:
        return rows
    return rows[np.lexsort(rows[:, :4].T[::-1])]


def _bigger(name, workdir, w, h):
    """The slim zoo nets on a larger input: more grid cells -> a few hundred candidates per image."""
    build = {"tiny": cfgs.yolov3_tiny, "v3": cfgs.yolov3, "xnor": cfgs.tiny_yolo_obj_xnor, "v2voc": cfgs.yolov2_voc}[name]
    secs = cfgs.slim(build, 4 if name in ("v3", "v2voc") else 2, w, h)
    cfg = os.path.join(workdir, f"det_{name}_{w}x{h}.cfg")
    wts = os.path.join(workdir, f"det_{name}_{w}x{h}.weights")
    cfgs.write_cfg(secs, cfg)
    cfgs.write_weights(secs, wts, seed=41)
    return cfg, wts


@pytest.mark.parametrize("name,w,h,thresh,relative,letter", [
    ("tiny", 160, 160, 0.2, 1, 0),
    ("tiny", 224, 160, 0.2, 0, 1),      # non-square, absolute coordinates, letterbox correction
    ("v3", 128, 128, 0.2, 1, 0),         # three yolo layers
    ("xnor", 160, 160, 0.05, 1, 0),       # region layer (every box is a candidate), softmax classes
    ("v2voc", 96, 96, 0.02, 1, 1),        # region layer behind reorg / route
])
def test_device_detect_equals_host_decode(name, w, h, thresh, relative, letter, workdir):
    import yolo2_light_b200 as yb
    B = 3
    cfg, wts = _bigger(name, workdir, w, h)
    net = yb.load_network(cfg, wts, batch=B)
    x = cfgs.synthetic_images(B, 3, h, w, seed=43)
    net.predict(x)
    dets, counts = net.detect(640, 480, thresh, 0.45, relative, letter, max_rows=4096)
    assert max(counts) <= 4096
    seen = nms_active = 0
    for b in range(B):
        host = net.get_network_boxes(b, 640, 480, thresh, 0.45, relative, letter)
        assert counts[b] == host.shape[0], (b, counts[b], host.shape)
        a, e = _sorted(dets[b]), _sorted(host)
        # boxes: double exp() on both sides, identical up to libm's last bit; probabilities: exact
        assert np.allclose(a[:, :4], e[:, :4], rtol=1e-6, atol=1e-7), b
        assert np.array_equal(a[:, 4:], e[:, 4:]), (b, np.abs(a[:, 4:] - e[:, 4:]).max())
        seen += host.shape[0]
        # NMS really removed something and really kept something
        if host.shape[0] > 20:
            raw = net.get_network_boxes(b, 640, 480, thresh, 0.0, relative, letter)
            assert (host[:, 5:] > 0).sum() < (raw[:, 5:] > 0).sum()
            assert (host[:, 5:] > 0).sum() > 0
    assert seen > 50, seen
    # nms = 0: decode only
    dets0, counts0 = net.detect(640, 480, thresh, 0.0, relative, letter, max_rows=4096)
    for b in range(B):
        raw = net.get_network_boxes(b, 640, 480, thresh, 0.0, relative, letter)
        assert np.array_equal(_sorted(dets0[b])[:, 4:], _sorted(raw)[:, 4:])


def test_device_detect_cap_and_empty(workdir):
    import yolo2_light_b200 as yb
    cfg, wts = _bigger("tiny", workdir, 160, 160)
    net = yb.load_network(cfg, wts, batch=2)
    x = cfgs.synthetic_images(2, 3, 160, 160, seed=44)
    net.predict(x)
    dets, counts = net.detect(640, 480, 0.2, 0.45, max_rows=4096)
    full = [d.copy() for d in dets]
    # cap below the candidate count: the first max_rows candidates (reference order) are decoded, count reports all
    cap = max(1, int(min(counts)) // 2)
    dets_c, counts_c = net.detect(640, 480, 0.2, 0.0, max_rows=cap)
    dets_f, _ = net.detect(640, 480, 0.2, 0.0, max_rows=4096)
    for b in range(2):
        assert counts_c[b] == counts[b] and dets_c[b].shape[0] == cap
        assert np.array_equal(dets_c[b], dets_f[b][:cap])
    # threshold nothing passes: zero candidates, no kernel trouble
    dets_e, counts_e = net.detect(640, 480, 1.5, 0.45, max_rows=64)
    assert list(counts_e) == [0, 0] and all(d.shape[0] == 0 for d in dets_e)
    # repeatable
    again, _ = net.detect(640, 480, 0.2, 0.45, max_rows=4096)
    for b in range(2):
        assert np.array_equal(again[b], full[b])
    with pytest.raises(yb.YbError):
        net.detect(640, 480, 0.5, 0.45, max_rows=0)


REF_CASES = [("tiny", 0), ("tiny", 1), ("xnor", 0)]


@pytest.mark.parametrize("name,q", REF_CASES)
def test_device_detect_vs_reference_boxes(name, q, workdir):
    """Each image through the unmodified reference (batch 1: its decoder reads item 0 only) vs the batched device path
    in exact (FP32 / INT8 / XNOR) precision."""
    import yolo2_light_b200 as yb
    B = 3
    cfg, wts = _bigger(name, workdir, 160, 160)
    x = cfgs.synthetic_images(B, 3, 160, 160, seed=45)
    net = yb.load_network(cfg, wts, batch=B, quantized=q)
    net.set_precision(yb.YB_PREC_FP32)
    net.predict(x, quantized=bool(q))
    thresh = 0.2 if name == "tiny" else 0.05
    dets, counts = net.detect(640, 480, thresh, 0.45, max_rows=4096, quantized=bool(q))
    for b in range(B):
        theirs = util.reference_arrays()[f"detect_{name}_q{q}_b{b}"]
        # forward outputs differ in the last bits (f32 sum order): candidates sitting exactly at the threshold may flip
        assert abs(int(counts[b]) - theirs.shape[0]) <= max(1, theirs.shape[0] // 100), (b, counts[b], theirs.shape)
        if counts[b] == theirs.shape[0] and theirs.shape[0]:
            a, e = _sorted(dets[b]), _sorted(theirs)
            assert np.allclose(a[:, :5], e[:, :5], rtol=2e-3 if q else 1e-4, atol=1e-5)
            kept_a, kept_e = (a[:, 5:] > 0).sum(), (e[:, 5:] > 0).sum()
            assert abs(int(kept_a) - int(kept_e)) <= max(2, int(kept_e) // 50), (kept_a, kept_e)
