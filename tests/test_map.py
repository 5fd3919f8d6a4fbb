"""mAP accounting (SURVEY 8f row 4): yb_map_evaluate against the reference's validate_detector_map
(additionally.c:4541-4898) on a small synthetic dataset -- BMP images + label files on disk, the reference's own CPU
forward and decoder on both sides, so only the bookkeeping under test differs.  The reference's detections of each image
and what validate_detector_map printed are stored in tests/golden/reference.json / reference_arrays.npz ("map")."""
import os
import re

import numpy as np
import pytest

import ybtest_util as util

MAP_CASES = [("tiny64", 0.5), ("v3_32", 0.5), ("tiny64", 0.75)]


def _write_bmp(path, img):   # img: u8 [h, w, 3] RGB
    h, w, _ = img.shape
    row = (3 * w + 3) // 4 * 4
    data = bytearray()
    for y in range(h - 1, -1, -1):
        line = img[y, :, ::-1].tobytes()
        data += line + b"\0" * (row - len(line))
    hdr = b"BM" + (54 + len(data)).to_bytes(4, "little") + b"\0\0\0\0" + (54).to_bytes(4, "little")
    dib = (40).to_bytes(4, "little") + w.to_bytes(4, "little") + h.to_bytes(4, "little") + (1).to_bytes(2, "little") + \
        (24).to_bytes(2, "little") + (0).to_bytes(4, "little") + len(data).to_bytes(4, "little") + \
        (2835).to_bytes(4, "little") * 2 + (0).to_bytes(4, "little") * 2
    open(path, "wb").write(hdr + dib + bytes(data))


def write_mapset(name, iou_thresh, workdir, classes, boxes):
    """The on-disk validation set: 7 BMP images, labels made from the detections `boxes(k, img)` of image k.  Returns
    (root, detections per image, truth rows)."""
    root = os.path.join(workdir, f"mapset_{name}_{int(iou_thresh * 100)}")
    os.makedirs(os.path.join(root, "images"), exist_ok=True)
    os.makedirs(os.path.join(root, "labels"), exist_ok=True)
    rng = np.random.default_rng(11)
    nimg = 7
    rows, truth, paths = [], [], []
    for k in range(nimg):
        img = rng.integers(0, 256, size=(72 + 4 * k, 80, 3), dtype=np.uint8)
        path = os.path.join(root, "images", f"img{k}.bmp")
        _write_bmp(path, img)
        paths.append(path)
        r = boxes(k, img)
        rows.append(r)
        # labels: some of the strongest detections (true positives), jittered copies (IoU near the threshold), strays
        lab = []
        if r.shape[0]:
            best = np.argsort(-r[:, 5:].max(axis=1))[:4]
            for j, i in enumerate(best):
                cls = int(np.argmax(r[i, 5:]))
                box = r[i, :4].astype(np.float64)
                if j % 2:
                    box = box * (1.0 + 0.08 * rng.standard_normal(4))
                lab.append((cls, *[round(float(v), 4) for v in box]))
        lab.append((int(rng.integers(0, classes)), 0.5, 0.5, 0.2, 0.3))
        if k == 3:
            lab = []                                                     # an image without labels (no file at all)
        else:
            with open(os.path.join(root, "labels", f"img{k}.txt"), "w") as f:
                for cls, bx, by, bw, bh in lab:
                    f.write(f"{cls} {bx:.4f} {by:.4f} {bw:.4f} {bh:.4f}\n")
        for cls, bx, by, bw, bh in lab:
            truth.append((k, cls, float(f"{bx:.4f}"), float(f"{by:.4f}"), float(f"{bw:.4f}"), float(f"{bh:.4f}")))
    open(os.path.join(root, "valid.txt"), "w").write("\n".join(paths) + "\n")
    open(os.path.join(root, "names.txt"), "w").write("\n".join(f"c{i}" for i in range(classes)) + "\n")
    datacfg = os.path.join(root, "data.cfg")
    open(datacfg, "w").write(f"classes = {classes}\nvalid = {root}/valid.txt\nnames = {root}/names.txt\n")
    return root, rows, truth


def _reference_boxes(k, img, key="tiny64_50"):
    """The reference's get_network_boxes(net, 1, 1, .005, ...) + NMS on load_image + resize_image of image k."""
    return util.reference_arrays()[f"map_{key}_img{k}"]


@pytest.mark.parametrize("name,iou_thresh", MAP_CASES)
def test_map_accounting_equals_reference(name, iou_thresh, workdir):
    import yolo2_light_b200 as yb
    key = f"{name}_{int(iou_thresh * 100)}"
    rec = util.reference()["map"][key]
    classes = rec["classes"]
    root, rows, truth = write_mapset(name, iou_thresh, workdir, classes, lambda k, img: _reference_boxes(k, img, key))
    out = rec["stdout"]
    with open(os.path.join(root, "ref_stdout.txt"), "w") as f:
        f.write(out)
    ap_ref = {int(m.group(1)): float(m.group(2)) for m in re.finditer(r"class_id = (\d+), name = \S+,\s+ap = ([0-9.]+) %", out)}
    m = re.search(r"(?:mean average precision \(mAP\)|average precision \(AP\)) = ([0-9.]+)", out)
    assert m and len(ap_ref) == classes, out[-400:]
    map_ref = float(m.group(1))
    tp, fp, fn, aiou = re.search(r"TP = (\d+), FP = (\d+), FN = (\d+), average IoU = ([0-9.]+) %", out).groups()
    prf = re.search(r"precision = ([0-9.]+), recall = ([0-9.]+), F1-score = ([0-9.]+)", out).groups()
    ndet = int(re.search(r"detections_count = (\d+), unique_truth_count = (\d+)", out).group(1))

    mAP, ap, st = yb.api.map_evaluate(rows, np.array(truth, np.float32).reshape(-1, 6), classes, iou_thresh, 0.24)
    assert int(st["detections"]) == ndet
    assert (int(st["tp"]), int(st["fp"]), int(st["fn"])) == (int(tp), int(fp), int(fn))
    assert abs(mAP - map_ref) < 5e-7, (mAP, map_ref)                      # the reference prints %f
    for c in range(classes):
        assert abs(ap[c] * 100 - ap_ref[c]) <= 0.00501, (c, ap[c], ap_ref[c])   # printed with %2.2f
    assert abs(st["avg_iou"] * 100 - float(aiou)) <= 0.00501
    for mine, theirs in zip((st["precision"], st["recall"], st["f1"]), prf):
        assert abs(mine - float(theirs)) <= 0.00501 or (np.isnan(mine) and "nan" in theirs)
    assert int(tp) > 0 and mAP > 0                                       # the dataset exercises the matching at all


def test_dataset_reader_matches_what_the_reference_reads(workdir):
    """BMP / PPM decode, the label-path rewriting and the label parser of yolo2_light_b200.dataset on the files the
    mAP parity test writes: the reference's loader must see the same pixels (its resize of them == ours of them)."""
    from yolo2_light_b200 import dataset
    root = os.path.join(workdir, "reader")
    os.makedirs(os.path.join(root, "images"), exist_ok=True)
    os.makedirs(os.path.join(root, "labels"), exist_ok=True)
    rng = np.random.default_rng(3)
    for w, h in ((80, 72), (33, 50)):                       # a width whose rows need BMP padding, too
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        p = os.path.join(root, "images", f"i{w}.bmp")
        _write_bmp(p, img)
        assert np.array_equal(dataset.read_image_u8(p), img)
        ppm = os.path.join(root, "images", f"i{w}.ppm")
        open(ppm, "wb").write(b"P6\n# c\n%d %d\n255\n" % (w, h) + img.tobytes())
        assert np.array_equal(dataset.read_image_u8(ppm), img)
        assert dataset.label_path(p) == os.path.join(root, "labels", f"i{w}.txt")
    lab = os.path.join(root, "labels", "i80.txt")
    open(lab, "w").write("3 0.5 0.25 0.125 0.0625\n7 0.1 0.2 0.3 0.4\n")
    got = dataset.read_labels(lab)
    assert got.shape == (2, 5) and got[1, 0] == 7 and np.allclose(got[0], [3, 0.5, 0.25, 0.125, 0.0625])
    assert dataset.read_labels(os.path.join(root, "labels", "missing.txt")).shape == (0, 5)
    open(os.path.join(root, "valid.txt"), "w").write(os.path.join(root, "images", "i80.bmp") + "\n")
    open(os.path.join(root, "names.txt"), "w").write("a\nb\n")
    open(os.path.join(root, "d.cfg"), "w").write(f"classes= 2\nvalid  = {root}/valid.txt\nnames = {root}/names.txt\n# x\n")
    paths, names, truth = dataset.load_validation_set(os.path.join(root, "d.cfg"))
    assert len(paths) == 1 and names == ["a", "b"] and truth.shape == (2, 6) and truth[1, 1] == 7


def test_map_driver_loop_equals_reference_end_to_end(workdir):
    """dataset.evaluate_map (the loop of tools/map.py) with the forward + decoder supplied by the reference through a
    stand-in object: same files in, same mAP out as validate_detector_map.  (The GPU stand-ins of the two calls are
    parity-tested on their own: test_gpu_detect.py, test_device_input_pipeline_bit_exact.)"""
    from yolo2_light_b200 import dataset
    name = "tiny64"
    classes = util.reference()["map"]["tiny64_50"]["classes"]
    root = os.path.join(workdir, "mapset_tiny64_50")          # written by test_map_accounting_equals_reference
    if not os.path.exists(os.path.join(root, "ref_stdout.txt")):
        test_map_accounting_equals_reference(name, 0.5, workdir)
    paths, names, truth = dataset.load_validation_set(os.path.join(root, "data.cfg"))
    assert len(paths) == 7 and len(names) == classes and truth.shape[0] > 0
    image_index = {dataset.read_image_u8(p).tobytes(): k for k, p in enumerate(paths)}

    class RefBacked:
        batch = 2                                               # exercises the padded last batch (7 images)

        def predict_image_u8(self, imgs, quantized=False):
            self.imgs = imgs

        def detect(self, w, h, thresh, nms, relative=1, letter=0, max_rows=1024, quantized=False):
            assert (w, h, thresh, nms) == (1, 1, 0.005, 0.45)   # the settings the stored detections were made with
            dets = [_reference_boxes(image_index[im.tobytes()], im) for im in self.imgs]
            return dets, np.array([d.shape[0] for d in dets], np.int32)

    mAP, aps, st = dataset.evaluate_map(RefBacked(), paths, truth, classes, 0.5, 0.24)
    out = open(os.path.join(root, "ref_stdout.txt")).read()
    map_ref = float(re.search(r"mean average precision \(mAP\) = ([0-9.]+)", out).group(1))
    tp, fp, fn = re.search(r"TP = (\d+), FP = (\d+), FN = (\d+)", out).groups()
    assert abs(mAP - map_ref) < 5e-7
    assert (int(st["tp"]), int(st["fp"]), int(st["fn"])) == (int(tp), int(fp), int(fn))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_map_driver_on_the_gpu_equals_validate_detector_map(precision, workdir):
    """SURVEY 8f row 4 on the device: dataset.evaluate_map with the REAL Network -- u8 frames -> yb_network_predict_image_u8
    (device resize) -> forward -> yb_network_detect (device decode + NMS) -> yb_map_evaluate -- on the on-disk dataset the
    reference's validate_detector_map (src/additionally.c:4541-4898) was run on: same TP / FP / FN, same mAP."""
    import yolo2_light_b200 as yb
    from yolo2_light_b200 import dataset
    name = "tiny64"
    cfg, wts = util.model_files(name, workdir)
    root = os.path.join(workdir, "mapset_tiny64_50")          # written by test_map_accounting_equals_reference
    if not os.path.exists(os.path.join(root, "ref_stdout.txt")):
        test_map_accounting_equals_reference(name, 0.5, workdir)
    paths, names, truth = dataset.load_validation_set(os.path.join(root, "data.cfg"))
    net = yb.load_network(cfg, wts, batch=2)                  # 7 images: exercises the padded last batch
    if precision == "fp32":
        net.set_precision(yb.YB_PREC_FP32)
    classes = len(names)
    mAP, aps, st = dataset.evaluate_map(net, paths, truth, classes, 0.5, 0.24)
    out = open(os.path.join(root, "ref_stdout.txt")).read()
    map_ref = float(re.search(r"mean average precision \(mAP\) = ([0-9.]+)", out).group(1))
    tp, fp, fn = (int(v) for v in re.search(r"TP = (\d+), FP = (\d+), FN = (\d+)", out).groups())
    if precision == "fp32":
        assert abs(mAP - map_ref) < 5e-6
        assert (int(st["tp"]), int(st["fp"]), int(st["fn"])) == (tp, fp, fn)
    else:   # bf16 tensor cores: detections within 1e-3 of the reference's; a borderline box may change sides
        assert abs(mAP - map_ref) < 0.02
        assert abs(int(st["tp"]) - tp) <= 2 and abs(int(st["fn"]) - fn) <= 2
