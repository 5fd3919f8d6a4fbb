"""Generates tests/golden/reference.json and tests/golden/reference_arrays.npz: what the tests that compare with the
original yolo2_light compare against, computed once by its UNMODIFIED CPU code so that the suite runs without it.

    make -C oracle REF=<yolo2_light checkout>          # builds oracle/_ref/libyolo2ref_{scalar,fast}.so from it
    python tests/golden/make_reference_golden.py <yolo2_light checkout>

Bit-exact comparisons store a sha256 of the reference's values (tests/ybtest_util.digest); tolerance comparisons store
the values, or -- for full-size detection tensors -- a fixed random sample of them together with its indices.
"""
import json
import os
import re
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ybtest_util as util  # noqa: E402
from oracle import ref  # noqa: E402
from yolo2_light_b200 import cfgs  # noqa: E402

SAMPLE = 2048            # values kept per full-size detection tensor and image


def parse_record(arrays, key, path, batch, q):
    """The reference parser's view of a .cfg: the fields the product parser mirrors (test_cfgs.FIELDS) as one row per layer,
    the anchors / masks / route sources and the input calibration."""
    import test_cfgs
    r = ref.RefNet(path, None, batch, q, 0)
    arrays[f"parse_{key}_net"] = np.array([r.n, r.batch, r.height, r.width, r.channels, r.inputs], np.int32)
    arrays[f"parse_{key}_layers"] = np.array([[L[k] for k in test_cfgs.FIELDS] for L in r.layers], np.int32)
    arrays[f"parse_{key}_input_calibration"] = r.input_calibration()
    for i, L in enumerate(r.layers):
        if L["type_name"] == "YOLO":
            arrays[f"parse_{key}_l{i}_mask"] = r.array(i, "mask", L["n"], np.int32)
            arrays[f"parse_{key}_l{i}_biases"] = r.array(i, "biases", 2 * L["total"])
        elif L["type_name"] == "REGION":
            arrays[f"parse_{key}_l{i}_biases"] = r.array(i, "biases", 2 * L["n"])
        elif L["type_name"] == "ROUTE":
            arrays[f"parse_{key}_l{i}_input_layers"] = r.array(i, "input_layers", L["n"], np.int32)


def sample(arrays, key, out, seed):
    """A fixed random sample of each image of `out` [batch, ...]: indices and values."""
    rng = np.random.default_rng(seed)
    for b in range(out.shape[0]):
        flat = out[b].ravel()
        idx = np.sort(rng.choice(flat.size, min(SAMPLE, flat.size), replace=False)).astype(np.int32)
        arrays[f"{key}_b{b}_idx"] = idx
        arrays[f"{key}_b{b}_val"] = flat[idx].astype(np.float32)


def detection_outputs(rnet, x):
    outs = []
    for b in range(x.shape[0]):
        rnet.predict(x[b:b + 1])
        outs.append({i: rnet.output(i)[0].copy() for i, L in enumerate(rnet.layers) if L["type_name"] in ("YOLO", "REGION")})
    return {i: np.stack([o[i] for o in outs]) for i in outs[0]}


def main(reference_tree):
    import test_calibration
    import test_cfgs
    import test_host_prep
    import test_map
    import test_oracle_vs_reference
    wd = tempfile.mkdtemp()
    g, arrays = {}, {}
    os.environ.setdefault("OMP_NUM_THREADS", str(min(os.cpu_count() or 1, 32)))

    # entropy_calibration (test_calibration)
    g["calibration"] = {}
    for bw, mb in test_calibration.PARAMS:
        g["calibration"][f"{bw},{mb}"] = [ref.entropy_calibration(np.asarray(a, np.float32), bw, mb)
                                          for _, a in test_calibration._cases()]

    # the shipped model definitions and the reference parser (test_cfgs)
    g["cfg_assets"] = {}
    for name, build, asset in test_cfgs.ASSETS:
        path = os.path.join(reference_tree, "bin", asset)
        g["cfg_assets"][asset] = cfgs.parse_text(open(path).read())
        if name in ("tiny", "xnor", "yolov3"):
            for q in (0, 1):
                parse_record(arrays, f"{asset}_q{q}", path, 1, q)
    for name in list(util.ZOO) + ["full_tiny", "full_xnor"]:
        if name.startswith("full_"):
            secs = cfgs.yolov3_tiny() if name == "full_tiny" else cfgs.tiny_yolo_obj_xnor()
            cfg = cfgs.write_cfg(secs, os.path.join(wd, name + ".cfg"))
        else:
            cfg, _ = util.model_files(name, wd)
        for q in (0, 1):
            parse_record(arrays, f"{name}_q{q}", cfg, 3, q)

    # host-side model preparation (test_host_prep, test_gpu_parity.test_dropin_from_reference_prepared_layers)
    g["prepared"] = {}
    for name, q in test_host_prep.PREP_CASES + [("tiny64", 0)]:
        cfg, wts = util.model_files(name, wd)
        r = ref.RefNet(cfg, wts, 1, q, 7)
        rec = {}
        for i, L in enumerate(r.layers):
            if L["type_name"] != "CONVOLUTIONAL":
                continue
            nw = L["n"] * L["c"] * L["size"] ** 2
            d = {"batch_normalize": L["batch_normalize"], "weights": util.digest(r.array(i, "weights", nw)),
                 "biases": util.digest(r.array(i, "biases", L["n"]))}
            if q:
                d["weights_int8"] = util.digest(r.array(i, "weights_int8", nw, np.int8), np.int8)
                d["weights_quant_multipler"] = L["weights_quant_multipler"]
                d["input_quant_multipler"] = L["input_quant_multipler"]
            if L["xnor"]:
                d["mean_arr"] = util.digest(r.array(i, "mean_arr", L["n"]))
            rec[str(i)] = d
        g["prepared"][f"{name}_q{q}"] = rec
    cfg, wts = util.model_files("tiny64", wd)
    r = ref.RefNet(cfg, wts, 1, 0, 0)
    g["unprepared_tiny64"] = {}
    for i, L in enumerate(r.layers):
        if L["type_name"] == "CONVOLUTIONAL":
            g["unprepared_tiny64"][str(i)] = {}
            for arr in ("weights", "biases", "scales", "rolling_mean", "rolling_variance"):
                a = r.array(i, arr, L["n"] * L["c"] * L["size"] ** 2 if arr == "weights" else L["n"])
                g["unprepared_tiny64"][str(i)][arr] = None if a is None else util.digest(a)

    # every layer output of whole networks (test_oracle_vs_reference)
    g["layers"] = {}
    for name, q, batch in [c + (1,) for c in test_oracle_vs_reference.WHOLE_NETWORK_CASES] + [("xnor64", 0, 2)]:
        cfg, wts = util.model_files(name, wd)
        r = ref.RefNet(cfg, wts, batch, q, 7)
        r.predict(util.images(name, batch))
        g["layers"][f"{name}_q{q}_b{batch}"] = [[L["type_name"], list(r.output(i).shape), util.digest(r.output(i))]
                                                for i, L in enumerate(r.layers)]
    g["resize"] = {}
    for h, w, oh, ow in test_oracle_vs_reference.RESIZE_SHAPES:
        img = test_oracle_vs_reference.resize_input(h, w)
        g["resize"][f"{h},{w},{oh},{ow}"] = util.digest(ref.load_resize_u8(img, ow, oh))

    # mAP accounting (test_map): the reference's detections of each image and what validate_detector_map printed
    g["map"] = {}
    for name, iou in test_map.MAP_CASES:
        cfg, wts = util.model_files(name, wd)
        rnet = ref.RefNet(cfg, wts, 1, 0, 7)
        classes = rnet.layers[-1]["classes"]

        def boxes(k, img):
            rnet.predict(ref.load_resize_u8(img, rnet.width, rnet.height)[None])
            return np.delete(rnet.get_boxes(1, 1, 0.005, 0.45), 5, axis=1)

        root, rows, _ = test_map.write_mapset(name, iou, wd, classes, boxes)
        out = ref.validate_map(os.path.join(root, "data.cfg"), cfg, wts, 0.24, 0, iou, os.path.join(root, "out.txt"))
        keep = re.compile(r"class_id = |mean average precision|average precision \(AP\)|TP = |precision = |detections_count = ")
        g["map"][f"{name}_{int(iou * 100)}"] = {"classes": classes, "stdout": "\n".join(
            line for line in out.splitlines() if keep.search(line))}
        for k, r in enumerate(rows):
            arrays[f"map_{name}_{int(iou * 100)}_img{k}"] = r

    # ---- what the GPU tests compare against ----------------------------------------------------------------
    import test_gpu_detect
    import test_gpu_fullsize
    import test_gpu_parity
    for name, q in test_gpu_detect.REF_CASES:
        cfg, wts = test_gpu_detect._bigger(name, wd, 160, 160)
        x = cfgs.synthetic_images(3, 3, 160, 160, seed=45)
        r = ref.RefNet(cfg, wts, 1, q, 7)
        thresh = 0.2 if name == "tiny" else 0.05
        for b in range(3):
            r.predict(x[b:b + 1])
            arrays[f"detect_{name}_q{q}_b{b}"] = np.delete(r.get_boxes(640, 480, thresh, 0.45), 5, axis=1)

    for key, (fname, secs, seed, q, kind, nimg, iseed) in test_gpu_fullsize.REF_RUNS.items():
        cfg, wts = test_gpu_fullsize._files(wd, fname, secs, seed=seed)
        x = cfgs.synthetic_images(nimg, 3, int(secs[0][1]["height"]), int(secs[0][1]["width"]), seed=iseed)
        for i, o in detection_outputs(ref.RefNet(cfg, wts, 1, q, 7, kind=kind), x).items():
            sample(arrays, f"full_{key}_l{i}", o, seed=len(arrays))
        print(key, "done", flush=True)

    for name, q in test_gpu_parity.DROPIN_CASES:
        cfg, wts = util.model_files(name, wd)
        r = ref.RefNet(cfg, wts, 1, q, 7)
        r.predict(util.images(name, 1))
        arrays[f"dropin_{name}_q{q}_boxes"] = r.get_boxes(640, 480, 0.3, 0.45)

    g["device_calibration"] = {}
    for name in test_gpu_parity.CALIB_NAMES:
        cfg, wts = util.model_files(name, wd)
        r = ref.RefNet(cfg, wts, 1, 0, 7)
        x = util.images(name, 2)
        convs = [i for i, L in enumerate(r.layers) if L["type_name"] == "CONVOLUTIONAL"]
        per_image = []
        for b in range(2):
            r.predict(x[b:b + 1])
            per_image.append([ref.entropy_calibration(x[b] if i == 0 else r.output(i - 1)) for i in convs])
        g["device_calibration"][name] = per_image

    secs = test_gpu_parity.xnor_fallback_model()
    cfg = cfgs.write_cfg(secs, os.path.join(wd, "xnor_fb.cfg"))
    wts = cfgs.write_weights(secs, os.path.join(wd, "xnor_fb.weights"), seed=23)
    x = cfgs.synthetic_images(2, 3, 32, 32, seed=24)
    r = ref.RefNet(cfg, wts, 1, 0, 7)
    g["xnor_fallback"] = []
    for b in range(2):
        r.predict(x[b:b + 1])
        g["xnor_fallback"].append([util.digest(r.output(i)[0]) for i in range(4)])
        arrays[f"xnor_fallback_b{b}"] = r.output(len(r.layers) - 1)[0]

    with open(os.path.join(HERE, "reference.json"), "w") as f:
        json.dump(g, f, indent=0, sort_keys=True, separators=(",", ":"))
        f.write("\n")
    np.savez_compressed(os.path.join(HERE, "reference_arrays.npz"), **arrays)
    for fn in ("reference.json", "reference_arrays.npz"):
        print(fn, os.path.getsize(os.path.join(HERE, fn)) // 1024, "KiB")


if __name__ == "__main__":
    if len(sys.argv) != 2 or not ref.available("scalar"):
        sys.exit(__doc__)
    main(sys.argv[1])
