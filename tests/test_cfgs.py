"""Generated model definitions == the reference's shipped assets, as seen by the reference's own parser; and the
product parser == the reference parser on every generated model.  The assets and the reference parser's view of each
model are stored in tests/golden/reference.json ("cfg_assets") and reference_arrays.npz ("parse_*")."""
import os

import numpy as np
import pytest

import ybtest_util as util
from yolo2_light_b200 import cfgs

ASSETS = [("yolov3", lambda: cfgs.yolov3(416, 416), "yolov3.cfg"), ("spp", cfgs.yolov3_spp, "yolov3-spp.cfg"),
          ("tiny", cfgs.yolov3_tiny, "yolov3-tiny.cfg"), ("xnor", cfgs.tiny_yolo_obj_xnor, "tiny-yolo-obj_xnor.cfg"),
          ("v2voc", cfgs.yolov2_voc, "yolov2-voc.cfg"), ("tinyvoc", cfgs.tiny_yolo_voc, "tiny-yolo-voc.cfg")]
FIELDS = ["type", "activation", "batch_normalize", "h", "w", "c", "n", "size", "stride", "pad", "out_h", "out_w",
          "out_c", "xnor", "quantized", "index", "classes", "coords", "softmax", "total", "reverse", "outputs"]


# keys of the shipped assets that only matter for training / drawing and are not emitted by the generators
TRAINING_KEYS = {"momentum", "decay", "angle", "saturation", "exposure", "hue", "learning_rate", "burn_in",
                 "max_batches", "policy", "steps", "scales", "jitter", "ignore_thresh", "truth_thresh", "random",
                 "rescore", "object_scale", "noobject_scale", "class_scale", "coord_scale", "absolute", "thresh",
                 "bias_match"}


@pytest.mark.parametrize("name,build,asset", ASSETS)
def test_generated_cfg_text_equals_reference_asset(name, build, asset):
    """Section by section, every option the forward path reads has the same value in the generated model and in
    the shipped asset (text level, with the reference's own line grammar)."""
    gen = cfgs.parse_text(cfgs.to_text(build()))
    ref = util.reference()["cfg_assets"][asset]
    assert len(gen) == len(ref)
    for i, ((tg, og), (tr, orf)) in enumerate(zip(gen, ref)):
        assert tg == tr, (i, tg, tr)
        keys = (set(og) | set(orf)) - TRAINING_KEYS
        if i == 0:
            keys -= {"batch", "subdivisions"}   # the app always overrides the batch (main.c:160)
        for k in keys:
            vg, vr = og.get(k), orf.get(k)
            if k in ("anchors", "input_calibration", "layers", "mask"):
                vg = [float(t) for t in vg.split(",")]; vr = [float(t) for t in vr.split(",")]
            elif vg is not None and vr is not None and k != "activation":
                vg, vr = float(vg), float(vr)
            assert vg == vr, (name, i, tg, k, vg, vr)


def _assert_same_network(a, key):
    """The product parser's network `a` == the reference parser's recorded view of the same model (tests/golden/
    reference_arrays.npz, "parse_<key>_*")."""
    g = {k[len(key) + 7:]: v for k, v in util.reference_arrays().items() if k.startswith(f"parse_{key}_")}
    n, batch, h, w, c, inputs = g["net"].tolist()
    assert a.n == n and a.batch == batch, (key, a.n, n, a.batch, batch)
    assert (a.h, a.w, a.c, a.inputs) == (h, w, c, inputs), key
    for i, lb in enumerate(g["layers"].tolist()):
        la = a.layer(i)
        for k, v in zip(FIELDS, lb):
            assert la[k] == v, (key, i, k, la[k], v)
        if la["type_name"] == "YOLO":
            assert np.array_equal(la["mask"], g[f"l{i}_mask"]), (key, i)
            assert np.array_equal(la["anchors"], g[f"l{i}_biases"]), (key, i)
        if la["type_name"] == "REGION":
            assert np.array_equal(la["anchors"][:2 * la["n"]], g[f"l{i}_biases"]), (key, i)
        if la["type_name"] == "ROUTE":
            assert np.array_equal(la["input_layers"], g[f"l{i}_input_layers"]), (key, i)
    assert np.array_equal(a.input_calibration(), g["input_calibration"]), key


@pytest.mark.parametrize("name,build,asset,qs", [(a[0], a[1], a[2], (0, 1) if a[0] in ("tiny", "xnor") else (1,))
                                                 for a in ASSETS if a[0] in ("tiny", "xnor", "yolov3")])
def test_generated_cfg_equals_reference_asset(name, build, asset, qs, workdir):
    """...and the generated file builds the network the reference's own parser builds from the shipped asset."""
    import yolo2_light_b200 as yb
    p = cfgs.write_cfg(build(), os.path.join(workdir, "gen_" + name + ".cfg"))
    for q in qs:
        _assert_same_network(yb.parse_network_cfg(p, 1, q), f"{asset}_q{q}")


@pytest.mark.parametrize("name", list(util.ZOO) + ["full_tiny", "full_xnor"])
def test_product_parser_equals_reference_parser(name, workdir):
    import yolo2_light_b200 as yb
    if name.startswith("full_"):
        secs = cfgs.yolov3_tiny() if name == "full_tiny" else cfgs.tiny_yolo_obj_xnor()
        cfg = cfgs.write_cfg(secs, os.path.join(workdir, name + ".cfg"))
    else:
        cfg, _ = util.model_files(name, workdir)
    for q in (0, 1):
        a = yb.parse_network_cfg(cfg, 3, q)
        assert a.batch == 3
        _assert_same_network(a, f"{name}_q{q}")


def test_shape_tracer_agrees_with_product_parser(workdir):
    import yolo2_light_b200 as yb
    for name in util.ZOO:
        build = util.ZOO[name][0]
        cfg, _ = util.model_files(name, workdir)
        net = yb.parse_network_cfg(cfg, 1, 0)
        shapes = cfgs.conv_shapes(build())
        assert len(shapes) == net.n
        for i, s in enumerate(shapes):
            l = net.layer(i)
            if l["type_name"] in ("CONVOLUTIONAL", "MAXPOOL", "UPSAMPLE", "REORG", "ROUTE", "SHORTCUT"):
                assert (s["out_h"], s["out_w"], s["out_c"]) == (l["out_h"], l["out_w"], l["out_c"]), (name, i)


def test_parser_rejects_bad_input(workdir):
    import yolo2_light_b200 as yb
    with pytest.raises(yb.YbError):
        yb.parse_network_cfg(os.path.join(workdir, "does_not_exist.cfg"), 1, 0)
    p = os.path.join(workdir, "bad.cfg")
    open(p, "w").write("[net]\nwidth=32\nheight=32\nchannels=3\n[convolutional]\nfilters=8\nsize=1\n"
                       "[yolo]\nmask=0\nnum=1\nclasses=80\n")
    with pytest.raises(yb.YbError):   # filters= does not match classes/mask (additionally.c:3656-3660)
        yb.parse_network_cfg(p, 1, 0)
