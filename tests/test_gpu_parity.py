"""Parity of the CUDA engine (through the C ABI) against the CPU oracle, the reference build (oracle/_ref), and the
golden vectors made by the reference (tests/golden).  GPU box only:  python -m pytest tests -m gpu

Bars (BASELINE.json north_star): XNOR popcounts and INT8 s32 accumulators bit-exact; the float epilogues of
those paths bit-exact too (same op order as the reference); FP32-variant convolutions: f32 CUDA-core path
<= 1e-5 rel-L2 per layer, bf16 tensor-core path <= 1e-3 rel-L2 on the activated detection tensors.
"""
import os

import numpy as np
import pytest

import ybtest_util as util
from yolo2_light_b200 import cfgs

pytestmark = pytest.mark.gpu


def _load(name, workdir, batch, q, precision=None, fuse=None, keep_counts=False):
    import yolo2_light_b200 as yb
    cfg, wts = util.model_files(name, workdir)
    net = yb.load_network(cfg, wts, batch=batch, quantized=q)
    if precision is not None:
        net.set_precision(precision)
    if fuse is not None:
        net.set_option("fuse", int(fuse))
    if keep_counts:
        net.set_option("keep_counts", 1)
    return net


def _oracle_outs(net, x, q):
    from oracle import port
    layers = net.layers
    per_image = [port.run_network(layers, x[b:b + 1], quantized=bool(q)) for b in range(x.shape[0])]
    return [np.concatenate([pi[i] for pi in per_image], axis=0) for i in range(len(layers))]


# ---- exact f32 mode: every layer of every model family against the oracle ---------------------------------
@pytest.mark.parametrize("name", ["tiny64", "v3_32", "spp32", "v2voc32", "tinyvoc64", "tiny_w96_h64", "v3_w64_h96"])
def test_fp32_mode_every_layer(name, workdir):
    import yolo2_light_b200 as yb
    B = 2
    net = _load(name, workdir, B, 0, precision=yb.YB_PREC_FP32, fuse=False)
    x = util.images(name, B)
    net.predict(x)
    outs = _oracle_outs(net, x, 0)
    for i, o in enumerate(outs):
        got = net.fetch_layer(i)
        t = net.layer(i)["type_name"]
        err = util.rel_l2(got, o.reshape(got.shape))
        assert err <= 1e-5, (name, i, t, err)
        # f32 mode runs the reference's own summation order (c, ky, kx) with separately rounded products and sums
        # (additionally.c:1272-1286): everything but the transcendental layers is bit-identical to the scalar build
        if t not in ("YOLO", "REGION"):
            assert util.bits_equal(got, o.reshape(got.shape)), (name, i, t, float(np.abs(got - o.reshape(got.shape)).max()))
    # the returned pointer is the last layer's host output, as network_predict_cpu returns it
    last = net.layer_output(net.n - 1)
    assert util.rel_l2(last, outs[-1].reshape(last.shape)) <= 1e-5


@pytest.mark.parametrize("name", ["v3_32", "spp32", "v2voc32"])
def test_fp32_mode_fused_equals_unfused(name, workdir):
    """conv+shortcut fusion and route aliasing change the plan, not the results."""
    import yolo2_light_b200 as yb
    B = 2
    x = util.images(name, B)
    a = _load(name, workdir, B, 0, precision=yb.YB_PREC_FP32, fuse=False)
    b = _load(name, workdir, B, 0, precision=yb.YB_PREC_FP32, fuse=True)
    a.predict(x); b.predict(x)
    assert b.last_launches() < a.last_launches()
    for i, oa in a.detection_outputs().items():
        assert util.bits_equal(oa, b.layer_output(i)), (name, i)


# ---- XNOR path --------------------------------------------------------------------------------------------
def test_xnor_counts_and_outputs_bit_exact_per_layer(workdir):
    """Each XNOR conv fed the oracle's own input: popcounts equal as integers, outputs equal bit-for-bit."""
    from oracle import port
    name, B = "xnor64", 2
    net = _load(name, workdir, B, 0, fuse=False, keep_counts=True)
    x = util.images(name, B)
    outs = _oracle_outs(net, x, 0)
    layers = net.layers
    n_x = 0
    for i, l in enumerate(layers):
        if l["type_name"] != "CONVOLUTIONAL" or not l["xnor"]:
            continue
        n_x += 1
        xin = outs[i - 1]
        got = net.forward_convolutional_layer(i, xin, variant=0)
        exp, cnt = port.conv_xnor(xin, l["weights"], l["biases"], l["mean_arr"], l["n"], l["size"], l["activation"],
                                  want_counts=True)
        assert util.bits_equal(got, exp), (i, np.abs(got - exp).max())
    assert n_x == 7


def test_xnor_network_counts_bit_exact(workdir):
    """Whole network, end to end: the f32 stem reproduces the reference's summation order bit for bit, so every XNOR
    layer sees exactly the reference's signs: ALL raw popcounts and every XNOR layer's float output are identical."""
    from oracle import port
    name, B = "xnor64", 2
    net = _load(name, workdir, B, 0, fuse=False, keep_counts=True)
    x = util.images(name, B)
    net.predict(x)
    outs = _oracle_outs(net, x, 0)
    layers = net.layers
    for i, l in enumerate(layers):
        if l["type_name"] == "CONVOLUTIONAL" and l["xnor"]:
            got = net.fetch_counts(i)
            _, cnt = port.conv_xnor(outs[i - 1], l["weights"], l["biases"], l["mean_arr"], l["n"], l["size"],
                                    l["activation"], want_counts=True)
            same = float((got == cnt).mean())
            assert same == 1.0, (i, same)
            out = net.fetch_layer(i)
            assert util.bits_equal(out, outs[i].reshape(out.shape)), i
    reg = net.layer_output(net.n - 1)
    assert util.rel_l2(reg, outs[-1].reshape(reg.shape)) <= 1e-3


# ---- INT8 path --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny64", "tinyvoc64", "v3_32"])
def test_int8_accumulators_and_outputs_bit_exact_per_layer(name, workdir):
    from oracle import port
    B = 2
    net = _load(name, workdir, B, 1, fuse=False)
    x = util.images(name, B)
    outs = _oracle_outs(net, x, 1)
    layers = net.layers
    n_q = 0
    for i, l in enumerate(layers):
        if l["type_name"] != "CONVOLUTIONAL" or i < 1 or l["activation"] == 3:
            continue
        n_q += 1
        if name == "v3_32" and n_q > 12:
            break
        xin = outs[i - 1]
        got = net.forward_convolutional_layer(i, xin, variant=1)
        exp = port.conv_int8(xin, l["weights_int8"], l["biases"], l["input_quant_multipler"],
                             l["weights_quant_multipler"], l["n"], l["size"], l["stride"], l["pad"], l["activation"])
        assert util.bits_equal(got, exp), (name, i, np.abs(got - exp).max())
    assert n_q >= 7


def test_int8_network_accumulators(workdir):
    from oracle import port
    name, B = "tiny64", 2
    net = _load(name, workdir, B, 1, fuse=False, keep_counts=True)
    x = util.images(name, B)
    net.predict(x, quantized=True)
    outs = _oracle_outs(net, x, 1)
    layers = net.layers
    for i, l in enumerate(layers):
        if l["type_name"] == "CONVOLUTIONAL" and i >= 1 and l["activation"] != 3:
            got = net.fetch_counts(i, quantized=True)
            _, acc = port.conv_int8(outs[i - 1], l["weights_int8"], l["biases"], l["input_quant_multipler"],
                                    l["weights_quant_multipler"], l["n"], l["size"], l["stride"], l["pad"],
                                    l["activation"], want_acc=True)
            same = float((got == acc).mean())
            assert same == 1.0, (i, same)   # bit-exact stem -> bit-exact s8 inputs -> identical s32 accumulators end to end
            out = net.fetch_layer(i, quantized=True)
            assert util.bits_equal(out, outs[i].reshape(out.shape)), i
    for i, o in net.detection_outputs().items():
        assert util.rel_l2(o, outs[i].reshape(o.shape)) <= 2e-3, i


# ---- golden vectors produced by the reference itself ------------------------------------------------------
@pytest.mark.parametrize("name,q", [("tiny64", 0), ("tiny64", 1), ("xnor64", 0), ("v3_32", 0), ("spp32", 0),
                                    ("v2voc32", 0), ("tinyvoc64", 1), ("v3_32", 1)])
def test_detection_outputs_vs_reference_golden(name, q, workdir):
    import yolo2_light_b200 as yb
    g = np.load(os.path.join(util.GOLDEN, f"{name}_q{q}.npz"))
    B = 2
    net = _load(name, workdir, B, q, precision=yb.YB_PREC_FP32)
    x = util.images(name, B)
    net.predict(x, quantized=bool(q))
    n = 0
    for i, o in net.detection_outputs().items():
        for b in range(B):
            ref = g[f"b{b}_out{i}"]
            err = util.rel_l2(o[b], ref.reshape(o[b].shape))
            assert err <= (2e-3 if q else 1e-5), (name, q, i, b, err)
            n += 1
    assert n >= 2


# ---- the drop-in path behind the reference's own loader -----------------------------------------------------
DROPIN_CASES = [("tiny64", 0), ("tiny64", 1), ("xnor64", 0)]


@pytest.mark.parametrize("name,q", DROPIN_CASES)
def test_dropin_from_reference_prepared_layers(name, q, workdir):
    """Model parsed, loaded, folded, binarised and quantised the way the REFERENCE's host code does it (arrays bit-identical
    to its own, checked against their digests); those arrays handed to the engine as yb_layer_desc[] (what INTEGRATION.md's
    glue does); result vs the reference's own predict and decoder (tests/golden)."""
    import ctypes as C
    import yolo2_light_b200 as yb
    from test_host_prep import assert_prepared_like_reference
    cfg, wts = util.model_files(name, workdir)
    prepared = yb.load_network(cfg, wts, batch=1, quantized=q)
    layers = prepared.layers
    assert_prepared_like_reference(layers, name, q)
    keep, descs = [], []

    def ptr(arr, ctype):
        if arr is None:
            return None
        keep.append(arr)
        return arr.ctypes.data_as(C.POINTER(ctype))

    for i, L in enumerate(layers):
        d = yb.LayerDesc()
        for k in ("type", "activation", "batch_normalize", "h", "w", "c", "n", "size", "stride", "pad", "out_h",
                  "out_w", "out_c", "xnor", "quantized", "index", "classes", "coords", "softmax", "total", "reverse"):
            setattr(d, k, L[k])
        d.scale = L["scale"]
        t = L["type_name"]
        if t == "CONVOLUTIONAL":
            d.weights = ptr(np.ascontiguousarray(L["weights"], np.float32), C.c_float)
            d.biases = ptr(np.ascontiguousarray(L["biases"], np.float32), C.c_float)
            if q:
                d.weights_int8 = ptr(np.ascontiguousarray(L["weights_int8"], np.int8), C.c_int8)
                d.weights_quant_multipler = L["weights_quant_multipler"]
                d.input_quant_multipler = L["input_quant_multipler"]
            if L["xnor"]:
                d.mean_arr = ptr(np.ascontiguousarray(L["mean_arr"], np.float32), C.c_float)
        elif t == "ROUTE":
            d.input_layers = ptr(np.ascontiguousarray(L["input_layers"], np.int32), C.c_int)
        elif t == "YOLO":
            d.mask = ptr(np.ascontiguousarray(L["mask"], np.int32), C.c_int)
            d.anchors = ptr(np.ascontiguousarray(L["anchors"], np.float32), C.c_float)
        elif t == "REGION":
            d.anchors = ptr(np.ascontiguousarray(L["anchors"], np.float32), C.c_float)
        descs.append(d)
    net = yb.network_from_layers(descs, 1, prepared.h, prepared.w, prepared.c, q)
    net.set_precision(yb.YB_PREC_FP32)
    x = util.images(name, 1)
    net.predict(x, quantized=bool(q))
    g = np.load(os.path.join(util.GOLDEN, f"{name}_q{q}.npz"))          # the reference's predict of this very image
    for i, o in net.detection_outputs().items():
        r = g[f"b0_out{i}"]
        assert util.rel_l2(o, r.reshape(o.shape)) <= (2e-3 if q else 1e-5), (name, q, i)
    # decoded boxes agree with the reference's get_network_boxes + do_nms_sort
    mine = net.get_network_boxes(0, 640, 480, 0.3, 0.45)
    theirs = util.reference_arrays()[f"dropin_{name}_q{q}_boxes"]
    assert mine.shape[0] == theirs.shape[0]
    if mine.shape[0]:
        a = mine[np.lexsort(mine[:, :4].T[::-1])]
        t2 = np.delete(theirs, 5, axis=1)
        b = t2[np.lexsort(t2[:, :4].T[::-1])]
        assert np.allclose(a[:, :5], b[:, :5], rtol=2e-3 if q else 1e-4, atol=1e-5)


@pytest.mark.parametrize("name,q", [("tiny_w96_h64", 0), ("tiny_w96_h64", 1), ("v3_w64_h96", 0)])
def test_non_square_inputs_default_precision(name, q, workdir):
    """H != W through the default (tensor-core where the shape allows) paths, batch 3 (odd)."""
    B = 3
    net = _load(name, workdir, B, q)
    x = util.images(name, B)
    net.predict(x, quantized=bool(q))
    outs = _oracle_outs(net, x, q)
    for i, o in net.detection_outputs().items():
        assert util.rel_l2(o, outs[i].reshape(o.shape)) <= 3e-3, (name, q, i)


def test_empty_and_edge_inputs(workdir):
    """All-zero and all-one images, batch 1 and 3, odd batch through the same engine path."""
    import yolo2_light_b200 as yb
    name = "tiny64"
    for B in (1, 3):
        net = _load(name, workdir, B, 0, precision=yb.YB_PREC_FP32)
        for val in (0.0, 1.0):
            x = np.full((B, 3, 64, 64), val, np.float32)
            net.predict(x)
            outs = _oracle_outs(net, x, 0)
            for i, o in net.detection_outputs().items():
                assert util.rel_l2(o, outs[i].reshape(o.shape)) <= 1e-5
    with pytest.raises(yb.YbError):
        net.predict(np.zeros((1, 3, 8, 8), np.float32))


@pytest.mark.skipif(not __import__("oracle.ref", fromlist=["x"]).available("dropin"), reason="drop-in build absent")
@pytest.mark.parametrize("name,q", [("tiny64", 0), ("tiny64", 1), ("xnor64", 0), ("v3_32", 0)])
def test_true_dropin_behind_reference_host_code(name, q, workdir):
    """oracle/_ref/libyolo2ref_dropin.so = the reference's UNMODIFIED host code (parser, loader, BN fold, binary
    weights, quantisation, get_network_boxes, do_nms_sort) + integration/yolo2_light_b200_glue.c + our engine:
    network_predict_b200(net, input) in the slot of network_predict_cpu; detections through the reference's own
    decoder must agree with its CPU path."""
    from oracle import ref
    cfg, wts = util.model_files(name, workdir)
    x = util.images(name, 1)
    net = ref.RefNet(cfg, wts, 1, q, 7, kind="dropin")
    net.predict(x)                                   # reference CPU forward
    det_idx = [i for i, L in enumerate(net.layers) if L["type_name"] in ("YOLO", "REGION")]
    cpu_out = {i: net.output(i).copy() for i in det_idx}
    cpu_boxes = net.get_boxes(640, 480, 0.25, 0.45)
    net.predict_b200(x)                              # same `network`, forward on the B200
    tol = 3e-3
    for i in det_idx:
        assert util.rel_l2(net.output(i), cpu_out[i]) <= tol, (name, q, i)
    gpu_boxes = net.get_boxes(640, 480, 0.25, 0.45)
    assert abs(gpu_boxes.shape[0] - cpu_boxes.shape[0]) <= max(2, cpu_boxes.shape[0] // 50)
    # the glue's device-side decode + NMS (get_network_boxes_nms_b200) == the reference's decoder run on the very
    # tensors network_predict_b200 put into l.output
    dev = net.get_boxes_b200(640, 480, 0.25, 0.45)
    assert dev.shape[0] == gpu_boxes.shape[0]
    if dev.shape[0]:
        a = np.delete(dev, 5, axis=1); e = np.delete(gpu_boxes, 5, axis=1)
        a = a[np.lexsort(a[:, :4].T[::-1])]; e = e[np.lexsort(e[:, :4].T[::-1])]
        assert np.allclose(a[:, :4], e[:, :4], rtol=1e-6, atol=1e-7)
        assert np.array_equal(a[:, 4:], e[:, 4:])


@pytest.mark.parametrize("src_hw", [(48, 80), (64, 64), (97, 131), (200, 33)])
def test_device_input_pipeline_bit_exact(src_hw, workdir):
    """u8 HWC -> /255 -> resize_image on the device == the reference's load_image_stb + resize_image bit-for-bit
    (oracle port, itself pinned to the reference in tests/test_oracle_vs_reference.py), then the same forward."""
    import yolo2_light_b200 as yb
    from oracle import port
    name, B = "tiny64", 2
    net = _load(name, workdir, B, 0, precision=yb.YB_PREC_FP32)
    rng = np.random.default_rng(7)
    imgs = rng.integers(0, 256, (B, src_hw[0], src_hw[1], 3), dtype=np.uint8)
    net.predict_image_u8(imgs)
    got = net.fetch_input()
    exp = np.stack([port.load_resize_u8(imgs[b], net.w, net.h) for b in range(B)])
    assert util.bits_equal(got, exp), float(np.abs(got - exp).max())
    a = {i: o.copy() for i, o in net.detection_outputs().items()}
    net.predict(exp)
    for i, o in net.detection_outputs().items():
        assert util.bits_equal(o, a[i])


CALIB_NAMES = ["tiny64", "v3_32"]


@pytest.mark.parametrize("name", CALIB_NAMES)
def test_int8_calibration_on_device(name, workdir):
    """SURVEY 8f row 3: |x| histograms of every convolution input on the GPU (exact integers) + the reference's KL
    search; multipliers against entropy_calibration run by the reference on ITS activations, image by image
    (tests/golden/reference.json, "device_calibration")."""
    import yolo2_light_b200 as yb
    B = 2
    cfg, wts = util.model_files(name, workdir)
    x = util.images(name, B)
    net = yb.load_network(cfg, wts, batch=B)
    net.set_precision(yb.YB_PREC_FP32)
    # (1) the histogram kernel counts exactly what the reference's binning counts
    net.set_option("fuse", 0)
    net.predict(x)
    convs = [i for i, l in enumerate(net.layers) if l["type_name"] == "CONVOLUTIONAL"]
    for i in convs[:6]:
        for b in range(B):
            src = x[b] if i == 0 else net.fetch_layer(i - 1)[b]
            bins = np.minimum(np.floor(np.abs(src.astype(np.float64)) * 16.0 + 0.5).astype(np.int64), 4095)
            exp = np.bincount(bins.ravel(), minlength=4096).astype(np.uint32)
            assert np.array_equal(net.input_histogram(i, b), exp), (i, b)
    # (2) whole tool
    mult = net.calibrate(x)
    assert mult.shape == (B, len(convs)) and np.all(mult > 0)
    expected = util.reference()["device_calibration"][name]
    same = total = 0
    for b in range(B):
        assert len(expected[b]) == len(convs)
        for k, i in enumerate(convs):
            theirs = expected[b][k]
            total += 1
            same += np.float32(theirs) == mult[b, k]
            # activations differ in the last bit (f32 summation order): a count may cross a bin edge and move the optimum
            assert abs(mult[b, k] - theirs) <= 0.05 * theirs, (b, i, mult[b, k], theirs)
    assert same >= 0.8 * total, (same, total)
    line = yb.api.format_input_calibration(mult)
    assert line.startswith("input_calibration = ") and line.endswith(", 16") and line.count(",") == len(convs)
    # the engine is back in its normal (fused) configuration and still right
    net.set_option("fuse", 1)
    net.predict(x)


@pytest.mark.parametrize("name,q", [("tiny64", 1), ("xnor64", 0), ("tinyvoc64", 1), ("tiny_w96_h64", 1)])
def test_maxpool_fused_with_quantise_or_binarise_is_bit_exact(name, q, workdir):
    """fuse=1 lets a max-pool write the s8 / sign input of the integer convolution that follows (k_maxpool_fused):
    the same values in the same order as max-pool + quantise / binarise, so everything downstream is bit-identical."""
    import yolo2_light_b200 as yb
    B = 3
    x = util.images(name, B)
    res = []
    for fuse in (0, 1):
        net = _load(name, workdir, B, q, precision=yb.YB_PREC_FP32)
        net.set_option("fuse", fuse)
        net.set_option("keep_counts", 1)
        net.predict(x, quantized=bool(q))
        kinds = [k for _, k, _ in net.profile(quantized=bool(q))]
        ints = [i for i, l in enumerate(net.layers)
                if l["type_name"] == "CONVOLUTIONAL" and (l["xnor"] or (q and i >= 1 and l["activation"] != 3))]
        res.append((kinds, {i: o.copy() for i, o in net.detection_outputs().items()},
                    [net.fetch_counts(i, quantized=bool(q)) for i in ints]))
    k0, k1 = res[0][0], res[1][0]
    assert (k1.count("quantize") + k1.count("binarize")) < (k0.count("quantize") + k0.count("binarize")), (k0, k1)
    for i in res[0][1]:
        assert np.array_equal(res[0][1][i], res[1][1][i]), (name, i)
    for a, b in zip(res[0][2], res[1][2]):
        assert np.array_equal(a, b)


# ---- XNOR layers outside the bit GEMM's shape (stride != 1 or pad != 1): the reference's float-GEMM fallback ----------
def xnor_fallback_model():
    return [cfgs._net(32, 32), cfgs._conv(8, 3), cfgs._conv(16, 3, 2, xnor=1), cfgs._conv(16, 1, xnor=1),
            cfgs._conv(16, 3, xnor=1),                      # an ordinary XNOR layer behind them
            cfgs._conv(18, 1, bn=False, act="linear"), cfgs._yolo("0,1,2", cfgs.COCO_ANCHORS, 9, classes=1)]


def test_xnor_stride_pad_fallback_matches_reference(workdir):
    """yolov2_forward_network.c:40-50 + :204: such layers binarise the input to +-1 floats, swap in +-mean weights and run the
    ordinary im2col + gemm_nn.  The engine does the same (k_binarize_pm1 + exact-order float conv): bit-identical to the
    reference's outputs (tests/golden/reference.json, "xnor_fallback")."""
    import yolo2_light_b200 as yb
    secs = xnor_fallback_model()
    cfg = cfgs.write_cfg(secs, os.path.join(workdir, "xnor_fb.cfg"))
    wts = cfgs.write_weights(secs, os.path.join(workdir, "xnor_fb.weights"), seed=23)
    B = 2
    x = cfgs.synthetic_images(B, 3, 32, 32, seed=24)
    net = yb.load_network(cfg, wts, batch=B)
    net.set_option("fuse", 0)
    net.predict(x)
    for b in range(B):
        for i in range(4):
            assert util.digest(net.fetch_layer(i)[b]) == util.reference()["xnor_fallback"][b][i], (b, i)
        outs = net.detection_outputs()
        assert list(outs) == [len(secs) - 2]
        for i, o in outs.items():
            exp = util.reference_arrays()[f"xnor_fallback_b{b}"]
            assert util.rel_l2(o[b], exp.reshape(o[b].shape)) <= 1e-3


# ---- stem + max-pool + quantise / binarise in one kernel (exact nets) ------------------------------------------------------
@pytest.mark.parametrize("builder,w,h,q", [(cfgs.yolov3_tiny, 64, 64, 1), (cfgs.tiny_yolo_obj_xnor, 64, 64, 0), (cfgs.yolov3_tiny, 96, 64, 1)])
def test_fused_stem_pool_is_bit_identical_to_the_three_kernels(builder, w, h, q, workdir):
    """k_stem_pool (layers 0-1 + the integer layer's input conversion; full-width models: the stem has 16 filters) against the
    unfused plan: the first integer convolution, every later layer and the detections are bit-identical; layers 0 and 1 are
    no longer materialised."""
    import yolo2_light_b200 as yb
    B = 3
    secs = builder(w, h)
    cfg = cfgs.write_cfg(secs, os.path.join(workdir, f"sp_{builder.__name__}_{w}x{h}.cfg"))
    wts = cfgs.write_weights(secs, os.path.join(workdir, f"sp_{builder.__name__}_{w}x{h}.weights"), seed=61)
    x = cfgs.synthetic_images(B, 3, h, w, seed=62)
    nets = []
    for fuse in (0, 1):
        net = yb.load_network(cfg, wts, batch=B, quantized=q)
        net.set_option("fuse", fuse)
        net.set_option("keep_counts", 1)
        net.predict(x, quantized=bool(q))
        nets.append(net)
    a, b = nets
    assert b.last_launches() <= a.last_launches() - 3        # stem, max-pool and quantise / binarise became one launch
    with pytest.raises(yb.YbError):
        b.fetch_layer(0, quantized=bool(q))
    assert np.array_equal(a.fetch_counts(2, quantized=bool(q)), b.fetch_counts(2, quantized=bool(q)))
    assert util.bits_equal(a.fetch_layer(2, quantized=bool(q)), b.fetch_layer(2, quantized=bool(q)))
    # every later integer layer sees identical inputs: raw accumulators / popcounts equal to the end of the trunk
    n_int = 0
    for i, l in enumerate(a.layers):
        if l["type_name"] == "CONVOLUTIONAL" and i >= 2 and (l["xnor"] or (q and l["activation"] != 3)):
            assert np.array_equal(a.fetch_counts(i, quantized=bool(q)), b.fetch_counts(i, quantized=bool(q))), i
            n_int += 1
    assert n_int >= 6
    # the detection tensors differ only by the head's fused [yolo] epilogue (fast logistic) that `fuse` also switches on
    for i, o in a.detection_outputs().items():
        assert util.rel_l2(o, b.layer_output(i)) <= 1e-5, (builder.__name__, i)
    # production configuration (no raw-accumulator dump): the max-pools behind the integer convolutions run in their epilogues
    # (tc_plan_fuse_pool) -- every integer layer that is still materialised is bit-identical to the unfused plan
    c = yb.load_network(cfg, wts, batch=B, quantized=q)
    c.predict(x, quantized=bool(q))
    assert c.last_launches() < b.last_launches()
    n_cmp = n_gone = 0
    for i, l in enumerate(a.layers):
        if not (l["type_name"] == "CONVOLUTIONAL" and i >= 2 and (l["xnor"] or (q and l["activation"] != 3))):
            continue
        try:
            got = c.fetch_layer(i, quantized=bool(q))
        except yb.YbError:
            n_gone += 1
            continue
        assert util.bits_equal(got, a.fetch_layer(i, quantized=bool(q))), i
        n_cmp += 1
    assert n_cmp >= 3 and n_gone >= 2, (n_cmp, n_gone)
    for i, o in a.detection_outputs().items():
        assert util.rel_l2(o, c.layer_output(i)) <= 1e-5, (builder.__name__, i)
