"""Full-size BASELINE.json configurations on the GPU against the reference's CPU path (a fixed random sample of each of
its detection tensors is stored in tests/golden/reference_arrays.npz, "full_*"), plus size-independent properties."""
import os

import numpy as np
import pytest

import ybtest_util as util
from yolo2_light_b200 import cfgs

pytestmark = pytest.mark.gpu


def _files(workdir, name, secs, seed=1):
    cfg = os.path.join(workdir, name + ".cfg")
    wts = os.path.join(workdir, name + ".weights")
    if not os.path.exists(cfg):
        cfgs.write_cfg(secs, cfg)
        cfgs.write_weights(secs, wts, seed=seed)
    return cfg, wts


# key -> (model file name, sections, weight seed, quantized, reference build, images, image seed) of each reference run
REF_RUNS = {
    "yolov3_608": ("yolov3_608", cfgs.yolov3(608, 608), 1, 0, "fast", 2, 1234),
    "tiny_416_fp32": ("tiny_416", cfgs.yolov3_tiny(416, 416), 1, 0, "fast", 2, 1234),
    "tiny_416_int8": ("tiny_416", cfgs.yolov3_tiny(416, 416), 1, 1, "scalar", 2, 1234),
    "xnor_416": ("xnor_416", cfgs.tiny_yolo_obj_xnor(416, 416), 2, 0, "scalar", 2, 1234),
    "spp_608": ("spp_608", cfgs.yolov3_spp(608, 608), 3, 0, "scalar", 1, 11),
}


def _ref_rel_l2(outputs, key, nimg):
    """rel_l2 of every detection tensor and image against the stored sample of the reference run `key`."""
    assert outputs
    return {(i, b): util.sampled_rel_l2(o, f"full_{key}_l{i}", b) for i, o in outputs.items() for b in range(nimg)}


def test_yolov3_608_bf16_tensor_core_vs_reference(workdir):
    """BASELINE configs[1] (batch reduced to 2 for the CPU side): FP32 detections <= 1e-3 rel (rel-L2 on the
    activated yolo tensors, SURVEY 7.3) against the reference CPU path on the same weights and images."""
    import yolo2_light_b200 as yb
    secs = cfgs.yolov3(608, 608)
    cfg, wts = _files(workdir, "yolov3_608", secs)
    x = cfgs.synthetic_images(2, 3, 608, 608)
    net = yb.load_network(cfg, wts, batch=2)
    net.predict(x)
    for ib, err in _ref_rel_l2(net.detection_outputs(), "yolov3_608", 2).items():
        assert err <= 1e-3, (ib, err)
    prof = net.profile()
    assert sum(1 for _, k, _ in prof if k in ("conv_tc", "conv_tc2")) >= 70
    assert sum(1 for _, k, _ in prof if k == "conv_tc2") >= 30   # CTA-pair kernel carries the wide layers


def test_yolov3_tiny_416_fp32_and_int8_vs_reference(workdir):
    import yolo2_light_b200 as yb
    secs = cfgs.yolov3_tiny(416, 416)
    cfg, wts = _files(workdir, "tiny_416", secs)
    x = cfgs.synthetic_images(2, 3, 416, 416)
    net = yb.load_network(cfg, wts, batch=2)
    net.predict(x)
    for ib, err in _ref_rel_l2(net.detection_outputs(), "tiny_416_fp32", 2).items():
        assert err <= 1e-3, ib
    netq = yb.load_network(cfg, wts, batch=2, quantized=1)
    netq.predict(x, quantized=True)
    kinds = [k for _, k, _ in netq.profile(quantized=True)]
    assert kinds.count("conv_tc_i8") >= 8, kinds   # the s8 x s8 -> s32 tcgen05 path carries the INT8 layers
    for ib, err in _ref_rel_l2(netq.detection_outputs(), "tiny_416_int8", 2).items():
        assert err <= 2e-3, ib


def test_xnor_416_vs_reference(workdir):
    import yolo2_light_b200 as yb
    secs = cfgs.tiny_yolo_obj_xnor(416, 416)
    cfg, wts = _files(workdir, "xnor_416", secs, seed=2)
    x = cfgs.synthetic_images(2, 3, 416, 416)
    net = yb.load_network(cfg, wts, batch=2)
    net.predict(x)
    for ib, err in _ref_rel_l2(net.detection_outputs(), "xnor_416", 2).items():
        assert err <= 2e-3, ib


def test_batch_invariance_and_determinism_at_full_size(workdir):
    """Images are independent: image k of a batch of 16 == the same image run in a batch of 1 (bit-for-bit: the
    kernels' reduction order does not depend on the batch), and two runs of the same batch are identical."""
    import yolo2_light_b200 as yb
    secs = cfgs.yolov3(608, 608)
    cfg, wts = _files(workdir, "yolov3_608", secs)
    x = cfgs.synthetic_images(16, 3, 608, 608)
    net = yb.load_network(cfg, wts, batch=16)
    net.predict(x)
    a = {i: o.copy() for i, o in net.detection_outputs().items()}
    net.predict(x)
    for i, o in net.detection_outputs().items():
        assert util.bits_equal(o, a[i])
        assert np.isfinite(o).all()
    one = yb.load_network(cfg, wts, batch=1)
    for k in (0, 7, 15):
        one.predict(x[k:k + 1])
        for i, o in one.detection_outputs().items():
            assert util.bits_equal(o[0], a[i][k]), (k, i)


def test_spp_608_runs_and_matches_f32_cuda_core_path(workdir):
    """yolov3-spp (BASELINE configs[4] model): tensor-core bf16 result vs the engine's own f32 CUDA-core path
    (which the slim-model tests pin to the oracle); covers the 5/9/13 max-pools and the 4-way concat at 19x19."""
    import yolo2_light_b200 as yb
    secs = cfgs.yolov3_spp(608, 608)
    cfg, wts = _files(workdir, "spp_608", secs, seed=3)
    x = cfgs.synthetic_images(2, 3, 608, 608)
    a = yb.load_network(cfg, wts, batch=2)
    a.predict(x)
    b = yb.load_network(cfg, wts, batch=2)
    b.set_precision(yb.YB_PREC_FP32)
    b.predict(x)
    for i, o in a.detection_outputs().items():
        assert util.rel_l2(o, b.layer_output(i)) <= 1e-3, i


def test_pipelined_submit_collect_equals_predict(workdir):
    """yb_network_submit/collect (copies overlapped with compute, 3 batches in flight) returns exactly what the
    synchronous predict returns, batch after batch, including when slots are reused."""
    import yolo2_light_b200 as yb
    secs = cfgs.yolov3_tiny(416, 416)
    cfg, wts = _files(workdir, "tiny_416", secs)
    B = 4
    net = yb.load_network(cfg, wts, batch=B)
    batches = [cfgs.synthetic_images(B, 3, 416, 416, seed=100 + 10 * k) for k in range(7)]
    expect = []
    for x in batches:
        net.predict(x)
        expect.append({i: o.copy() for i, o in net.detection_outputs().items()})
    pinned = [yb.PinnedBuffer(B * 3 * 416 * 416) for _ in range(3)]
    inflight, got = [], []
    for k, x in enumerate(batches):
        if len(inflight) == 3:
            got.append({i: o.copy() for i, o in net.collect(inflight.pop(0)).items()})
        pinned[k % 3].array[:] = x.ravel()
        inflight.append(net.submit(pinned[k % 3].array))
    while inflight:
        got.append({i: o.copy() for i, o in net.collect(inflight.pop(0)).items()})
    assert len(got) == len(expect)
    for g, e in zip(got, expect):
        for i in e:
            assert util.bits_equal(g[i], e[i])
    with pytest.raises(yb.YbError):
        net.collect(0)   # nothing in flight


# ---- per-layer bit-exactness of the integer variants at the REAL BASELINE shapes (configs[2], configs[3]) ----------------------
def _saturating_input(l, B, rng, image, f0=0, py=6, px=6):
    """Random activations, plus -- in image `image` around pixel (py, px) -- the pattern that drives filter f0 of an INT8 layer
    into the int16 clamp of the reference (acc / 32 > 32767, yolov2_forward_network_quantized.c:474-490): every tap gets the
    sign of its own weight at full scale."""
    c, h, w, size, pad = l["c"], l["h"], l["w"], l["size"], l["pad"]
    x = rng.standard_normal((B, c, h, w)).astype(np.float32) * 2.0
    wq = np.asarray(l["weights_int8"], np.int8).reshape(l["n"], c, size, size)
    big = np.float32(200.0 / l["input_quant_multipler"])
    for ky in range(size):
        for kx in range(size):
            x[image, :, py + ky - pad, px + kx - pad] = np.where(wq[f0, :, ky, kx] >= 0, big, -big)
    return x


@pytest.mark.parametrize("layer", [2, 4, 8, 12, 13, 14, 21])
def test_c3_int8_layers_bit_exact_at_full_shape(layer, workdir):
    """yolov3-tiny 416 -quantized, batch 64 (BASELINE configs[2]): conv `layer` alone on the GPU at its real shape (K up to 4608,
    multi-wave tiles, CTA pairs) against the oracle on three images of the batch: s32 accumulators identical, float outputs
    bit-identical, including outputs that hit the int16 saturation."""
    import yolo2_light_b200 as yb
    from oracle import port
    B = 64
    cfg, wts = _files(workdir, "tiny_416", cfgs.yolov3_tiny(416, 416))
    net = yb.load_network(cfg, wts, batch=B, quantized=1)
    l = net.layers[layer]
    rng = np.random.default_rng(700 + layer)
    x = _saturating_input(l, B, rng, image=31)
    got = net.forward_convolutional_layer(layer, x, variant=1)
    saturated = []
    for b in (0, 31, 63):
        exp, acc = port.conv_int8(x[b:b + 1], l["weights_int8"], l["biases"], l["input_quant_multipler"], l["weights_quant_multipler"],
                                  l["n"], l["size"], l["stride"], l["pad"], l["activation"], want_acc=True)
        assert util.bits_equal(got[b:b + 1], exp), (layer, b, float(np.abs(got[b:b + 1] - exp).max()))
        if b == 31:
            # filter 0 at full-scale inputs: sum |wq| * 127; shallow layers (K = 144) cannot reach the clamp at all
            reach = int(np.abs(np.asarray(l["weights_int8"], np.int64).reshape(l["n"], -1)[0]).sum()) * 127 // 32
            if reach > 40000:
                assert (np.abs(acc // 32) > 32767).any(), "the test input was meant to saturate the int16 clamp"
                saturated.append(layer)
    if layer in (12, 14, 21):
        assert saturated, "deep-K layers must exercise the int16 clamp"


@pytest.mark.parametrize("layer", [2, 4, 6, 10, 12, 13])
def test_c4_xnor_layers_bit_exact_at_full_shape(layer, workdir):
    """tiny-yolo-obj_xnor 416, batch 64 (BASELINE configs[3]): every XNOR layer class at its real shape (K up to 9216) --
    popcount kernels for the narrow layers, +-1 on kind::i8 for the wide ones -- against the oracle on three images."""
    import yolo2_light_b200 as yb
    from oracle import port
    B = 64
    cfg, wts = _files(workdir, "xnor_416", cfgs.tiny_yolo_obj_xnor(416, 416))
    net = yb.load_network(cfg, wts, batch=B)
    l = net.layers[layer]
    assert l["xnor"]
    rng = np.random.default_rng(800 + layer)
    x = rng.standard_normal((B, l["c"], l["h"], l["w"])).astype(np.float32)
    x[:, :, ::3, ::5] = 0.0                      # exact zeros: sign(0) = -1 in the reference (x > 0)
    got = net.forward_convolutional_layer(layer, x, variant=0)
    for b in (0, 40, 63):
        exp = port.conv_xnor(x[b:b + 1], l["weights"], l["biases"], l["mean_arr"], l["n"], l["size"], l["activation"])
        assert util.bits_equal(got[b:b + 1], exp), (layer, b, float(np.abs(got[b:b + 1] - exp).max()))


def test_c4_all_popcount_configuration(workdir, monkeypatch):
    """YB_XNOR_TC=0: every XNOR layer on the xor + __popc kernels (what north_star describes), whole network bit-identical to the
    default configuration (wide layers as +-1 on the tensor cores) on every XNOR layer's output."""
    import yolo2_light_b200 as yb
    cfg, wts = _files(workdir, "xnor_416", cfgs.tiny_yolo_obj_xnor(416, 416))
    B = 4
    x = cfgs.synthetic_images(B, 3, 416, 416, seed=5)
    a = yb.load_network(cfg, wts, batch=B); a.set_option("fuse", 0); a.predict(x)
    monkeypatch.setenv("YB_XNOR_TC", "0")
    b = yb.load_network(cfg, wts, batch=B); b.set_option("fuse", 0); b.predict(x)
    kinds = {k for _, k, _ in b.profile()}
    assert "conv_xnor" in kinds and "conv_tc_i8" not in kinds
    assert "conv_tc_i8" in {k for _, k, _ in a.profile()}
    n = 0
    for i, l in enumerate(a.layers):
        if l["type_name"] == "CONVOLUTIONAL" and l["xnor"]:
            assert util.bits_equal(a.fetch_layer(i), b.fetch_layer(i)), i
            n += 1
    assert n == 7
    for i, o in a.detection_outputs().items():
        assert util.bits_equal(o, b.layer_output(i)), i


# ---- BASELINE configs[4]: the SPP block at its real size against the UNMODIFIED reference (scalar build) ---------------------------
def test_spp_608_against_scalar_reference(workdir):
    """yolov3-spp 608 (BASELINE configs[4], one image): the 5 / 9 / 13 max-pools on 19x19x512, the 2048-channel concat and the
    convolution behind it, layer by layer against the oracle's restatement of the reference's scalar code (forward_maxpool_layer,
    forward_route_layer, forward_convolutional_layer_cpu; additionally.c:1448-1482 -- the AVX max-pool is wrong for these pools,
    SURVEY F6; the restatement is pinned to the reference in test_oracle_vs_reference.py) fed with the engine's own activations;
    then the whole network's detections against the reference's CPU path."""
    import yolo2_light_b200 as yb
    from oracle import port
    secs = cfgs.yolov3_spp(608, 608)
    cfg, wts = _files(workdir, "spp_608", secs, seed=3)
    x = cfgs.synthetic_images(1, 3, 608, 608, seed=11)
    net = yb.load_network(cfg, wts, batch=1)
    net.set_precision(yb.YB_PREC_FP32)            # f32 engine: data-movement layers are then comparable bit for bit
    net.set_option("fuse", 0)
    net.predict(x)
    layers = net.layers
    types = [L["type_name"] for L in layers]
    first_pool = types.index("MAXPOOL")
    assert types[first_pool:first_pool + 6] == ["MAXPOOL", "ROUTE", "MAXPOOL", "ROUTE", "MAXPOOL", "ROUTE"]
    # start from the engine's activation of the layer in front of the SPP block, then run the restatement layer by layer through
    # the block and the convolution behind it (route layers read their sources from these outputs)
    outs = {first_pool - 1: net.fetch_layer(first_pool - 1)}
    cur = outs[first_pool - 1]
    for i in range(first_pool, first_pool + 7):
        L = layers[i]
        if types[i] == "MAXPOOL":
            cur = port.maxpool(cur, L["size"], L["stride"], L["pad"])
        elif types[i] == "ROUTE":
            cur = np.concatenate([outs[int(j)] for j in L["input_layers"]], axis=1)
        else:
            assert types[i] == "CONVOLUTIONAL", types[i]
            cur = port.conv_fp32(cur, L["weights"], L["biases"], L["n"], L["size"], L["stride"], L["pad"], L["activation"])
        outs[i] = cur
        got = net.fetch_layer(i)
        if types[i] == "CONVOLUTIONAL":
            assert util.bits_equal(got, cur.reshape(got.shape)), (i, types[i], float(np.abs(got - cur.reshape(got.shape)).max()))
        else:
            assert util.bits_equal(got, cur.reshape(got.shape)), (i, types[i])
    assert layers[first_pool + 5]["out_c"] == 2048
    # default precision (bf16 tensor cores), the whole network against the reference's scalar CPU path on the same image
    # (~1 minute of single-thread CPU): FP32-variant bar of north_star, <= 1e-3 rel on the activated detection tensors
    fast = yb.load_network(cfg, wts, batch=1)
    fast.predict(x)
    n = 0
    for i, o in fast.detection_outputs().items():
        err = util.sampled_rel_l2(o, f"full_spp_608_l{i}", 0)
        assert err <= 1e-3, (i, err)
        assert util.sampled_rel_l2(net.layer_output(i), f"full_spp_608_l{i}", 0) <= 1e-5, i     # the f32 engine, too
        n += 1
    assert n == 3
