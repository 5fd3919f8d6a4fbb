"""Pins the CPU restatement (oracle/yolo_oracle.c) against the UNMODIFIED reference: whole networks, every layer,
bit-for-bit (digests of the reference's outputs in tests/golden/reference.json, "layers" and "resize")."""
import numpy as np
import pytest

import ybtest_util as util

WHOLE_NETWORK_CASES = [("tiny64", 0), ("tiny64", 1), ("xnor64", 0), ("v3_32", 0), ("spp32", 0), ("v2voc32", 0),
                       ("tinyvoc64", 1), ("v3_32", 1), ("tiny_w96_h64", 0), ("tiny_w96_h64", 1), ("v3_w64_h96", 0)]
RESIZE_SHAPES = [(480, 640, 608, 608), (37, 53, 64, 96), (64, 64, 64, 64), (1, 7, 32, 32), (100, 1, 32, 32)]


def _assert_port_equals_reference(name, workdir, quantized, batch=1):
    import yolo2_light_b200 as yb
    from oracle import port
    cfg, wts = util.model_files(name, workdir)
    x = util.images(name, batch)
    net = yb.load_network(cfg, wts, batch=batch, quantized=quantized)
    outs = port.run_network(net.layers, x, quantized=bool(quantized))
    rec = util.reference()["layers"][f"{name}_q{quantized}_b{batch}"]
    assert len(outs) == len(rec)
    for i, (o, (type_name, shape, dig)) in enumerate(zip(outs, rec)):
        assert o.size == np.prod(shape), (i, o.shape, shape)
        assert util.digest(o) == dig, f"{name} q={quantized} layer {i} {type_name}"


@pytest.mark.parametrize("name,quantized", WHOLE_NETWORK_CASES)
def test_whole_network_bit_exact(name, quantized, workdir):
    """Same cfg, same generated .weights, same image -> every layer output of the restatement equals the
    reference's l.output bit-for-bit (FP32 conv: identical k-ascending float accumulation; XNOR / INT8: exact
    integers + identical float epilogue; small layers: copies / compares / libm)."""
    _assert_port_equals_reference(name, workdir, quantized)


def test_batch_two_fp32(workdir):
    """The reference's FP32/XNOR loops handle l.batch > 1 (yolov2_forward_network.c:111, :212); so does the port."""
    _assert_port_equals_reference("xnor64", workdir, 0, batch=2)


def test_quantize_input_matches_reference_cast():
    """(int16_t)(x*mult) with x86 semantics, clamp +-127 (yolov2_forward_network_quantized.c:556-560), including
    values around the truncation boundaries and large magnitudes."""
    from oracle import port
    x = np.array([0.0, 0.49, -0.49, 1.0, -1.0, 7.999, -7.999, 126.9, 127.2, -127.2, 300.0, -300.0,
                  32767.9, 32768.5, -32769.5, 65536.0 + 5, 1e9, -1e9, 1e20, np.nan], np.float32)
    q = port.quantize_input(x, 1.0)
    exp = []
    for v in x:
        f = np.float32(v)
        if not (f > -2147483648.0 and f < 2147483648.0):
            i = -2147483648
        else:
            i = int(f)
        s = ((i & 0xffff) ^ 0x8000) - 0x8000
        exp.append(max(-127, min(127, s)))
    assert q.tolist() == exp


def resize_input(h, w):
    return np.random.default_rng(h * 1000 + w).integers(0, 256, (h, w, 3), dtype=np.uint8)


@pytest.mark.parametrize("shape", RESIZE_SHAPES)
def test_image_pipeline_port_equals_reference(shape):
    """u8 -> float/255 -> resize_image: the port against the reference's own functions, bit-for-bit."""
    from oracle import port
    h, w, oh, ow = shape
    got = port.load_resize_u8(resize_input(h, w), ow, oh)
    assert got.shape == (3, oh, ow)
    assert util.digest(got) == util.reference()["resize"][f"{h},{w},{oh},{ow}"]
