"""Host-side model preparation of the product (loader, BN fold, XNOR statistics, INT8 quantisation) against the
reference's own functions, bit-for-bit (main.c:160-171 sequence; digests of the reference's arrays in
tests/golden/reference.json, "prepared" and "unprepared_tiny64")."""
import numpy as np
import pytest

import ybtest_util as util

PREP_CASES = [("tiny64", 1), ("xnor64", 0), ("v3_32", 1), ("v2voc32", 1), ("tinyvoc64", 1), ("spp32", 0)]


def assert_prepared_like_reference(layers, name, q):
    """Every convolution's prepared arrays (list of layer dicts) bit-identical to what the reference prepared."""
    rec = util.reference()["prepared"][f"{name}_q{q}"]
    convs = [i for i, la in enumerate(layers) if la["type_name"] == "CONVOLUTIONAL"]
    assert convs == sorted(int(i) for i in rec)
    for i in convs:
        la, lb = layers[i], rec[str(i)]
        assert la["batch_normalize"] == lb["batch_normalize"] == 0
        assert util.digest(la["weights"]) == lb["weights"], (i, "weights")
        assert util.digest(la["biases"]) == lb["biases"], (i, "biases")
        if q:
            assert util.digest(la["weights_int8"], np.int8) == lb["weights_int8"], (i, "int8")
            assert la["weights_quant_multipler"] == lb["weights_quant_multipler"], i
            assert la["input_quant_multipler"] == lb["input_quant_multipler"], i
        assert bool(la["xnor"]) == ("mean_arr" in lb), i
        if la["xnor"]:
            assert util.digest(la["mean_arr"]) == lb["mean_arr"], (i, "mean_arr")
    assert convs


@pytest.mark.parametrize("name,q", PREP_CASES)
def test_prepared_arrays_bit_exact(name, q, workdir):
    import yolo2_light_b200 as yb
    cfg, wts = util.model_files(name, workdir)
    net = yb.load_network(cfg, wts, batch=1, quantized=q)      # the layer arrays are views into the network
    assert_prepared_like_reference(net.layers, name, q)


def test_unprepared_weights_equal_file(workdir):
    """load_weights_upto_cpu alone (no fold): arrays are the file contents in cfg order (additionally.c:3459-3468)."""
    import yolo2_light_b200 as yb
    cfg, wts = util.model_files("tiny64", workdir)
    a = yb.parse_network_cfg(cfg, 1, 0)
    yb.load_weights_upto_cpu(a, wts)
    rec = util.reference()["unprepared_tiny64"]
    convs = [i for i in range(a.n) if a.layer(i)["type_name"] == "CONVOLUTIONAL"]
    assert convs == sorted(int(i) for i in rec)
    for i in convs:
        la = a.layer(i)
        for arr, rb in rec[str(i)].items():
            if rb is None:
                assert la[arr] is None
            else:
                assert util.digest(la[arr]) == rb, (i, arr)


def test_cutoff_and_short_file(workdir):
    """cutoff stops loading after `cutoff` layers; a truncated file is not an error (the reference ignores short
    reads, additionally.c:3459-3468)."""
    import os
    import yolo2_light_b200 as yb
    cfg, wts = util.model_files("tiny64", workdir)
    a = yb.parse_network_cfg(cfg, 1, 0)
    yb.load_weights_upto_cpu(a, wts, cutoff=1)
    assert np.abs(a.layer(0)["weights"]).max() > 0
    assert np.abs(a.layer(2)["weights"]).max() == 0
    short = os.path.join(workdir, "short.weights")
    data = open(wts, "rb").read()
    open(short, "wb").write(data[:len(data) // 2])
    b = yb.parse_network_cfg(cfg, 1, 0)
    yb.load_weights_upto_cpu(b, short)
    assert np.abs(b.layer(0)["weights"]).max() > 0
    with pytest.raises(yb.YbError):
        yb.load_weights_upto_cpu(b, os.path.join(workdir, "missing.weights"))
