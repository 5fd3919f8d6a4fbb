"""INT8 input calibration (SURVEY 8f row 3): the host half -- histogram + KL search restated from
entropy_calibration (yolov2_forward_network_quantized.c:1292-1398) -- must return the reference's multiplier bit for bit
(tests/golden/reference.json, "calibration")."""
import numpy as np
import pytest

import ybtest_util as util

PARAMS = [(1.0 / 16, 4096), (1.0 / 4, 1024)]


def _cases():
    rng = np.random.default_rng(7)
    yield "leaky activations", np.where(rng.standard_normal(200000) > 0, 1.0, 0.1) * rng.standard_normal(200000) * 3.0
    yield "image in [0,1)", rng.random(3 * 64 * 64)
    yield "heavy tail with outliers beyond the last bin", rng.standard_cauchy(50000) * 20.0
    yield "mostly zeros", np.concatenate([np.zeros(90000), rng.random(10000) * 40.0])
    yield "tiny", rng.standard_normal(300) * 8.0
    yield "wide uniform", rng.random(400000) * 250.0


@pytest.mark.parametrize("bin_width,max_bin", PARAMS)
def test_entropy_calibration_bit_identical_to_reference(bin_width, max_bin):
    import yolo2_light_b200 as yb
    expected = util.reference()["calibration"][f"{bin_width},{max_bin}"]
    for (name, arr), theirs in zip(_cases(), expected, strict=True):
        a = np.asarray(arr, np.float32)
        mine = yb.api.entropy_calibration(a, bin_width, max_bin)
        assert np.float32(mine) == np.float32(theirs), (name, mine, theirs)


def test_format_input_calibration_line():
    import yolo2_light_b200 as yb
    m = np.array([[4.5, 9.25, 16.0], [5.5, 8.75, 15.0]], np.float32)
    assert yb.api.format_input_calibration(m) == "input_calibration = 5, 9, 15.5, 16"
