"""Shared helpers for the test-suite: small model zoo (generated cfg + seeded weights), the stored results of the
reference (tests/golden)."""
import functools
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from yolo2_light_b200 import cfgs  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# name -> (section builder, input size, weight seed, image seed)
ZOO = {
    "tiny64": (lambda: cfgs.slim(cfgs.yolov3_tiny, 2, 64, 64), 64, 11, 101),
    "xnor64": (lambda: cfgs.slim(cfgs.tiny_yolo_obj_xnor, 2, 64, 64), 64, 12, 102),
    "v3_32": (lambda: cfgs.slim(cfgs.yolov3, 4, 32, 32), 32, 13, 103),
    "spp32": (lambda: cfgs.slim(cfgs.yolov3_spp, 4, 32, 32), 32, 14, 104),
    "v2voc32": (lambda: cfgs.slim(cfgs.yolov2_voc, 4, 32, 32), 32, 15, 105),
    # non-square inputs (H != W): name -> builder uses (width, height)
    "tiny_w96_h64": (lambda: cfgs.slim(cfgs.yolov3_tiny, 2, 96, 64), (64, 96), 17, 107),
    "v3_w64_h96": (lambda: cfgs.slim(cfgs.yolov3, 4, 64, 96), (96, 64), 18, 108),
    "tinyvoc64": (lambda: cfgs.slim(cfgs.tiny_yolo_voc, 2, 64, 64), 64, 16, 106),
}


def model_files(name, workdir):
    build, size, wseed, _ = ZOO[name]
    secs = build()
    cfg = os.path.join(workdir, name + ".cfg")
    wts = os.path.join(workdir, name + ".weights")
    if not os.path.exists(cfg):
        cfgs.write_cfg(secs, cfg)
        cfgs.write_weights(secs, wts, seed=wseed)
    return cfg, wts


def images(name, batch):
    _, size, _, iseed = ZOO[name]
    h, w = size if isinstance(size, tuple) else (size, size)
    return cfgs.synthetic_images(batch, 3, h, w, seed=iseed)


@functools.lru_cache(maxsize=None)
def reference():
    """What the original project's CPU code computed for the tests that compare with it (tests/golden/make_reference_golden.py)."""
    with open(os.path.join(GOLDEN, "reference.json")) as f:
        return json.load(f)


@functools.lru_cache(maxsize=None)
def reference_arrays():
    return dict(np.load(os.path.join(GOLDEN, "reference_arrays.npz")))


def digest(a, dtype=np.float32):
    """The first 64 bits of the sha256 of the values of `a` as `dtype`: a fingerprint of the flattened array's bits."""
    return hashlib.sha256(np.ascontiguousarray(a, dtype).tobytes()).hexdigest()[:16]


def sampled_rel_l2(out, key, b):
    """rel_l2 of image `b` of `out` [batch, ...] against the stored sample `key` of the reference's tensor."""
    g = reference_arrays()
    idx = g[f"{key}_b{b}_idx"]
    return rel_l2(np.asarray(out[b]).ravel()[idx], g[f"{key}_b{b}_val"])


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel(); b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def bits_equal(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))
