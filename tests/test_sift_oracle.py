"""CPU checks of the SIFT extractor: the oracle's wrapper glue on hand-built cases, the host-side Gaussian kernels and
octave count against cv2, and the C struct layout."""
import ctypes
import math
import subprocess
from pathlib import Path

import cv2
import numpy as np
import torch

from oracle import sift as osift

ROOT = Path(__file__).resolve().parent.parent
CONF = {"n_octave_layers": 4, "contrast_threshold": 0.0066667, "edge_threshold": 10, "sigma": 1.6, "max_keypoints": 4096,
        "nms_radius": 0, "rootsift": True}


def test_pixel_dedupe_score_then_ori():
    # pixels: (0,0) x3 -> best score wins; (2,1) x3 -> score tie, lowest |ori| wins; (3,3) x2 -> exact tie, both stay
    pts = np.array([[0.6, 0.4], [0.9, 0.7], [0.2, 0.9],
                    [2.4, 1.3], [2.6, 1.4], [2.5, 1.5],
                    [3.2, 3.2], [3.3, 3.1]], np.float32)
    scores = np.array([1.0, 3.0, 2.0, 5.0, 5.0, 4.0, 7.0, 7.0], np.float32)
    oris = np.array([0.0, 0.5, 0.1, -0.3, 0.2, 0.0, -0.4, 0.4], np.float32)
    keep = osift.filter_dog_point(pts, scores, oris, (8, 8), 0, scores)
    assert sorted(keep.tolist()) == [1, 4, 6, 7]
    # round(pt - 0.5) rounds half to even: 2.5 - 0.5 = 2.0 and 1.5 - 0.5 = 1.0 -> pixel (1, 2); 3.0 -> 2 (half to even)
    ij = np.round(np.array([[3.0, 1.0]], np.float32) - 0.5)
    assert ij.tolist() == [[2.0, 0.0]]


def test_uint8_truncates():
    x = np.array([1 / 255 - 1e-7, 0.5, 1.0, 254.9 / 255], np.float32)
    assert osift.to_uint8(x).tolist() == [0, 127, 255, 254]


def test_rootsift():
    d = torch.tensor([[4.0, 0.0, 12.0, 0.0], [0.0, 0.0, 0.0, 0.0]])
    r = osift.sift_to_rootsift(d.clone())
    ref = torch.sqrt(torch.tensor([0.25, 1e-6, 0.75, 1e-6]))
    assert torch.allclose(r[0], ref / ref.norm(), atol=1e-7)
    assert torch.allclose(r[1].norm(), torch.tensor(1.0))   # eps keeps empty descriptors finite


def _sigmas(L, sigma=1.6):
    k = 2 ** (1 / L)
    sf = np.float32(sigma)   # the base blur sigma is float arithmetic in createInitialImage
    base = float(np.sqrt(np.maximum(sf * sf - np.float32(0.5) * np.float32(0.5) * np.float32(4), np.float32(0.01))))
    return [base] + \
        [math.sqrt((k ** i * sigma) ** 2 - (k ** (i - 1) * sigma) ** 2) for i in range(1, L + 3)]


def test_host_taps_equal_cv2_and_octave_count():
    from imcui_b200 import ops
    for L, (h, w) in ((4, (480, 640)), (3, (240, 320)), (4, (123, 457))):
        n_oct, taps = ops.sift_plan({**CONF, "n_octave_layers": L}, h, w)
        assert n_oct == int(np.rint(np.log2(min(2 * h, 2 * w)) - 2)) + 1
        for s, (ks, t) in zip(_sigmas(L), taps):
            ref = cv2.getGaussianKernel(int(np.rint(s * 8 + 1)) | 1, s, cv2.CV_32F).ravel()
            assert ks == len(ref) and np.array_equal(t, ref), (L, s)
    assert ops.sift_plan(CONF, 480, 640)[0] == 9


def test_bad_confs_raise():
    import pytest
    from imcui_b200 import ops
    with pytest.raises(ValueError):
        ops.sift_plan({**CONF, "nms_radius": 3}, 480, 640)
    with pytest.raises(ValueError):
        ops.sift_plan({**CONF, "n_octave_layers": 0}, 480, 640)


def test_plugin_rejects_unbuilt_options():
    import pytest
    from imcui_b200.hloc import extractors
    from imcui_b200.hloc.utils.base_model import dynamic_load
    cls = dynamic_load(extractors, "sift")
    for bad in ({"backend": "pycolmap"}, {"nms_radius": 3}):
        with pytest.raises(NotImplementedError):
            cls(bad)


def test_sift_conf_struct_size(tmp_path):
    from imcui_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "imw_b200.h"\nint main(void){printf("%zu\\n", sizeof(imw_sift_conf));return 0;}')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)])
    assert ctypes.sizeof(_lib.SiftConf) == int(subprocess.check_output([str(exe)], text=True))
