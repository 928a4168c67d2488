"""SIFT oracle (opencv backend): cv2.SIFT_create(...).detectAndCompute plus the wrapper glue of hloc's SIFT extractor,
which follows LightGlue's lightglue/sift.py (run_opencv_sift, filter_dog_point, top-k, sift_to_rootsift).

The wrapper glue is restated from lightglue/sift.py: hloc's SIFT wrapper is not in this tree, so its defaults are not
pinned against the reference (DESIGN.md).  cv2 is the arithmetic the reference itself calls."""
import cv2
import numpy as np
import torch

DEFAULT_CONF = {"rootsift": True, "nms_radius": 0, "max_num_keypoints": 4096, "backend": "opencv",
                "detection_threshold": 0.0066667, "edge_threshold": 10, "first_octave": -1, "num_octaves": 4}


def to_uint8(image):
    """(image_np * 255.0).astype(np.uint8): truncation of the fp32 product, not rounding"""
    return (np.asarray(image, np.float32) * 255.0).astype(np.uint8)


def create(conf):
    # the wrapper passes num_octaves as nOctaveLayers
    return cv2.SIFT_create(contrastThreshold=conf["detection_threshold"], nfeatures=conf["max_num_keypoints"] or 0,
                           edgeThreshold=conf["edge_threshold"], nOctaveLayers=conf["num_octaves"])


def run_opencv_sift(sift, image_u8):
    """lightglue/sift.py run_opencv_sift: points, scores (response), scales (size), angles (radians), descriptors"""
    det, desc = sift.detectAndCompute(image_u8, None)
    points = np.array([k.pt for k in det], dtype=np.float32).reshape(-1, 2)
    scores = np.array([k.response for k in det], dtype=np.float32)
    scales = np.array([k.size for k in det], dtype=np.float32)
    angles = np.deg2rad(np.array([k.angle for k in det], dtype=np.float32))
    if desc is None:
        desc = np.zeros((0, 128), np.float32)
    return points, scores, scales, angles, desc


def filter_dog_point(points, scales, angles, image_shape, nms_radius, scores=None):
    """lightglue/sift.py filter_dog_point for nms_radius 0: one keypoint per pixel round(pt - 0.5) (half to even), the
    highest score, then the lowest |angle|; exact ties all stay."""
    assert nms_radius == 0
    h, w = image_shape
    ij = np.round(points - 0.5).astype(int).T[::-1]
    s = scales if scores is None else scores
    buffer = np.zeros((h, w))
    np.maximum.at(buffer, tuple(ij), s)
    keep = np.where(buffer[tuple(ij)] == s)[0]
    ij = ij[:, keep]
    buffer[:] = np.inf
    o_abs = np.abs(angles[keep])
    np.minimum.at(buffer, tuple(ij), o_abs)
    mask = buffer[tuple(ij)] == o_abs
    return keep[mask]


def sift_to_rootsift(x, eps=1e-6):
    x = torch.nn.functional.normalize(x, p=1, dim=-1, eps=eps)
    x.clip_(min=eps).sqrt_()
    return torch.nn.functional.normalize(x, p=2, dim=-1, eps=eps)


def extract(image, conf=None):
    """image [H,W] float in [0,1] -> dict of keypoints [N,2], scores [N], scales [N], oris [N], descriptors [N,128]
    (torch, the wrapper's order: cv2's, filtered, then top-k)."""
    conf = {**DEFAULT_CONF, **(conf or {})}
    points, scores, scales, angles, desc = run_opencv_sift(create(conf), to_uint8(image))
    pred = {"keypoints": points, "scales": scales, "oris": angles, "descriptors": desc, "scores": scores}
    if conf["nms_radius"] is not None:
        keep = filter_dog_point(points, scales, angles, np.asarray(image).shape, conf["nms_radius"], scores)
        pred = {k: v[keep] for k, v in pred.items()}
    pred = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in pred.items()}
    n = conf["max_num_keypoints"]
    if n is not None and n > 0 and len(pred["keypoints"]) > n:
        idx = torch.topk(pred["scores"], n).indices
        pred = {k: v[idx] for k, v in pred.items()}
    if conf["rootsift"]:
        pred["descriptors"] = sift_to_rootsift(pred["descriptors"].float())
    return pred


def pyramid(image_u8, n_layers=4, sigma=1.6, n_octaves=None):
    """The Gaussian pyramid cv2.SIFT builds (createInitialImage with firstOctave -1, buildGaussianPyramid), from cv2
    calls: a list per octave of [L+3, h, w] float32 arrays on the 0-255 scale."""
    img = image_u8.astype(np.float32)
    h, w = img.shape
    base = cv2.resize(img, (2 * w, 2 * h), interpolation=cv2.INTER_LINEAR)
    # createInitialImage computes this blur sigma in float (sqrtf of a float expression), the layer sigmas in double
    sf = np.float32(sigma)
    sd = float(np.sqrt(np.maximum(sf * sf - np.float32(0.5) * np.float32(0.5) * np.float32(4), np.float32(0.01))))
    base = cv2.GaussianBlur(base, (0, 0), sd, sigmaY=sd)
    if n_octaves is None:
        n_octaves = int(np.rint(np.log2(min(2 * h, 2 * w)) - 2)) + 1
    k = 2 ** (1.0 / n_layers)
    sig = [sigma] + [np.sqrt((k ** i * sigma) ** 2 - (k ** (i - 1) * sigma) ** 2) for i in range(1, n_layers + 3)]
    out = []
    for o in range(n_octaves):
        layers = []
        for i in range(n_layers + 3):
            if o == 0 and i == 0:
                layers.append(base)
            elif i == 0:
                src = out[-1][n_layers]
                layers.append(cv2.resize(src, (src.shape[1] // 2, src.shape[0] // 2), interpolation=cv2.INTER_NEAREST))
            else:
                layers.append(cv2.GaussianBlur(layers[-1], (0, 0), sig[i], sigmaY=sig[i]))
        out.append(np.stack(layers))
    return out
