"""Matching driver -- drop-in for `match_images` of imcui/hloc/match_features.py:204-275, with the result preparation on
the GPU.

The reference copies every matcher output to the host and builds the matched-keypoint arrays with NumPy
(:236-257).  Here `PairResult.sparse` gathers the matched keypoints, rescales all coordinates to the original frames
((k + 0.5) * s - 0.5 in fp32, as torch does) and fetches everything with one packed D2H (csrc/prepost.cu)."""
import torch

from .configs import confs_dict
from .pipeline import PairResult

confs = confs_dict["matchers"]


def _first(x):
    """extractors hand back lists / tuples of per-image tensors or tensors with a leading batch dimension of 1"""
    return x[0]


def pair_inputs(feat0, feat1):
    """The matcher's input dict (match_features.py:207-234): keypoints [1,N,2], scores [1,N], descriptors [1,D,N]."""
    data = {}
    for side, f in (("0", feat0), ("1", feat1)):
        desc = _first(f["descriptors"])
        kpts = f["keypoints"]
        kpts = _first(kpts)[None] if isinstance(kpts, (list, tuple)) else kpts
        data["image" + side] = f["image"]
        data["keypoints" + side] = kpts
        data["scores" + side] = _first(f["scores"]).unsqueeze(0)
        data["descriptors" + side] = desc.unsqueeze(0) if desc.dim() == 2 else desc
        for extra in ("scales", "oris"):
            if extra in f:
                x = f[extra]
                data[extra + side] = _first(x)[None] if isinstance(x, (list, tuple)) else x
    return data


@torch.no_grad()
def match_images(model, feat0, feat1):
    """match_features.py:204-275: features of two images (outputs of `extract`) -> the reference's result dict (NumPy)."""
    data = pair_inputs(feat0, feat1)
    pred = model(data)
    s0 = feat0["original_size"] / feat0["size"]
    s1 = feat1["original_size"] / feat1["size"]
    res = PairResult.sparse(data["keypoints0"][0], data["keypoints1"][0], pred["matches0"][0], pred["matching_scores0"][0], s0, s1)
    # (the reference calls torch.cuda.empty_cache() for every pair, :273; the engine's workspaces are cached on purpose)
    return {"image0_orig": feat0["image_orig"], "image1_orig": feat1["image_orig"], **res}
