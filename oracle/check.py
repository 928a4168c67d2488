"""Checker for the batched SuperPoint -> LightGlue pair stream (TEST INFRASTRUCTURE, see oracle/__init__.py).

Runs the CPU oracle (oracle.superpoint / oracle.lightglue: restatements of
third_party/SuperGluePretrainedNetwork/models/superpoint.py:145-206 and
third_party/LightGlue/lightglue/lightglue.py:488-634) on the same uint8 images a PairEngine step
consumed and compares per pair:

  * keypoint SET identity per image (integer pixel coordinates, bit-exact);
  * the LightGlue stop layer;
  * match-F1 (SURVEY.md 8(d)): F1 of the set of matches.  Top-k keypoint ORDER is a sort on fp32
    scores and may swap near-ties, so matches are compared as coordinate 4-tuples (x0, y0, x1, y1)
    "within 0 px" -- identical to index identity whenever the keypoint order is identical;
  * exact: the two match sets are identical.
"""
import numpy as np
import torch

from . import lightglue as olg
from . import synthetic_weights
from . import superpoint as osp

LG_CONF_CUDA = {"depth_confidence": 0.95, "width_confidence": 0.99, "filter_threshold": 0.2, "pruning_min_kpts": 1536}


def to_float(images_u8):
    """extract_features.py:139: float64 division by 255, then .float()."""
    return torch.from_numpy(np.asarray(images_u8).astype(np.float64) / 255.0).float()[:, None]


def oracle_pairs(images_u8, sp_conf, lg_conf=None, weights=None):
    """images_u8 [2n,H,W] uint8 (slot 2p+side) -> list of per-pair dicts
    {kpts0, kpts1 [N,2] f32, scores0/1, matches0 [N0] int64, mscores0, stop}."""
    ws, wl = weights or (synthetic_weights("superpoint"), synthetic_weights("lightglue"))
    lg_conf = {**LG_CONF_CUDA, **(lg_conf or {})}
    out = []
    imgs = to_float(images_u8)
    for p in range(len(imgs) // 2):
        f0 = osp.forward(ws, imgs[2 * p:2 * p + 1], sp_conf)
        f1 = osp.forward(ws, imgs[2 * p + 1:2 * p + 2], sp_conf)
        r = olg.forward(wl, f0["keypoints"][0][None], f0["descriptors"][0].t().contiguous()[None],
                        f1["keypoints"][0][None], f1["descriptors"][0].t().contiguous()[None], lg_conf)
        out.append({"kpts0": f0["keypoints"][0].numpy(), "kpts1": f1["keypoints"][0].numpy(),
                    "scores0": f0["scores"][0].numpy(), "scores1": f1["scores"][0].numpy(),
                    "desc0": f0["descriptors"][0].numpy(), "desc1": f1["descriptors"][0].numpy(),
                    "matches0": r["matches0"][0].numpy(), "mscores0": r["matching_scores0"][0].numpy(), "stop": int(r["stop"])})
    return out


def match_tuples(kpts0, kpts1, matches0):
    k0, k1, m = np.asarray(kpts0), np.asarray(kpts1), np.asarray(matches0)
    v = np.nonzero(m > -1)[0]
    q = np.concatenate([k0[v], k1[m[v]]], 1).astype(np.int64) if len(v) else np.zeros((0, 4), np.int64)
    return {tuple(r) for r in q.tolist()}


def kpt_set(k):
    k = np.asarray(k).astype(np.int64)
    return set((k[:, 1] * 100000 + k[:, 0]).tolist())


def compare_pair(eng, ref):
    """eng / ref: dicts with kpts0, kpts1, matches0, stop.  -> per-pair report."""
    a, b = match_tuples(eng["kpts0"], eng["kpts1"], eng["matches0"]), match_tuples(ref["kpts0"], ref["kpts1"], ref["matches0"])
    tp = len(a & b)
    f1 = 1.0 if not a and not b else 2.0 * tp / max(len(a) + len(b), 1)
    same_order = all(np.array_equal(np.asarray(eng[k]), np.asarray(ref[k])) for k in ("kpts0", "kpts1"))
    return {"kpts_set_equal": kpt_set(eng["kpts0"]) == kpt_set(ref["kpts0"]) and kpt_set(eng["kpts1"]) == kpt_set(ref["kpts1"]),
            "kpts_order_equal": same_order,
            "index_exact": bool(same_order and np.array_equal(np.asarray(eng["matches0"]), np.asarray(ref["matches0"]))),
            "stop_equal": int(eng["stop"]) == int(ref["stop"]), "stop": (int(eng["stop"]), int(ref["stop"])),
            "f1": f1, "exact": a == b, "n_eng": len(a), "n_ref": len(b)}


def engine_pairs(h_matches, h_kpts, h_counts, h_stop, n_pairs):
    """PairEngine.match_host() host buffers -> the per-pair dicts compare_pair() takes."""
    out = []
    for p in range(n_pairs):
        n0, n1 = int(h_counts[0][2 * p]), int(h_counts[0][2 * p + 1])
        out.append({"kpts0": np.asarray(h_kpts[2 * p][:n0]), "kpts1": np.asarray(h_kpts[2 * p + 1][:n1]),
                    "matches0": np.asarray(h_matches[2 * p][:n0]).astype(np.int64), "stop": int(h_stop[p])})
    return out


def summarize(reports):
    n = max(len(reports), 1)
    tp2 = sum(r["f1"] * (r["n_eng"] + r["n_ref"]) for r in reports)
    tot = sum(r["n_eng"] + r["n_ref"] for r in reports)
    return {"pairs": len(reports), "match_f1": (tp2 / tot) if tot else 1.0, "min_pair_f1": min((r["f1"] for r in reports), default=1.0),
            "exact_pairs": sum(r["exact"] for r in reports) / n, "index_exact_pairs": sum(r["index_exact"] for r in reports) / n,
            "kpts_set_equal": sum(r["kpts_set_equal"] for r in reports) / n, "stop_equal": sum(r["stop_equal"] for r in reports) / n}
