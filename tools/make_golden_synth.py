"""Regenerate the fixtures whose values depend on the SuperPoint / LightGlue / SuperGlue parameters.

    python tools/make_golden_synth.py

The pretrained checkpoints are not part of the repository, so the tests run these three networks on the deterministic
synthetic parameters of image-matching-webui_b200/utils/synth_weights.py.  This script computes the expected outputs
with the CPU oracle on the inputs already stored under tests/golden/ (images, keypoints, descriptors) and writes:

  sp_sw.npz                       SuperPoint outputs on the images of sp_real / sp_synth / sp_fix (keypoints and scores in
                                  full, descriptors at a seeded sample of keypoints, dense maps sampled)
  lg_*.npz, aliked_lg.npz, sg.npz the output keys of the matcher fixtures, rewritten in place.  lg_proj / lg_so keep no
                                  descriptors: the tests derive their 128-d inputs from the sp_* descriptors
                                  (conftest.compressed_descriptors).  aliked_lg keeps the ALIKED descriptors as float16
                                  and gets a whitening input_proj fitted on them (see aliked_input_proj).

CPU fp32.
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import oracle  # noqa: E402
from oracle import lightglue as olg  # noqa: E402
from oracle import superglue as osg  # noqa: E402
from oracle import superpoint as osp  # noqa: E402

OUT = ROOT / "tests" / "golden"
DESC_SAMPLE = 48          # descriptor columns kept per image
DENSE_SAMPLE = 4096       # dense-score pixels kept per image
SP_CONFS = {
    "api": {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.015, "remove_borders": 4},
    "max1024": {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.005, "remove_borders": 4},
    "nocap": {"nms_radius": 4, "max_keypoints": -1, "keypoint_threshold": 0.005, "remove_borders": 4},
    "max2048": {"nms_radius": 3, "max_keypoints": 2048, "keypoint_threshold": 0.005, "remove_borders": 4},
}
SP_FIX_CONF = {"nms_radius": 3, "max_keypoints": 256, "keypoint_threshold": 0.005, "remove_borders": 4, "fix_sampling": True}
LG_MODES = {
    "full": dict(depth_confidence=-1, width_confidence=-1, pruning_min_kpts=-1),
    "cuda": dict(depth_confidence=0.95, width_confidence=0.99, pruning_min_kpts=1536),
    "cpu": dict(depth_confidence=0.95, width_confidence=0.99, pruning_min_kpts=-1),
}


def load(name):
    return dict(np.load(OUT / f"{name}.npz"))


def save(name, blob):
    np.savez_compressed(OUT / f"{name}.npz", **blob)
    print("wrote", name, f"{(OUT / f'{name}.npz').stat().st_size / 1e3:.0f} kB")


def sp_entry(blob, pre, out, rng):
    k, s, d = out["keypoints"][0], out["scores"][0], out["descriptors"][0]
    cols = np.sort(rng.choice(len(k), min(DESC_SAMPLE, len(k)), replace=False)).astype(np.int32)
    blob[pre + "keypoints"] = k.numpy().astype(np.int16)
    blob[pre + "scores"] = s.numpy()
    blob[pre + "desc_cols"] = cols
    blob[pre + "descriptors"] = d.numpy()[:, cols]


def sp_fixtures():
    w = oracle.synthetic_weights("superpoint")
    rng = np.random.default_rng(0)
    blob = {}
    for case, confs in (("sp_real", ["api", "max1024", "nocap"]), ("sp_synth", ["max1024", "max2048"])):
        images = torch.from_numpy(load(case)["images"])
        for c in confs:
            for b in range(images.shape[0]):
                sp_entry(blob, f"{case}/{c}/{b}/", osp.forward(w, images[b:b + 1], SP_CONFS[c]), rng)
    images = torch.from_numpy(load("sp_fix")["images"])
    for b in range(images.shape[0]):
        sp_entry(blob, f"fix/{b}/", osp.forward(w, images[b:b + 1], SP_FIX_CONF), rng)
    images = torch.from_numpy(load("sp_real")["images"])
    out = osp.forward(w, images, SP_CONFS["api"], return_dense=True)
    for b in range(images.shape[0]):
        dense = out["dense_scores"][b].numpy().ravel()
        idx = np.sort(rng.choice(dense.size, DENSE_SAMPLE, replace=False)).astype(np.int32)
        blob[f"dense/{b}/idx"], blob[f"dense/{b}/scores"] = idx, dense[idx]
        blob[f"dense/{b}/nms3_bits"] = np.packbits(out["nms_scores"][b].numpy().ravel() > 0)
        blob[f"dense/{b}/desc_sub"] = out["dense_descriptors"][b, :, ::16, ::16].numpy()
    # the registry pipeline's pair (sp_real images, API keypoint settings): raw LightGlue match count, CUDA semantics
    f = osp.forward(w, images, SP_CONFS["api"])
    r = olg.forward(oracle.synthetic_weights("lightglue"), f["keypoints"][0][None], f["descriptors"][0].t().contiguous()[None],
                    f["keypoints"][1][None], f["descriptors"][1].t().contiguous()[None], LG_MODES["cuda"])
    blob["registry/n_matches"] = np.int32((r["matches0"] > -1).sum())
    # the registry pipeline's synthetic pair (seed 0 as RGB frames, superpoint_max pre-processing forced to 640x480)
    import importlib.util
    from oracle import preprocess as opre
    spec = importlib.util.spec_from_file_location("synth", ROOT / "image-matching-webui_b200/utils/synth.py")
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    pre = {"grayscale": True, "resize_max": 1600, "dfactor": 8, "force_resize": True, "width": 640, "height": 480}
    a, c, _ = synth.make_pair(0, 480, 640)
    x = torch.cat([torch.from_numpy(opre.preprocess(synth.to_rgb(im), pre)[0])[None] for im in (a, c)])
    f = osp.forward(w, x, SP_CONFS["api"])
    r = olg.forward(oracle.synthetic_weights("lightglue"), f["keypoints"][0][None], f["descriptors"][0].t().contiguous()[None],
                    f["keypoints"][1][None], f["descriptors"][1].t().contiguous()[None], LG_MODES["cuda"])
    blob["registry/synth/n_matches"] = np.int32((r["matches0"] > -1).sum())
    save("sp_sw", blob)


def lg_outputs(blob, pre, out, keys):
    for k in keys:
        v = out[k][0].numpy()
        blob[pre + k] = v.astype(np.int32) if k in ("matches0", "matches1", "prune0", "prune1") else v
    blob[pre + "stop"] = np.int32(out["stop"])


def aliked_input_proj(descs, dim=256, seed=7):
    """Linear(128 -> 256) for the ALIKED composition: the ALIKED descriptors nearly share one direction, so input_proj
    subtracts their mean, whitens them (PCA over all stored descriptors) and lifts them by a seeded orthonormal map; rows
    come out with unit norm on average.  The synthetic LightGlue then matches by the similarity of these rows."""
    d = np.concatenate(descs).astype(np.float64)
    mu = d.mean(0)
    _, s, vt = np.linalg.svd(d - mu, full_matrices=False)
    q, _ = np.linalg.qr(np.random.default_rng(seed).standard_normal((dim, d.shape[1])))
    w = q @ (vt / s[:, None]) * np.sqrt(len(d) / d.shape[1])
    return w.astype(np.float32), (-w @ mu).astype(np.float32)


def lg_fixtures():
    from conftest import compressed_descriptors, lg_pair_from_source
    w = oracle.synthetic_weights("lightglue")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))[None]
    cache = {}
    golden = lambda n: cache.setdefault(n, load(n))
    all_keys = ("matches0", "matches1", "matching_scores0", "matching_scores1", "prune0", "prune1")
    for case in ("lg_real", "lg_synth"):
        blob = load(case)
        for mode, mconf in LG_MODES.items():
            for p, src in enumerate(blob["sources"]):
                k0, d0, k1, d1 = lg_pair_from_source(golden, src)
                out = olg.forward(w, t(k0), t(d0.T), t(k1), t(d1.T), mconf)
                lg_outputs(blob, f"{mode}/{p}/", out, all_keys)
                print(case, mode, p, "stop", out["stop"], "matches", int((out["matches0"] > -1).sum()))
        save(case, blob)
    for case in ("lg_proj", "lg_so"):
        blob = load(case)
        wp = {**w, "input_proj.weight": torch.from_numpy(blob["input_proj_w"]), "input_proj.bias": torch.from_numpy(blob["input_proj_b"])}
        if case == "lg_so":
            wp["posenc.Wr.weight"] = torch.from_numpy(blob["posenc_wr"])
        for p, src in enumerate(blob["sources"]):
            k0, d0, k1, d1 = lg_pair_from_source(golden, src)
            blob.pop(f"{p}/descriptors0", None), blob.pop(f"{p}/descriptors1", None)
            c0, c1 = (t(compressed_descriptors(d, blob["input_proj_w"])) for d in (d0, d1))
            so = tuple(t(blob[f"{p}/{n}"]) for n in ("scales0", "oris0", "scales1", "oris1")) if case == "lg_so" else None
            out = olg.forward(wp, t(k0), c0, t(k1), c1, LG_MODES["cuda"], scale_ori=so)
            lg_outputs(blob, f"{p}/", out, all_keys if case == "lg_proj" else ("matches0", "matches1", "matching_scores0"))
            print(case, p, "stop", out["stop"], "matches", int((out["matches0"] > -1).sum()))
        save(case, blob)
    blob = load("aliked_lg")
    n_pairs = len(blob["eval_seeds"])
    for p in range(n_pairs):
        for i in range(2):
            blob[f"{p}/descriptors{i}"] = blob[f"{p}/descriptors{i}"].astype(np.float16)
    blob["input_proj_w"], blob["input_proj_b"] = aliked_input_proj([blob[f"{p}/descriptors{i}"] for p in range(n_pairs) for i in range(2)])
    wp = {**w, "input_proj.weight": torch.from_numpy(blob["input_proj_w"]), "input_proj.bias": torch.from_numpy(blob["input_proj_b"])}
    for p in range(n_pairs):
        g = lambda n: t(blob[f"{p}/{n}"].astype(np.float32))
        out = olg.forward(wp, g("keypoints0"), g("descriptors0"), g("keypoints1"), g("descriptors1"), LG_MODES["cuda"])
        lg_outputs(blob, f"{p}/", out, ("matches0", "matching_scores0"))
        print("aliked_lg", p, "stop", out["stop"], "matches", int((out["matches0"] > -1).sum()))
    save("aliked_lg", blob)


def sg_fixtures():
    w = oracle.synthetic_weights("superglue")
    blob = load("sg")
    t = torch.from_numpy
    for it in (50, 20):
        for p, src in enumerate(blob["sources"]):
            f, conf, i, j = str(src).split(":")
            b = load(f)
            data = {"image0": torch.empty(1, 1, 480, 640), "image1": torch.empty(1, 1, 480, 640),
                    "keypoints0": t(b[f"{conf}/{i}/keypoints"].astype(np.float32))[None], "keypoints1": t(b[f"{conf}/{j}/keypoints"].astype(np.float32))[None],
                    "scores0": t(b[f"{conf}/{i}/scores"])[None], "scores1": t(b[f"{conf}/{j}/scores"])[None],
                    "descriptors0": t(b[f"{conf}/{i}/descriptors"])[None], "descriptors1": t(b[f"{conf}/{j}/descriptors"])[None]}
            out = osg.forward(w, data, sinkhorn_iterations=it, match_threshold=0.2)
            pre = f"it{it}/{p}/"
            for k in ("matches0", "matches1"):
                blob[pre + k] = out[k][0].numpy().astype(np.int32)
            for k in ("matching_scores0", "matching_scores1"):
                blob[pre + k] = out[k][0].numpy()
            print("sg", it, p, "matches", int((out["matches0"] > -1).sum()))
    save("sg", blob)


if __name__ == "__main__":
    torch.set_grad_enabled(False)
    sp_fixtures()
    lg_fixtures()
    sg_fixtures()
