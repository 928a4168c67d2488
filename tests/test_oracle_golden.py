"""Pin the CPU oracle (oracle/) against fixtures produced by the unmodified reference modules
(tools/make_golden.py) and, for the networks that run on synthetic parameters (SuperPoint, LightGlue, SuperGlue), against
the oracle's own outputs on the stored inputs (tools/make_golden_synth.py).  CPU only."""
import numpy as np
import pytest
import torch

import oracle
from oracle import lightglue as olg
from oracle import matchers as om
from oracle import superpoint as osp
from conftest import ROOT, compressed_descriptors, lg_pair_from_source, match_f1

SP_CONFS = {
    "api": {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.015, "remove_borders": 4},
    "max1024": {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.005, "remove_borders": 4},
    "nocap": {"nms_radius": 4, "max_keypoints": -1, "keypoint_threshold": 0.005, "remove_borders": 4},
    "max2048": {"nms_radius": 3, "max_keypoints": 2048, "keypoint_threshold": 0.005, "remove_borders": 4},
}


@pytest.mark.parametrize("case,confs", [("sp_real", ["api", "max1024", "nocap"]), ("sp_synth", ["max1024", "max2048"])])
def test_superpoint_oracle_matches_reference(golden, case, confs):
    g, s = golden(case), golden("sp_sw")
    w = oracle.synthetic_weights("superpoint")
    images = torch.from_numpy(g["images"])
    for c in confs:
        for b in range(images.shape[0]):
            out = osp.forward(w, images[b:b + 1], SP_CONFS[c])
            pre = f"{case}/{c}/{b}/"
            # keypoint set + order bit-exact, scores/descriptors to 1e-5 (same machine class: ~0)
            assert np.array_equal(out["keypoints"][0].numpy().astype(np.int16), s[pre + "keypoints"]), (case, c, b)
            np.testing.assert_allclose(out["scores"][0].numpy(), s[pre + "scores"], atol=1e-5)
            np.testing.assert_allclose(out["descriptors"][0].numpy()[:, s[pre + "desc_cols"]], s[pre + "descriptors"], atol=1e-4)


def test_superpoint_oracle_fix_sampling(golden):
    """oracle.sample_descriptors_fix_sampling (fix_sampling=True) on the sp_fix images."""
    g, s = golden("sp_fix"), golden("sp_sw")
    w = oracle.synthetic_weights("superpoint")
    conf = {"nms_radius": 3, "max_keypoints": 256, "keypoint_threshold": 0.005, "remove_borders": 4, "fix_sampling": True}
    images = torch.from_numpy(g["images"])
    for b in range(images.shape[0]):
        out = osp.forward(w, images[b:b + 1], conf)
        cols = s[f"fix/{b}/desc_cols"]
        assert np.array_equal(out["keypoints"][0].numpy().astype(np.int16), s[f"fix/{b}/keypoints"])
        np.testing.assert_allclose(out["descriptors"][0].numpy()[:, cols], s[f"fix/{b}/descriptors"], atol=1e-4)
        plain = osp.forward(w, images[b:b + 1], {**conf, "fix_sampling": False})
        assert np.abs(plain["descriptors"][0].numpy()[:, cols] - s[f"fix/{b}/descriptors"]).max() > 1e-2


def test_superpoint_oracle_dense_maps(golden):
    g, s = golden("sp_real"), golden("sp_sw")
    w = oracle.synthetic_weights("superpoint")
    out = osp.forward(w, torch.from_numpy(g["images"]), SP_CONFS["api"], return_dense=True)
    for b in range(2):
        np.testing.assert_allclose(out["dense_scores"][b].numpy().ravel()[s[f"dense/{b}/idx"]], s[f"dense/{b}/scores"], atol=2e-6)
        assert np.array_equal(np.packbits(out["nms_scores"][b].numpy().ravel() > 0), s[f"dense/{b}/nms3_bits"])
        np.testing.assert_allclose(out["dense_descriptors"][b, :, ::16, ::16].numpy(), s[f"dense/{b}/desc_sub"], atol=1e-5)


def test_superpoint_oracle_rejects_bad_max_keypoints():
    w = oracle.synthetic_weights("superpoint")
    with pytest.raises(ValueError):
        osp.forward(w, torch.zeros(1, 1, 16, 16), {"max_keypoints": 0})


MODES = {
    "full": dict(depth_confidence=-1, width_confidence=-1, pruning_min_kpts=-1),
    "cuda": dict(depth_confidence=0.95, width_confidence=0.99, pruning_min_kpts=1536),
    "cpu": dict(depth_confidence=0.95, width_confidence=0.99, pruning_min_kpts=-1),
}


@pytest.mark.parametrize("case", ["lg_real", "lg_synth"])
@pytest.mark.parametrize("mode", ["full", "cuda", "cpu"])
def test_lightglue_oracle_matches_reference(golden, case, mode):
    g = golden(case)
    w = oracle.synthetic_weights("lightglue")
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        out = olg.forward(w, torch.from_numpy(k0)[None], torch.from_numpy(d0).t().contiguous()[None],
                          torch.from_numpy(k1)[None], torch.from_numpy(d1).t().contiguous()[None], MODES[mode])
        pre = f"{mode}/{p}/"
        assert out["stop"] == int(g[pre + "stop"])
        assert np.array_equal(out["matches0"][0].numpy(), g[pre + "matches0"]), (case, mode, p, match_f1(out["matches0"][0].numpy(), g[pre + "matches0"]))
        assert np.array_equal(out["matches1"][0].numpy(), g[pre + "matches1"])
        np.testing.assert_allclose(out["matching_scores0"][0].numpy(), g[pre + "matching_scores0"], atol=1e-4)
        assert np.array_equal(out["prune0"][0].numpy().astype(np.int32), g[pre + "prune0"])
        assert np.array_equal(out["prune1"][0].numpy().astype(np.int32), g[pre + "prune1"])


def _lg_proj_weights(g):
    w = dict(oracle.synthetic_weights("lightglue"))
    w["input_proj.weight"], w["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    return w


def test_lightglue_input_proj_oracle_matches_reference(golden):
    """LightGlue with a Linear(128 -> 256) input_proj (aliked / disk architecture, lightglue.py:392-395,519-520)."""
    g = golden("lg_proj")
    w = _lg_proj_weights(g)
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        c0, c1 = (torch.from_numpy(compressed_descriptors(d, g["input_proj_w"]))[None] for d in (d0, d1))
        out = olg.forward(w, torch.from_numpy(k0)[None], c0, torch.from_numpy(k1)[None], c1, MODES["cuda"])
        assert out["stop"] == int(g[f"{p}/stop"])
        assert np.array_equal(out["matches0"][0].numpy(), g[f"{p}/matches0"])
        np.testing.assert_allclose(out["matching_scores0"][0].numpy(), g[f"{p}/matching_scores0"], atol=1e-4)


def test_aliked_lightglue_fitted_input_proj_oracle_matches_reference(golden):
    """BASELINE configs[3] composition on the reference's own outputs: reference ALIKED features -> LightGlue(input_dim=128) with the
    fitted input_proj (tools/make_golden.py aliked_lg_case).  The oracle reproduces matches0 / stop, and the matches are real:
    most of them lie within 3 px of the ground-truth warp."""
    g = golden("aliked_lg")
    w = _lg_proj_weights(g)
    for p in range(len(g["eval_seeds"])):
        t = lambda n: torch.from_numpy(g[f"{p}/{n}"].astype(np.float32))[None]
        out = olg.forward(w, t("keypoints0"), t("descriptors0"), t("keypoints1"), t("descriptors1"), MODES["cuda"])
        assert out["stop"] == int(g[f"{p}/stop"])
        m = out["matches0"][0].numpy()
        assert np.array_equal(m, g[f"{p}/matches0"])
        np.testing.assert_allclose(out["matching_scores0"][0].numpy(), g[f"{p}/matching_scores0"], atol=1e-4)
        v = m > -1
        q = np.concatenate([g[f"{p}/keypoints0"][v], np.ones((v.sum(), 1))], 1) @ g[f"{p}/H"].T
        err = np.linalg.norm(q[:, :2] / q[:, 2:] - g[f"{p}/keypoints1"][m[v]], axis=1)
        assert v.sum() > 300 and (err < 3).mean() > 0.8


def test_lightglue_scale_ori_oracle_matches_reference(golden):
    """LightGlue with add_scale_ori (sift / doghardnet architecture, lightglue.py:366-377,500-506): posenc over
    (x, y, scale, orientation)."""
    g = golden("lg_so")
    w = _lg_proj_weights(g)
    w["posenc.Wr.weight"] = torch.from_numpy(g["posenc_wr"])
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        c0, c1 = (torch.from_numpy(compressed_descriptors(d, g["input_proj_w"]))[None] for d in (d0, d1))
        so = tuple(torch.from_numpy(g[f"{p}/{n}"])[None] for n in ("scales0", "oris0", "scales1", "oris1"))
        out = olg.forward(w, torch.from_numpy(k0)[None], c0, torch.from_numpy(k1)[None], c1, MODES["cuda"], scale_ori=so)
        assert out["stop"] == int(g[f"{p}/stop"])
        assert np.array_equal(out["matches0"][0].numpy(), g[f"{p}/matches0"])
        np.testing.assert_allclose(out["matching_scores0"][0].numpy(), g[f"{p}/matching_scores0"], atol=1e-4)


def _sg_data(golden, src):
    f, conf, i, j = str(src).split(":")
    b = golden(f)
    t = torch.from_numpy
    return {"image0": torch.empty(1, 1, 480, 640), "image1": torch.empty(1, 1, 480, 640),
            "keypoints0": t(b[f"{conf}/{i}/keypoints"].astype(np.float32))[None], "keypoints1": t(b[f"{conf}/{j}/keypoints"].astype(np.float32))[None],
            "scores0": t(b[f"{conf}/{i}/scores"])[None], "scores1": t(b[f"{conf}/{j}/scores"])[None],
            "descriptors0": t(b[f"{conf}/{i}/descriptors"])[None], "descriptors1": t(b[f"{conf}/{j}/descriptors"])[None]}


@pytest.mark.parametrize("iters", [50, 20])
def test_superglue_oracle_matches_reference(golden, iters):
    from oracle import superglue as osg
    g = golden("sg")
    w = oracle.synthetic_weights("superglue")
    for p, src in enumerate(g["sources"]):
        out = osg.forward(w, _sg_data(golden, src), sinkhorn_iterations=iters, match_threshold=0.2)
        pre = f"it{iters}/{p}/"
        assert np.array_equal(out["matches0"][0].numpy(), g[pre + "matches0"])
        assert np.array_equal(out["matches1"][0].numpy(), g[pre + "matches1"])
        np.testing.assert_allclose(out["matching_scores0"][0].numpy(), g[pre + "matching_scores0"], atol=1e-5)


@pytest.mark.parametrize("tag", ["s", "m"])
def test_loftr_oracle_matches_reference(golden, tag):
    """Oracle == the in-tree LoFTR module (SE2LoFTR copy) with the same deterministic random weights."""
    import importlib.util
    from conftest import ROOT
    from oracle import loftr as ol
    spec = importlib.util.spec_from_file_location("synth", ROOT / "image-matching-webui_b200/utils/synth.py")
    synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
    g = golden("loftr")
    H, W = (int(v) for v in g[tag + "/hw"])
    a, b, _ = synth.make_pair(0, H, W)
    x0 = torch.from_numpy(a.astype(np.float32) / 255.0)[None, None]; x1 = torch.from_numpy(b.astype(np.float32) / 255.0)[None, None]
    o = ol.forward(ol.random_weights(0), x0, x1, thr=float(g[tag + "/thr"]))
    assert np.array_equal(o["i_ids"].numpy(), g[tag + "/i_ids"]) and np.array_equal(o["j_ids"].numpy(), g[tag + "/j_ids"])
    assert np.array_equal(o["keypoints0"].numpy(), g[tag + "/keypoints0"])
    np.testing.assert_allclose(o["keypoints1"].numpy(), g[tag + "/keypoints1"], atol=1e-4)
    np.testing.assert_allclose(o["confidence"].numpy(), g[tag + "/confidence"], rtol=1e-4)
    np.testing.assert_allclose(o["conf_matrix"][0].max(1)[0].numpy(), g[tag + "/conf_rowmax"], rtol=1e-4)


@pytest.mark.parametrize("tag", ["d", "e"])
def test_loftr_oracle_different_sizes(golden, tag):
    """Pairs whose two images differ in size (backbone per image, loftr.py:48-56): oracle == the unmodified module."""
    from oracle import loftr as ol
    g = golden("loftr_hw")
    x0 = torch.from_numpy(g[tag + "/image0"].astype(np.float32) / 255.0)[None, None]
    x1 = torch.from_numpy(g[tag + "/image1"].astype(np.float32) / 255.0)[None, None]
    o = ol.forward(ol.random_weights(0), x0, x1, thr=float(g[tag + "/thr"]))
    assert len(g[tag + "/i_ids"]) > 0
    assert np.array_equal(o["i_ids"].numpy(), g[tag + "/i_ids"]) and np.array_equal(o["j_ids"].numpy(), g[tag + "/j_ids"])
    assert np.array_equal(o["keypoints0"].numpy(), g[tag + "/keypoints0"])
    np.testing.assert_allclose(o["keypoints1"].numpy(), g[tag + "/keypoints1"], atol=1e-4)
    np.testing.assert_allclose(o["confidence"].numpy(), g[tag + "/confidence"], rtol=1e-4)


def _matcher_inputs(golden, p):
    g = golden("matchers")
    if p == 0:
        s = golden("sp_real")
        return s["api/0/descriptors"], s["api/1/descriptors"]
    return g[f"in/{p}/descriptors0"], g[f"in/{p}/descriptors1"]


@pytest.mark.parametrize("p", [0, 1])
def test_matchers_oracle_matches_reference(golden, p):
    g = golden("matchers")
    d0, d1 = (torch.from_numpy(x)[None] for x in _matcher_inputs(golden, p))
    cases = {
        "nn": om.nearest_neighbor(d0, d1),
        "nn_ratio": om.nearest_neighbor(d0, d1, ratio_threshold=0.9, distance_threshold=0.9),
        "nn_nomutual": om.nearest_neighbor(d0, d1, do_mutual_check=False),
        "dsm": om.dual_softmax(d0, d1, match_threshold=0.01, inv_temperature=20),
    }
    for tag, out in cases.items():
        assert np.array_equal(out["matches0"][0].numpy(), g[f"{tag}/{p}/matches0"]), tag
        np.testing.assert_allclose(out["matching_scores0"][0].numpy(), g[f"{tag}/{p}/matching_scores0"], atol=1e-6)
    assert cases["dsm"]["matching_scores0"].dtype == torch.float64


def test_matchers_oracle_empty_inputs():
    e = torch.zeros(1, 128, 0)
    d = torch.randn(1, 128, 5)
    for fn in (om.nearest_neighbor, om.dual_softmax):
        out = fn(e, d)
        assert out["matches0"].shape == (1, 128) or out["matches0"].shape == (1, 128)  # reference quirk: shape[:2]
        assert (out["matches0"] == -1).all()


# ---- ALIKED -------------------------------------------------------------------------------------------------------
def _aliked_input(tag):
    import importlib.util
    spec = importlib.util.spec_from_file_location("synth", ROOT / "image-matching-webui_b200/utils/synth.py")
    synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
    from aliked_cases import ALIKED_CASES
    seed, H, W, rgb, conf = ALIKED_CASES[tag]
    a, _, _ = synth.make_pair(seed, H, W)
    if rgb:
        return torch.from_numpy(synth.to_rgb(a).astype(np.float32) / 255.0).permute(2, 0, 1)[None], conf
    return torch.from_numpy(a.astype(np.float32) / 255.0)[None, None], conf


@pytest.mark.parametrize("tag", ["s", "cap", "pad", "topk", "mean", "densecap"])
def test_aliked_oracle_matches_reference(golden, tag):
    from oracle import aliked as oa
    g = golden("aliked")
    img, conf = _aliked_input(tag)
    with torch.no_grad():
        o = oa.forward(oa.random_weights(0), img, **conf)
    assert o["keypoints"].shape == g[tag + "/keypoints"].shape
    np.testing.assert_allclose(o["keypoints"].numpy(), g[tag + "/keypoints"], atol=1e-4)
    np.testing.assert_allclose(o["keypoint_scores"].numpy(), g[tag + "/scores"], atol=1e-6)
    np.testing.assert_allclose(o["descriptors"].numpy(), g[tag + "/descriptors"], atol=2e-5)
    if tag + "/score_map" in g:
        np.testing.assert_allclose(o["score_map"][0, 0].numpy(), g[tag + "/score_map"], atol=1e-6)
        np.testing.assert_allclose(o["feature_map"][0, :, ::40].numpy(), g[tag + "/feature_map_rows"], atol=1e-6)
