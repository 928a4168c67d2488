"""SIFT extractor on the GPU against cv2 (oracle/sift.py): pyramid, detector, descriptors, the plugin with the wrapper's
defaults, and SIFT + mutual NN / LightGlue(features="sift") end to end."""
from pathlib import Path

import numpy as np
import pytest
import torch
from scipy.spatial import cKDTree

from oracle import sift as osift

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"
RAW = {"n_octave_layers": 4, "contrast_threshold": 0.0066667, "edge_threshold": 10, "sigma": 1.6, "max_keypoints": 0,
       "nms_radius": None, "rootsift": False}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _images():
    """[H,W] float32 in [0,1]: synthetic seeds 0-1 (both sides) and the two real frames force-resized to 640x480"""
    from imcui_b200 import ops
    from imcui_b200.utils import synth
    out = []
    for s in (0, 1):
        a, b, _ = synth.make_pair(s, 480, 640)
        out += [a.astype(np.float32) / 255.0, b.astype(np.float32) / 255.0]
    pre = {"grayscale": True, "resize_max": 0, "force_resize": True, "width": 640, "height": 480, "dfactor": 1}
    for name in ("02928139_3448003521", "17295357_9106075285"):
        rgb = np.load(GOLDEN / "data" / f"{name}.npz")["rgb"]
        x = ops.preprocess(torch.from_numpy(rgb).cuda()[None], pre)
        out.append(x[0, 0].cpu().numpy())
    return out


def _match_sets(k_gpu, s_gpu, a_gpu, k_ref, s_ref, a_ref, pt_tol=1e-2, size_rel=1e-3, ang_tol=np.deg2rad(0.5)):
    """pairs (i_gpu, i_ref) with |dpt| <= pt_tol, relative size within size_rel and angle within ang_tol (one-to-one)"""
    tree = cKDTree(k_gpu)
    pairs, used = [], set()
    for j, cands in enumerate(tree.query_ball_point(k_ref, pt_tol)):
        for i in cands:
            da = abs((a_gpu[i] - a_ref[j] + np.pi) % (2 * np.pi) - np.pi)
            if i not in used and abs(s_gpu[i] - s_ref[j]) <= size_rel * s_ref[j] and da <= ang_tol:
                pairs.append((i, j)); used.add(i)
                break
    return np.array(pairs, dtype=np.int64).reshape(-1, 2)


def _gpu(imgs, conf, dev, cap=16384, debug=False):
    from imcui_b200 import ops
    x = torch.from_numpy(np.stack(imgs))[:, None].to(dev)
    out = ops.sift_forward(x, conf, cap, debug=debug)
    torch.cuda.synchronize()
    return out


def test_pyramid_matches_cv2(dev):
    from imcui_b200.utils import synth
    a, _, _ = synth.make_pair(0, 480, 640)
    img = a.astype(np.float32) / 255.0
    out = _gpu([img, img], RAW, dev, cap=64, debug=True)
    ref = osift.pyramid(osift.to_uint8(img))
    for o in range(4):   # octaves -1 .. 2
        g = out["pyramid"][o][0].cpu().numpy()
        err = np.abs(g - ref[o]).max()
        print(f"[sift pyramid] octave {o - 1}: max abs err {err:.2e}")
        assert g.shape == ref[o].shape and err <= 1e-3
    assert torch.equal(out["pyramid"][0][0], out["pyramid"][0][1])


def test_detector_uncapped(dev):
    imgs = _images()
    out = _gpu(imgs, RAW, dev)
    counts = out["counts"].cpu()
    sift = osift.create({**osift.DEFAULT_CONF, "max_num_keypoints": 0})
    for b, img in enumerate(imgs):
        n = int(counts[0, b])
        assert n == int(counts[1, b]) > 0
        kr, sr, scr, ar, _ = osift.run_opencv_sift(sift, osift.to_uint8(img))
        kg, sg = out["keypoints"][b, :n].cpu().numpy(), out["scores"][b, :n].cpu().numpy()
        scg, ag = out["scales"][b, :n].cpu().numpy(), out["oris"][b, :n].cpu().numpy()
        pr = _match_sets(kg, scg, ag, kr, scr, ar)
        recall, precision = len(pr) / len(kr), len(pr) / n
        rerr = np.abs(sg[pr[:, 0]] - sr[pr[:, 1]]).max()
        print(f"[sift detect] image {b}: gpu {n} cv2 {len(kr)} recall {recall:.4f} precision {precision:.4f} response err {rerr:.1e}")
        assert recall >= 0.98 and precision >= 0.98 and rerr <= 1e-5
        assert np.all(np.diff(sg) <= 0)   # descending response


def test_descriptors_raw(dev):
    imgs = _images()
    out = _gpu(imgs, RAW, dev)
    sift = osift.create({**osift.DEFAULT_CONF, "max_num_keypoints": 0})
    tot = close = 0
    for b, img in enumerate(imgs):
        n = int(out["counts"][0, b])
        kr, sr, scr, ar, dr = osift.run_opencv_sift(sift, osift.to_uint8(img))
        kg, ag = out["keypoints"][b, :n].cpu().numpy(), out["oris"][b, :n].cpu().numpy()
        pr = _match_sets(kg, out["scales"][b, :n].cpu().numpy(), ag, kr, scr, ar, ang_tol=np.deg2rad(0.05))
        dg = out["descriptors"][b, :n].cpu().numpy()[pr[:, 0]]
        diff = np.abs(dg - dr[pr[:, 1]])
        assert np.array_equal(dg, np.round(dg)) and dg.max() <= 255
        tot += diff.size
        close += int((diff <= 1).sum())
    print(f"[sift desc] {close / tot:.5f} of entries within +-1 ({tot // 128} keypoints)")
    assert close / tot >= 0.999


def _plugin(dev, conf=None):
    from imcui_b200.hloc import extractors
    from imcui_b200.hloc.utils.base_model import dynamic_load
    return dynamic_load(extractors, "sift")(conf or {}).eval().to(dev)


def test_plugin_defaults(dev):
    from imcui_b200.utils import synth
    model = _plugin(dev)
    a, b, _ = synth.make_pair(0, 480, 640)
    x0, x1 = (torch.from_numpy(v.astype(np.float32) / 255.0) for v in (a, b))
    batch = torch.stack([x0, torch.flip(x0, (1,)), x0])[:, None].to(dev)
    with torch.no_grad():
        out = model({"image": batch})
    for k in ("keypoints", "scores", "descriptors", "scales", "oris"):
        assert torch.equal(out[k][0], out[k][2]), k   # same image, same bits in any slot
    n = out["keypoints"][0].shape[0]
    assert out["keypoints"][0].shape == (n, 2) and out["descriptors"][0].shape == (128, n)
    assert out["scores"][0].shape == out["scales"][0].shape == out["oris"][0].shape == (n,)
    assert torch.allclose(out["descriptors"][0].norm(dim=0), torch.ones(n, device=dev), atol=1e-5)
    ref = osift.extract(x0.numpy())
    nr = len(ref["keypoints"])
    pr = _match_sets(out["keypoints"][0].cpu().numpy(), out["scales"][0].cpu().numpy(), out["oris"][0].cpu().numpy(),
                     ref["keypoints"].numpy(), ref["scales"].numpy(), ref["oris"].numpy())
    print(f"[sift plugin] kept {n} oracle {nr} set recall {len(pr) / nr:.4f}")
    assert abs(n - nr) <= 0.01 * nr and len(pr) / nr >= 0.98 and n <= 4096
    with pytest.raises(NotImplementedError):
        model({"image": batch[:1].repeat(1, 3, 1, 1)})


def _nn_inliers(k0, d0, k1, d1, Hm):
    from imcui_b200 import ops
    from oracle import matchers as om
    m = om.nearest_neighbor(d0.t()[None].cpu(), d1.t()[None].cpu(), do_mutual_check=True)["matches0"][0].numpy()
    v = m > -1
    p0, p1 = k0[v].cpu().numpy(), k1[m[v]].cpu().numpy()
    q = np.c_[p0, np.ones(len(p0))] @ Hm.T
    return int((np.linalg.norm(q[:, :2] / q[:, 2:] - p1, axis=1) <= 3).sum()), int(v.sum())


def test_sift_nearest_neighbor(dev):
    from imcui_b200.hloc import matchers
    from imcui_b200.hloc.utils.base_model import dynamic_load
    from imcui_b200.utils import synth
    model = _plugin(dev)
    nn = dynamic_load(matchers, "nearest_neighbor")({"do_mutual_check": True}).eval().to(dev)
    for seed in range(4):
        a, b, Hm = synth.make_pair(seed, 480, 640)
        x = torch.from_numpy(np.stack([a, b]).astype(np.float32) / 255.0)[:, None].to(dev)
        with torch.no_grad():
            f = model({"image": x})
            pred = nn({"descriptors0": f["descriptors"][0][None], "descriptors1": f["descriptors"][1][None]})
        m = pred["matches0"][0].cpu().numpy()
        v = m > -1
        p0, p1 = f["keypoints"][0].cpu().numpy()[v], f["keypoints"][1].cpu().numpy()[m[v]]
        q = np.c_[p0, np.ones(len(p0))] @ Hm.T
        good = int((np.linalg.norm(q[:, :2] / q[:, 2:] - p1, axis=1) <= 3).sum())
        r0, r1 = osift.extract(a.astype(np.float32) / 255.0), osift.extract(b.astype(np.float32) / 255.0)
        good_ref, n_ref = _nn_inliers(r0["keypoints"], r0["descriptors"], r1["keypoints"], r1["descriptors"], Hm)
        print(f"[sift+nn] seed {seed}: {int(v.sum())} matches, {good} within 3 px (oracle chain {n_ref} / {good_ref})")
        assert good >= 0.97 * good_ref


def test_sift_lightglue_magsac(dev):
    import oracle
    from oracle import lightglue as olg
    from imcui_b200.hloc import extract_features, match_features, matchers
    from imcui_b200.hloc.utils.base_model import dynamic_load
    from imcui_b200.ui import utils as U
    from imcui_b200.utils import synth
    from conftest import match_f1
    g = np.load(GOLDEN / "lg_so.npz")
    sd = dict(oracle.synthetic_weights("lightglue"))
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    sd["posenc.Wr.weight"] = torch.from_numpy(g["posenc_wr"])
    lg = dynamic_load(matchers, "lightglue")({"match_threshold": 0.2, "features": "sift", "state_dict": dict(sd)}).eval().to(dev)
    ext = _plugin(dev)
    pre = {"grayscale": True, "resize_max": 1024, "force_resize": False, "dfactor": 8}
    a, b, _ = synth.make_pair(0, 480, 640)
    f0, f1 = extract_features.extract(ext, a, pre), extract_features.extract(ext, b, pre)
    pred = match_features.match_images(lg, f0, f1)
    k0, k1 = f0["keypoints"][0][None].cpu(), f1["keypoints"][0][None].cpu()
    d0, d1 = f0["descriptors"][0].t()[None].cpu(), f1["descriptors"][0].t()[None].cpu()
    so = tuple(f[k][0][None].cpu() for f in (f0,) for k in ("scales", "oris")) + \
        tuple(f[k][0][None].cpu() for f in (f1,) for k in ("scales", "oris"))
    ref = olg.forward(sd, k0, d0, k1, d1, {"pruning_min_kpts": 1536}, scale_ori=so)
    data = match_features.pair_inputs(f0, f1)
    with torch.no_grad():
        out = lg(data)
    f1s = match_f1(out["matches0"][0].cpu().numpy(), ref["matches0"][0].numpy())
    geo = U.filter_matches(dict(pred), "B200_MAGSAC", 8, 0.9999, 10000)
    print(f"[sift+lg] {len(k0[0])}/{len(k1[0])} keypoints, {len(pred['mkeypoints0_orig'])} matches, F1 {f1s:.4f}, "
          f"verified {len(geo['mmkeypoints0_orig'])}, {geo.get('geom_info', {}).keys()}")
    assert f1s >= 0.999
    assert "Homography" in geo["geom_info"]


def test_export_features_and_match_from_paths(dev, tmp_path):
    """The batched exporters with a SIFT conf on 4 frames: stored features are the plugin's (fp16, scales / oris included),
    and the stored matches are the single-pair plugin call's on those stored features, for mutual NN and for LightGlue."""
    import cv2
    import oracle
    from imcui_b200.hloc import matchers, pairs_stream as ps
    from imcui_b200.hloc.configs import confs_dict
    from imcui_b200.hloc.utils.base_model import dynamic_load
    from imcui_b200.hloc.utils.store import open_store
    from imcui_b200.utils import synth
    root = tmp_path / "images"
    root.mkdir()
    names = []
    for s in (0, 1):
        a, b, _ = synth.make_pair(s, 480, 640)
        for tag, im in (("a", a), ("b", b)):
            cv2.imwrite(str(root / f"{s}{tag}.png"), im)
            names.append(f"{s}{tag}.png")
    econf = {"output": "feats-sift", "model": {"name": "sift", "max_num_keypoints": 4096},
             "preprocessing": {"grayscale": True, "resize_max": 1024}}
    fpath = ps.export_features(econf, root, feature_path=tmp_path / "feats.imw", batch=4)
    keys = ("keypoints", "scores", "descriptors", "scales", "oris")
    ext = _plugin(dev)
    with open_store(fpath, "r") as st:
        assert sorted(st.groups()) == sorted(names)
        for n in names:   # 640x480 <= resize_max: stored in the frame's own coordinates
            g = cv2.imread(str(root / n), cv2.IMREAD_GRAYSCALE).astype(np.float32) / 255.0
            with torch.no_grad():
                f = ext({"image": torch.from_numpy(g)[None, None].to(dev)})
            for k in keys:
                ref = f[k][0].cpu().numpy().astype(np.float16)
                assert st.read(n, k).dtype == np.float16 and np.array_equal(st.read(n, k), ref), (n, k)
    pairs = [("0a.png", "0b.png"), ("1a.png", "1b.png")]
    (tmp_path / "pairs.txt").write_text("".join(f"{a} {b}\n" for a, b in pairs))
    g = np.load(GOLDEN / "lg_so.npz")
    sd = dict(oracle.synthetic_weights("lightglue"))
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    sd["posenc.Wr.weight"] = torch.from_numpy(g["posenc_wr"])
    lg_conf = {"output": "matches-sift-lightglue",
               "model": {"name": "lightglue", "features": "sift", "match_threshold": 0.2, "state_dict": sd}}
    for mconf, plugin in ((confs_dict["matchers"]["NN-mutual"], "nearest_neighbor"), (lg_conf, "lightglue")):
        mpath = ps.match_from_paths(mconf, tmp_path / "pairs.txt", tmp_path / f"m_{plugin}.imw", fpath, fpath, batch=2)
        model = dynamic_load(matchers, plugin)({**mconf["model"], "state_dict": dict(sd)} if plugin == "lightglue"
                                               else mconf["model"]).eval().to(dev)
        with open_store(mpath, "r") as ms, open_store(fpath, "r") as fs:
            assert len(ms.groups()) == len(pairs)
            for a, b in pairs:
                f = [{k: torch.from_numpy(fs.read(n, k).astype(np.float32)).to(dev) for k in keys} for n in (a, b)]
                data = {f"{k}{i}": f[i][k][None] for i in (0, 1) for k in keys}
                data["image0"], data["image1"] = torch.empty(1, 1, 480, 640), torch.empty(1, 1, 480, 640)
                with torch.no_grad():
                    m_ref = model(data)["matches0"][0].cpu().short().numpy()
                stored = ms.read(f"{a}/{b}", "matches0")
                print(f"[sift export] {plugin} {a} x {b}: {int((m_ref > -1).sum())} matches, "
                      f"agreement with the single-pair call {(stored == m_ref).mean():.4f}")
                # LightGlue runs the batch at the largest padded size of the chunk (as tests/test_pairs_stream.py allows)
                assert stored.dtype == np.int16 and (stored == m_ref).mean() >= (1.0 if plugin == "nearest_neighbor" else 0.995)
