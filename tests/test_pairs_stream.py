"""Pair-stream exporters (SURVEY.md 8(f) rank 2): container layout, parsers, pair de-duplication, readers -- CPU;
export_features / match_from_paths end to end against the per-image / per-pair plugin calls -- GPU."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN


def test_record_file_roundtrip_overwrite_and_attrs(tmp_path):
    from imcui_b200.hloc.utils.store import open_store
    path = tmp_path / "feats.imw"
    a = {"keypoints": np.random.rand(5, 2).astype(np.float16), "descriptors": np.random.rand(8, 5).astype(np.float16),
         "image_size": np.array([640, 480])}
    with open_store(path, "a") as st:
        st.write_group("db/1.jpg", a, {"keypoints": {"uncertainty": np.float32(2.5)}})
        st.write_group("q/2.jpg", {"keypoints": np.zeros((0, 2), np.float16)})
    with open_store(path, "a") as st:          # reopen + supersede
        st.write_group("q/2.jpg", {"keypoints": np.ones((3, 2), np.float16), "scores": np.ones(3, np.float16)})
    with open_store(path, "r") as st:
        assert st.groups() == ["db/1.jpg", "q/2.jpg"] and "db/1.jpg" in st and "nope" not in st
        for k, v in a.items():
            got = st.read("db/1.jpg", k)
            assert got.dtype == v.dtype and np.array_equal(got, v)
        assert st.attrs("db/1.jpg", "keypoints")["uncertainty"] == 2.5
        assert st.read("q/2.jpg", "keypoints").shape == (3, 2) and sorted(st.datasets("q/2.jpg")) == ["keypoints", "scores"]
    with pytest.raises(FileNotFoundError):
        open_store(tmp_path / "missing.imw", "r")


def test_parsers_and_pair_keys(tmp_path):
    from imcui_b200.hloc.utils import parsers as P
    (tmp_path / "pairs.txt").write_text("q/a.jpg db/1.jpg\nq/a.jpg db/2.jpg\n\nq/b.jpg db/1.jpg\n")
    assert P.parse_retrieval(tmp_path / "pairs.txt") == {"q/a.jpg": ["db/1.jpg", "db/2.jpg"], "q/b.jpg": ["db/1.jpg"]}
    assert P.names_to_pair("q/a.jpg", "db/1.jpg") == "q-a.jpg/db-1.jpg" and P.names_to_pair_old("q/a.jpg", "db/1.jpg") == "q-a.jpg_db-1.jpg"
    (tmp_path / "list_1.txt").write_text("# comment\nq/a.jpg SIMPLE 1 2 3\n\nq/b.jpg\n")
    (tmp_path / "list_2.txt").write_text("db/1.jpg\n")
    assert P.parse_image_lists(tmp_path / "list_*.txt") == ["q/a.jpg", "q/b.jpg", "db/1.jpg"]


def test_find_unique_new_pairs_and_readers(tmp_path):
    from imcui_b200.hloc import pairs_stream as ps
    from imcui_b200.hloc.utils import io
    from imcui_b200.hloc.utils.parsers import names_to_pair, names_to_pair_old
    from imcui_b200.hloc.utils.store import open_store
    pairs = [("a", "b"), ("b", "a"), ("a", "c"), ("a", "b"), ("c", "d"), ("e", "f")]
    assert ps.find_unique_new_pairs(pairs) == [("a", "b"), ("a", "c"), ("c", "d"), ("e", "f")]
    mp = tmp_path / "m.imw"
    m = np.array([2, -1, 0, -1], np.int16); sc = np.array([0.9, 0, 0.5, 0], np.float16)
    with open_store(mp, "a") as st:
        st.write_group(names_to_pair("c", "a"), {"matches0": m, "matching_scores0": sc})       # stored reversed
        st.write_group(names_to_pair_old("c", "d"), {"matches0": m, "matching_scores0": sc})   # old-style key
    assert ps.find_unique_new_pairs(pairs, mp) == [("a", "b"), ("e", "f")]
    mm, ss = io.get_matches(mp, "a", "c")                                                     # reversed -> flipped columns
    assert mm.tolist() == [[2, 0], [0, 2]] and ss.tolist() == [np.float16(0.9), np.float16(0.5)]
    mm, _ = io.get_matches(mp, "c", "d")
    assert mm.tolist() == [[0, 2], [2, 0]]
    with pytest.raises(ValueError):
        io.get_matches(mp, "x", "y")
    assert sorted(io.list_h5_names(mp)) == sorted([names_to_pair("c", "a"), names_to_pair_old("c", "d")])


def test_list_images_and_dataset_size(tmp_path):
    import cv2
    from imcui_b200.hloc import pairs_stream as ps
    (tmp_path / "sub").mkdir()
    for n in ("b.png", "sub/a.jpg", "c.txt"):
        if n.endswith("txt"):
            (tmp_path / n).write_text("x")
        else:
            cv2.imwrite(str(tmp_path / n), np.zeros((4, 6, 3), np.uint8))
    assert ps.list_images(tmp_path) == ["b.png", "sub/a.jpg"]
    assert ps.list_images(tmp_path, ["sub/a.jpg"]) == ["sub/a.jpg"]
    with pytest.raises(ValueError):
        ps.list_images(tmp_path, ["nope.jpg"])
    # ImageDataset resize rule (extract_features.py:82-87)
    assert ps._dataset_size((1063, 780), {"resize_max": 1024}) == (751, 1024)
    assert ps._dataset_size((480, 640), {"resize_max": 1024}) is None
    assert ps._dataset_size((480, 640), {"resize_max": 1024, "force_resize": True}) == (1024, 768)
    assert ps.read_image(tmp_path / "b.png", grayscale=True).shape == (4, 6)


@pytest.mark.gpu
def test_export_features_and_match_from_paths(tmp_path):
    """Files written by the batched exporters == what the reference's per-image / per-pair loops store: keypoints in the original
    frame as fp16, descriptors fp16, matches0 int16 equal to the single-pair plugin result on the stored features."""
    import cv2
    import oracle
    from imcui_b200.hloc import extractors, matchers, pairs_stream as ps
    from imcui_b200.hloc.configs import confs_dict
    from imcui_b200.hloc.utils import io
    from imcui_b200.hloc.utils.base_model import dynamic_load
    from imcui_b200.hloc.utils.store import open_store
    from imcui_b200.utils import synth
    dev = torch.device("cuda:0")
    root = tmp_path / "images"
    (root / "db").mkdir(parents=True)
    names = []
    for s in range(3):
        a, b, _ = synth.make_pair(s, 480, 640)
        for tag, im in (("a", a), ("b", b)):
            n = f"db/{s}{tag}.png"
            cv2.imwrite(str(root / n), im)
            names.append(n)
    big = cv2.resize(synth.make_pair(7, 480, 640)[0], (1300, 975), interpolation=cv2.INTER_LINEAR)
    cv2.imwrite(str(root / "big.png"), big)                                  # larger than resize_max: area-resized to 1024x768
    names.append("big.png")
    econf = {"output": "feats-superpoint-n1024-r1024", "model": {**confs_dict["extractors"]["superpoint_aachen"]["model"], "max_keypoints": 1024,
                                                                  "state_dict": oracle.synthetic_weights("superpoint")},
             "preprocessing": {"grayscale": True, "resize_max": 1024}}
    fpath = ps.export_features(econf, root, feature_path=tmp_path / "feats.imw", batch=4)
    assert sorted(io.list_h5_names(fpath)) == sorted(names)
    ext = dynamic_load(extractors, "superpoint")(econf["model"]).eval().to(dev)
    with open_store(fpath, "r") as st:
        for n in ("db/1a.png", "big.png"):
            g = cv2.imread(str(root / n), cv2.IMREAD_GRAYSCALE).astype(np.float32)
            if n == "big.png":
                g = cv2.resize(g, (1024, 768), interpolation=cv2.INTER_AREA)
            pred = ext({"image": torch.from_numpy(g / 255.0)[None, None].to(dev)})
            k = pred["keypoints"][0].cpu().numpy()
            orig = np.array(cv2.imread(str(root / n), cv2.IMREAD_GRAYSCALE).shape[::-1])
            scales = (orig / np.array(g.shape[::-1])).astype(np.float32)
            ref_k = ((k + 0.5) * scales[None] - 0.5).astype(np.float16)
            assert st.read(n, "keypoints").dtype == np.float16 and np.array_equal(st.read(n, "keypoints"), ref_k), n
            assert np.array_equal(st.read(n, "descriptors"), pred["descriptors"][0].cpu().numpy().astype(np.float16))
            assert np.array_equal(st.read(n, "scores"), pred["scores"][0].cpu().numpy().astype(np.float16))
            assert st.read(n, "image_size").tolist() == orig.tolist()
            assert abs(st.attrs(n, "keypoints")["uncertainty"] - 2.0 * scales.mean()) < 1e-6
    # second call: everything is already there
    assert ps.export_features(econf, root, feature_path=fpath) == fpath
    (tmp_path / "pairs.txt").write_text("".join(f"db/{s}a.png db/{s}b.png\n" for s in range(3)) + "db/0b.png db/0a.png\ndb/0a.png big.png\n")
    for mname, plugin in (("NN-mutual", "nearest_neighbor"), ("superpoint-lightglue", "lightglue")):
        mconf = confs_dict["matchers"][mname]
        if plugin == "lightglue":
            mconf = {**mconf, "model": {**mconf["model"], "state_dict": oracle.synthetic_weights("lightglue")}}
        mpath = ps.match_from_paths(mconf, tmp_path / "pairs.txt", tmp_path / f"m_{plugin}.imw", fpath, fpath, batch=3)
        model = dynamic_load(matchers, plugin)(mconf["model"]).eval().to(dev)
        with open_store(mpath, "r") as ms, open_store(fpath, "r") as fs:
            assert len(ms.groups()) == 4                                     # the reversed duplicate is dropped
            for a, b in (("db/1a.png", "db/1b.png"), ("db/0a.png", "big.png")):
                f = [{k: torch.from_numpy(fs.read(n, k).astype(np.float32)).to(dev) for k in ("keypoints", "descriptors", "scores")} for n in (a, b)]
                data = {f"{k}{i}": f[i][k][None] for i in (0, 1) for k in ("keypoints", "descriptors", "scores")}
                data["image0"], data["image1"] = torch.empty(1, 1, 480, 640), torch.empty(1, 1, 480, 640)
                pred = model(data)
                m_ref = pred["matches0"][0].cpu().short().numpy()
                mm = io.get_matches(mpath, a, b)[0]
                key = f"{a.replace('/', '-')}/{b.replace('/', '-')}"
                stored = ms.read(key, "matches0")
                assert stored.dtype == np.int16 and ms.read(key, "matching_scores0").dtype == np.float16
                agree = (stored == m_ref).mean()
                print(f"[pairs_stream] {plugin} {a} x {b}: {int((m_ref > -1).sum())} matches, agreement with the per-pair plugin call {agree:.4f}")
                assert agree >= (1.0 if plugin == "nearest_neighbor" else 0.995) and len(mm) == int((stored > -1).sum())
    assert ps.match_from_paths(confs_dict["matchers"]["NN-mutual"], tmp_path / "pairs.txt", tmp_path / "m_nearest_neighbor.imw", fpath, fpath) is None
