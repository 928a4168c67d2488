"""Parity of the BENCHED path: PairEngine with its defaults (tcgen05 SuperPoint convs, tcgen05 LightGlue
linears / attention / assignment, batch of pairs from the bench stream incl. seeds >= 2) against the CPU oracle
on the same uint8 images.  bench.py times exactly this object; its `match_f1` comes from the same checker."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SP_CONF = {"nms_radius": 3, "keypoint_threshold": 0.005, "max_keypoints": 1024, "remove_borders": 4}
SEEDS = [0, 1, 2, 3, 17, 18, 31, 32, 40, 41, 47, 48, 55, 56, 62, 63]   # both halves of the 64-pair bench step


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def stream():
    """uint8 images of the bench stream + the oracle's answer on them (one oracle run for the module)."""
    from oracle import check
    from imcui_b200.utils import synth
    torch.set_num_threads(max(1, min(32, len(__import__("os").sched_getaffinity(0)))))
    imgs = np.empty((2 * len(SEEDS), 480, 640), np.uint8)
    for i, s in enumerate(SEEDS):
        imgs[2 * i], imgs[2 * i + 1], _ = synth.make_pair(s, 480, 640)
    return imgs, check.oracle_pairs(imgs, SP_CONF)


def test_engine_default_path_vs_oracle(dev, stream):
    """Keypoint set per image, stop layer per pair, match-F1 and exactness of the match sets."""
    from oracle import check
    import oracle
    from imcui_b200.engine import PairEngine
    imgs, ref = stream
    P = len(SEEDS)
    eng = PairEngine(dev, P, 480, 640, sp_state_dict=oracle.synthetic_weights("superpoint"), lg_state_dict=oracle.synthetic_weights("lightglue"))       # defaults == what bench.py constructs
    assert eng.sp_conf.get("tensor_cores", True) and eng.lg_conf["use_tensor_cores"] == 1
    eng.h_images.copy_(torch.from_numpy(imgs))
    hm, hs, hk, hc, hstop = eng.match_host()
    got = check.engine_pairs(hm.numpy(), hk.numpy(), hc.numpy(), hstop.numpy(), P)
    reports = [check.compare_pair(g, r) for g, r in zip(got, ref)]
    summ = check.summarize(reports)
    for s, r in zip(SEEDS, reports):
        print(f"[engine] seed {s}: kpts_set {r['kpts_set_equal']} order {r['kpts_order_equal']} stop {r['stop']} "
              f"F1 {r['f1']:.4f} exact {r['exact']} ({r['n_eng']}/{r['n_ref']} matches)")
    print("[engine]", summ)
    assert summ["kpts_set_equal"] == 1.0, "keypoint set differs from the oracle"
    assert summ["stop_equal"] == 1.0, [r["stop"] for r in reports]
    assert summ["match_f1"] >= 0.999 and summ["min_pair_f1"] >= 0.995, summ
    # scores of identical matches within the 1e-3 tolerance of north_star
    for g, r, p in zip(got, ref, range(P)):
        if not reports[p]["kpts_order_equal"]:
            continue
        both = (g["matches0"] > -1) & (r["matches0"] > -1) & (g["matches0"] == r["matches0"])
        err = np.abs(hs.numpy()[2 * p][: len(r["mscores0"])] - r["mscores0"])[both]
        assert err.size == 0 or err.max() < 1e-3, (p, err.max())


def test_engine_lightglue_on_oracle_features(dev, stream):
    """The batched tcgen05 LightGlue alone on the ORACLE's keypoints/descriptors (identical inputs, identical order):
    stop layer identical, matches0 compared index by index; reports the fraction of bit-identical pairs."""
    from oracle.check import compare_pair
    from imcui_b200 import ops
    import oracle
    from imcui_b200.engine import PairEngine
    _, ref = stream
    P, cap = len(SEEDS), 1024
    eng = PairEngine(dev, P, 480, 640, sp_state_dict=oracle.synthetic_weights("superpoint"), lg_state_dict=oracle.synthetic_weights("lightglue"))
    kp = torch.zeros(2 * P, cap, 2, device=dev); ds = torch.zeros(2 * P, cap, 256, device=dev)
    counts = torch.zeros(2 * P, dtype=torch.int32, device=dev)
    for p, r in enumerate(ref):
        for s in (0, 1):
            k, d = r[f"kpts{s}"], r[f"desc{s}"]
            kp[2 * p + s, : len(k)] = torch.from_numpy(k).to(dev)
            ds[2 * p + s, : len(k)] = torch.from_numpy(d).t().to(dev)
            counts[2 * p + s] = len(k)
    out = ops.lightglue_forward(eng.lg_w, eng.n_layers, kp, ds, counts, eng.lg_conf)
    m, stop = out["matches"].cpu().numpy(), out["stop"].cpu().numpy()
    n_exact, flips = 0, []
    for p, r in enumerate(ref):
        g = {"kpts0": r["kpts0"], "kpts1": r["kpts1"], "matches0": m[2 * p][: len(r["kpts0"])].astype(np.int64), "stop": int(stop[p])}
        rep = compare_pair(g, r)
        n_exact += rep["index_exact"]
        d = np.nonzero(g["matches0"] != r["matches0"])[0]
        flips.append(len(d))
        print(f"[engine-lg] seed {SEEDS[p]}: stop {rep['stop']} F1 {rep['f1']:.4f} index-exact {rep['index_exact']} flipped rows {len(d)}")
        assert rep["stop_equal"], rep["stop"]
        assert rep["f1"] >= 0.998, rep
    print(f"[engine-lg] bit-identical matches0 on {n_exact}/{P} pairs; flipped rows per pair {flips}")
    assert sum(flips) <= 2 * P, flips    # threshold-crossing scores (|score - 0.2| ~ 1e-6) at most: a handful over 16k rows


def test_engine_device_path_equals_host_path(dev, stream):
    """match_device (HBM-resident inputs: the timed `value`) and match_host (the `e2e` leg) give the same answer."""
    import oracle
    from imcui_b200.engine import PairEngine
    imgs, _ = stream
    P = 4
    eng = PairEngine(dev, P, 480, 640, sp_state_dict=oracle.synthetic_weights("superpoint"), lg_state_dict=oracle.synthetic_weights("lightglue"))
    eng.h_images.copy_(torch.from_numpy(imgs[: 2 * P]))
    hm, _, hk, hc, hstop = (t.clone() for t in eng.match_host())
    sp, lg = eng.match_device(eng.to_float(eng.h_images.to(dev)))
    torch.cuda.synchronize()
    assert torch.equal(lg["matches"].cpu(), hm) and torch.equal(lg["stop"].cpu(), hstop)
    assert torch.equal(sp["keypoints"].cpu(), hk) and torch.equal(sp["counts"].cpu(), hc)


def test_pair_stream_from_rgb_frames_equals_the_registry_path(dev, stream):
    """PairStream (double-buffered H2D / compute / D2H over three streams, buffers reused every other batch) on decoded RGB
    frames == the plugin path one pair at a time (extract -> match_images) on the same frames: identical matched keypoints
    in original-frame coordinates; and batch i's record is not disturbed by batches i+1, i+2 in flight."""
    import oracle
    from imcui_b200.engine import PairEngine, PairStream
    from imcui_b200.hloc import extract_features, match_features
    from imcui_b200.ui import utils as U
    from imcui_b200.utils import synth
    imgs, _ = stream
    P, NBATCH = 2, 5
    rgb = synth.to_rgb(imgs[: 2 * P * NBATCH])                                     # [20,480,640,3]
    pre = {"grayscale": True, "resize_max": 1600, "dfactor": 8}
    eng = PairEngine(dev, P, 480, 640, sp_state_dict=oracle.synthetic_weights("superpoint"), lg_state_dict=oracle.synthetic_weights("lightglue"), frame_shape=(480, 640, 3), pre_conf=pre)
    batches = [torch.from_numpy(rgb[2 * P * b: 2 * P * (b + 1)]).pin_memory() for b in range(NBATCH)]
    recs = []
    for rec in PairStream(eng).run(iter(batches)):
        recs.append({k: v.clone() for k, v in rec.items()})
    assert len(recs) == NBATCH
    conf = U.get_matcher_zoo({"x": {"matcher": "superpoint-lightglue", "feature": "superpoint_max", "dense": False, "standalone": False}})["x"]
    conf["feature"] = {**conf["feature"], "model": {**conf["feature"]["model"], "state_dict": oracle.synthetic_weights("superpoint")}}
    conf["matcher"] = {**conf["matcher"], "model": {**conf["matcher"]["model"], "state_dict": oracle.synthetic_weights("lightglue")}}
    ext, mat = U.get_feature_model(conf["feature"], dev), U.get_model(conf["matcher"], dev)
    ext.conf.update(SP_CONF)
    for b in (0, 3, 4):
        for p in range(P):
            f0 = extract_features.extract(ext, rgb[2 * (P * b + p)], pre)
            f1 = extract_features.extract(ext, rgb[2 * (P * b + p) + 1], pre)
            ref = match_features.match_images(mat, f0, f1)
            n = int(recs[b]["mcount"][p])
            a = {tuple(r) for r in np.concatenate([recs[b]["mkpts0_orig"][p, :n].numpy(), recs[b]["mkpts1_orig"][p, :n].numpy()], 1).tolist()}
            r = {tuple(r) for r in np.concatenate([ref["mkeypoints0_orig"], ref["mkeypoints1_orig"]], 1).tolist()}
            f1s = 2 * len(a & r) / max(len(a) + len(r), 1)
            print(f"[stream] batch {b} pair {p}: {n} matches, F1 vs plugin path {f1s:.4f}")
            assert f1s >= 0.995, (b, p, f1s)      # single-pair plugin call vs batch-of-2 engine: same kernels, same decisions
            assert int(recs[b]["n_kpts"][2 * p]) == len(ref["keypoints0"])
