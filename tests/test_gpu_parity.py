"""GPU parity: the CUDA path, called through the plugin classes -> ctypes -> C ABI, against the golden
vectors minted from the reference and against the CPU oracle on the same inputs."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN, assert_keypoints_equivalent, compressed_descriptors, lg_pair_from_source, match_f1

pytestmark = pytest.mark.gpu

SP_CONFS = {
    "api": {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.015, "remove_borders": 4},
    "max1024": {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.005, "remove_borders": 4},
    "nocap": {"nms_radius": 4, "max_keypoints": -1, "keypoint_threshold": 0.005, "remove_borders": 4},
    "max2048": {"nms_radius": 3, "max_keypoints": 2048, "keypoint_threshold": 0.005, "remove_borders": 4},
}
DESC_TOL = 1e-3   # north_star: descriptor/score tensors within 1e-3 fp32
SCORE_TOL = 1e-3


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _load(root, name, conf, dev):
    """The plugin on the synthetic parameters of the oracle (oracle.synthetic_weights) unless conf brings its own."""
    import oracle
    from imcui_b200.hloc.utils.base_model import dynamic_load
    if name in ("superpoint", "lightglue", "superglue") and conf.get("state_dict") is None:
        conf = {**conf, "state_dict": oracle.synthetic_weights(name)}
    return dynamic_load(root, name)(conf).eval().to(dev)


@pytest.mark.parametrize("tc", [False, True], ids=["cuda-core-fp32", "tcgen05-fp16x2"])
@pytest.mark.parametrize("case,confs", [("sp_real", ["api", "max1024", "nocap"]), ("sp_synth", ["max1024", "max2048"])])
def test_superpoint_matches_reference(golden, dev, case, confs, tc):
    from imcui_b200.hloc import extractors
    g, s = golden(case), golden("sp_sw")
    images = torch.from_numpy(g["images"]).to(dev)
    model = _load(extractors, "superpoint", {"tensor_cores": tc}, dev)
    for c in confs:
        model.conf.update(SP_CONFS[c])  # mutable conf, as the UI/API do
        for b in range(images.shape[0]):
            out = model({"image": images[b:b + 1]})
            pre = f"{case}/{c}/{b}/"
            moved = assert_keypoints_equivalent(
                out["keypoints"][0].cpu().numpy(), out["scores"][0].cpu().numpy(), out["descriptors"][0].cpu().numpy(),
                s[pre + "keypoints"], s[pre + "scores"], s[pre + "descriptors"], desc_cols=s[pre + "desc_cols"],
                score_tol=SCORE_TOL, desc_tol=DESC_TOL, order_noise=5e-5 if tc else 2e-5, what=f"{case}/{c}/{b}")
            if SP_CONFS[c]["max_keypoints"] < 0:
                assert moved == 0  # row-major order: exact


SP_FIX_CONF = {"nms_radius": 3, "max_keypoints": 256, "keypoint_threshold": 0.005, "remove_borders": 4, "fix_sampling": True}


def test_superpoint_fix_sampling_matches_reference_plugin(golden, dev):
    """conf["fix_sampling"] = True (hloc/extractors/superpoint.py:16-30,46-47)."""
    from imcui_b200.hloc import extractors
    g, s = golden("sp_fix"), golden("sp_sw")
    images = torch.from_numpy(g["images"]).to(dev)
    model = _load(extractors, "superpoint", dict(SP_FIX_CONF), dev)
    plain = _load(extractors, "superpoint", {**SP_FIX_CONF, "fix_sampling": False}, dev)
    for b in range(images.shape[0]):
        out = model({"image": images[b:b + 1]})
        assert_keypoints_equivalent(
            out["keypoints"][0].cpu().numpy(), out["scores"][0].cpu().numpy(), out["descriptors"][0].cpu().numpy(),
            s[f"fix/{b}/keypoints"], s[f"fix/{b}/scores"], s[f"fix/{b}/descriptors"], desc_cols=s[f"fix/{b}/desc_cols"],
            score_tol=SCORE_TOL, desc_tol=DESC_TOL, order_noise=5e-5, what=f"sp_fix/{b}")
        other = plain({"image": images[b:b + 1]})["descriptors"][0]
        assert (other - out["descriptors"][0]).abs().max() > 1e-2      # the switch does change the sampling


@pytest.mark.parametrize("hw", [(136, 208), (200, 336), (136, 200), (64, 64)], ids=lambda v: f"{v[0]}x{v[1]}")
def test_superpoint_ragged_sizes_vs_oracle(dev, hw):
    """Sizes that leave partial tiles in every conv kernel (H % 16 != 0, W % 16 != 0 -> CUDA-core convs, tiny maps):
    no cap, so the keypoint list is the exact row-major set; checked against the CPU oracle on the same image."""
    import oracle
    from oracle import superpoint as osp
    from imcui_b200.hloc import extractors
    from imcui_b200.utils import synth
    H, W = hw
    a, _, _ = synth.make_pair(5, H, W)
    img = torch.from_numpy(a.astype(np.float32) / 255.0)[None, None]
    conf = {"nms_radius": 3, "max_keypoints": -1, "keypoint_threshold": 0.01, "remove_borders": 4}
    ref = osp.forward(oracle.synthetic_weights("superpoint"), img, conf)
    out = _load(extractors, "superpoint", conf, dev)({"image": img.to(dev)})
    k, rk = out["keypoints"][0].cpu(), ref["keypoints"][0]
    assert k.shape == rk.shape and torch.equal(k, rk), f"{hw}: {k.shape[0]} vs {rk.shape[0]} keypoints"
    assert (out["scores"][0].cpu() - ref["scores"][0]).abs().max() < 1e-4
    assert (out["descriptors"][0].cpu() - ref["descriptors"][0]).abs().max() < 1e-3


@pytest.mark.parametrize("tc", [False, True], ids=["cuda-core-fp32", "tcgen05-fp16x2"])
def test_superpoint_dense_scores(golden, dev, tc):
    from imcui_b200 import ops
    from imcui_b200.hloc import extractors
    g, s = golden("sp_real"), golden("sp_sw")
    model = _load(extractors, "superpoint", {**SP_CONFS["api"], "tensor_cores": tc}, dev)
    out = ops.superpoint_forward(model._bufs(), torch.from_numpy(g["images"]).to(dev), model.conf, 1024, want_dense=True)
    for b in range(2):
        err = float(np.abs(out["dense_scores"][b].cpu().numpy().ravel()[s[f"dense/{b}/idx"]] - s[f"dense/{b}/scores"]).max())
        print(f"[sp dense] tensor_cores={tc} image {b}: max |score - reference| = {err:.2e}")
        assert err < (3e-5 if tc else 1e-5)


def test_superpoint_batch_equals_single(golden, dev):
    """Batched call == per-image calls (the reference loops over the batch in Python)."""
    from imcui_b200.hloc import extractors
    g = golden("sp_synth")
    images = torch.from_numpy(g["images"]).to(dev)
    model = _load(extractors, "superpoint", SP_CONFS["max1024"], dev)
    outb = model({"image": images})
    for b in range(images.shape[0]):
        o = model({"image": images[b:b + 1]})
        assert torch.equal(o["keypoints"][0], outb["keypoints"][b])
        assert torch.equal(o["descriptors"][0], outb["descriptors"][b])


def test_superpoint_bad_conf(dev):
    from imcui_b200.hloc import extractors
    from imcui_b200.hloc.utils.base_model import dynamic_load
    with pytest.raises(ValueError):
        dynamic_load(extractors, "superpoint")({"max_keypoints": 0})
    model = _load(extractors, "superpoint", {}, dev)
    with pytest.raises(AssertionError):
        model({})
    model.conf["max_keypoints"] = -5
    with pytest.raises(ValueError):
        model({"image": torch.zeros(1, 1, 64, 64, device=dev)})


def test_superpoint_blank_image(dev):
    """No keypoints is not an error."""
    from imcui_b200.hloc import extractors
    model = _load(extractors, "superpoint", {"max_keypoints": 128, "keypoint_threshold": 0.9}, dev)
    out = model({"image": torch.zeros(1, 1, 64, 96, device=dev)})
    assert out["keypoints"][0].shape == (0, 2) and out["descriptors"][0].shape == (256, 0)


LG_MODES = {
    "full": dict(depth_confidence=-1, width_confidence=-1, pruning_min_kpts=-1),
    "cuda": dict(depth_confidence=0.95, width_confidence=0.99, pruning_min_kpts=1536),
    "cpu": dict(depth_confidence=0.95, width_confidence=0.99, pruning_min_kpts=-1),
}


def _lg_inputs(k0, d0, k1, d1, dev):
    t = lambda a: torch.from_numpy(a).to(dev)
    return {"image0": torch.empty(1, 1, 480, 640, device=dev), "image1": torch.empty(1, 1, 480, 640, device=dev),
            "keypoints0": t(k0)[None], "keypoints1": t(k1)[None],
            "scores0": torch.ones(1, len(k0), device=dev), "scores1": torch.ones(1, len(k1), device=dev),
            "descriptors0": t(d0)[None], "descriptors1": t(d1)[None]}


@pytest.mark.parametrize("case", ["lg_real", "lg_synth"])
@pytest.mark.parametrize("mode", ["full", "cuda", "cpu"])
def test_lightglue_matches_reference(golden, dev, case, mode):
    """Exact-fp32 path: match indices, stop layer and pruning bit-identical to the reference."""
    from imcui_b200.hloc import matchers
    g = golden(case)
    model = _load(matchers, "lightglue", {"match_threshold": 0.2, "tensor_cores": False, **LG_MODES[mode]}, dev)
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        out = model(_lg_inputs(k0, d0, k1, d1, dev))
        pre = f"{mode}/{p}/"
        m0 = out["matches0"][0].cpu().numpy()
        f1 = match_f1(m0, g[pre + "matches0"])
        assert out["stop"] == int(g[pre + "stop"]), (case, mode, p, out["stop"], int(g[pre + "stop"]), f1)
        assert np.array_equal(m0, g[pre + "matches0"]), (case, mode, p, "F1", f1)
        assert np.array_equal(out["matches1"][0].cpu().numpy(), g[pre + "matches1"])
        np.testing.assert_allclose(out["matching_scores0"][0].cpu().numpy(), g[pre + "matching_scores0"], atol=SCORE_TOL)
        np.testing.assert_allclose(out["matching_scores1"][0].cpu().numpy(), g[pre + "matching_scores1"], atol=SCORE_TOL)
        assert np.array_equal(out["prune0"][0].cpu().numpy().astype(np.int32), g[pre + "prune0"])
        assert np.array_equal(out["prune1"][0].cpu().numpy().astype(np.int32), g[pre + "prune1"])
        assert out["matches0"].dtype == torch.int64 and out["matches"][0].shape[1] == 2


@pytest.mark.parametrize("case", ["lg_real", "lg_synth"])
@pytest.mark.parametrize("mode", ["full", "cuda"])
@pytest.mark.parametrize("tc", ["3xtf32", "tf32"])
def test_lightglue_tensor_core_path(golden, dev, case, mode, tc):
    """tcgen05 linears.  3xTF32 (default, fp32-equivalent): same stop layer, match-F1 >= 0.999, scores within
    the 1e-3 parity tolerance.  Single TF32 (fast mode): F1 >= 0.99, scores within 3e-2."""
    from imcui_b200.hloc import matchers
    g = golden(case)
    model = _load(matchers, "lightglue", {"match_threshold": 0.2, "tensor_cores": tc, **LG_MODES[mode]}, dev)
    f1_min, tol = (0.999, SCORE_TOL) if tc == "3xtf32" else (0.98, 0.15)   # single TF32: documented fast mode, outside the parity tolerance
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        out = model(_lg_inputs(k0, d0, k1, d1, dev))
        pre = f"{mode}/{p}/"
        m0 = out["matches0"][0].cpu().numpy()
        f1 = match_f1(m0, g[pre + "matches0"])
        both = (m0 > -1) & (g[pre + "matches0"] > -1)
        err = np.abs(out["matching_scores0"][0].cpu().numpy() - g[pre + "matching_scores0"])[both].max()
        print(f"[tc:{tc}] {case}/{mode}/{p}: F1 {f1:.4f} exact {np.array_equal(m0, g[pre + 'matches0'])} "
              f"stop {out['stop']}/{int(g[pre + 'stop'])} score err {err:.2e}")
        assert out["stop"] == int(g[pre + "stop"])
        assert f1 >= f1_min, (case, mode, p, f1)
        assert err < tol, (case, mode, p, err)


@pytest.mark.parametrize("tc", [False, "3xtf32"], ids=["cuda-core-fp32", "tcgen05-3xtf32"])
def test_lightglue_input_proj_128d(golden, dev, tc):
    """features="aliked" architecture: 128-d descriptors through the Linear input_proj (lightglue.py:392-395,519-520)."""
    import oracle
    from imcui_b200.hloc import matchers
    g = golden("lg_proj")
    sd = dict(oracle.synthetic_weights("lightglue"))
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    model = _load(matchers, "lightglue", {"match_threshold": 0.2, "features": "aliked", "state_dict": sd, "tensor_cores": tc, **LG_MODES["cuda"]}, dev)
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        c0, c1 = (np.ascontiguousarray(compressed_descriptors(d, g["input_proj_w"]).T) for d in (d0, d1))
        out = model(_lg_inputs(k0, c0, k1, c1, dev))
        m0 = out["matches0"][0].cpu().numpy()
        f1 = match_f1(m0, g[f"{p}/matches0"])
        both = (m0 > -1) & (g[f"{p}/matches0"] > -1)
        err = np.abs(out["matching_scores0"][0].cpu().numpy() - g[f"{p}/matching_scores0"])[both].max()
        print(f"[lg-proj tc={tc}] pair {p}: F1 {f1:.4f} stop {out['stop']}/{int(g[f'{p}/stop'])} score err {err:.2e}")
        assert out["stop"] == int(g[f"{p}/stop"]) and err < SCORE_TOL
        if tc is False:
            assert np.array_equal(m0, g[f"{p}/matches0"]) and np.array_equal(out["matches1"][0].cpu().numpy(), g[f"{p}/matches1"])
        else:
            assert f1 >= 0.999


@pytest.mark.parametrize("tc", [False, "3xtf32"], ids=["cuda-core-fp32", "tcgen05-3xtf32"])
def test_aliked_lightglue_composition(golden, dev, tc):
    """BASELINE configs[3] composition: ALIKED (CUDA) -> LightGlue features="aliked" with the fitted input_proj, against the
    UNMODIFIED reference modules run end to end on the same two synthetic pairs (tests/golden/aliked_lg.npz)."""
    import oracle
    from imcui_b200 import ops
    from imcui_b200.hloc import matchers
    from imcui_b200.utils import synth, synth_weights
    g = golden("aliked_lg")
    sd = dict(oracle.synthetic_weights("lightglue"))
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    model = _load(matchers, "lightglue", {"match_threshold": 0.2, "features": "aliked", "state_dict": sd, "tensor_cores": tc, **LG_MODES["cuda"]}, dev)
    aw = {k: v.to(dev) for k, v in ops.aliked_pack_weights(synth_weights.aliked_random_weights(0)).items()}
    for p, seed in enumerate(g["eval_seeds"]):
        a, c, _ = synth.make_pair(int(seed), 480, 640)
        rgb = torch.from_numpy(synth.to_rgb(np.stack([a, c])).astype(np.float32) / 255.0).permute(0, 3, 1, 2).contiguous().to(dev)
        f = ops.aliked_forward(aw, rgb, {"detection_threshold": 0.1, "max_num_keypoints": 1024, "nms_radius": 2}, 1024)
        n = [int(v) for v in f["counts"][0].cpu()]
        kp = [f["keypoints"][i, :n[i]] for i in range(2)]
        ds = [f["descriptors"][i, :n[i]] for i in range(2)]
        # the extractor against the reference's features (score-sorted selection: same set, near-tie swaps allowed)
        for i in range(2):
            rk = g[f"{p}/keypoints{i}"]
            assert n[i] == len(rk)
            d = np.abs(kp[i].cpu().numpy()[:, None] - rk[None]).max(-1)
            j = d.argmin(1)
            assert d[np.arange(len(j)), j].max() < 2e-3 and len(set(j.tolist())) == len(j)
            assert np.abs(ds[i].cpu().numpy() - g[f"{p}/descriptors{i}"][j]).max() < 1e-3
        # the matcher on the reference's features: indices comparable one to one
        out = model(_lg_inputs(g[f"{p}/keypoints0"], np.ascontiguousarray(g[f"{p}/descriptors0"].T, np.float32), g[f"{p}/keypoints1"],
                               np.ascontiguousarray(g[f"{p}/descriptors1"].T, np.float32), dev))
        m0 = out["matches0"][0].cpu().numpy()
        f1 = match_f1(m0, g[f"{p}/matches0"])
        print(f"[aliked-lg tc={tc}] pair {p}: F1 {f1:.4f} stop {out['stop']}/{int(g[f'{p}/stop'])} matches {(m0 > -1).sum()}")
        assert out["stop"] == int(g[f"{p}/stop"])
        assert np.array_equal(m0, g[f"{p}/matches0"]) if tc is False else f1 >= 0.999
        # and end to end on our own features: the matches are geometrically real
        out = model(_lg_inputs(kp[0].cpu().numpy(), np.ascontiguousarray(ds[0].t().cpu().numpy()), kp[1].cpu().numpy(),
                               np.ascontiguousarray(ds[1].t().cpu().numpy()), dev))
        m = out["matches0"][0].cpu().numpy(); v = m > -1
        q = np.concatenate([kp[0].cpu().numpy()[v], np.ones((v.sum(), 1))], 1) @ g[f"{p}/H"].T
        err = np.linalg.norm(q[:, :2] / q[:, 2:] - kp[1].cpu().numpy()[m[v]], axis=1)
        assert v.sum() > 300 and (err < 3).mean() > 0.8


@pytest.mark.parametrize("tc", [False, "3xtf32"], ids=["cuda-core-fp32", "tcgen05-3xtf32"])
def test_lightglue_scale_ori_inputs(golden, dev, tc):
    """features="sift" architecture (SURVEY.md 8(f) rank 4): 128-d descriptors + per-keypoint scales / orientations in the
    positional encoding (lightglue.py:500-506), forwarded by the plugin exactly as hloc/matchers/lightglue.py:61-73 does."""
    import oracle
    from imcui_b200.hloc import matchers
    g = golden("lg_so")
    sd = dict(oracle.synthetic_weights("lightglue"))
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    sd["posenc.Wr.weight"] = torch.from_numpy(g["posenc_wr"])
    model = _load(matchers, "lightglue", {"match_threshold": 0.2, "features": "sift", "state_dict": sd, "tensor_cores": tc, **LG_MODES["cuda"]}, dev)
    for p, src in enumerate(g["sources"]):
        k0, d0, k1, d1 = lg_pair_from_source(golden, src)
        c0, c1 = (np.ascontiguousarray(compressed_descriptors(d, g["input_proj_w"]).T) for d in (d0, d1))
        data = _lg_inputs(k0, c0, k1, c1, dev)
        for n in ("scales0", "oris0", "scales1", "oris1"):
            data[n] = torch.from_numpy(g[f"{p}/{n}"])[None].to(dev)
        out = model(data)
        m0 = out["matches0"][0].cpu().numpy()
        f1 = match_f1(m0, g[f"{p}/matches0"])
        both = (m0 > -1) & (g[f"{p}/matches0"] > -1)
        err = np.abs(out["matching_scores0"][0].cpu().numpy() - g[f"{p}/matching_scores0"])[both].max()
        print(f"[lg-so tc={tc}] pair {p}: F1 {f1:.4f} stop {out['stop']}/{int(g[f'{p}/stop'])} score err {err:.2e}")
        assert out["stop"] == int(g[f"{p}/stop"]) and err < SCORE_TOL and f1 >= 0.995
    with pytest.raises(AssertionError):
        model(_lg_inputs(k0, c0, k1, c1, dev))   # scales / oris missing


def test_tcgen05_gemm_unit(dev):
    """tcgen05/TMA GEMM against the CUDA-core GEMM and torch fp64."""
    from imcui_b200 import ops
    torch.manual_seed(0)
    for (M, N, K) in ((128, 128, 32), (256, 256, 256), (1024, 768, 256), (512, 512, 512), (4096, 256, 512), (2048, 512, 128)):
        A = torch.randn(M, K, device=dev); Wt = torch.randn(N, K, device=dev) / K ** 0.5; b = torch.randn(N, device=dev)
        ref = (A.double() @ Wt.double().t() + b.double()).float()
        simt = ops.debug_gemm(A, Wt, b, "fp32")
        tf32 = ops.debug_gemm(A, Wt, b, "tf32")
        x3 = ops.debug_gemm(A, Wt, b, "3xtf32")
        x3w = ops.debug_gemm(A, Wt, b, "3xtf32_wlo")      # host-provided W lo plane
        f16 = ops.debug_gemm(A, Wt, b, "f16x2")           # split-fp16 with host-packed weight planes (what the LightGlue / LoFTR linears use)
        torch.cuda.synchronize()
        e_f16 = float((f16 - ref).abs().max())
        print(f"[gemm] {M}x{N}x{K}: split-fp16 {e_f16:.2e}")
        assert e_f16 < 3e-5, (M, N, K, e_f16)
        if K % 64 == 0:   # activations handed over as planes by their producer (no splitter warps): the same operands, bit for bit
            assert torch.equal(ops.debug_gemm(A, Wt, b, "f16x2_ap"), f16)
        e_simt, e_tf32, e_x3, e_x3w = (float((t - ref).abs().max()) for t in (simt, tf32, x3, x3w))
        print(f"[gemm] {M}x{N}x{K}: fp32 {e_simt:.2e} tf32 {e_tf32:.2e} 3xtf32 {e_x3:.2e} 3xtf32+wlo {e_x3w:.2e}")
        assert e_simt < 1e-4 and e_tf32 < 2e-2 and e_x3 < 3e-5 and e_x3w < 3e-5, (M, N, K, e_simt, e_tf32, e_x3, e_x3w)
        assert torch.equal(x3, x3w)                       # same products in the same order: bit-identical
    # exactly representable operands -> exact result (layout / descriptor correctness independent of rounding)
    A = torch.randint(-4, 5, (256, 64), device=dev).float(); Wt = torch.randint(-4, 5, (128, 64), device=dev).float()
    for mode in ("tf32", "3xtf32", "3xtf32_wlo", "f16x2"):
        assert torch.equal(ops.debug_gemm(A, Wt, torch.zeros(128, device=dev), mode), A @ Wt.t())
    # split-fp16 over a wide dynamic range (LightGlue residual-stream magnitudes, tiny values next to large ones)
    A = torch.randn(256, 512, device=dev) * torch.logspace(-4, 2, 512, device=dev)[None]; Wt = torch.randn(256, 512, device=dev) / 512 ** 0.5
    ref = (A.double() @ Wt.double().t()).float()
    out = ops.debug_gemm(A, Wt, torch.zeros(256, device=dev), "f16x2")
    assert float((out - ref).abs().max() / ref.abs().max()) < 2e-6


def test_tcgen05_conv_unit(dev):
    """tcgen05 split-fp16 implicit-GEMM conv == fp32 CUDA-core conv to fp32 rounding noise, incl. zero padding,
    fused ReLU / 2x2 max-pool, partial tiles (H % 8 != 0) and both Cout tile widths."""
    from imcui_b200 import _lib, ops
    torch.manual_seed(1)
    for (B, H, W, Cin, Cout, pool) in ((1, 16, 32, 64, 64, False), (2, 48, 64, 64, 64, True), (1, 24, 48, 64, 64, True),
                                       (1, 40, 16, 64, 64, False), (1, 24, 32, 64, 128, False),
                                       (2, 32, 48, 128, 128, True), (1, 60, 80, 128, 256, False),
                                       (1, 24, 48, 128, 128, False), (3, 40, 24, 256, 256, False), (1, 20, 40, 64, 256, True)):
        x = torch.rand(B, H, W, Cin, device=dev)
        w = torch.randn(9, Cin, Cout, device=dev) / (9 * Cin) ** 0.5
        b = torch.randn(Cout, device=dev) * 0.1
        ref = ops.debug_conv3x3(x, w, b, relu=True, pool=pool, tensor_cores=False)
        # halo kernels (default for W % 8 == 0) and the per-tap generic kernel
        for halo, pair in ((1, 1), (1, 0), (0, 1)):   # pair = 1: CTA-pair kernels (cta_group::2), 0: their single-CTA predecessors
            _lib.lib().imw_debug_set_conv_halo(halo)
            _lib.lib().imw_debug_set_conv_pair(pair)
            out = ops.debug_conv3x3(x, w, b, relu=True, pool=pool, tensor_cores=True)
            torch.cuda.synchronize()
            err = float((out - ref).abs().max())
            print(f"[conv] {B}x{H}x{W} {Cin}->{Cout} pool={pool} halo={halo} pair={pair}: max |tc - fp32| = {err:.2e} (ref max {float(ref.abs().max()):.2f})")
            assert err < 1e-5, (B, H, W, Cin, Cout, pool, halo, pair, err)
        _lib.lib().imw_debug_set_conv_halo(1)
        _lib.lib().imw_debug_set_conv_pair(1)
    # against torch (NCHW) once, to pin the CUDA-core conv itself
    x = torch.rand(1, 16, 32, 64, device=dev); w = torch.randn(9, 64, 64, device=dev) * 0.05; b = torch.zeros(64, device=dev)
    ref = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).double(), w.view(3, 3, 64, 64).permute(3, 2, 0, 1).double(), padding=1).relu()
    out = ops.debug_conv3x3(x, w, b, relu=True, pool=False, tensor_cores=True)
    assert float((out.permute(0, 3, 1, 2) - ref.float()).abs().max()) < 1e-5


def test_tcgen05_fused_first_layer_unit(dev):
    """SuperPoint conv1a + conv1b in one kernel (conv1a evaluated by producer warps straight into the tcgen05 operand tile) == torch
    fp64 conv -> ReLU -> conv -> ReLU -> max-pool, on the CTA-pair kernel (default) and the single-CTA kernel; odd tile counts, partial
    tiles (H % 16 != 0), several images."""
    from imcui_b200 import _lib as L, ops
    torch.manual_seed(3)
    lib = L.lib()
    for (B, H, W, pool) in ((1, 16, 16, False), (2, 48, 64, True), (1, 40, 24, True), (3, 16, 8, False), (1, 120, 160, True)):
        img = torch.rand(B, H, W, device=dev)
        w1a = torch.randn(9, 64, device=dev) / 3.0; b1a = torch.randn(64, device=dev) * 0.1
        w1b = torch.randn(9, 64, 64, device=dev) / 24.0; b1b = torch.randn(64, device=dev) * 0.1
        y = torch.nn.functional.conv2d(img[:, None].double(), w1a.view(3, 3, 1, 64).permute(3, 2, 0, 1).double(), b1a.double(), padding=1).relu()
        y = torch.nn.functional.conv2d(y.float().double(), w1b.view(3, 3, 64, 64).permute(3, 2, 0, 1).double(), b1b.double(), padding=1).relu()
        if pool: y = torch.nn.functional.max_pool2d(y, 2)
        ref = y.permute(0, 2, 3, 1).float()
        wp = ops.split_f16_planes(w1b.permute(0, 2, 1).contiguous()).to(dev)   # [2][9][Cout][Cin]
        for pair in (1, 0):
            lib.imw_debug_set_conv_pair(pair)
            out = torch.empty(2, *ref.shape, dtype=torch.float16, device=dev)
            L.check(lib.imw_debug_conv1ab_fused(L.ptr(img), L.ptr(w1a), L.ptr(b1a), L.ptr(wp), L.ptr(b1b), L.ptr(out), B, H, W, int(pool), L.stream_ptr(dev)))
            torch.cuda.synchronize()
            err = float((out[0].float() + out[1].float() / 2048.0 - ref).abs().max())
            print(f"[conv1ab] {B}x{H}x{W} pool={pool} pair={pair}: max err {err:.2e}")
            assert err < 5e-6, (B, H, W, pool, pair, err)
        lib.imw_debug_set_conv_pair(1)


def test_tcgen05_attention_unit(dev):
    """tcgen05 3xTF32 flash attention == fp32 CUDA-core attention == torch SDPA (fp64), ragged key/query counts,
    self and cross pairing."""
    from imcui_b200 import ops
    torch.manual_seed(2)
    S, cap = 4, 256
    q, k, v = (torch.randn(S, 4, cap, 64, device=dev) for _ in range(3))
    counts = torch.tensor([256, 200, 131, 64], dtype=torch.int32, device=dev)
    for cross in (False, True):
        simt = ops.debug_attention(q, k, v, counts, 0.125, cross, tensor_cores=False)
        tcg = ops.debug_attention(q, k, v, counts, 0.125, cross, tensor_cores=True)
        torch.cuda.synchronize()
        for z in range(S):
            zk = z ^ 1 if cross else z
            nq, nk = int(counts[z]), int(counts[zk])
            ref = torch.nn.functional.scaled_dot_product_attention(q[z, :, :nq].double(), k[zk, :, :nk].double(), v[zk, :, :nk].double())
            ref = ref.transpose(0, 1).reshape(nq, 256).float()
            e_simt = float((simt[z, :nq] - ref).abs().max()); e_tc = float((tcg[z, :nq] - ref).abs().max())
            print(f"[attn] cross={cross} slot {z} ({nq}x{nk}): fp32 {e_simt:.2e} tcgen05 {e_tc:.2e}")
            assert e_simt < 1e-5 and e_tc < 2e-5, (cross, z, e_simt, e_tc)


def test_lightglue_empty_and_tiny(dev):
    from imcui_b200.hloc import matchers
    model = _load(matchers, "lightglue", {}, dev)
    k = np.zeros((0, 2), np.float32); d = np.zeros((256, 0), np.float32)
    k1 = np.random.RandomState(0).rand(7, 2).astype(np.float32) * 100
    d1 = np.random.RandomState(1).randn(256, 7).astype(np.float32)
    out = model(_lg_inputs(k, d, k1, d1, dev))
    assert out["matches0"].shape == (1, 0) and (out["matches1"] == -1).all() and out["stop"] == 1


def test_lightglue_batched_pairs_independent(golden, dev):
    """A batch of pairs == the same pairs run one by one (per-pair early exit, ragged counts)."""
    from imcui_b200 import ops
    from imcui_b200.hloc import matchers
    g = golden("lg_synth")
    model = _load(matchers, "lightglue", {"match_threshold": 0.2, "tensor_cores": False, **LG_MODES["cuda"]}, dev)
    pairs = [lg_pair_from_source(golden, s) for s in g["sources"][:2]] + [lg_pair_from_source(golden, golden("lg_real")["sources"][0])]
    cap = 1024
    kp = torch.zeros(6, cap, 2, device=dev); ds = torch.zeros(6, cap, 256, device=dev)
    counts = torch.zeros(6, dtype=torch.int32, device=dev)
    for p, (k0, d0, k1, d1) in enumerate(pairs):
        for s, (k, d) in enumerate(((k0, d0), (k1, d1))):
            kp[2 * p + s, :len(k)] = torch.from_numpy(k).to(dev)
            ds[2 * p + s, :len(k)] = torch.from_numpy(d).t().to(dev)
            counts[2 * p + s] = len(k)
    out = ops.lightglue_forward(model._bufs(), 9, kp, ds, counts, model._kernel_conf())
    golds = [("lg_synth", 0), ("lg_synth", 1), ("lg_real", 0)]
    for p, (case, q) in enumerate(golds):
        gg = golden(case)
        n0 = len(pairs[p][0])
        assert int(out["stop"][p]) == int(gg[f"cuda/{q}/stop"])
        assert np.array_equal(out["matches"][2 * p, :n0].cpu().numpy(), gg[f"cuda/{q}/matches0"])


@pytest.mark.parametrize("tc", [False, True], ids=["cuda-core-fp32", "tcgen05-3xtf32"])
@pytest.mark.parametrize("iters", [50, 20])
def test_superglue_matches_reference(golden, dev, iters, tc):
    from imcui_b200.hloc import matchers
    g = golden("sg")
    model = _load(matchers, "superglue", {"weights": "outdoor", "sinkhorn_iterations": iters, "match_threshold": 0.2, "tensor_cores": tc}, dev)
    for p, src in enumerate(g["sources"]):
        f, conf, i, j = str(src).split(":")
        b = golden(f)
        t = lambda a: torch.from_numpy(a).to(dev)
        data = {"image0": torch.empty(1, 1, 480, 640, device=dev), "image1": torch.empty(1, 1, 480, 640, device=dev),
                "keypoints0": t(b[f"{conf}/{i}/keypoints"].astype(np.float32))[None], "keypoints1": t(b[f"{conf}/{j}/keypoints"].astype(np.float32))[None],
                "scores0": t(b[f"{conf}/{i}/scores"])[None], "scores1": t(b[f"{conf}/{j}/scores"])[None],
                "descriptors0": t(b[f"{conf}/{i}/descriptors"])[None], "descriptors1": t(b[f"{conf}/{j}/descriptors"])[None]}
        out = model(data)
        pre = f"it{iters}/{p}/"
        m0 = out["matches0"][0].cpu().numpy()
        f1 = match_f1(m0, g[pre + "matches0"])
        err = float(np.abs(out["matching_scores0"][0].cpu().numpy() - g[pre + "matching_scores0"]).max())
        print(f"[sg] tc={tc} it={iters} pair {p}: F1 {f1:.4f} exact {np.array_equal(m0, g[pre + 'matches0'])} score err {err:.2e}")
        assert np.array_equal(m0, g[pre + "matches0"]), (p, f1)
        assert np.array_equal(out["matches1"][0].cpu().numpy(), g[pre + "matches1"])
        assert err < SCORE_TOL
        assert out["matches0"].dtype == torch.int64


def _matcher_inputs(golden, p):
    g = golden("matchers")
    if p == 0:
        s = golden("sp_real")
        return s["api/0/descriptors"], s["api/1/descriptors"]
    return g[f"in/{p}/descriptors0"], g[f"in/{p}/descriptors1"]


@pytest.mark.parametrize("tc", [False, True], ids=["cuda-core-fp32", "tcgen05-3xtf32"])
@pytest.mark.parametrize("p", [0, 1])
def test_matchers_match_reference(golden, dev, p, tc):
    from imcui_b200.hloc import matchers
    g = golden("matchers")
    d0, d1 = (torch.from_numpy(x).to(dev)[None] for x in _matcher_inputs(golden, p))
    data = {"descriptors0": d0, "descriptors1": d1}
    cases = {
        "nn": _load(matchers, "nearest_neighbor", {"do_mutual_check": True, "tensor_cores": tc}, dev),
        "nn_ratio": _load(matchers, "nearest_neighbor", {"do_mutual_check": True, "ratio_threshold": 0.9, "distance_threshold": 0.9, "tensor_cores": tc}, dev),
        "nn_nomutual": _load(matchers, "nearest_neighbor", {"do_mutual_check": False, "tensor_cores": tc}, dev),
        "dsm": _load(matchers, "dual_softmax", {"match_threshold": 0.01, "inv_temperature": 20, "tensor_cores": tc}, dev),
    }
    for tag, model in cases.items():
        out = model(data)
        m = out["matches0"][0].cpu().numpy()
        assert np.array_equal(m, g[f"{tag}/{p}/matches0"]), (tag, match_f1(m, g[f"{tag}/{p}/matches0"]))
        np.testing.assert_allclose(out["matching_scores0"][0].cpu().numpy(), g[f"{tag}/{p}/matching_scores0"], atol=1e-4)
    assert cases["dsm"](data)["matching_scores0"].dtype == torch.float64


def test_matchers_empty(dev):
    from imcui_b200.hloc import matchers
    for name in ("nearest_neighbor", "dual_softmax"):
        model = _load(matchers, name, {}, dev)
        out = model({"descriptors0": torch.zeros(1, 128, 0, device=dev), "descriptors1": torch.randn(1, 128, 5, device=dev)})
        assert (out["matches0"] == -1).all()


@pytest.mark.parametrize("tc", [False, True], ids=["cuda-core-fp32", "tcgen05-3xtf32"])
def test_dual_softmax_large_property(dev, tc):
    """BASELINE config 5 size (4096 x 4096 x 128): planted permutation is recovered and the result equals
    the oracle formula evaluated with torch on the GPU for a random subset of rows."""
    import importlib.util
    from pathlib import Path
    from imcui_b200 import ops
    spec = importlib.util.spec_from_file_location("synth", Path(__file__).parent.parent / "image-matching-webui_b200/utils/synth.py")
    synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
    d0, d1 = synth.make_descriptor_pair(7, n=4096, dim=128)
    ds = torch.stack([torch.from_numpy(d0).t(), torch.from_numpy(d1).t()]).contiguous().to(dev)
    counts = torch.tensor([4096, 4096], dtype=torch.int32, device=dev)
    m0, s0 = ops.dual_softmax(ds, counts, 0.01, 20.0, tensor_cores=tc)
    a, b = ds[0], ds[1]
    sim = (a / a.norm(dim=1, keepdim=True)) @ (b / b.norm(dim=1, keepdim=True)).t() * 20
    P = sim.softmax(0) * sim.softmax(1)
    mask = (P == P.max(1, keepdim=True).values) & (P == P.max(0, keepdim=True).values) & (P > 0.01)
    ref = torch.where(mask.any(1), mask.float().argmax(1), torch.full((4096,), -1, device=dev))
    agree = (ref == m0[0].long()).float().mean().item()
    assert agree > 0.999, agree
    assert (m0[0] > -1).sum() > 1500


def test_registry_pipeline_end_to_end(golden, dev):
    """The registry path a Gradio / API caller drives: zoo entry -> get_feature_model / get_model -> extract x2 (GPU
    pre-processing from the decoded RGB frames) -> match_images (GPU post-processing) -> filter_matches (GPU MAGSAC++).
    On the real photo pair the pre-processed image equals the reference's and the raw match count equals the oracle's
    SuperPoint -> LightGlue result (golden sp_sw, CUDA semantics).  The synthetic parameters find few consistent matches
    across that wide baseline, so geometric verification is checked on the synthetic pair of seed 0 (a homography of
    one texture): raw count equal to the oracle's, and MAGSAC++ keeps at least 8 matches and reports a fundamental matrix."""
    import oracle
    from imcui_b200.hloc import extract_features, match_features
    from imcui_b200.ui import utils as U
    from imcui_b200.utils import synth
    conf = U.get_matcher_zoo({"superpoint+lightglue": {"matcher": "superpoint-lightglue", "feature": "superpoint_max", "dense": False,
                                                       "standalone": False}})["superpoint+lightglue"]
    conf["feature"] = {**conf["feature"], "model": {**conf["feature"]["model"], "state_dict": oracle.synthetic_weights("superpoint")}}
    conf["matcher"] = {**conf["matcher"], "model": {**conf["matcher"]["model"], "state_dict": oracle.synthetic_weights("lightglue")}}
    extractor, matcher = U.get_feature_model(conf["feature"], dev), U.get_model(conf["matcher"], dev)
    extractor.conf["max_keypoints"], extractor.conf["keypoint_threshold"] = 1024, 0.015          # api/core.py:78-96 overrides
    pre = {**conf["feature"]["preprocessing"], "force_resize": True, "width": 640, "height": 480}
    rgb0 = np.load(GOLDEN / "data" / "02928139_3448003521.npz")["rgb"]
    rgb1 = np.load(GOLDEN / "data" / "17295357_9106075285.npz")["rgb"]
    a, b, _ = synth.make_pair(0, 480, 640)
    s = golden("sp_sw")
    for tag, (im0, im1), n_ref in (("real", (rgb0, rgb1), int(s["registry/n_matches"])),
                                   ("synth", (synth.to_rgb(a), synth.to_rgb(b)), int(s["registry/synth/n_matches"]))):
        f0, f1 = extract_features.extract(extractor, im0, pre), extract_features.extract(extractor, im1, pre)
        if tag == "real":
            g = golden("sp_real")
            assert torch.equal(f0["image"].cpu(), torch.from_numpy(g["images"][0])[None]) and tuple(f0["size"]) == (640, 480)
        pred = match_features.match_images(matcher, f0, f1)
        pred = U.filter_matches(pred, "B200_MAGSAC", 8, 0.9999, 10000)
        n = len(pred["mkeypoints0_orig"])
        print(f"[registry] {tag}: raw matches {n} (reference {n_ref}), verified {len(pred['mmkeypoints0_orig'])}")
        assert abs(n - n_ref) <= 2 and pred["mconf"].shape == (n,) and pred["keypoints0"].shape[1] == 2
        s0 = f0["original_size"] / f0["size"]
        assert np.allclose(pred["mkeypoints0_orig"], (pred["mkeypoints0"] + 0.5) * s0 - 0.5, atol=1e-3)
        assert len(pred["mmkeypoints0_orig"]) <= n and "geom_info" in pred
        if tag == "synth":
            assert len(pred["mmkeypoints0_orig"]) >= 8 and "Fundamental" in pred["geom_info"]
    f0, f1 = extract_features.extract(extractor, rgb0, pre), extract_features.extract(extractor, rgb1, pre)
    # the batch sibling gives the same features
    fb = extract_features.extract_batch(extractor, [rgb0, rgb1, rgb0], pre)
    assert torch.equal(fb[2]["keypoints"][0], f0["keypoints"][0]) and torch.equal(fb[1]["descriptors"][0], f1["descriptors"][0])
