"""Per-row device timings of the SURVEY.md 8(a) stages that the headline bench (SuperPoint+LightGlue) does not cover:
SuperGlue, LoFTR (480x640 and 1024x1024), ALIKED, mutual NN / dual-softmax at 4096 x 128, MAGSAC++.
One JSON line per row (CUDA events on the launching stream, after warm-up, inputs resident in HBM).
Secondary evidence for DESIGN.md / profiles/ -- bench.py stays the contract line.

  gpurun -- python tools/bench_rows.py [--rows sg,loftr,aliked,nn,magsac] [--iters 5]
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import imcui_b200  # noqa: E402,F401
from imcui_b200 import _lib as L, engine, ops  # noqa: E402
from imcui_b200.utils import synth, synth_weights  # noqa: E402


def timed(fn, iters, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = L.lib().imw_launch_count()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters, (L.lib().imw_launch_count() - n0) // iters


def emit(row, **kw):
    print(json.dumps({"row": row, **kw}), flush=True)


def sp_features(dev, P, cap=1024):
    """SuperPoint features of P synthetic pairs -> keypoints / scores / descriptors / counts in slot order."""
    eng = engine.PairEngine(dev, P)
    a, b = synth.make_pair_batch(list(range(P)))
    imgs = torch.from_numpy(np.stack([a, b], 1).reshape(2 * P, 480, 640)).to(dev)
    sp, _ = eng.match_device(eng.to_float(imgs))
    return {k: v.clone() for k, v in sp.items()}


def row_superglue(dev, iters):
    P = 16
    sp = sp_features(dev, P)
    sd = synth_weights.superglue_random_weights(0)
    w = {k: v.to(dev) for k, v in ops.sg_pack_weights(sd).items()}
    wh = torch.tensor([[640, 480]] * (2 * P), dtype=torch.int32, device=dev)
    counts = sp["counts"][0].contiguous()
    for it in (50, 20):
        conf = {"sinkhorn_iterations": it, "match_threshold": 0.2}
        f = lambda: ops.superglue_forward(w, float(sd["bin_score"]), sp["keypoints"], sp["scores"], sp["descriptors"], counts, wh, conf)
        ms, nl = timed(f, iters)
        m, _ = f()
        emit("a7 SuperGlue", pairs=P, keypoints=1024, sinkhorn_iterations=it, ms=round(ms, 3), pairs_per_s=round(P / ms * 1e3, 1),
             launches=nl, mean_matches=float((m[0::2] > -1).sum(1).float().mean()))


def row_loftr(dev, iters):
    wd = ops.loftr_to_device(ops.loftr_pack_weights(synth_weights.loftr_random_weights(0)), dev)   # no checkpoint offline
    for (H, W, P, thr) in ((480, 640, 16, 1e-6), (1024, 1024, 32, 1e-7)):   # BASELINE configs[2]: batch = 32 at 1024x1024
        a, b = synth.make_pair_batch(list(range(P)), H, W)
        imgs = torch.from_numpy(np.stack([a, b], 1).reshape(2 * P, H, W).astype(np.float32) / 255.0).to(dev)
        for tc in (1,):
            f = lambda: ops.loftr_forward(wd, imgs, {"match_threshold": thr, "use_tensor_cores": tc}, max_matches=4096)
            ms, nl = timed(f, iters)
            out = f()
            flop = 709e9 * (H * W) / (480 * 640)   # SURVEY 8(a) a11: 709 GFLOP/pair at 480x640, ~linear in pixels (2.5 T at 1024^2)
            emit("a10/a11 LoFTR", pairs=P, size=[H, W], linears="3xTF32", ms=round(ms, 2), pairs_per_s=round(P / ms * 1e3, 2),
                 launches=nl, mean_matches=float(out["counts"].float().mean()), fp32_equiv_tflops=round(flop * P / ms / 1e9, 1),
                 weights="random (no LoFTR checkpoint offline)")


def row_aliked(dev, iters):
    w = {k: v.to(dev) for k, v in ops.aliked_pack_weights(synth_weights.aliked_random_weights(0)).items()}
    B = 32
    a, _ = synth.make_pair_batch(list(range(B)))
    rgb = torch.from_numpy(synth.to_rgb(a).astype(np.float32) / 255.0).permute(0, 3, 1, 2).contiguous().to(dev)
    for thr, mk in ((0.2, -1), (0.1, 1024)):
        conf = {"detection_threshold": thr, "max_num_keypoints": mk, "nms_radius": 2}
        f = lambda: ops.aliked_forward(w, rgb, conf, 1024 if mk > 0 else 8192)
        ms, nl = timed(f, iters)
        out = f()
        emit("a3 ALIKED", images=B, size=[480, 640], conf=conf, ms=round(ms, 2), images_per_s=round(B / ms * 1e3, 1), launches=nl,
             mean_keypoints=float(out["counts"][0].float().mean()), weights="random (no aliked-n16.pth offline)")


def row_nn(dev, iters):
    P, n, dim = 64, 4096, 128
    d = []
    for s in range(4):
        d0, d1 = synth.make_descriptor_pair(s, n=n, dim=dim)
        d += [d0.T, d1.T]
    desc = torch.from_numpy(np.stack(d * (P // 4))).contiguous().to(dev)
    counts = torch.full((2 * P,), n, dtype=torch.int32, device=dev)
    flop = 2.0 * n * n * dim * P
    for name, f in (("a8 mutual NN", lambda: ops.nearest_neighbor(desc, counts)),
                    ("a8 mutual NN + ratio", lambda: ops.nearest_neighbor(desc, counts, ratio_threshold=0.9, distance_threshold=0.9)),
                    ("a9 dual-softmax", lambda: ops.dual_softmax(desc, counts, 0.01, 20.0))):
        ms, nl = timed(f, iters)
        m0, _ = f()
        emit(name, pairs=P, keypoints=n, dim=dim, ms=round(ms, 3), pairs_per_s=round(P / ms * 1e3, 1), launches=nl,
             sim_tflops=round(flop * (2 if "dual" in name or "NN" in name else 1) / ms / 1e9, 1), mean_matches=float((m0 > -1).sum(1).float().mean()))


def row_magsac(dev, iters):
    import cv2
    P, n = 64, 800
    rng = np.random.default_rng(0)
    p0 = np.zeros((P, 1024, 2), np.float32); p1 = np.zeros((P, 1024, 2), np.float32)
    for p in range(P):
        _, _, Hm = synth.make_pair(p)
        x = rng.uniform([0, 0], [640, 480], (n, 2)).astype(np.float32)
        y = cv2.perspectiveTransform(x[None], Hm)[0] + rng.normal(0, 0.7, (n, 2)).astype(np.float32)
        out = rng.uniform(size=n) < 0.3
        y[out] = rng.uniform([0, 0], [640, 480], (int(out.sum()), 2)).astype(np.float32)
        p0[p, :n], p1[p, :n] = x, y
    t0, t1 = torch.from_numpy(p0).to(dev), torch.from_numpy(p1).to(dev)
    counts = torch.full((P,), n, dtype=torch.int32, device=dev)
    for gt in ("Homography", "Fundamental"):
        f = lambda: ops.magsac(t0, t1, counts, gt, 3.0, 0.9999, 10000)
        ms, nl = timed(f, iters)
        _, masks, ninl, nit = f()
        emit("a12 MAGSAC++ " + gt, pairs=P, matches=n, ms=round(ms, 3), pairs_per_s=round(P / ms * 1e3, 1), launches=nl,
             mean_inliers=float(ninl.float().mean()), mean_iterations=float(nit.float().mean()))


def row_config4(dev, iters):
    """BASELINE configs[3] on one GPU: ALIKED (RGB 640x480, 1024 keypoints) -> LightGlue (128-d input_proj) -> MAGSAC++ F.
    Random ALIKED weights and GIM LightGlue weights with the synthetic input_proj of the goldens (no checkpoints offline):
    a throughput configuration, parity is covered by the per-stage tests."""
    P, cap = 32, 1024
    aw = {k: v.to(dev) for k, v in ops.aliked_pack_weights(synth_weights.aliked_random_weights(0)).items()}
    g = np.load(ROOT / "tests/golden/lg_proj.npz")
    sd = synth_weights.lightglue_random_weights(0)
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    lw = {k: v.to(dev) for k, v in ops.lg_pack_weights(sd, 9).items()}
    a, b = synth.make_pair_batch(list(range(P)))
    rgb = torch.from_numpy(synth.to_rgb(np.stack([a, b], 1).reshape(2 * P, 480, 640)).astype(np.float32) / 255.0).permute(0, 3, 1, 2).contiguous().to(dev)
    aconf = {"detection_threshold": 0.1, "max_num_keypoints": cap, "nms_radius": 2}
    # no trained ALIKED / ALIKED-LightGlue weights offline: with random descriptors the early exit fires at layer 1, so the
    # matcher is forced to full depth (9 layers, no pruning) = an upper bound of its cost
    lconf = {"depth_confidence": -1.0, "width_confidence": -1.0, "filter_threshold": 0.2, "pruning_min_kpts": 1536, "use_tensor_cores": 1}
    ar = torch.arange(cap, device=dev)

    def step():
        f = ops.aliked_forward(aw, rgb, aconf, cap)
        counts = f["counts"][0].contiguous()
        lg = ops.lightglue_forward(lw, 9, f["keypoints"], f["descriptors"], counts, lconf)
        m0 = lg["matches"][0::2]                                       # [P,cap] matches0 per pair
        valid = (m0 > -1) & (ar[None] < counts[0::2, None])
        order = torch.argsort((~valid).to(torch.int8), dim=1, stable=True)   # matched keypoints first (device-side compaction)
        k0 = torch.gather(f["keypoints"][0::2], 1, order[..., None].expand(-1, -1, 2))
        j = torch.gather(m0, 1, order).clamp(min=0).long()
        k1 = torch.gather(f["keypoints"][1::2], 1, j[..., None].expand(-1, -1, 2))
        nm = valid.sum(1).to(torch.int32)
        _, masks, ninl, _ = ops.magsac(k0.contiguous(), k1.contiguous(), nm, "Fundamental", 3.0, 0.9999, 10000)
        return nm, ninl, lg["stop"]
    ms, nl = timed(step, iters)
    nm, ninl, stop = step()
    emit("config 4: ALIKED + LightGlue(128-d) + MAGSAC++ F", pairs=P, keypoints=cap, ms=round(ms, 2), pairs_per_s=round(P / ms * 1e3, 1), launches=nl,
         mean_matches=float(nm.float().mean()), mean_inliers=float(ninl.float().mean()), mean_stop_layer=float(stop.float().mean()),
         weights="random ALIKED, GIM LightGlue + synthetic input_proj; LightGlue forced to full depth")


ROWS = {"config4": row_config4, "sg": row_superglue, "loftr": row_loftr, "aliked": row_aliked, "nn": row_nn, "magsac": row_magsac}

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="sg,loftr,aliked,nn,magsac,config4")
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    with torch.no_grad():
        for r in args.rows.split(","):
            try:
                ROWS[r](dev, args.iters)
            except Exception as e:  # keep the other rows
                emit(r, error=f"{type(e).__name__}: {e}")
