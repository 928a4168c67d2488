"""SIFT throughput on one GPU: SIFT images/s (B = 64, 640x480, 5 distinct seeded batches dealt round-robin), SIFT +
mutual-NN pairs/s, SIFT + LightGlue(features="sift", synthetic weights) pairs/s, per-stage kernel times with the pyramid
bytes computed from shapes, and cv2.SIFT on the host cores as the CPU baseline.  Prints one JSON line (and writes it to
--out when given).  The GPU name and power limit are queried in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_info():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                    text=True).splitlines()[0]
        name, power, clk = (s.strip() for s in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:   # query only: a missing nvidia-smi leaves the fields empty
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e.__class__.__name__})"}


def timed(fn, iters):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--cpu-images", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sift: no CUDA device (timings are only taken on the GPU)")
    import cv2
    import oracle
    from oracle import sift as osift
    from imcui_b200 import _lib, ops
    from imcui_b200.hloc import extractors, matchers
    from imcui_b200.hloc.utils.base_model import dynamic_load
    from imcui_b200.utils import synth

    torch.set_grad_enabled(False)
    dev = torch.device("cuda:0")
    B, H, W = a.batch, a.height, a.width
    # 5 distinct batches of seeded synthetic frames (pairs: slot 2p / 2p+1), dealt round-robin over the timed steps
    batches = []
    for k in range(5):
        x0, x1 = synth.make_pair_batch(range(k * B // 2, (k + 1) * B // 2), H, W)
        frames = np.stack([x0, x1], 1).reshape(B, H, W)
        batches.append(torch.from_numpy(frames.astype(np.float32) / 255.0)[:, None].to(dev))
    ext = dynamic_load(extractors, "sift")({}).eval().to(dev)
    kc = ext.kernel_conf()
    res = {"metric": "sift", "batch": B, "height": H, "width": W, **gpu_info()}

    for x in batches:   # warm-up of every shape
        ext({"image": x})
    ms = timed(lambda i: ext({"image": batches[i % 5]}), a.iters)
    res["sift_ms_per_batch"] = ms
    res["sift_images_per_s"] = B / ms * 1e3

    # per-stage kernel time (library launch profiler), pyramid bytes from shapes
    with _lib.launch_profile(dev) as prof:
        ops.sift_forward(batches[0], kc, kc["max_keypoints"])
    stages = {}
    for site, n, t in prof.sites:
        name = site.rsplit(":", 1)[0]
        stages[name] = stages.get(name, 0.0) + t
    res["stage_ms"] = {k: round(v, 4) for k, v in sorted(stages.items(), key=lambda kv: -kv[1])}
    shapes = ops.sift_pyramid_shapes(kc, H, W)
    pyr_bytes = 4 * B * sum(l * h * w for _, l, h, w in shapes)
    res["pyramid_bytes_per_batch"] = pyr_bytes
    blur_ms = sum(v for k, v in stages.items() if "blur" in k or "base" in k or "downsample" in k)
    # each layer is written once by the column pass and read by the row pass of the next (plus the tmp round trip)
    res["pyramid_write_GBps"] = pyr_bytes / (blur_ms * 1e-3) / 1e9 if blur_ms > 0 else None

    # SIFT + mutual NN: B / 2 pairs per batch
    nn = dynamic_load(matchers, "nearest_neighbor")({"do_mutual_check": True}).eval().to(dev)

    def sift_nn(i):
        f = ext({"image": batches[i % 5]})
        for p in range(B // 2):
            nn({"descriptors0": f["descriptors"][2 * p][None], "descriptors1": f["descriptors"][2 * p + 1][None]})
    sift_nn(0)
    ms = timed(sift_nn, max(2, a.iters // 2))
    res["sift_nn_pairs_per_s"] = (B // 2) / ms * 1e3

    # SIFT + LightGlue(features="sift") on synthetic weights
    g = np.load(ROOT / "tests" / "golden" / "lg_so.npz")
    sd = dict(oracle.synthetic_weights("lightglue"))
    sd["input_proj.weight"], sd["input_proj.bias"] = torch.from_numpy(g["input_proj_w"]), torch.from_numpy(g["input_proj_b"])
    sd["posenc.Wr.weight"] = torch.from_numpy(g["posenc_wr"])
    lg = dynamic_load(matchers, "lightglue")({"match_threshold": 0.2, "features": "sift", "state_dict": sd}).eval().to(dev)

    def sift_lg(i):
        x = batches[i % 5]
        f = ext({"image": x})
        for p in range(B // 2):
            d = {}
            for side, s in (("0", 2 * p), ("1", 2 * p + 1)):
                d.update({"image" + side: x[s:s + 1], "keypoints" + side: f["keypoints"][s][None], "scores" + side: f["scores"][s][None],
                          "descriptors" + side: f["descriptors"][s][None], "scales" + side: f["scales"][s][None],
                          "oris" + side: f["oris"][s][None]})
            lg(d)
    sift_lg(0)
    ms = timed(sift_lg, 2)
    res["sift_lightglue_pairs_per_s"] = (B // 2) / ms * 1e3

    # CPU baseline: the oracle's cv2 path on the host cores
    sift = osift.create(osift.DEFAULT_CONF)
    imgs = [osift.to_uint8(batches[0][i, 0].cpu().numpy()) for i in range(min(a.cpu_images, B))]
    sift.detectAndCompute(imgs[0], None)
    t0 = time.perf_counter()
    for im in imgs:
        sift.detectAndCompute(im, None)
    res["cv2_cpu_images_per_s"] = len(imgs) / (time.perf_counter() - t0)
    res["cv2_threads"] = cv2.getNumThreads()
    res["host_cpus"] = os.cpu_count()
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
