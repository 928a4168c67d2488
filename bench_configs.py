"""bench.py --config {1,3,4,5}: the other BASELINE.json configurations behind the same measurement contract as the
headline config (bench.Config2): value (inputs resident in HBM), e2e (host buffers in, host results out), roofline of the
dominant kernel from the live launch-site profile, cpu_baseline / --impl reference from the oracle port.

  1  SuperPoint extract + mutual-NN matcher + MAGSAC on the reference's two test images (tests/test_basic.py path)
  3  LoFTR coarse-to-fine, batch = 32 synthetic 1024x1024 pairs           (random weights: no checkpoint offline)
  4  ALIKED + LightGlue(128-d input_proj) + MAGSAC++ fundamental matrix, RGB 640x480 stream (random ALIKED weights)
  5  dual-softmax (and mutual NN) on 4096 x 128-d descriptors -- the matcher side of DISK+NN (DISK net: not in the tree)
"""
import json
import time
from pathlib import Path

import numpy as np
import torch

import bench
from bench import NB, ROOT, roofline_from_sites


def _pin(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


class _Base:
    ref_pairs_per_step = 1
    cpu_sample_pairs = 2

    def __init__(self, dev, rank, world, args):
        self.dev, self.args, self.P = dev, args, args.pairs or self.default_pairs
        self.host_only = dev is None
        self.last_stats = {}

    def workload(self, world):
        return {"workload": self.workload_desc, "pairs_per_gpu": self.P, **self.last_stats,
                "stream": f"cycle of {NB} distinct batches dealt round-robin over ranks",
                "l2": "consecutive steps take different batches; per-step working set >> 126 MB L2 (config 1: single pair, L2-resident by nature)"}


# =========================================================================================================
class Config5(_Base):
    metric = "image-pairs/sec dual-softmax mutual matching @4096 x 128-d descriptors"
    default_pairs = 64
    workload_desc = ("dual-softmax matcher (inv_temperature 20, threshold 0.01) on 4096 x 128-d synthetic descriptor pairs with a planted "
                     "50 % partial permutation (BASELINE configs[4]: the matcher side of DISK+NN; the DISK net is not in the reference tree)")
    dtype = "f32-equivalent: split-fp16 (2 planes, 3 products) tcgen05 similarity tiles, f32 softmax statistics"
    N, D = 4096, 128
    cpu_sample_desc = "hloc DualSoftMax restated (oracle/matchers.py): torch CPU fp32 einsum + two softmax passes + host scatter"

    def __init__(self, dev, rank, world, args):
        super().__init__(dev, rank, world, args)
        from imcui_b200.utils import synth
        P = self.ref_pairs_per_step if self.host_only else self.P
        self.h_batches = []
        for b in range(1 if self.host_only else NB):
            d = np.empty((2 * P, self.N, self.D), np.float32)
            for p in range(P):
                d0, d1 = synth.make_descriptor_pair(b * self.P + p, n=self.N, dim=self.D)
                d[2 * p], d[2 * p + 1] = d0.T, d1.T
            self.h_batches.append(torch.from_numpy(d) if self.host_only else _pin(d))
        if self.host_only:
            return
        self.d_batches = [h.to(dev) for h in self.h_batches]
        self.counts = torch.full((2 * self.P,), self.N, dtype=torch.int32, device=dev)
        self.d_stage = torch.empty_like(self.d_batches[0])
        self.h_m = torch.empty(self.P, self.N, dtype=torch.int32).pin_memory()
        self.h_s = torch.empty(self.P, self.N, dtype=torch.float32).pin_memory()

    def _match(self, desc):
        from imcui_b200 import ops
        return ops.dual_softmax(desc, self.counts, 0.01, 20.0)

    def step_device(self, b):
        m0, _ = self._match(self.d_batches[b])
        return (m0 > -1).sum(1, dtype=torch.int32)

    def step_host(self, b):
        self.d_stage.copy_(self.h_batches[b], non_blocking=True)
        m0, s0 = self._match(self.d_stage)
        self.h_m.copy_(m0, non_blocking=True); self.h_s.copy_(s0, non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()
        return self.h_m, self.h_s

    h2d_bytes = property(lambda self: self.h_batches[0].numel() * 4)
    d2h_bytes = property(lambda self: self.h_m.numel() * 8)

    def gflop_per_pair(self):
        return 2.0 * self.N * self.N * self.D / 1e9

    def roofline(self, prof):
        return roofline_from_sites(prof, ["launch_tc_simreduce"], self.gflop_per_pair() * self.P, "TFLOP/s", "tensor",
                                   "tc_simreduce_kernel<dual-softmax ops> (streaming 128x128 split-fp16 similarity tiles in TMEM, never materialised)",
                                   note="algorithmic = ONE 4096x4096x128 similarity per pair (4.29 GFLOP); every extra sweep over the tiles and the "
                                        "split-precision products (three fp16 partial products per product) are overheads of the implementation")

    def cpu_unit(self):
        from oracle import matchers as om
        d = self.h_batches[0]
        return lambda: om.dual_softmax(d[0].t()[None], d[1].t()[None], 0.01, 20)

    def cpu_pairs(self, n, first=0):
        from oracle import matchers as om
        d = self.h_batches[0]
        t0 = time.perf_counter()
        for p in range(first, first + n):
            om.dual_softmax(d[2 * p].t()[None].contiguous(), d[2 * p + 1].t()[None].contiguous(), 0.01, 20)
        return time.perf_counter() - t0

    def match_f1(self, n):
        from oracle import matchers as om
        m0, _ = self._match(self.d_batches[0])
        m0 = m0.cpu().numpy()
        d = self.h_batches[0]
        tp = a = r = exact = 0
        for p in range(n):
            ref = om.dual_softmax(d[2 * p].t()[None].contiguous(), d[2 * p + 1].t()[None].contiguous(), 0.01, 20)["matches0"][0].numpy()
            g = m0[p]
            tp += int(((g == ref) & (g > -1)).sum()); a += int((g > -1).sum()); r += int((ref > -1).sum())
            exact += int(np.array_equal(g, ref))
        return {"pairs": n, "match_f1": 2 * tp / max(a + r, 1), "exact_pairs": exact / n, "kpts_set_equal": 1.0, "stop_equal": 1.0}


# =========================================================================================================
class Config3(_Base):
    metric = "image-pairs/sec @1024x1024 LoFTR coarse-to-fine"
    default_pairs = 32
    cpu_sample_pairs = 1
    workload_desc = ("LoFTR (ResNet-FPN 8/2, 4x(self,cross) linear-attention coarse transformer, dual-softmax coarse matching, fine refinement), "
                     "batch=32 synthetic 1024x1024 grayscale pairs per GPU (BASELINE configs[2]); seeded random weights (no LoFTR checkpoint "
                     "offline), coarse threshold lowered so that the fine stage is loaded")
    dtype = "f32-equivalent: split-fp16 tcgen05 convs (backbone), split-fp16 tcgen05 linears / coarse similarity, f32 linear attention"
    HW = 1024
    THR = 1e-9
    cpu_sample_desc = "SE2LoFTR module restated (oracle/loftr.py), torch CPU fp32, one 1024x1024 pair (materialises the 1.07 GB confidence matrix)"

    def __init__(self, dev, rank, world, args):
        super().__init__(dev, rank, world, args)
        from imcui_b200.utils import synth, synth_weights
        P = self.ref_pairs_per_step if self.host_only else self.P
        self.h_batches = []
        for b in range(1 if self.host_only else NB):
            a, c = synth.make_pair_batch(range(b * self.P, b * self.P + P), self.HW, self.HW)
            u8 = np.empty((2 * P, self.HW, self.HW), np.uint8)
            u8[0::2], u8[1::2] = a, c
            self.h_batches.append(torch.from_numpy(u8) if self.host_only else _pin(u8))
        self.sd = synth_weights.loftr_random_weights(0)
        if self.host_only:
            return
        from imcui_b200 import ops
        self.wd = ops.loftr_to_device(ops.loftr_pack_weights(self.sd), dev)
        self.d_batches = [h.to(dev) for h in self.h_batches]
        self.d_stage = torch.empty_like(self.d_batches[0])
        self.mcap = 4096
        self.h_k0 = torch.empty(self.P, self.mcap, 2).pin_memory(); self.h_k1 = torch.empty(self.P, self.mcap, 2).pin_memory()
        self.h_c = torch.empty(self.P, self.mcap).pin_memory(); self.h_n = torch.empty(self.P, dtype=torch.int32).pin_memory()

    def _fwd(self, u8):
        from imcui_b200 import ops
        imgs = (u8.double() / 255.0).float()
        return ops.loftr_forward(self.wd, imgs, {"match_threshold": self.THR, "use_tensor_cores": 1}, max_matches=self.mcap)

    def step_device(self, b):
        out = self._fwd(self.d_batches[b])
        self.last_stats = {"coarse_threshold": self.THR, "max_matches": self.mcap}
        return out["counts"]

    def step_host(self, b):
        self.d_stage.copy_(self.h_batches[b], non_blocking=True)
        out = self._fwd(self.d_stage)
        self.h_k0.copy_(out["keypoints0"], non_blocking=True); self.h_k1.copy_(out["keypoints1"], non_blocking=True)
        self.h_c.copy_(out["confidence"], non_blocking=True); self.h_n.copy_(out["counts"], non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()

    h2d_bytes = property(lambda self: self.h_batches[0].numel())
    d2h_bytes = property(lambda self: (self.h_k0.numel() * 2 + self.h_c.numel() + self.h_n.numel()) * 4)

    def gflop_per_pair(self):
        return 2520.0     # SURVEY.md 8(d): backbone 2 x 1014 + coarse transformer 352 + similarity 137

    def roofline(self, prof):
        # all tcgen05 implicit-GEMM conv launches of the ResNet-FPN backbone: 1.014 TFLOP / image minus the 7x7 stem (3.3 GFLOP, CUDA cores)
        return roofline_from_sites(prof, ["tc_conv"], (1014.0 - 3.3) * 2 * self.P, "TFLOP/s", "tensor",
                                   "tc_conv3x3_halo_pair_kernel / tc_conv3x3_kernel<BN,KS,RES> (LoFTR ResNet-FPN backbone @1024x1024: every 3x3 / 1x1 conv, tcgen05 split-fp16 = fp32-equivalent)",
                                   note="split precision: three fp16 partial products per fp32-equivalent product; 196-channel layers zero-padded to 256 (padding FLOPs not counted)")

    def cpu_unit(self):
        from oracle import loftr as ol
        img = (self.h_batches[0][:2, :256, :256].double() / 255.0).float()[:, None]
        return lambda: ol.forward(self.sd, img[:1], img[1:], thr=self.THR)

    def cpu_pairs(self, n, first=0):
        from oracle import loftr as ol
        t0 = time.perf_counter()
        for p in range(first, first + n):
            img = (self.h_batches[0][2 * p: 2 * p + 2].double() / 255.0).float()[:, None]
            ol.forward(self.sd, img[:1], img[1:], thr=self.THR)
        return time.perf_counter() - t0


# =========================================================================================================
class Config4(_Base):
    metric = "image-pairs/sec @640x480 ALIKED+LightGlue+MAGSAC++ (fundamental matrix)"
    default_pairs = 64
    cpu_sample_pairs = 2
    workload_desc = ("ALIKED-n16 (RGB 640x480, top-1024 keypoints) -> LightGlue features='aliked' architecture (128-d input_proj, 9 layers) -> "
                     "MAGSAC++ fundamental matrix 3 px / 0.9999 / 10000 on the matched keypoints (BASELINE configs[3]); seeded random ALIKED "
                     "weights + synthetic LightGlue weights (utils/synth_weights.py) with an input_proj FITTED (ridge regression, tools/make_golden.py aliked_lg_case) so that "
                     "the trained matcher sees SuperPoint-like descriptors: no aliked checkpoints offline, yet hundreds of geometrically "
                     "correct matches per pair reach MAGSAC; reference LightGlue semantics (depth 0.95 / width 0.99 / threshold 0.2)")
    dtype = "f32 (ALIKED, CUDA cores), split-fp16 tcgen05 = f32-equivalent (LightGlue), f64 (MAGSAC++ solvers)"
    cpu_sample_desc = "ALIKED x2 + LightGlue restated in torch CPU fp32 (oracle/aliked.py, oracle/lightglue.py) + cv2.findFundamentalMat(USAC_MAGSAC)"
    ACONF = {"detection_threshold": 0.1, "max_num_keypoints": 1024, "nms_radius": 2}
    # the reference's defaults (lightglue.py:331-344; hloc passes match_threshold 0.2 as filter_threshold): early stop + CUDA pruning
    LCONF = {"depth_confidence": 0.95, "width_confidence": 0.99, "filter_threshold": 0.2, "pruning_min_kpts": 1536, "use_tensor_cores": 1}

    def __init__(self, dev, rank, world, args):
        super().__init__(dev, rank, world, args)
        from imcui_b200.utils import synth, synth_weights
        P = self.ref_pairs_per_step if self.host_only else self.P
        self.h_batches = []
        for b in range(1 if self.host_only else NB):
            a, c = synth.make_pair_batch(range(b * self.P, b * self.P + P), 480, 640)
            g = np.empty((2 * P, 480, 640), np.uint8)
            g[0::2], g[1::2] = a, c
            rgb = synth.to_rgb(g)                                             # [2P,H,W,3] uint8
            self.h_batches.append(torch.from_numpy(rgb) if self.host_only else _pin(rgb))
        self.asd = synth_weights.aliked_random_weights(0)
        gz = np.load(ROOT / "tests/golden/aliked_lg.npz")    # fitted input_proj (see workload_desc)
        self.lsd = synth_weights.lightglue_random_weights(0)
        self.lsd["input_proj.weight"], self.lsd["input_proj.bias"] = torch.from_numpy(gz["input_proj_w"]), torch.from_numpy(gz["input_proj_b"])
        if self.host_only:
            return
        from imcui_b200 import ops
        self.aw = {k: v.to(dev) for k, v in ops.aliked_pack_weights(self.asd).items()}
        self.lw = {k: v.to(dev) for k, v in ops.lg_pack_weights(self.lsd, 9).items()}
        self.d_batches = [h.to(dev) for h in self.h_batches]
        self.d_stage = torch.empty_like(self.d_batches[0])
        self.cap = 1024
        self.ar = torch.arange(self.cap, device=dev)
        self.h_F = torch.empty(self.P, 3, 3, dtype=torch.float64).pin_memory()
        self.h_mask = torch.empty(self.P, self.cap, dtype=torch.bool).pin_memory()
        self.h_k0 = torch.empty(self.P, self.cap, 2).pin_memory(); self.h_k1 = torch.empty(self.P, self.cap, 2).pin_memory()
        self.h_n = torch.empty(2, self.P, dtype=torch.int32).pin_memory()

    def _pipeline(self, rgb_u8):
        from imcui_b200 import ops
        img = (rgb_u8.permute(0, 3, 1, 2).double() / 255.0).float().contiguous()
        f = ops.aliked_forward(self.aw, img, self.ACONF, self.cap)
        counts = f["counts"][0].contiguous()
        lg = ops.lightglue_forward(self.lw, 9, f["keypoints"], f["descriptors"], counts, self.LCONF)
        k0, k1, nm = ops.gather_matches(f["keypoints"], lg["matches"], counts)
        Fm, masks, ninl, _ = ops.magsac(k0, k1, nm, "Fundamental", 3.0, 0.9999, 10000)
        return k0, k1, nm, Fm, masks, ninl, lg

    def step_device(self, b):
        k0, k1, nm, Fm, masks, ninl, lg = self._pipeline(self.d_batches[b])
        self._last = (nm, ninl, lg["stop"])
        return nm

    def workload(self, world):
        nm, ninl, stop = self._last
        self.last_stats = {"mean_inliers": float(ninl.float().mean()), "mean_stop_layer": float(stop.float().mean()),
                           "pairs_verified": int((nm >= 8).sum()), "max_keypoints": 1024}
        return super().workload(world)

    def step_host(self, b):
        self.d_stage.copy_(self.h_batches[b], non_blocking=True)
        k0, k1, nm, Fm, masks, ninl, _ = self._pipeline(self.d_stage)
        self.h_F.copy_(Fm, non_blocking=True); self.h_mask.copy_(masks, non_blocking=True)
        self.h_k0.copy_(k0, non_blocking=True); self.h_k1.copy_(k1, non_blocking=True)
        self.h_n[0].copy_(nm, non_blocking=True); self.h_n[1].copy_(ninl, non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()

    h2d_bytes = property(lambda self: self.h_batches[0].numel())
    d2h_bytes = property(lambda self: self.h_F.numel() * 8 + self.h_mask.numel() + self.h_k0.numel() * 8 + self.h_n.numel() * 4)

    def gflop_per_pair(self):
        stop = float(self._last[2].float().mean()) if getattr(self, "_last", None) is not None else 9.0
        return 2 * 5.5 + bench.lg_gflop(1024, stop)

    def roofline(self, prof):
        # ALIKED is the HBM-bound class (SURVEY 8(d)): its dominant kernel is the fused 1x1 head + upsample + concat + L2 norm +
        # score_head.0, which writes the 128-channel full-resolution map once: 128 x H x W x 4 B out + the four pyramid levels in
        n_img = 2 * self.P
        by = (128 * 480 * 640 * 4 + (16 * 480 * 640 + 32 * 240 * 320 + 64 * 60 * 80 + 128 * 15 * 20) * 4 + 8 * 480 * 640 * 4) / 1e9
        return roofline_from_sites(prof, ["ak_fuse_kernel"], by * n_img, "GB/s", "hbm",
                                   "ak_fuse_kernel (ALIKED: four 1x1 heads + x2/x8/x32 bilinear upsampling + concat + L2 norm + score_head.0; the 128-channel map is written once)",
                                   note="algorithmic bytes = 128-ch fp32 feature map written + 8-ch score features written + pyramid levels read")

    def cpu_unit(self):
        from oracle import aliked as oa
        img = (self.h_batches[0][:1, :240, :320].permute(0, 3, 1, 2).double() / 255.0).float()
        return lambda: oa.forward(self.asd, img, 0.1, 1024, 2)

    def cpu_pairs(self, n, first=0):
        import cv2
        from oracle import aliked as oa, lightglue as olg
        t0 = time.perf_counter()
        for p in range(first, first + n):
            img = (self.h_batches[0][2 * p: 2 * p + 2].permute(0, 3, 1, 2).double() / 255.0).float()
            f0, f1 = oa.forward(self.asd, img[:1], 0.1, 1024, 2), oa.forward(self.asd, img[1:], 0.1, 1024, 2)
            r = olg.forward(self.lsd, f0["keypoints"][None], f0["descriptors"][None], f1["keypoints"][None], f1["descriptors"][None],
                            {"depth_confidence": 0.95, "width_confidence": 0.99, "filter_threshold": 0.2})
            m = r["matches0"][0].numpy()
            v = m > -1
            if v.sum() >= 8:
                try:
                    cv2.findFundamentalMat(f0["keypoints"].numpy()[v], f1["keypoints"].numpy()[m[v]], method=cv2.USAC_MAGSAC,
                                           ransacReprojThreshold=3.0, confidence=0.9999, maxIters=10000)
                except cv2.error:
                    pass
        return time.perf_counter() - t0


# =========================================================================================================
class Config1(_Base):
    metric = "image-pairs/sec SuperPoint + mutual-NN + MAGSAC on the reference test pair (640x480)"
    default_pairs = 1
    cpu_sample_pairs = 2
    workload_desc = ("the reference's CPU-runnable case (tests/test_basic.py `test_one`, BASELINE configs[0]): tests/data pair (780x1063 and "
                     "1013x673 RGB JPEGs) -> RGB2GRAY, INTER_AREA force-resize to 640x480 -> SuperPoint (nms 3, thr 0.015, max 1024) -> mutual NN "
                     "-> MAGSAC F + H 3 px / 0.9999 / 10000; ONE pair per step (latency-bound by construction)")
    dtype = "f32-equivalent: split-fp16 tcgen05 convs and similarity tiles, f64 MAGSAC++ solvers"
    cpu_sample_desc = "cv2 pre-processing + SuperPoint x2 + NearestNeighbor (oracle ports, torch CPU fp32) + cv2 USAC_MAGSAC F and H"
    SP = {"nms_radius": 3, "max_keypoints": 1024, "keypoint_threshold": 0.015, "remove_borders": 4}
    PRE = {"grayscale": True, "resize_max": 1024, "dfactor": 8, "force_resize": True, "width": 640, "height": 480}

    def __init__(self, dev, rank, world, args):
        super().__init__(dev, rank, world, args)
        self.P = 1
        names = ["02928139_3448003521", "17295357_9106075285"]
        self.rgb = [np.load(ROOT / "tests/golden/data" / f"{n}.npz")["rgb"] for n in names]
        if self.host_only:
            return
        from imcui_b200.hloc import extractors, matchers
        from imcui_b200.hloc.utils.base_model import dynamic_load
        from imcui_b200.utils import synth_weights
        self.sp = dynamic_load(extractors, "superpoint")({**self.SP, "state_dict": synth_weights.superpoint_random_weights(0)}).eval().to(dev)
        self.nn = dynamic_load(matchers, "nearest_neighbor")({"do_mutual_check": True}).eval().to(dev)
        from imcui_b200.hloc.pipeline import FramePrep
        pre = FramePrep(self.PRE, dev)(self.rgb)
        self.d_img = torch.cat([p[0] for p in pre])            # [2,1,480,640] resident
        self.scales = [p[1] / p[2] for p in pre]

    def _match_device(self):
        from imcui_b200 import ops
        f = self.sp({"image": self.d_img})
        d0, d1 = f["descriptors"][0][None], f["descriptors"][1][None]
        pred = self.nn({"descriptors0": d0, "descriptors1": d1})
        m0 = pred["matches0"][0]
        v = m0 > -1
        k0 = f["keypoints"][0][v]; k1 = f["keypoints"][1][m0[v]]
        n = int(v.sum())
        cap = max(128, (n + 127) // 128 * 128)
        p0 = torch.zeros(2, cap, 2, device=self.dev); p1 = torch.zeros(2, cap, 2, device=self.dev)
        s0 = torch.as_tensor(self.scales[0], dtype=torch.float32, device=self.dev); s1 = torch.as_tensor(self.scales[1], dtype=torch.float32, device=self.dev)
        p0[:, :n] = (k0 + 0.5) * s0 - 0.5; p1[:, :n] = (k1 + 0.5) * s1 - 0.5
        cnt = torch.tensor([n, n], dtype=torch.int32, device=self.dev)
        _, _, ninl_f, _ = ops.magsac(p0[:1], p1[:1], cnt[:1], "Fundamental", 3.0, 0.9999, 10000)
        _, _, ninl_h, _ = ops.magsac(p0[1:], p1[1:], cnt[1:], "Homography", 3.0, 0.9999, 10000)
        self.last_stats = {"keypoints": [int(len(f["keypoints"][0])), int(len(f["keypoints"][1]))], "inliers_F": int(ninl_f[0]), "inliers_H": int(ninl_h[0])}
        return torch.tensor([n], dtype=torch.int32, device=self.dev)

    def step_device(self, b):
        return self._match_device()

    def step_host(self, b):
        from imcui_b200.hloc import extract_features as ef, match_features as mf
        from imcui_b200.ui import utils as uu
        conf = {**self.PRE}
        f0, f1 = ef.extract(self.sp, self.rgb[0], conf), ef.extract(self.sp, self.rgb[1], conf)
        pred = mf.match_images(self.nn, f0, f1)
        return uu.filter_matches(pred, ransac_method="B200_MAGSAC", ransac_reproj_threshold=3.0, ransac_confidence=0.9999, ransac_max_iter=10000)

    h2d_bytes = property(lambda self: sum(r.size for r in self.rgb))
    d2h_bytes = property(lambda self: 2 * 1024 * (2 + 1 + 256) * 4)

    def gflop_per_pair(self):
        return 2 * bench.SP_GFLOP_PER_IMAGE + 2 * 1024 * 1024 * 256 / 1e9

    def roofline(self, prof):
        return roofline_from_sites(prof, ["tc_conv1ab_fused"], (bench.SP_LAYER_GFLOP["conv1a"] + bench.SP_LAYER_GFLOP["conv1b"]) * 2, "TFLOP/s", "tensor",
                                   "tc_conv3x3_c64_pair_kernel<fused conv1a> at batch 2 (one pair): 2 x 2400 tiles over 74 persistent CTA pairs",
                                   note="single-pair latency case: the grid covers the SMs but nothing amortises launch gaps")

    def _cpu_pair(self):
        import cv2
        import oracle
        from oracle import matchers as om, superpoint as osp
        ws = oracle.synthetic_weights("superpoint")
        feats = []
        for r in self.rgb:
            g = cv2.cvtColor(r, cv2.COLOR_RGB2GRAY).astype(np.float32)
            g = cv2.resize(g, (640, 480), interpolation=cv2.INTER_AREA)
            feats.append(osp.forward(ws, torch.from_numpy(g / 255.0).float()[None, None], self.SP))
        r = om.nearest_neighbor(feats[0]["descriptors"][0][None], feats[1]["descriptors"][0][None])
        m = r["matches0"][0].numpy(); v = m > -1
        k0 = feats[0]["keypoints"][0].numpy()[v]; k1 = feats[1]["keypoints"][0].numpy()[m[v]]
        if len(k0) >= 8:
            cv2.findFundamentalMat(k0, k1, method=cv2.USAC_MAGSAC, ransacReprojThreshold=3.0, confidence=0.9999, maxIters=10000)
            cv2.findHomography(k0, k1, method=cv2.USAC_MAGSAC, ransacReprojThreshold=3.0, confidence=0.9999, maxIters=10000)

    def cpu_unit(self):
        return self._cpu_pair

    def cpu_pairs(self, n, first=0):
        t0 = time.perf_counter()
        for _ in range(n):
            self._cpu_pair()
        return time.perf_counter() - t0


def make(n, dev, rank, world, args):
    return {1: Config1, 3: Config3, 4: Config4, 5: Config5}[n](dev, rank, world, args)
