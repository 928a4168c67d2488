"""Batched SuperPoint -> LightGlue pair pipeline (the BASELINE config-2 hot path as one device-resident stream).

  PairEngine   P pairs per step: decoded frames (uint8, HBM) -> imw_preprocess -> SuperPoint -> LightGlue ->
               imw_gather_matches, no host synchronisation between the stages.  `match_device` is the model part alone
               (what bench.py times as `value`), `match_frames_device` the whole step from decoded frames.
  PairStream   the host side of a pair stream: pinned frame batches in, compact match records out, double-buffered over
               three CUDA streams so that H2D(i+1), compute(i) and D2H(i-1) overlap (bench.py's `e2e`; the
               match_from_paths-style exporter in hloc/pairs_stream.py drives it the same way).

The single-pair plugin classes under hloc/ go through the same C-ABI entry points."""
import torch

from . import _lib as L
from . import ops
from .hloc import WEIGHTS_DIR

SP_CONF_DEFAULT = {"nms_radius": 3, "keypoint_threshold": 0.005, "max_keypoints": 1024, "remove_borders": 4}
LG_CONF_DEFAULT = {"depth_confidence": 0.95, "width_confidence": 0.99, "filter_threshold": 0.2, "pruning_min_kpts": 1536,
                   "use_tensor_cores": 1}


class PairEngine:
    def __init__(self, device, n_pairs, height=480, width=640, sp_conf=None, lg_conf=None, n_layers=9, frame_shape=None, pre_conf=None,
                 sp_state_dict=None, lg_state_dict=None):
        """height/width: size of the network input.  frame_shape (H0, W0[, 3]) + pre_conf (the registry's `preprocessing`
        dict): decoded frames of that shape are prepared on the device; their prepared size must equal (height, width).
        sp_state_dict / lg_state_dict: in-memory checkpoints (reference key names) instead of weights/*.pt."""
        self.device = torch.device(device)
        self.P, self.H, self.W = n_pairs, height, width
        self.sp_conf = {**SP_CONF_DEFAULT, **(sp_conf or {})}
        self.lg_conf = {**LG_CONF_DEFAULT, **(lg_conf or {})}
        self.n_layers = n_layers
        L.lib()  # fail loudly now if the CUDA library is missing
        sp_sd = sp_state_dict if sp_state_dict is not None else torch.load(str(WEIGHTS_DIR / "superpoint_v1.pt"), map_location="cpu")
        lg_sd = lg_state_dict if lg_state_dict is not None else torch.load(str(WEIGHTS_DIR / "superpoint_lightglue.pt"), map_location="cpu")
        self.sp_w = {k: v.to(self.device) for k, v in ops.sp_pack_weights(sp_sd).items()}
        self.lg_w = {k: v.to(self.device) for k, v in ops.lg_pack_weights(lg_sd, n_layers).items()}
        mk = self.sp_conf["max_keypoints"]
        assert mk > 0, "the batched engine needs a keypoint cap"
        self.cap = (mk + 127) // 128 * 128
        S, dev = 2 * n_pairs, self.device
        self.sp_out = {
            "keypoints": torch.zeros(S, self.cap, 2, device=dev),
            "scores": torch.zeros(S, self.cap, device=dev),
            "descriptors": torch.zeros(S, self.cap, 256, device=dev),
            "counts": torch.zeros(2, S, dtype=torch.int32, device=dev),
        }
        self.lg_out = {
            "matches": torch.empty(S, self.cap, dtype=torch.int32, device=dev),
            "scores": torch.empty(S, self.cap, device=dev),
            "stop": torch.empty(n_pairs, dtype=torch.int32, device=dev),
            "prune": torch.empty(S, self.cap, dtype=torch.int32, device=dev),
        }
        # decoded-frame front end
        self.frame_shape, self.pre_conf = None, None
        if frame_shape is not None:
            self.pre_conf = dict(pre_conf or {})
            self.frame_shape = tuple(frame_shape)
            ch = self.frame_shape[2] if len(self.frame_shape) == 3 else 1
            oc, oh, ow = ops.preprocess_plan(self.pre_conf, self.frame_shape[0], self.frame_shape[1], ch)
            assert (oc, oh, ow) == (1, height, width), f"frames {frame_shape} prepare to {(oc, oh, ow)}, engine built for (1, {height}, {width})"
            self.d_image = torch.empty(S, 1, height, width, device=dev)
            # scales = original_size / size per image (w, h), as match_features.py:249-250 computes them (float64 -> fp32)
            s = torch.tensor([self.frame_shape[1] / width, self.frame_shape[0] / height], dtype=torch.float64).float()
            self.scales = s[None].repeat(S, 1).contiguous().to(dev)
        # pinned host staging for the synchronous end-to-end path (match_host)
        self.h_images = torch.empty(S, height, width, dtype=torch.uint8).pin_memory()
        self.d_images_u8 = torch.empty(S, height, width, dtype=torch.uint8, device=dev)
        self.h_matches = torch.empty(S, self.cap, dtype=torch.int32).pin_memory()
        self.h_mscores = torch.empty(S, self.cap, dtype=torch.float32).pin_memory()
        self.h_kpts = torch.empty(S, self.cap, 2, dtype=torch.float32).pin_memory()
        self.h_counts = torch.empty(2, S, dtype=torch.int32).pin_memory()
        self.h_stop = torch.empty(n_pairs, dtype=torch.int32).pin_memory()

    # ---- model part ------------------------------------------------------------------------------------------------
    def match_device(self, images):
        """images [2P,1,H,W] fp32 on the device, slot 2p+side.  Everything stays on the device."""
        sp = ops.superpoint_forward(self.sp_w, images, self.sp_conf, self.cap, out=self.sp_out)
        lg = ops.lightglue_forward(self.lg_w, self.n_layers, sp["keypoints"], sp["descriptors"], sp["counts"][0],
                                   self.lg_conf, out=self.lg_out)
        return sp, lg

    def to_float(self, images_u8):
        """gray uint8 [2P,H,W] at network size -> fp32 in [0,1] exactly as the reference does (extract_features.py:139),
        through the pre-processing kernel (no resize: conversion and /255 only)."""
        return ops.preprocess(images_u8, {"grayscale": True, "resize_max": 0, "force_resize": False, "dfactor": 1})

    # ---- whole step from decoded frames ----------------------------------------------------------------------------------
    def new_record(self):
        """device buffers of one step's compact result (PairStream keeps two)"""
        P, cap, dev = self.P, self.cap, self.device
        return {"mkpts0": torch.zeros(P, cap, 2, device=dev), "mkpts1": torch.zeros(P, cap, 2, device=dev),
                "mkpts0_orig": torch.zeros(P, cap, 2, device=dev), "mkpts1_orig": torch.zeros(P, cap, 2, device=dev),
                "mconf": torch.zeros(P, cap, device=dev), "mcount": torch.zeros(P, dtype=torch.int32, device=dev),
                "stop": torch.zeros(P, dtype=torch.int32, device=dev), "n_kpts": torch.zeros(2 * P, dtype=torch.int32, device=dev)}

    def match_frames_device(self, frames_u8, record):
        """frames_u8 [2P,H0,W0(,3)] uint8 on the device (decoded frames) -> `record` (see new_record) on the device."""
        assert self.frame_shape is not None and tuple(frames_u8.shape[1:]) == self.frame_shape
        ops.preprocess(frames_u8, self.pre_conf, out=self.d_image)
        sp, lg = self.match_device(self.d_image)
        counts = sp["counts"][0]
        ops.gather_matches(sp["keypoints"], lg["matches"], counts, scores=lg["scores"], scales=self.scales, out=record)
        record["stop"].copy_(lg["stop"])
        record["n_kpts"].copy_(counts)
        return record

    # ---- synchronous end-to-end path at network size -----------------------------------------------------------------------
    def match_host(self, images_u8_pinned=None):
        """pinned gray uint8 host images at network size -> H2D -> SuperPoint -> LightGlue -> D2H of matches, scores,
        keypoints, counts, stop into pinned host buffers.  One stream synchronisation at the end."""
        src = self.h_images if images_u8_pinned is None else images_u8_pinned
        self.d_images_u8.copy_(src, non_blocking=True)
        sp, lg = self.match_device(self.to_float(self.d_images_u8))
        self.h_matches.copy_(lg["matches"], non_blocking=True)
        self.h_mscores.copy_(lg["scores"], non_blocking=True)
        self.h_kpts.copy_(sp["keypoints"], non_blocking=True)
        self.h_counts.copy_(sp["counts"], non_blocking=True)
        self.h_stop.copy_(lg["stop"], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self.h_matches, self.h_mscores, self.h_kpts, self.h_counts, self.h_stop

    @property
    def h2d_bytes(self):
        return self.h_images.numel()

    @property
    def d2h_bytes(self):
        return sum(t.numel() * t.element_size() for t in (self.h_matches, self.h_mscores, self.h_kpts, self.h_counts, self.h_stop))


class PairStream:
    """Double-buffered host pipeline around a PairEngine built with `frame_shape`.

    for rec in PairStream(engine).run(batches): ...   `batches` yields pinned uint8 tensors [2P,H0,W0(,3)] (decoded frames,
    slot 2p+side); `rec` holds pinned host arrays of that batch: mkpts0_orig / mkpts1_orig [P,cap,2] (original-frame
    coordinates), mconf [P,cap], mcount [P], stop [P], n_kpts [2P] -- valid until the next-but-one batch is yielded.

    Three streams: H2D of batch i+1 and D2H of batch i-1 run while batch i computes; two input buffers, two device
    records, two host records; the host only ever waits for the D2H event of the batch it hands out."""
    KEYS = ("mkpts0_orig", "mkpts1_orig", "mconf", "mcount", "stop", "n_kpts")

    def __init__(self, engine: PairEngine):
        assert engine.frame_shape is not None, "PairStream needs an engine built with frame_shape / pre_conf"
        self.eng, dev = engine, engine.device
        self.s_in, self.s_comp, self.s_out = (torch.cuda.Stream(dev) for _ in range(3))
        shape = (2 * engine.P, *engine.frame_shape)
        self.d_in = [torch.empty(shape, dtype=torch.uint8, device=dev) for _ in range(2)]
        self.d_rec = [engine.new_record() for _ in range(2)]
        self.h_rec = [{k: torch.empty_like(self.d_rec[0][k], device="cpu").pin_memory() for k in self.KEYS} for _ in range(2)]
        self.ev_in = [torch.cuda.Event() for _ in range(2)]
        self.ev_comp = [torch.cuda.Event() for _ in range(2)]
        self.ev_out = [torch.cuda.Event() for _ in range(2)]
        self.h2d_bytes = self.d_in[0].numel()
        self.d2h_bytes = sum(t.numel() * t.element_size() for t in self.h_rec[0].values())

    def _enqueue(self, i, frames):
        s = i % 2
        with torch.cuda.stream(self.s_in):
            if i >= 2:
                self.s_in.wait_event(self.ev_comp[s])       # batch i-2 has consumed this input buffer
            self.d_in[s].copy_(frames, non_blocking=True)
            self.ev_in[s].record(self.s_in)
        with torch.cuda.stream(self.s_comp):
            self.s_comp.wait_event(self.ev_in[s])
            if i >= 2:
                self.s_comp.wait_event(self.ev_out[s])      # batch i-2's record has left the device
            self.eng.match_frames_device(self.d_in[s], self.d_rec[s])
            self.ev_comp[s].record(self.s_comp)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.ev_comp[s])
            for k in self.KEYS:
                self.h_rec[s][k].copy_(self.d_rec[s][k], non_blocking=True)
            self.ev_out[s].record(self.s_out)

    def run(self, batches):
        cur = torch.cuda.current_stream(self.eng.device)
        self.s_comp.wait_stream(cur)
        pending = None
        i = 0
        for frames in batches:
            self._enqueue(i, frames)
            if pending is not None:
                self.ev_out[pending % 2].synchronize()
                yield self.h_rec[pending % 2]
            pending = i
            i += 1
        if pending is not None:
            self.ev_out[pending % 2].synchronize()
            yield self.h_rec[pending % 2]
        cur.wait_stream(self.s_comp)
