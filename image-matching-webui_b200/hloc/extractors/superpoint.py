"""SuperPoint extractor plugin -- drop-in for imcui/hloc/extractors/superpoint.py:33-57.
Same default_conf / required_inputs / output dict; the forward pass runs in libimw_b200.so
(imw_superpoint_forward) instead of third_party/SuperGluePretrainedNetwork/models/superpoint.py."""
import torch

from .. import MODEL_REPO_ID, logger
from ..utils.base_model import BaseModel
from ... import ops


class SuperPoint(BaseModel):
    default_conf = {
        "nms_radius": 4,
        "model_name": "superpoint_v1.pth",
        "keypoint_threshold": 0.005,
        "max_keypoints": -1,
        "remove_borders": 4,
        "fix_sampling": False,
        "state_dict": None,  # B200 engine: in-memory checkpoint (reference key names) instead of model_name
        # B200 engine switch (not in the reference): encoder convs on tcgen05 with split-fp16 operands (2 planes, 3 products)
        # (fp32-equivalent products, needs W % 128 == 0); False = fp32 CUDA-core convs
        "tensor_cores": True,
    }
    required_inputs = ["image"]
    detection_noise = 2.0

    def _init(self, conf):
        mk = conf["max_keypoints"]
        if mk == 0 or mk < -1:  # superpoint.py:139-141
            raise ValueError('"max_keypoints" must be positive or "-1"')
        sd = conf.get("state_dict")
        if sd is None:
            weights_path = self._download_model(
                repo_id=MODEL_REPO_ID, filename="{}/{}".format("superglue", self.conf["model_name"]))
            sd = torch.load(str(weights_path), map_location="cpu")
        self.conf["state_dict"] = None
        for k, v in ops.sp_pack_weights(sd).items():
            self.register_buffer(k, v, persistent=False)
        self._uncapped_cap = 8192
        logger.info("Load SuperPoint model done.")

    def _bufs(self):
        return dict(self.named_buffers())

    def _forward(self, data):
        conf = self.conf  # mutable: UI/API overwrite max_keypoints / keypoint_threshold per call
        image = data["image"]
        if image.shape[1] != 1:
            raise AssertionError(f"SuperPoint expects a grayscale image, got {tuple(image.shape)}")
        mk = int(conf["max_keypoints"])
        cap = mk if mk > 0 else self._uncapped_cap
        out = ops.superpoint_forward(self._bufs(), image.float(), conf, cap)
        counts = out["counts"].cpu()  # the reference API returns ragged tensors: one host sync
        if int((counts[1] > counts[0]).any()):  # only possible with max_keypoints = -1
            self._uncapped_cap = cap = int(counts[1].max())
            out = ops.superpoint_forward(self._bufs(), image.float(), conf, cap)
            counts = out["counts"].cpu()
        n = [int(c) for c in counts[0]]
        B = image.shape[0]
        return {
            "keypoints": [out["keypoints"][b, : n[b]] for b in range(B)],
            "scores": tuple(out["scores"][b, : n[b]] for b in range(B)),
            "descriptors": [out["descriptors"][b, : n[b]].t() for b in range(B)],  # [256,N] view
        }
