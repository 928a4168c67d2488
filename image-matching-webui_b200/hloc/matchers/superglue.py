"""SuperGlue matcher plugin -- drop-in for imcui/hloc/matchers/superglue.py:13-43.  Same default_conf /
required_inputs / output dict; the forward pass runs in libimw_b200.so (imw_superglue_forward) instead of
third_party/SuperGluePretrainedNetwork/models/superglue.py."""
import torch

from .. import MODEL_REPO_ID, logger
from ..utils.base_model import BaseModel
from ... import ops


class SuperGlue(BaseModel):
    default_conf = {
        "weights": "outdoor",
        "model_name": "superglue_outdoor.pth",
        "sinkhorn_iterations": 100,
        "match_threshold": 0.2,
        "state_dict": None,  # B200 engine: in-memory checkpoint (reference key names) instead of model_name
        "tensor_cores": True,  # B200 engine switch: True/"3xtf32", "tf32", False (see matchers/lightglue.py)
    }
    required_inputs = ["image0", "keypoints0", "scores0", "descriptors0", "image1", "keypoints1", "scores1", "descriptors1"]

    def _init(self, conf):
        assert conf["weights"] in ["indoor", "outdoor"]  # superglue.py:221
        sd = conf.get("state_dict")
        if sd is None:
            weights_path = self._download_model(repo_id=MODEL_REPO_ID, filename="{}/{}".format("superglue", self.conf["model_name"]))
            sd = torch.load(str(weights_path), map_location="cpu")
        self.conf["state_dict"] = None
        self.bin_score = float(sd["bin_score"])
        for k, v in ops.sg_pack_weights(sd).items():
            self.register_buffer(k.replace(".", "__"), v, persistent=False)
        logger.info('Loaded SuperGlue model ("{}" weights)'.format(self.conf["weights"]))

    def _bufs(self):
        return {k.replace("__", "."): v for k, v in self.named_buffers()}

    def _forward(self, data):
        k0, k1 = data["keypoints0"], data["keypoints1"]
        if k0.shape[1] == 0 or k1.shape[1] == 0:  # superglue.py:233-240
            s0, s1 = k0.shape[:-1], k1.shape[:-1]
            return {"matches0": k0.new_full(s0, -1, dtype=torch.int), "matches1": k1.new_full(s1, -1, dtype=torch.int),
                    "matching_scores0": k0.new_zeros(s0), "matching_scores1": k1.new_zeros(s1)}
        assert k0.shape[0] == 1, "one pair per call"
        m, n, dev = k0.shape[1], k1.shape[1], k0.device
        cap = max(128, (max(m, n) + 127) // 128 * 128)
        kp = torch.zeros(2, cap, 2, device=dev); sc = torch.zeros(2, cap, device=dev); ds = torch.zeros(2, cap, 256, device=dev)
        kp[0, :m], kp[1, :n] = k0[0].float(), k1[0].float()
        sc[0, :m], sc[1, :n] = data["scores0"][0].float(), data["scores1"][0].float()
        ds[0, :m], ds[1, :n] = data["descriptors0"][0].t().float(), data["descriptors1"][0].t().float()
        counts = torch.tensor([m, n], dtype=torch.int32, device=dev)
        # normalize_keypoints uses the image tensor shapes (superglue.py:65-72)
        wh = torch.tensor([[data["image0"].shape[-1], data["image0"].shape[-2]], [data["image1"].shape[-1], data["image1"].shape[-2]]],
                          dtype=torch.int32, device=dev)
        tc = {False: 0, True: 1, "3xtf32": 1, "tf32": 2}[self.conf["tensor_cores"]]
        matches, ms = ops.superglue_forward(self._bufs(), self.bin_score, kp, sc, ds, counts, wh,
                                            {"sinkhorn_iterations": self.conf["sinkhorn_iterations"],
                                             "match_threshold": self.conf["match_threshold"], "use_tensor_cores": tc})
        return {"matches0": matches[0, :m].long()[None], "matches1": matches[1, :n].long()[None],
                "matching_scores0": ms[0, :m][None], "matching_scores1": ms[1, :n][None]}

    def match_batch(self, batch):
        """see LightGlue.match_batch (image_wh [2P,2] int32 feeds the keypoint normalisation, superglue.py:65-72)"""
        tc = {False: 0, True: 1, "3xtf32": 1, "tf32": 2}[self.conf["tensor_cores"]]
        matches, ms = ops.superglue_forward(self._bufs(), self.bin_score, batch["keypoints"], batch["scores"], batch["descriptors"],
                                            batch["counts"], batch["image_wh"],
                                            {"sinkhorn_iterations": self.conf["sinkhorn_iterations"],
                                             "match_threshold": self.conf["match_threshold"], "use_tensor_cores": tc})
        return matches[0::2], ms[0::2]
