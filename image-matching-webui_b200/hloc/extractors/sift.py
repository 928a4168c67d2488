"""SIFT extractor plugin -- the opencv backend of hloc's SIFT wrapper (which follows LightGlue's lightglue/sift.py):
cv2.SIFT_create(contrastThreshold=detection_threshold, nfeatures=max_num_keypoints, edgeThreshold=edge_threshold,
nOctaveLayers=num_octaves).detectAndCompute on uint8(trunc(image * 255)), then filter_dog_point (nms_radius 0), top-k on
the response and RootSIFT.  The whole chain runs in libimw_b200.so (imw_sift_forward).

Outputs are lists per image: keypoints [N,2], scores [N] (response), descriptors [128,N], scales [N] (keypoint size) and
oris [N] (radians), in descending response order -- the scales / oris LightGlue's features="sift" encoding reads."""
from ..utils.base_model import BaseModel
from ... import ops


class SIFT(BaseModel):
    default_conf = {
        "rootsift": True,
        "nms_radius": 0,
        "max_num_keypoints": 4096,
        "backend": "opencv",
        "detection_threshold": 0.0066667,
        "edge_threshold": 10,
        "first_octave": -1,   # read by the pycolmap backend only; cv2.SIFT always starts at octave -1
        "num_octaves": 4,
    }
    required_inputs = ["image"]

    def _init(self, conf):
        if conf["backend"] != "opencv":
            raise NotImplementedError(f"SIFT backend {conf['backend']!r}: only the opencv arithmetic is built")
        if conf["nms_radius"] is not None and conf["nms_radius"] > 0:
            raise NotImplementedError("SIFT nms_radius > 0: only None and 0 (one keypoint per pixel) are built")
        self._uncapped_cap = 8192

    def kernel_conf(self):
        c = self.conf
        mk = c["max_num_keypoints"]
        # the wrapper hands num_octaves to cv2 as nOctaveLayers
        return {"n_octave_layers": int(c["num_octaves"]), "contrast_threshold": float(c["detection_threshold"]),
                "edge_threshold": float(c["edge_threshold"]), "sigma": 1.6, "max_keypoints": int(mk) if mk else 0,
                "nms_radius": c["nms_radius"], "rootsift": bool(c["rootsift"])}

    def _forward(self, data):
        image = data["image"].float()
        if image.shape[1] != 1:
            raise NotImplementedError("SIFT takes gray images (conf['preprocessing']['grayscale'] = True)")
        kc = self.kernel_conf()
        cap = kc["max_keypoints"] if kc["max_keypoints"] > 0 else self._uncapped_cap
        out = ops.sift_forward(image, kc, cap)
        counts = out["counts"].cpu()  # ragged outputs: one host sync
        if int((counts[1] < 0).any()):
            raise RuntimeError("SIFT: more extrema than the per-image capacity of the kernel")
        if int((counts[1] > counts[0]).any()):
            self._uncapped_cap = cap = int(counts[1].max())
            out = ops.sift_forward(image, kc, cap)
            counts = out["counts"].cpu()
        n = [int(c) for c in counts[0]]
        B = image.shape[0]
        return {
            "keypoints": [out["keypoints"][b, : n[b]] for b in range(B)],
            "scores": [out["scores"][b, : n[b]] for b in range(B)],
            "descriptors": [out["descriptors"][b, : n[b]].t() for b in range(B)],
            "scales": [out["scales"][b, : n[b]] for b in range(B)],
            "oris": [out["oris"][b, : n[b]] for b in range(B)],
        }
