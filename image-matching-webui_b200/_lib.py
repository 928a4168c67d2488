"""ctypes binding of libimw_b200.so (include/imw_b200.h).  Fails loudly when the library is missing:
there is no CPU or PyTorch fallback in the product path."""
import ctypes as C
from pathlib import Path

import torch

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "lib" / "libimw_b200.so"
IMW_LG_MAX_LAYERS = 16
fp = C.POINTER(C.c_float)


class SPWeights(C.Structure):
    _fields_ = [("w", C.c_void_p * 12), ("b", C.c_void_p * 12), ("wp", C.c_void_p * 12)]


class SPConf(C.Structure):
    _fields_ = [("nms_radius", C.c_int), ("keypoint_threshold", C.c_float), ("max_keypoints", C.c_int),
                ("remove_borders", C.c_int), ("use_tensor_cores", C.c_int), ("fix_sampling", C.c_int)]


class LGBlock(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("qkv_w", "qkv_b", "out_w", "out_b", "ffn0_w", "ffn0_b", "ln_g", "ln_b", "ffn3_w", "ffn3_b")]


class LGLayer(C.Structure):
    _fields_ = [("self_blk", LGBlock), ("cross_blk", LGBlock)]


class LGWeights(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("input_dim", C.c_int), ("posenc_wr", C.c_void_p),
                ("token_w", C.c_void_p), ("token_b", C.c_void_p), ("final_w", C.c_void_p), ("final_b", C.c_void_p),
                ("match_w", C.c_void_p), ("match_b", C.c_void_p), ("layers", LGLayer * IMW_LG_MAX_LAYERS),
                ("input_proj_w", C.c_void_p), ("input_proj_b", C.c_void_p), ("has_lo_planes", C.c_int), ("posenc_dim", C.c_int)]


IMW_SG_MAX_LAYERS = 32


class SGLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("qkv_w", "qkv_b", "merge_w", "merge_b", "mlp0_w", "mlp0_b", "mlp1_w", "mlp1_b")] + \
               [("is_cross", C.c_int), ("pad_", C.c_int)]


class SGWeights(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("bin_score", C.c_float), ("kenc_w", C.c_void_p * 5), ("kenc_b", C.c_void_p * 5),
                ("final_w", C.c_void_p), ("final_b", C.c_void_p), ("layers", SGLayer * IMW_SG_MAX_LAYERS)]


class SGConf(C.Structure):
    _fields_ = [("sinkhorn_iterations", C.c_int), ("match_threshold", C.c_float), ("use_tensor_cores", C.c_int)]


ALIKED_FIELDS = ("b1c1_w b1c1_b b1c2_w b1c2_b b2c1_w b2c1_b b2c2_w b2c2_b b2ds_w b2ds_b "
                 "b3o1_w b3o1_b b3c1_w b3c1_b b3o2_w b3o2_b b3c2_w b3c2_b b3ds_w b3ds_b "
                 "b4o1_w b4o1_b b4c1_w b4c1_b b4o2_w b4o2_b b4c2_w b4c2_b b4ds_w b4ds_b "
                 "conv1_w conv2_w conv3_w conv4_w s0_w s2_w s4_w s6_w sd_off0_w sd_off0_b sd_off2_w sd_off2_b sd_sf_w sd_agg").split()


class AlikedWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ALIKED_FIELDS]


class AlikedConf(C.Structure):
    _fields_ = [("detection_threshold", C.c_float), ("max_num_keypoints", C.c_int), ("nms_radius", C.c_int)]


IMW_SIFT_MAX_TAPS = 64


class SiftConf(C.Structure):
    _fields_ = [("n_octave_layers", C.c_int), ("contrast_threshold", C.c_float), ("edge_threshold", C.c_float), ("sigma", C.c_double),
                ("max_keypoints", C.c_int), ("nms_radius", C.c_int), ("rootsift", C.c_int)]


class LoftrConv(C.Structure):
    _fields_ = [("w", C.c_void_p), ("b", C.c_void_p), ("cin", C.c_int), ("cout", C.c_int), ("ksize", C.c_int), ("stride", C.c_int)]


class LoftrBackbone(C.Structure):
    _fields_ = [("conv1_w", C.c_void_p), ("conv1_b", C.c_void_p), ("l1", LoftrConv * 4), ("l2", LoftrConv * 4), ("l2_down", LoftrConv),
                ("l3", LoftrConv * 4), ("l3_down", LoftrConv), ("l3_out", LoftrConv), ("l2_out", LoftrConv), ("l2_out2", LoftrConv * 2),
                ("l1_out", LoftrConv), ("l1_out2", LoftrConv * 2)]


class LoftrLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("qkv_w", "merge_w", "mlp0_w", "mlp2_w", "norm1_g", "norm1_b", "norm2_g", "norm2_b")] + \
               [("is_cross", C.c_int), ("pad_", C.c_int)]


class LoftrWeights(C.Structure):
    _fields_ = [("backbone", LoftrBackbone), ("pos_enc", C.c_void_p), ("n_coarse", C.c_int), ("n_fine", C.c_int),
                ("coarse", LoftrLayer * 8), ("fine", LoftrLayer * 2), ("down_proj_w", C.c_void_p), ("down_proj_b", C.c_void_p),
                ("merge_feat_w", C.c_void_p), ("merge_feat_b", C.c_void_p), ("has_f16_planes", C.c_int)]


class LoftrConf(C.Structure):
    _fields_ = [("match_threshold", C.c_float), ("temperature", C.c_float), ("border_rm", C.c_int), ("use_tensor_cores", C.c_int)]


class PreConf(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("grayscale", "resize_max", "force_resize", "width", "height", "dfactor")]


class LGConf(C.Structure):
    _fields_ = [("depth_confidence", C.c_float), ("width_confidence", C.c_float), ("filter_threshold", C.c_float),
                ("pruning_min_kpts", C.c_int), ("use_tensor_cores", C.c_int)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  The B200 engine has no CPU/PyTorch fallback.")
        L = C.CDLL(str(LIB_PATH))
        L.imw_last_error.restype = C.c_char_p
        L.imw_version.restype = C.c_int
        L.imw_launch_count.restype = C.c_ulonglong
        for name in ("imw_superpoint_workspace_bytes", "imw_lightglue_workspace_bytes", "imw_matcher_workspace_bytes",
                     "imw_superglue_workspace_bytes"):
            getattr(L, name).restype = C.c_size_t
        L.imw_superpoint_workspace_bytes.argtypes = [C.c_int] * 3
        L.imw_lightglue_workspace_bytes.argtypes = [C.c_int] * 2
        L.imw_matcher_workspace_bytes.argtypes = [C.c_int] * 2
        L.imw_superglue_workspace_bytes.argtypes = [C.c_int] * 2
        L.imw_aliked_workspace_bytes.restype = C.c_size_t
        L.imw_aliked_workspace_bytes.argtypes = [C.c_int] * 4
        L.imw_aliked_forward.restype = C.c_int
        L.imw_aliked_forward.argtypes = [C.POINTER(AlikedWeights), C.POINTER(AlikedConf), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_void_p]
        L.imw_sift_plan.restype = C.c_int
        L.imw_sift_plan.argtypes = [C.POINTER(SiftConf), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.imw_sift_workspace_bytes.restype = C.c_size_t
        L.imw_sift_workspace_bytes.argtypes = [C.POINTER(SiftConf), C.c_int, C.c_int, C.c_int]
        L.imw_sift_forward.restype = C.c_int
        L.imw_sift_forward.argtypes = [C.POINTER(SiftConf), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 8 + \
                                      [C.c_size_t, C.c_void_p]
        L.imw_loftr_workspace_bytes.restype = C.c_size_t
        L.imw_loftr_workspace_bytes.argtypes = [C.c_int] * 4
        L.imw_loftr_workspace_bytes_hw.restype = C.c_size_t
        L.imw_loftr_workspace_bytes_hw.argtypes = [C.c_int] * 6
        L.imw_loftr_forward_hw.restype = C.c_int
        L.imw_loftr_forward_hw.argtypes = [C.POINTER(LoftrWeights), C.POINTER(LoftrConf), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                           C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_int,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                           C.c_void_p]
        L.imw_loftr_forward.restype = C.c_int
        L.imw_loftr_forward.argtypes = [C.POINTER(LoftrWeights), C.POINTER(LoftrConf), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_void_p]
        vp = C.c_void_p
        L.imw_superpoint_forward.restype = C.c_int
        L.imw_superpoint_forward.argtypes = [C.POINTER(SPWeights), C.POINTER(SPConf), C.c_int, C.c_int, C.c_int, vp,
                                             C.c_int, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
        L.imw_lightglue_forward.restype = C.c_int
        L.imw_lightglue_forward.argtypes = [C.POINTER(LGWeights), C.POINTER(LGConf), C.c_int, C.c_int, vp, vp, vp, vp,
                                            vp, vp, vp, vp, C.c_size_t, vp]
        L.imw_lightglue_forward_so.restype = C.c_int
        L.imw_lightglue_forward_so.argtypes = [C.POINTER(LGWeights), C.POINTER(LGConf), C.c_int, C.c_int, vp, vp, vp, vp, vp, vp,
                                               vp, vp, vp, vp, C.c_size_t, vp]
        L.imw_superglue_forward.restype = C.c_int
        L.imw_superglue_forward.argtypes = [C.POINTER(SGWeights), C.POINTER(SGConf), C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                            vp, C.c_size_t, vp]
        L.imw_magsac.restype = C.c_int
        L.imw_magsac.argtypes = [C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_float, C.c_float, C.c_int, C.c_uint, vp, vp, vp, vp, vp]
        L.imw_nearest_neighbor.restype = C.c_int
        L.imw_nearest_neighbor.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, C.c_float, C.c_float, C.c_int, C.c_int, vp, vp,
                                           vp, C.c_size_t, vp]
        L.imw_dual_softmax.restype = C.c_int
        L.imw_dual_softmax.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, C.c_float, C.c_float, C.c_int, vp, vp, vp,
                                       C.c_size_t, vp]
        L.imw_debug_set_gemm_ablate.restype = C.c_int
        L.imw_debug_set_gemm_ablate.argtypes = [C.c_int]
        L.imw_debug_set_conv_pair.restype = C.c_int
        L.imw_debug_set_conv_pair.argtypes = [C.c_int]
        L.imw_debug_conv1ab_fused.restype = C.c_int
        L.imw_debug_conv1ab_fused.argtypes = [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
        L.imw_debug_gemm_tf32.restype = C.c_int
        L.imw_debug_gemm_tf32.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
        L.imw_debug_gemm_fp32.restype = C.c_int
        L.imw_debug_gemm_fp32.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
        L.imw_debug_conv3x3.restype = C.c_int
        L.imw_debug_conv3x3.argtypes = [vp] * 4 + [C.c_int] * 7 + [vp]
        L.imw_debug_conv3x3_tc_planes.restype = C.c_int
        L.imw_debug_conv3x3_tc_planes.argtypes = [vp] * 4 + [C.c_int] * 7 + [vp]
        L.imw_debug_attention.restype = C.c_int
        L.imw_debug_attention.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, vp, vp, C.c_size_t, vp]
        L.imw_debug_conv3x3_tc.restype = C.c_int
        L.imw_debug_conv3x3_tc.argtypes = [vp] * 4 + [C.c_int] * 7 + [vp, C.c_size_t, vp]
        L.imw_preprocess_plan.restype = C.c_int
        L.imw_preprocess_plan.argtypes = [C.POINTER(PreConf), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                          C.POINTER(C.c_int), C.POINTER(C.c_size_t)]
        L.imw_preprocess_workspace_bytes.restype = C.c_size_t
        L.imw_preprocess_workspace_bytes.argtypes = [C.POINTER(PreConf), C.c_int, C.c_int, C.c_int, C.c_int]
        L.imw_preprocess.restype = C.c_int
        L.imw_preprocess.argtypes = [C.POINTER(PreConf), C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_size_t, vp]
        L.imw_gather_matches.restype = C.c_int
        L.imw_gather_matches.argtypes = [C.c_int, C.c_int] + [vp] * 12
        L.imw_rescale_keypoints.restype = C.c_int
        L.imw_rescale_keypoints.argtypes = [C.c_int, C.c_int, vp, vp, vp, vp, vp]
        L.imw_quantize_keypoints.restype = C.c_int
        L.imw_quantize_keypoints.argtypes = [C.c_int, C.c_int, vp, vp, C.c_float, vp, vp, vp]
        L.imw_nearest_point.restype = C.c_int
        L.imw_nearest_point.argtypes = [C.c_int, vp, C.c_int, vp, C.c_float, vp, vp]
        L.imw_unique_matches_workspace_bytes.restype = C.c_size_t
        L.imw_unique_matches_workspace_bytes.argtypes = [C.c_int, C.c_int]
        L.imw_unique_matches.restype = C.c_int
        L.imw_unique_matches.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
        L.imw_prof_begin.restype = C.c_int
        L.imw_prof_begin.argtypes = [vp]
        L.imw_prof_end.restype = C.c_longlong
        L.imw_prof_end.argtypes = [C.c_char_p, C.c_size_t]
        _lib = L
    return _lib


class launch_profile:
    """with launch_profile(device) as p: step()  ->  p.sites = [(site, launches, total_ms)] sorted by time, p.total_ms.
    Library-side CUDA events behind every launch on the current stream (include/imw_b200.h: imw_prof_begin/end)."""

    def __init__(self, device=None):
        self.device, self.sites, self.total_ms, self.launches = device, [], 0.0, 0

    def __enter__(self):
        check(lib().imw_prof_begin(stream_ptr(self.device)))
        return self

    def __exit__(self, *exc):
        buf = C.create_string_buffer(1 << 18)
        n = lib().imw_prof_end(buf, len(buf))
        if n < 0:
            check(int(n))
        self.launches = int(n)
        for line in buf.value.decode().splitlines():
            site, cnt, ms = line.rsplit("\t", 2)
            self.sites.append((site, int(cnt), float(ms)))
        self.sites.sort(key=lambda t: -t[2])
        self.total_ms = sum(t[2] for t in self.sites)
        return False

    def find(self, *needles):
        """Sites whose signature contains every needle (kernel family / template arguments)."""
        return [t for t in self.sites if all(n in t[0] for n in needles)]


class ImwError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = lib().imw_last_error().decode()
        if rc == -1:  # IMW_ERR_ARG: the reference raises ValueError for bad conf values
            raise ValueError(msg)
        raise ImwError(f"imw error {rc}: {msg}")


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: tensor is on {t.device}; the B200 engine only runs on CUDA devices "
                           "(no CPU fallback)")


class WorkspaceCache:
    """One growing scratch tensor per (device, tag): no allocation in the steady state."""

    def __init__(self):
        self.bufs = {}

    def get(self, device, nbytes, tag="ws"):
        key = (str(device), tag)
        buf = self.bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
            self.bufs[key] = buf
        return buf


workspaces = WorkspaceCache()
