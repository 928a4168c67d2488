"""Thin torch-tensor front-ends of the C ABI (include/imw_b200.h): allocate outputs + workspace with
torch (plumbing), pass raw pointers and the current CUDA stream to the library."""
import ctypes as C

import torch

from . import _lib as L


# ---------------------------------------------------------------------------------------------------
# pre- / post-processing of the hloc drivers
# ---------------------------------------------------------------------------------------------------
PRE_DEFAULT = {"grayscale": True, "resize_max": 1024, "dfactor": 8, "force_resize": False, "width": 320, "height": 240}


def pre_conf_struct(conf):
    c = {**PRE_DEFAULT, **{k: v for k, v in (conf or {}).items() if k in PRE_DEFAULT}}
    return L.PreConf(int(bool(c["grayscale"])), int(c["resize_max"] or 0), int(bool(c["force_resize"])), int(c["width"]), int(c["height"]),
                     int(c["dfactor"] or 1))


def preprocess_plan(conf, height, width, channels):
    """(out_channels, out_height, out_width) of ops.preprocess for frames of this size (host arithmetic only)."""
    oc, oh, ow, wsb = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
    pc = pre_conf_struct(conf)
    L.check(L.lib().imw_preprocess_plan(C.byref(pc), int(height), int(width), int(channels), C.byref(oc), C.byref(oh), C.byref(ow), C.byref(wsb)))
    return oc.value, oh.value, ow.value


def preprocess(images_u8, conf, out=None):
    """images_u8 [B,H,W] or [B,H,W,3] uint8 CUDA (decoded frames) -> fp32 [B,C,H',W'] in [0,1], exactly the tensor the
    reference's extract() feeds the extractor (extract_features.py:120-162)."""
    L.require_cuda(images_u8, "preprocess(images)")
    assert images_u8.dtype == torch.uint8 and images_u8.dim() in (3, 4)
    x = images_u8.contiguous()
    B, H, W = x.shape[:3]
    Cc = x.shape[3] if x.dim() == 4 else 1
    oc, oh, ow = preprocess_plan(conf, H, W, Cc)
    dev = x.device
    if out is None:
        out = torch.empty(B, oc, oh, ow, device=dev)
    assert out.shape == (B, oc, oh, ow) and out.is_contiguous()
    pc = pre_conf_struct(conf)
    lib = L.lib()
    ws = L.workspaces.get(dev, lib.imw_preprocess_workspace_bytes(C.byref(pc), B, H, W, Cc), "pre")
    with torch.cuda.device(dev):
        L.check(lib.imw_preprocess(C.byref(pc), B, H, W, Cc, L.ptr(x), L.ptr(out), L.ptr(ws), ws.numel(), L.stream_ptr(dev)))
    return out


def gather_matches(keypoints, matches, counts, scores=None, scales=None, out=None):
    """Device-side match_features.py:244-257 for a batch: keypoints [2P,cap,2], matches [2P,cap] int32 (matches0 in even
    slots), counts [2P], scores [2P,cap] (optional), scales [2P,2] fp32 = original_size / size (optional).
    Returns (mkpts0 [P,cap,2], mkpts1 [P,cap,2], mcount [P]) or, with `out` (dict of preallocated buffers incl. the
    *_orig / mconf ones), fills and returns it."""
    L.require_cuda(keypoints, "gather_matches(keypoints)")
    S, cap, _ = keypoints.shape
    P, dev = S // 2, keypoints.device
    assert matches.shape == (S, cap) and matches.dtype == torch.int32 and counts.dtype == torch.int32 and counts.numel() == S
    simple = out is None
    if out is None:
        out = {"mkpts0": torch.empty(P, cap, 2, device=dev), "mkpts1": torch.empty(P, cap, 2, device=dev),
               "mcount": torch.empty(P, dtype=torch.int32, device=dev)}
    with torch.cuda.device(dev):
        L.check(L.lib().imw_gather_matches(P, cap, L.ptr(keypoints.contiguous()), L.ptr(matches.contiguous()),
                                           L.ptr(scores.contiguous() if scores is not None else None), L.ptr(counts.contiguous()),
                                           L.ptr(scales.contiguous() if scales is not None else None), L.ptr(out["mkpts0"]), L.ptr(out["mkpts1"]),
                                           L.ptr(out.get("mkpts0_orig")), L.ptr(out.get("mkpts1_orig")), L.ptr(out.get("mconf")),
                                           L.ptr(out["mcount"]), L.stream_ptr(dev)))
    return (out["mkpts0"], out["mkpts1"], out["mcount"]) if simple else out


def quantize_keypoints(keypoints, cell_size, counts=None):
    """`to_cpts` (match_dense.py:37-40): keypoints [S,cap,2] fp32 -> (cells [S,cap,2] int32, coords [S,cap,2] fp32)."""
    L.require_cuda(keypoints, "quantize_keypoints(keypoints)")
    S, cap, _ = keypoints.shape
    dev = keypoints.device
    cells = torch.zeros(S, cap, 2, dtype=torch.int32, device=dev)
    coords = torch.zeros(S, cap, 2, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().imw_quantize_keypoints(S, cap, L.ptr(keypoints.contiguous()), L.ptr(counts), float(cell_size), L.ptr(cells), L.ptr(coords),
                                               L.stream_ptr(dev)))
    return cells, coords


def nearest_point(query, points, max_error):
    """`assign_keypoints(update=False)` (match_dense.py:52-59): query [K,2], points [M,2] fp32 -> ids [K] int32 (-1 beyond max_error)."""
    L.require_cuda(query, "nearest_point(query)")
    K, M = query.shape[0], points.shape[0]
    ids = torch.full((K,), -1, dtype=torch.int32, device=query.device)
    if K == 0 or M == 0:
        return ids
    with torch.cuda.device(query.device):
        L.check(L.lib().imw_nearest_point(K, L.ptr(query.float().contiguous()), M, L.ptr(points.float().contiguous()), float(max_error), L.ptr(ids),
                                          L.stream_ptr(query.device)))
    return ids


def unique_matches(ids0, ids1, scores, counts, id_cap):
    """`kpids_to_matches0` (match_dense.py:99-121) for a batch: ids0/ids1 [P,cap] int32, scores [P,cap] fp32, counts [P] ->
    (matches0 [P,id_cap] int32, scores0 [P,id_cap] fp16, n_kps0 [P] int32)."""
    L.require_cuda(ids0, "unique_matches(ids0)")
    P, cap = ids0.shape
    dev = ids0.device
    m0 = torch.empty(P, id_cap, dtype=torch.int32, device=dev)
    s0 = torch.empty(P, id_cap, dtype=torch.float16, device=dev)
    nk = torch.empty(P, dtype=torch.int32, device=dev)
    lib = L.lib()
    ws = L.workspaces.get(dev, lib.imw_unique_matches_workspace_bytes(P, id_cap), "dense_agg")
    with torch.cuda.device(dev):
        L.check(lib.imw_unique_matches(P, cap, int(id_cap), L.ptr(ids0.contiguous()), L.ptr(ids1.contiguous()), L.ptr(scores.float().contiguous()),
                                       L.ptr(counts.contiguous()), L.ptr(m0), L.ptr(s0), L.ptr(nk), L.ptr(ws), ws.numel(), L.stream_ptr(dev)))
    return m0, s0, nk


def rescale_keypoints(keypoints, scales, counts=None, out=None):
    """keypoints [S,cap,2] fp32, scales [S,2] fp32 -> (k + 0.5) * s - 0.5 (match_features.py:251-254)."""
    L.require_cuda(keypoints, "rescale_keypoints(keypoints)")
    S, cap, _ = keypoints.shape
    dev = keypoints.device
    if out is None:
        out = torch.empty_like(keypoints)
    with torch.cuda.device(dev):
        L.check(L.lib().imw_rescale_keypoints(S, cap, L.ptr(keypoints.contiguous()), L.ptr(counts), L.ptr(scales.contiguous()), L.ptr(out),
                                              L.stream_ptr(dev)))
    return out


# ---------------------------------------------------------------------------------------------------
# SuperPoint
# ---------------------------------------------------------------------------------------------------
SP_LAYERS = ["conv1a", "conv1b", "conv2a", "conv2b", "conv3a", "conv3b", "conv4a", "conv4b", "convPa", "convPb",
             "convDa", "convDb"]


def sp_pack_weights(state_dict):
    """Re-lay the reference's Conv2d parameters ([Cout,Cin,kh,kw]) for the kernels:
    3x3 -> [ky*3+kx][Cin][Cout]; 1x1 -> [Cout][Cin].  Returns {name: tensor} (CPU fp32)."""
    out = {}
    for name in SP_LAYERS:
        w = state_dict[name + ".weight"].float()
        if w.shape[-1] == 3:
            w = w.permute(2, 3, 1, 0).reshape(9, w.shape[1], w.shape[0])
        else:
            w = w.reshape(w.shape[0], w.shape[1])
        out[name + "_w"] = w.contiguous()
        out[name + "_b"] = state_dict[name + ".bias"].float().contiguous()
        if name in SP_TC_LAYERS:  # [2 planes][tap][Cout][Cin] fp16, w = hi + lo * 2^-11 (tcgen05 split-precision path)
            wt = state_dict[name + ".weight"].float().permute(2, 3, 0, 1).reshape(9, w.shape[2], w.shape[1]).contiguous()
            out[name + "_wp"] = split_f16_planes(wt)
        elif name in ("convPb", "convDb"):  # 1x1 heads on the same path: [2][1][Cout_p][Cin], the 65 detector outputs padded to 128
            co, ci = w.shape
            cop = (co + 127) // 128 * 128
            wt = torch.zeros(1, cop, ci); wt[0, :co] = w
            out[name + "_wp"] = split_f16_planes(wt)
            bp = torch.zeros(cop); bp[:co] = out[name + "_b"]
            out[name + "_b"] = bp
    return out


SP_TC_LAYERS = ["conv1b", "conv2a", "conv2b", "conv3a", "conv3b", "conv4a", "conv4b", "convPa", "convDa"]


PLANE_LO_SCALE = 2048.0   # csrc/split_planes.cuh


def split_f16_planes(x):
    """fp32 -> [2, ...] fp16 planes (hi, lo * 2^11) with x == hi + lo * 2^-11 to 2^-22 relative (csrc/split_planes.cuh)."""
    x = x.float().clamp(-65504.0, 65504.0)
    hi = x.half()
    lo = ((x - hi.float()) * PLANE_LO_SCALE).half()
    return torch.stack([hi, lo]).contiguous()


def sp_weights_struct(bufs):
    s = L.SPWeights()
    for i, name in enumerate(SP_LAYERS):
        s.w[i] = bufs[name + "_w"].data_ptr()
        s.b[i] = bufs[name + "_b"].data_ptr()
        s.wp[i] = bufs[name + "_wp"].data_ptr() if (name + "_wp") in bufs else None
    return s


def superpoint_forward(bufs, image, conf, cap, out=None, want_dense=False):
    """image [B,1,H,W] fp32 CUDA.  Returns dict of batch buffers: keypoints [B,cap,2], scores [B,cap],
    descriptors [B,cap,256], counts [2,B] int32 (written, total)."""
    L.require_cuda(image, "superpoint_forward(image)")
    assert image.dim() == 4 and image.shape[1] == 1 and image.dtype == torch.float32
    image = image.contiguous()
    B, _, H, W = image.shape
    dev = image.device
    if out is None:
        out = {
            "keypoints": torch.empty(B, cap, 2, device=dev),
            "scores": torch.empty(B, cap, device=dev),
            "descriptors": torch.empty(B, cap, 256, device=dev),
            "counts": torch.empty(2, B, dtype=torch.int32, device=dev),
        }
    dense = torch.empty(B, H, W, device=dev) if want_dense else None
    lib = L.lib()
    nbytes = lib.imw_superpoint_workspace_bytes(B, H, W)
    ws = L.workspaces.get(dev, nbytes, "sp")
    use_tc = bool(conf.get("tensor_cores", True)) and W % 16 == 0
    c = L.SPConf(int(conf["nms_radius"]), float(conf["keypoint_threshold"]), int(conf["max_keypoints"]),
                 int(conf["remove_borders"]), int(use_tc), int(bool(conf.get("fix_sampling", False))))
    wstruct = sp_weights_struct(bufs)
    with torch.cuda.device(dev):
        rc = lib.imw_superpoint_forward(C.byref(wstruct), C.byref(c), B, H, W, L.ptr(image), cap, L.ptr(out["keypoints"]),
                                        L.ptr(out["scores"]), L.ptr(out["descriptors"]), L.ptr(out["counts"]), L.ptr(dense),
                                        L.ptr(ws), ws.numel(), L.stream_ptr(dev))
    L.check(rc)
    if want_dense:
        out["dense_scores"] = dense
    return out


# ---------------------------------------------------------------------------------------------------
# LightGlue
# ---------------------------------------------------------------------------------------------------
def lg_pack_weights(sd, n_layers=9, heads=4):
    """Flat reference state dict -> kernel layout (CPU fp32 tensors).
    Wqkv rows are permuted from [head][dim][q,k,v] (lightglue.py:166) to [q|k|v][head][dim];
    cross to_qk / to_v are stacked to one [512,256] projection."""
    out = {"posenc_wr": sd["posenc.Wr.weight"].float().contiguous()}
    d = sd["transformers.0.self_attn.out_proj.weight"].shape[0]
    hd = d // heads
    for i in range(n_layers):
        p = f"transformers.{i}.self_attn."
        w = sd[p + "Wqkv.weight"].float().view(heads, hd, 3, d).permute(2, 0, 1, 3).reshape(3 * d, d)
        b = sd[p + "Wqkv.bias"].float().view(heads, hd, 3).permute(2, 0, 1).reshape(3 * d)
        out[f"l{i}.self.qkv_w"], out[f"l{i}.self.qkv_b"] = w.contiguous(), b.contiguous()
        out[f"l{i}.self.out_w"], out[f"l{i}.self.out_b"] = sd[p + "out_proj.weight"].float(), sd[p + "out_proj.bias"].float()
        c = f"transformers.{i}.cross_attn."
        out[f"l{i}.cross.qkv_w"] = torch.cat([sd[c + "to_qk.weight"], sd[c + "to_v.weight"]], 0).float().contiguous()
        out[f"l{i}.cross.qkv_b"] = torch.cat([sd[c + "to_qk.bias"], sd[c + "to_v.bias"]], 0).float().contiguous()
        out[f"l{i}.cross.out_w"], out[f"l{i}.cross.out_b"] = sd[c + "to_out.weight"].float(), sd[c + "to_out.bias"].float()
        for blk, pre in (("self", p), ("cross", c)):
            out[f"l{i}.{blk}.ffn0_w"], out[f"l{i}.{blk}.ffn0_b"] = sd[pre + "ffn.0.weight"].float(), sd[pre + "ffn.0.bias"].float()
            out[f"l{i}.{blk}.ln_g"], out[f"l{i}.{blk}.ln_b"] = sd[pre + "ffn.1.weight"].float(), sd[pre + "ffn.1.bias"].float()
            out[f"l{i}.{blk}.ffn3_w"], out[f"l{i}.{blk}.ffn3_b"] = sd[pre + "ffn.3.weight"].float(), sd[pre + "ffn.3.bias"].float()
    out["token_w"] = torch.stack([sd[f"token_confidence.{i}.token.0.weight"].float().reshape(d) for i in range(n_layers - 1)])
    out["token_b"] = torch.stack([sd[f"token_confidence.{i}.token.0.bias"].float().reshape(()) for i in range(n_layers - 1)])
    out["final_w"] = torch.stack([sd[f"log_assignment.{i}.final_proj.weight"].float() for i in range(n_layers)])
    out["final_b"] = torch.stack([sd[f"log_assignment.{i}.final_proj.bias"].float() for i in range(n_layers)])
    out["match_w"] = torch.stack([sd[f"log_assignment.{i}.matchability.weight"].float().reshape(d) for i in range(n_layers)])
    out["match_b"] = torch.stack([sd[f"log_assignment.{i}.matchability.bias"].float().reshape(()) for i in range(n_layers)])
    if "input_proj.weight" in sd:  # Linear(input_dim -> 256) for 128-d features (lightglue.py:392-395)
        out["input_proj_w"], out["input_proj_b"] = sd["input_proj.weight"].float(), sd["input_proj.bias"].float()
    # split-fp16 tcgen05 GEMM: every linear weight matrix carries its two fp16 planes behind it ([W fp32 ; hi | lo]: the same
    # bytes as a second fp32 matrix), so the kernel splits activations only.  The fp32 CUDA-core path reads the first N rows.
    for k in list(out):
        if k.endswith(("qkv_w", "out_w", "ffn0_w", "ffn3_w")) or k == "input_proj_w":
            out[k] = with_f16_planes(out[k])
    return {k: v.contiguous() for k, v in out.items()}


def tf32_lo(w):
    """w - trunc_tf32(w): what kind::tf32 drops when it ignores the 13 low mantissa bits of an fp32 operand"""
    w = w.float().contiguous()
    hi = (w.view(torch.int32) & -8192).view(torch.float32)
    return w - hi


def with_tf32_lo_plane(w):
    return torch.cat([w.float(), tf32_lo(w)], 0).contiguous()


def f16_planes(w):
    """csrc/split_planes.cuh on the host: hi = fp16(w), lo = fp16((w - hi) * 2^11) -> [2, N, K] float16"""
    w = w.float().clamp(-65504.0, 65504.0).contiguous()
    hi = w.half()
    lo = ((w - hi.float()) * 2048.0).half()
    return torch.stack([hi, lo]).contiguous()


def with_f16_planes(w):
    """[N, K] fp32 -> [2N, K] fp32 storage: the matrix followed by its split-fp16 planes (2 * N * K halves = N * K floats)"""
    n, k = w.shape
    return torch.cat([w.float(), f16_planes(w).view(torch.float32).reshape(n, k)], 0).contiguous()


def lg_weights_struct(bufs, n_layers=9):
    s = L.LGWeights()
    s.n_layers, s.input_dim = n_layers, 256
    s.has_lo_planes = 2
    s.posenc_dim = bufs["posenc_wr"].shape[1]
    if "input_proj_w" in bufs:
        s.input_dim = bufs["input_proj_w"].shape[1]
        s.input_proj_w, s.input_proj_b = bufs["input_proj_w"].data_ptr(), bufs["input_proj_b"].data_ptr()
    s.posenc_wr = bufs["posenc_wr"].data_ptr()
    for k in ("token_w", "token_b", "final_w", "final_b", "match_w", "match_b"):
        setattr(s, k, bufs[k].data_ptr())
    for i in range(n_layers):
        for blk, dst in (("self", s.layers[i].self_blk), ("cross", s.layers[i].cross_blk)):
            for f in ("qkv_w", "qkv_b", "out_w", "out_b", "ffn0_w", "ffn0_b", "ln_g", "ln_b", "ffn3_w", "ffn3_b"):
                setattr(dst, f, bufs[f"l{i}.{blk}.{f}"].data_ptr())
    return s


def lightglue_forward(bufs, n_layers, keypoints, descriptors, counts, conf, out=None, scales=None, oris=None):
    """keypoints [2P,cap,2], descriptors [2P,cap,input_dim], counts [2P] int32 (all CUDA, contiguous); scales / oris [2P,cap]
    for the add_scale_ori features (posenc over (x, y, scale, orientation), lightglue.py:500-506).
    Returns dict: matches [2P,cap] int32, scores [2P,cap], stop [P] int32, prune [2P,cap] int32."""
    L.require_cuda(keypoints, "lightglue_forward(keypoints)")
    S, cap, _ = keypoints.shape
    in_dim = bufs["input_proj_w"].shape[1] if "input_proj_w" in bufs else 256
    assert bufs["l0.self.out_w"].shape[0] == 512, "lg_pack_weights output expected (weights followed by their split-fp16 planes)"
    assert S % 2 == 0 and descriptors.shape == (S, cap, in_dim) and counts.numel() == S and counts.dtype == torch.int32
    assert keypoints.is_contiguous() and descriptors.is_contiguous() and counts.is_contiguous()
    P, dev = S // 2, keypoints.device
    if out is None:
        out = {
            "matches": torch.empty(S, cap, dtype=torch.int32, device=dev),
            "scores": torch.empty(S, cap, device=dev),
            "stop": torch.empty(P, dtype=torch.int32, device=dev),
            "prune": torch.empty(S, cap, dtype=torch.int32, device=dev),
        }
    lib = L.lib()
    ws = L.workspaces.get(dev, lib.imw_lightglue_workspace_bytes(P, cap), "lg")
    c = L.LGConf(float(conf["depth_confidence"]), float(conf["width_confidence"]), float(conf["filter_threshold"]),
                 int(conf["pruning_min_kpts"]), int(conf.get("use_tensor_cores", 1)) if cap % 128 == 0 else 0)
    wstruct = lg_weights_struct(bufs, n_layers)
    with torch.cuda.device(dev):
        rc = lib.imw_lightglue_forward_so(C.byref(wstruct), C.byref(c), P, cap, L.ptr(keypoints),
                                          L.ptr(scales.contiguous() if scales is not None else None), L.ptr(oris.contiguous() if oris is not None else None),
                                          L.ptr(descriptors), L.ptr(counts), L.ptr(out["matches"]), L.ptr(out["scores"]), L.ptr(out["stop"]),
                                          L.ptr(out["prune"]), L.ptr(ws), ws.numel(), L.stream_ptr(dev))
    L.check(rc)
    return out


# ---------------------------------------------------------------------------------------------------
# SuperGlue
# ---------------------------------------------------------------------------------------------------
def _fold_bn(w, b, sd, p):
    """Conv1d(k=1) followed by BatchNorm1d in eval mode -> one affine layer."""
    g = sd[p + "weight"] / torch.sqrt(sd[p + "running_var"] + 1e-5)
    return w * g[:, None], (b - sd[p + "running_mean"]) * g + sd[p + "bias"]


def sg_pack_weights(sd, layer_names=("self", "cross") * 9, heads=4):
    """Reference state dict (superglue.py) -> kernel layout (CPU fp32): BN folded, attention projections permuted
    from channel order d*heads+h (superglue.py:106 `view(b, dim, heads, N)`) to h*dim+d, kenc layer 0 padded 3 -> 16."""
    out = {}
    for l in range(5):
        w, b = sd[f"kenc.encoder.{3 * l}.weight"][:, :, 0].float(), sd[f"kenc.encoder.{3 * l}.bias"].float()
        if l < 4:
            w, b = _fold_bn(w, b, sd, f"kenc.encoder.{3 * l + 1}.")
        if l == 0:
            w = torch.cat([w, torch.zeros(w.shape[0], 13)], 1)
        out[f"kenc_w{l}"], out[f"kenc_b{l}"] = w.contiguous(), b.contiguous()
    d = sd["final_proj.weight"].shape[0]
    hd = d // heads
    perm_rows = lambda w: w.view(hd, heads, -1).permute(1, 0, 2).reshape(d, -1)
    for i, _ in enumerate(layer_names):
        p = f"gnn.layers.{i}."
        ws = [perm_rows(sd[p + f"attn.proj.{j}.weight"][:, :, 0].float()) for j in range(3)]
        bs = [sd[p + f"attn.proj.{j}.bias"].float().view(hd, heads).t().reshape(d) for j in range(3)]
        out[f"l{i}.qkv_w"], out[f"l{i}.qkv_b"] = torch.cat(ws, 0).contiguous(), torch.cat(bs, 0).contiguous()
        mw = sd[p + "attn.merge.weight"][:, :, 0].float()
        out[f"l{i}.merge_w"] = mw.view(d, hd, heads).permute(0, 2, 1).reshape(d, d).contiguous()
        out[f"l{i}.merge_b"] = sd[p + "attn.merge.bias"].float().contiguous()
        w0, b0 = _fold_bn(sd[p + "mlp.0.weight"][:, :, 0].float(), sd[p + "mlp.0.bias"].float(), sd, p + "mlp.1.")
        out[f"l{i}.mlp0_w"], out[f"l{i}.mlp0_b"] = w0.contiguous(), b0.contiguous()
        out[f"l{i}.mlp1_w"], out[f"l{i}.mlp1_b"] = sd[p + "mlp.3.weight"][:, :, 0].float().contiguous(), sd[p + "mlp.3.bias"].float().contiguous()
    out["final_w"], out["final_b"] = sd["final_proj.weight"][:, :, 0].float().contiguous(), sd["final_proj.bias"].float().contiguous()
    return out


def sg_weights_struct(bufs, bin_score, layer_names=("self", "cross") * 9):
    s = L.SGWeights()
    s.n_layers, s.bin_score = len(layer_names), float(bin_score)
    for l in range(5):
        s.kenc_w[l], s.kenc_b[l] = bufs[f"kenc_w{l}"].data_ptr(), bufs[f"kenc_b{l}"].data_ptr()
    s.final_w, s.final_b = bufs["final_w"].data_ptr(), bufs["final_b"].data_ptr()
    for i, name in enumerate(layer_names):
        for f in ("qkv_w", "qkv_b", "merge_w", "merge_b", "mlp0_w", "mlp0_b", "mlp1_w", "mlp1_b"):
            setattr(s.layers[i], f, bufs[f"l{i}.{f}"].data_ptr())
        s.layers[i].is_cross = int(name == "cross")
    return s


def superglue_forward(bufs, bin_score, keypoints, scores, descriptors, counts, image_wh, conf):
    """keypoints [2P,cap,2], scores [2P,cap], descriptors [2P,cap,256], counts [2P] int32, image_wh [2P,2] int32.
    Returns matches [2P,cap] int32, matching_scores [2P,cap]."""
    L.require_cuda(keypoints, "superglue_forward(keypoints)")
    S, cap, _ = keypoints.shape
    assert S % 2 == 0 and descriptors.shape == (S, cap, 256) and counts.dtype == torch.int32 and image_wh.dtype == torch.int32
    dev = keypoints.device
    matches = torch.empty(S, cap, dtype=torch.int32, device=dev)
    mscores = torch.empty(S, cap, device=dev)
    lib = L.lib()
    ws = L.workspaces.get(dev, lib.imw_superglue_workspace_bytes(S // 2, cap), "sg")
    c = L.SGConf(int(conf["sinkhorn_iterations"]), float(conf["match_threshold"]),
                 int(conf.get("use_tensor_cores", 1)) if cap % 128 == 0 else 0)
    wstruct = sg_weights_struct(bufs, bin_score)
    with torch.cuda.device(dev):
        rc = lib.imw_superglue_forward(C.byref(wstruct), C.byref(c), S // 2, cap, L.ptr(keypoints.contiguous()), L.ptr(scores.contiguous()),
                                       L.ptr(descriptors.contiguous()), L.ptr(counts), L.ptr(image_wh.contiguous()), L.ptr(matches),
                                       L.ptr(mscores), L.ptr(ws), ws.numel(), L.stream_ptr(dev))
    L.check(rc)
    return matches, mscores


# ---------------------------------------------------------------------------------------------------
# ALIKED
# ---------------------------------------------------------------------------------------------------
def aliked_pack_weights(sd):
    """Reference aliked-n16 state dict (lightglue/aliked.py naming) -> kernel layout (CPU fp32 tensors keyed by the
    imw_aliked_weights field names): BatchNorm folded, 3x3 kernels as [tap][Cin][Cout], 1x1 kernels as [Cin][Cout]."""
    f = lambda k: sd[k].float()

    def fold(wkey, bn):
        w = f(wkey)
        g = f(bn + "weight") / torch.sqrt(f(bn + "running_var") + 1e-5)
        return w * g[:, None, None, None], f(bn + "bias") - f(bn + "running_mean") * g

    def taps(w, cin_pad=None, cout_pad=None):  # [Co][Ci][3][3] -> [9][Ci_p][Co_p]
        co, ci = w.shape[:2]
        t = torch.zeros(9, cin_pad or ci, cout_pad or co)
        t[:, :ci, :co] = w.permute(2, 3, 1, 0).reshape(9, ci, co)
        return t.contiguous()

    def padv(b, n):
        o = torch.zeros(n); o[: len(b)] = b
        return o

    out = {}
    w, b = fold("block1.conv1.weight", "block1.bn1."); out["b1c1_w"], out["b1c1_b"] = taps(w, cin_pad=4), b
    w, b = fold("block1.conv2.weight", "block1.bn2."); out["b1c2_w"], out["b1c2_b"] = taps(w), b
    w, b = fold("block2.conv1.weight", "block2.bn1."); out["b2c1_w"], out["b2c1_b"] = taps(w), b
    w, b = fold("block2.conv2.weight", "block2.bn2."); out["b2c2_w"], out["b2c2_b"] = taps(w), b
    for i in (2, 3, 4):
        out[f"b{i}ds_w"] = f(f"block{i}.downsample.weight")[:, :, 0, 0].t().contiguous()
        out[f"b{i}ds_b"] = f(f"block{i}.downsample.bias")
    for i in (3, 4):
        for j in (1, 2):
            out[f"b{i}o{j}_w"] = taps(f(f"block{i}.conv{j}.offset_conv.weight"), cout_pad=24)
            out[f"b{i}o{j}_b"] = padv(f(f"block{i}.conv{j}.offset_conv.bias"), 24)
            w, b = fold(f"block{i}.conv{j}.regular_conv.weight", f"block{i}.bn{j}.")
            out[f"b{i}c{j}_w"], out[f"b{i}c{j}_b"] = taps(w), b
    for i in (1, 2, 3, 4):
        out[f"conv{i}_w"] = f(f"conv{i}.weight")[:, :, 0, 0].t().contiguous()
    out["s0_w"] = f("score_head.0.weight")[:, :, 0, 0].t().contiguous()
    out["s2_w"], out["s4_w"], out["s6_w"] = taps(f("score_head.2.weight")), taps(f("score_head.4.weight")), taps(f("score_head.6.weight"))
    out["sd_off0_w"], out["sd_off0_b"] = taps(f("desc_head.offset_conv.0.weight")), f("desc_head.offset_conv.0.bias")
    out["sd_off2_w"], out["sd_off2_b"] = f("desc_head.offset_conv.2.weight")[:, :, 0, 0].t().contiguous(), f("desc_head.offset_conv.2.bias")
    out["sd_sf_w"] = f("desc_head.sf_conv.weight")[:, :, 0, 0].t().contiguous()
    out["sd_agg"] = f("desc_head.agg_weights").contiguous()
    assert set(out) == set(L.ALIKED_FIELDS)
    return {k: v.contiguous() for k, v in out.items()}


def aliked_forward(bufs, image, conf, cap, debug=False):
    """image [B,1|3,H,W] fp32 CUDA in [0,1].  Returns batch buffers: keypoints [B,cap,2], scores [B,cap],
    descriptors [B,cap,128], counts [2,B] int32 (written, total) (+ score_map / feature_map with debug)."""
    L.require_cuda(image, "aliked_forward(image)")
    assert image.dim() == 4 and image.shape[1] in (1, 3) and image.dtype == torch.float32
    image = image.contiguous()
    B, Cc, H, W = image.shape
    dev = image.device
    out = {"keypoints": torch.empty(B, cap, 2, device=dev), "scores": torch.empty(B, cap, device=dev),
           "descriptors": torch.empty(B, cap, 128, device=dev), "counts": torch.empty(2, B, dtype=torch.int32, device=dev)}
    smap = torch.empty(B, H, W, device=dev) if debug else None
    fmap = torch.empty(B, H, W, 128, device=dev) if debug else None
    lib = L.lib()
    ws = L.workspaces.get(dev, lib.imw_aliked_workspace_bytes(B, H, W, cap), "aliked")
    c = L.AlikedConf(float(conf["detection_threshold"]), int(conf["max_num_keypoints"]), int(conf["nms_radius"]))
    wstruct = L.AlikedWeights(**{k: bufs[k].data_ptr() for k in L.ALIKED_FIELDS})
    with torch.cuda.device(dev):
        rc = lib.imw_aliked_forward(C.byref(wstruct), C.byref(c), B, Cc, H, W, L.ptr(image), cap, L.ptr(out["keypoints"]), L.ptr(out["scores"]),
                                    L.ptr(out["descriptors"]), L.ptr(out["counts"]), L.ptr(smap), L.ptr(fmap), L.ptr(ws), ws.numel(),
                                    L.stream_ptr(dev))
    L.check(rc)
    if debug:
        out["score_map"], out["feature_map"] = smap, fmap
    return out


# ---------------------------------------------------------------------------------------------------
# SIFT
# ---------------------------------------------------------------------------------------------------
def sift_conf_struct(conf):
    """conf keys: n_octave_layers, contrast_threshold, edge_threshold, sigma, max_keypoints (<= 0: all),
    nms_radius (None or 0), rootsift"""
    nms = conf.get("nms_radius")
    return L.SiftConf(int(conf["n_octave_layers"]), float(conf["contrast_threshold"]), float(conf["edge_threshold"]),
                      float(conf.get("sigma", 1.6)), int(conf["max_keypoints"] or 0), -1 if nms is None else int(nms),
                      int(bool(conf["rootsift"])))


def sift_plan(conf, height, width):
    """Host-only: (octave count, [(ksize, taps as float32 numpy)] per pyramid layer; entry 0 blurs the doubled base)."""
    import numpy as np
    c = sift_conf_struct(conf)
    n_layers = c.n_octave_layers + 3
    n_oct = C.c_int()
    ks = (C.c_int * n_layers)()
    taps = np.zeros((n_layers, L.IMW_SIFT_MAX_TAPS), np.float32)
    L.check(L.lib().imw_sift_plan(C.byref(c), height, width, C.addressof(n_oct), C.addressof(ks), taps.ctypes.data))
    return n_oct.value, [(ks[i], taps[i, :ks[i]].copy()) for i in range(n_layers)]


def sift_pyramid_shapes(conf, height, width):
    """[(octave, layers, h, w)] of the Gaussian pyramid (octave -1 is the doubled image)."""
    n_oct, _ = sift_plan(conf, height, width)
    lay = int(conf["n_octave_layers"]) + 3
    return [(o - 1, lay, (2 * height) >> o, (2 * width) >> o) for o in range(n_oct)]


def sift_forward(image, conf, cap, debug=False):
    """image [B,1,H,W] fp32 CUDA in [0,1].  Returns batch buffers in descending response order: keypoints [B,cap,2],
    scores / scales / oris [B,cap], descriptors [B,cap,128], counts [2,B] int32 (written, total; total -1 = internal
    capacity exceeded) (+ pyramid: a list of [B, L+3, h, w] per octave with debug)."""
    L.require_cuda(image, "sift_forward(image)")
    assert image.dim() == 4 and image.shape[1] == 1 and image.dtype == torch.float32
    image = image.contiguous()
    B, _, H, W = image.shape
    dev = image.device
    c = sift_conf_struct(conf)
    out = {"keypoints": torch.empty(B, cap, 2, device=dev), "scores": torch.empty(B, cap, device=dev),
           "scales": torch.empty(B, cap, device=dev), "oris": torch.empty(B, cap, device=dev),
           "descriptors": torch.empty(B, cap, 128, device=dev), "counts": torch.empty(2, B, dtype=torch.int32, device=dev)}
    shapes = sift_pyramid_shapes(conf, H, W) if debug else []
    pyr = torch.empty(B, sum(l * h * w for _, l, h, w in shapes), device=dev) if debug else None
    lib = L.lib()
    nbytes = lib.imw_sift_workspace_bytes(C.byref(c), B, H, W)
    if nbytes == 0:
        L.check(lib.imw_sift_plan(C.byref(c), H, W, None, None, None))
    ws = L.workspaces.get(dev, nbytes, "sift")
    with torch.cuda.device(dev):
        rc = lib.imw_sift_forward(C.byref(c), B, H, W, L.ptr(image), cap, L.ptr(out["keypoints"]), L.ptr(out["scores"]),
                                  L.ptr(out["scales"]), L.ptr(out["oris"]), L.ptr(out["descriptors"]), L.ptr(out["counts"]),
                                  L.ptr(pyr), L.ptr(ws), ws.numel(), L.stream_ptr(dev))
    L.check(rc)
    if debug:
        levels, off = [], 0
        for _, l, h, w in shapes:
            levels.append(pyr[:, off:off + l * h * w].view(B, l, h, w))
            off += l * h * w
        out["pyramid"] = levels
    return out


# ---------------------------------------------------------------------------------------------------
# LoFTR
# ---------------------------------------------------------------------------------------------------
def _pad_to(n, m=64):
    return (n + m - 1) // m * m


def _loftr_conv(sd, conv_key, bn_prefix, stride):
    """Conv2d (bias-free) [+ BatchNorm2d eval] -> two fp16 planes [2][k*k][Cout_p][Cin_p] + fp32 bias [Cout_p];
    channel counts zero-padded to multiples of 64 (196 -> 256)."""
    w = sd[conv_key].float()
    co, ci, k, _ = w.shape
    b = None
    if bn_prefix is not None:
        g = sd[bn_prefix + "weight"] / torch.sqrt(sd[bn_prefix + "running_var"] + 1e-5)
        w = w * g[:, None, None, None]
        b = sd[bn_prefix + "bias"] - sd[bn_prefix + "running_mean"] * g
    cop, cip = _pad_to(co), _pad_to(ci)
    wt = torch.zeros(k * k, cop, cip)
    wt[:, :co, :ci] = w.permute(2, 3, 0, 1).reshape(k * k, co, ci)
    bias = torch.zeros(cop)
    if b is not None:
        bias[:co] = b
    return {"w": split_f16_planes(wt), "b": bias if b is not None else None, "cin": cip, "cout": cop, "ksize": k, "stride": stride}


def loftr_pack_weights(sd):
    """Reference LoFTR state dict (SE2LoFTR/src/loftr naming) -> kernel layout (CPU tensors + conv descriptors)."""
    out = {"convs": {}}
    g = sd["backbone.bn1.weight"] / torch.sqrt(sd["backbone.bn1.running_var"] + 1e-5)
    w1 = sd["backbone.conv1.weight"].float() * g[:, None, None, None]
    out["conv1_w"] = w1[:, 0].permute(1, 2, 0).reshape(49, 128).contiguous()
    out["conv1_b"] = (sd["backbone.bn1.bias"] - sd["backbone.bn1.running_mean"] * g).float().contiguous()
    cv = out["convs"]
    for li in (1, 2, 3):
        for bi in (0, 1):
            p = f"backbone.layer{li}.{bi}."
            s = 2 if (li > 1 and bi == 0) else 1
            cv[f"l{li}.{2 * bi}"] = _loftr_conv(sd, p + "conv1.weight", p + "bn1.", s)
            cv[f"l{li}.{2 * bi + 1}"] = _loftr_conv(sd, p + "conv2.weight", p + "bn2.", 1)
        if li > 1:
            p = f"backbone.layer{li}.0."
            cv[f"l{li}_down"] = _loftr_conv(sd, p + "downsample.0.weight", p + "downsample.1.", 2)
    cv["l3_out"] = _loftr_conv(sd, "backbone.layer3_outconv.weight", None, 1)
    cv["l2_out"] = _loftr_conv(sd, "backbone.layer2_outconv.weight", None, 1)
    cv["l2_out2.0"] = _loftr_conv(sd, "backbone.layer2_outconv2.0.weight", "backbone.layer2_outconv2.1.", 1)
    cv["l2_out2.1"] = _loftr_conv(sd, "backbone.layer2_outconv2.3.weight", None, 1)
    cv["l1_out"] = _loftr_conv(sd, "backbone.layer1_outconv.weight", None, 1)
    cv["l1_out2.0"] = _loftr_conv(sd, "backbone.layer1_outconv2.0.weight", "backbone.layer1_outconv2.1.", 1)
    cv["l1_out2.1"] = _loftr_conv(sd, "backbone.layer1_outconv2.3.weight", None, 1)
    for prefix, n, tag in (("loftr_coarse.", 8, "c"), ("loftr_fine.", 2, "f")):
        for i in range(n):
            p = f"{prefix}layers.{i}."
            # every matrix is followed by its split-fp16 planes (tcgen05 GEMM operands); the fp32 paths read the first N rows
            out[f"{tag}{i}.qkv_w"] = with_f16_planes(torch.cat([sd[p + "q_proj.weight"], sd[p + "k_proj.weight"], sd[p + "v_proj.weight"]], 0).float())
            out[f"{tag}{i}.merge_w"] = with_f16_planes(sd[p + "merge.weight"].float())
            out[f"{tag}{i}.mlp0_w"] = with_f16_planes(sd[p + "mlp.0.weight"].float())
            out[f"{tag}{i}.mlp2_w"] = with_f16_planes(sd[p + "mlp.2.weight"].float())
            for nm, k in (("norm1.weight", "norm1_g"), ("norm1.bias", "norm1_b"), ("norm2.weight", "norm2_g"), ("norm2.bias", "norm2_b")):
                out[f"{tag}{i}.{k}"] = sd[p + nm].float().contiguous()
    for k in ("down_proj.weight", "down_proj.bias", "merge_feat.weight", "merge_feat.bias"):
        out[k.replace(".weight", "_w").replace(".bias", "_b")] = sd["fine_preprocess." + k].float().contiguous()
    return out


def loftr_position_encoding(d_model, h, w, temp_bug_fix=False):
    """utils/position_encoding.py:6-42 as a token table [h*w][d_model] (the default keeps the reference's 'buggy' div_term)."""
    import math
    pe = torch.zeros((d_model, h, w))
    y_pos = torch.ones((h, w)).cumsum(0).float().unsqueeze(0)
    x_pos = torch.ones((h, w)).cumsum(1).float().unsqueeze(0)
    if temp_bug_fix:
        div = torch.exp(torch.arange(0, d_model // 2, 2).float() * (-math.log(10000.0) / (d_model // 2)))
    else:
        div = torch.exp(torch.arange(0, d_model // 2, 2).float() * (-math.log(10000.0) / d_model // 2))
    div = div[:, None, None]
    pe[0::4] = torch.sin(x_pos * div); pe[1::4] = torch.cos(x_pos * div)
    pe[2::4] = torch.sin(y_pos * div); pe[3::4] = torch.cos(y_pos * div)
    return pe.permute(1, 2, 0).reshape(h * w, d_model).contiguous()


def loftr_to_device(packed, device):
    dev = {k: v.to(device) for k, v in packed.items() if torch.is_tensor(v)}
    dev["convs"] = {k: {**c, "w": c["w"].to(device), "b": (c["b"].to(device) if c["b"] is not None else None)} for k, c in packed["convs"].items()}
    return dev


def _loftr_struct(wd, pos_enc):
    s = L.LoftrWeights()
    bb = s.backbone
    bb.conv1_w, bb.conv1_b = wd["conv1_w"].data_ptr(), wd["conv1_b"].data_ptr()

    def fill(dst, c):
        dst.w = c["w"].data_ptr(); dst.b = c["b"].data_ptr() if c["b"] is not None else None
        dst.cin, dst.cout, dst.ksize, dst.stride = c["cin"], c["cout"], c["ksize"], c["stride"]
    cv = wd["convs"]
    for i in range(4):
        fill(bb.l1[i], cv[f"l1.{i}"]); fill(bb.l2[i], cv[f"l2.{i}"]); fill(bb.l3[i], cv[f"l3.{i}"])
    fill(bb.l2_down, cv["l2_down"]); fill(bb.l3_down, cv["l3_down"]); fill(bb.l3_out, cv["l3_out"]); fill(bb.l2_out, cv["l2_out"])
    fill(bb.l2_out2[0], cv["l2_out2.0"]); fill(bb.l2_out2[1], cv["l2_out2.1"]); fill(bb.l1_out, cv["l1_out"])
    fill(bb.l1_out2[0], cv["l1_out2.0"]); fill(bb.l1_out2[1], cv["l1_out2.1"])
    s.pos_enc = pos_enc.data_ptr()
    s.n_coarse, s.n_fine = 8, 2
    for tag, arr, n in (("c", s.coarse, 8), ("f", s.fine, 2)):
        for i in range(n):
            for f in ("qkv_w", "merge_w", "mlp0_w", "mlp2_w", "norm1_g", "norm1_b", "norm2_g", "norm2_b"):
                setattr(arr[i], f, wd[f"{tag}{i}.{f}"].data_ptr())
            arr[i].is_cross = i % 2  # layer_names = ['self', 'cross'] * n
    s.down_proj_w, s.down_proj_b = wd["down_proj_w"].data_ptr(), wd["down_proj_b"].data_ptr()
    s.merge_feat_w, s.merge_feat_b = wd["merge_feat_w"].data_ptr(), wd["merge_feat_b"].data_ptr()
    s.has_f16_planes = 1
    return s


def loftr_forward(wd, images, conf, max_matches=None, debug=False, temp_bug_fix=False, max_workspace_bytes=48 << 30, images1=None):
    """images [2P,H,W] fp32 CUDA (slot 2p = rows of the confidence matrix), or -- for pairs whose two images differ in size --
    images [P,H0,W0] with images1 [P,H1,W1].  Returns dict of device tensors: keypoints0/1 [P,mcap,2], confidence [P,mcap],
    counts [P] (+ debug features)."""
    L.require_cuda(images, "loftr_forward(images)")
    images = images.contiguous()
    if images1 is None:
        S, H0, W0 = images.shape
        assert S % 2 == 0
        P, H1, W1 = S // 2, H0, W0
        im0, st0, im1, st1 = images, 2 * H0 * W0, images.view(-1)[H0 * W0:], 2 * H0 * W0
    else:
        images1 = images1.contiguous()
        P, H0, W0 = images.shape
        assert images1.shape[0] == P and images1.device == images.device
        H1, W1 = images1.shape[1:]
        im0, st0, im1, st1 = images, H0 * W0, images1, H1 * W1
    assert H0 % 8 == 0 and W0 % 8 == 0 and H1 % 8 == 0 and W1 % 8 == 0
    dev = images.device
    L0, L1 = (H0 // 8) * (W0 // 8), (H1 // 8) * (W1 // 8)
    Lc = max(L0, L1)
    cap = (Lc + 127) // 128 * 128
    mcap = int(max_matches or L0)
    pes = []
    for (hc, wc) in ((H0 // 8, W0 // 8), (H1 // 8, W1 // 8)):
        key = ("pe", hc, wc, temp_bug_fix)
        if key not in wd:
            wd[key] = loftr_position_encoding(256, hc, wc, temp_bug_fix).to(dev)
        pes.append(wd[key])
    out = {"keypoints0": torch.zeros(P, mcap, 2, device=dev), "keypoints1": torch.zeros(P, mcap, 2, device=dev),
           "confidence": torch.zeros(P, mcap, device=dev), "counts": torch.zeros(P, dtype=torch.int32, device=dev)}
    dbg_c = torch.zeros(2 * P, cap, 256, device=dev) if debug else None
    dbg_b = torch.zeros(2 * P, Lc, 256, device=dev) if debug else None
    lib = L.lib()
    # pairs per library call: bound the workspace -- BASELINE configs[2] is batch = 32
    per_pair = lib.imw_loftr_workspace_bytes_hw(1, H0, W0, H1, W1, mcap)
    chunk = max(1, min(P, int(max_workspace_bytes // max(per_pair, 1)), 65535 // mcap))   # grid.y of the fine stage = pairs * mcap
    ws = L.workspaces.get(dev, lib.imw_loftr_workspace_bytes_hw(chunk, H0, W0, H1, W1, mcap), "loftr")
    c = L.LoftrConf(float(conf.get("match_threshold", 0.2)), float(conf.get("temperature", 0.1)), int(conf.get("border_rm", 2)),
                    int(conf.get("use_tensor_cores", 1)))
    wstruct = _loftr_struct(wd, pes[0])
    f0, f1 = im0.view(-1), im1.view(-1)
    with torch.cuda.device(dev):
        for p0 in range(0, P, chunk):
            n = min(chunk, P - p0)
            rc = lib.imw_loftr_forward_hw(C.byref(wstruct), C.byref(c), n, H0, W0, H1, W1, L.ptr(f0[p0 * st0:]), st0, L.ptr(f1[p0 * st1:]), st1,
                                          L.ptr(pes[1]), mcap, L.ptr(out["keypoints0"][p0:]), L.ptr(out["keypoints1"][p0:]),
                                          L.ptr(out["confidence"][p0:]), L.ptr(out["counts"][p0:]),
                                          L.ptr(dbg_c[2 * p0:]) if debug else None, L.ptr(dbg_b[2 * p0:]) if debug else None,
                                          L.ptr(ws), ws.numel(), L.stream_ptr(dev))
            L.check(rc)
    if debug:
        out["feat_c"], out["backbone_c"] = dbg_c[:, :Lc], dbg_b
    return out


# ---------------------------------------------------------------------------------------------------
# hloc first-party matchers
# ---------------------------------------------------------------------------------------------------
def _matcher_common(descriptors, counts):
    L.require_cuda(descriptors, "matcher(descriptors)")
    S, cap, dim = descriptors.shape
    assert S % 2 == 0 and counts.numel() == S and counts.dtype == torch.int32 and descriptors.is_contiguous()
    dev = descriptors.device
    m0 = torch.empty(S // 2, cap, dtype=torch.int32, device=dev)
    s0 = torch.empty(S // 2, cap, device=dev)
    ws = L.workspaces.get(dev, L.lib().imw_matcher_workspace_bytes(S // 2, cap), "mt")
    return S // 2, cap, dim, dev, m0, s0, ws


def nearest_neighbor(descriptors, counts, ratio_threshold=None, distance_threshold=None, do_mutual_check=True, tensor_cores=True):
    """descriptors [2P,cap,dim] token-major, counts [2P].  -> matches0 [P,cap] int32, scores0 [P,cap]."""
    P, cap, dim, dev, m0, s0, ws = _matcher_common(descriptors, counts)
    with torch.cuda.device(dev):
        rc = L.lib().imw_nearest_neighbor(P, cap, dim, L.ptr(descriptors), L.ptr(counts), float(ratio_threshold or 0.0),
                                          float(distance_threshold or 0.0), int(bool(do_mutual_check)), int(bool(tensor_cores)), L.ptr(m0), L.ptr(s0),
                                          L.ptr(ws), ws.numel(), L.stream_ptr(dev))
    L.check(rc)
    return m0, s0


def dual_softmax(descriptors, counts, match_threshold=0.2, inv_temperature=20.0, tensor_cores=True):
    P, cap, dim, dev, m0, s0, ws = _matcher_common(descriptors, counts)
    with torch.cuda.device(dev):
        rc = L.lib().imw_dual_softmax(P, cap, dim, L.ptr(descriptors), L.ptr(counts), float(match_threshold),
                                      float(inv_temperature), int(bool(tensor_cores)), L.ptr(m0), L.ptr(s0), L.ptr(ws), ws.numel(),
                                      L.stream_ptr(dev))
    L.check(rc)
    return m0, s0


def magsac(pts0, pts1, counts, geometry_type="Homography", threshold=3.0, confidence=0.9999, max_iters=10000, seed=0):
    """Batched MAGSAC++.  pts0/pts1 [n,cap,2] fp32 CUDA, counts [n] int32.
    Returns models [n,3,3] float64, masks [n,cap] bool, n_inliers [n] int32, n_iters [n] int32 (all CUDA)."""
    L.require_cuda(pts0, "magsac(pts0)")
    n, cap, _ = pts0.shape
    dev = pts0.device
    models = torch.zeros(n, 9, dtype=torch.float64, device=dev)
    masks = torch.zeros(n, cap, dtype=torch.uint8, device=dev)
    n_inl = torch.zeros(n, dtype=torch.int32, device=dev)
    n_it = torch.zeros(n, dtype=torch.int32, device=dev)
    mt = {"Homography": 0, "Fundamental": 1}[geometry_type]
    with torch.cuda.device(dev):
        L.check(L.lib().imw_magsac(n, cap, L.ptr(pts0.contiguous()), L.ptr(pts1.contiguous()), L.ptr(counts), mt, float(threshold),
                                   float(confidence), int(max_iters), int(seed) & 0xFFFFFFFF, L.ptr(models), L.ptr(masks), L.ptr(n_inl),
                                   L.ptr(n_it), L.stream_ptr(dev)))
    return models.view(n, 3, 3), masks.bool(), n_inl, n_it


def debug_gemm(A, W, bias, mode="3xtf32"):
    """out = A @ W.T + bias through the tcgen05 GEMM ("tf32" / "3xtf32" / "3xtf32_wlo": host-provided W lo plane / "f16x2":
    split-fp16 with host-packed weight planes, what the LightGlue / LoFTR linears run) or the CUDA-core GEMM ("fp32")."""
    L.require_cuda(A, "debug_gemm(A)")
    M, K = A.shape
    N = W.shape[0]
    out = torch.empty(M, N, device=A.device)
    if mode == "3xtf32_wlo":
        W = with_tf32_lo_plane(W)
    if mode in ("f16x2", "f16x2_ap"):
        W = with_f16_planes(W)
    if mode == "f16x2_ap":   # the activations arrive as split-fp16 planes too (what a producer kernel writes)
        A = split_f16_planes(A)
    args = (L.ptr(A.contiguous()), L.ptr(W.contiguous()), L.ptr(bias.contiguous()), L.ptr(out), M, N, K)
    with torch.cuda.device(A.device):
        if mode == "fp32":
            L.check(L.lib().imw_debug_gemm_fp32(*args, L.stream_ptr(A.device)))
        else:
            L.check(L.lib().imw_debug_gemm_tf32(*args, {"3xtf32": 3, "3xtf32_wlo": 4, "f16x2": 5, "f16x2_ap": 6, "tf32": 1}[mode], L.stream_ptr(A.device)))
    return out


def debug_conv3x3(x, w, bias, relu=True, pool=False, tensor_cores=True):
    """One 3x3 conv layer, NHWC fp32 in/out; w [9][Cin][Cout] fp32.  tensor_cores: tcgen05 split-fp16 path."""
    L.require_cuda(x, "debug_conv3x3(x)")
    B, H, W_, Cin = x.shape
    Cout = w.shape[2]
    out = torch.empty(B, H // 2 if pool else H, W_ // 2 if pool else W_, Cout, device=x.device)
    with torch.cuda.device(x.device):
        if tensor_cores:
            scratch = torch.empty(int(6 * x.numel() + 10 * w.numel() + 4096), dtype=torch.uint8, device=x.device)
            L.check(L.lib().imw_debug_conv3x3_tc(L.ptr(x.contiguous()), L.ptr(w.contiguous()), L.ptr(bias), L.ptr(out), B, H, W_, Cin, Cout,
                                                 int(relu), int(pool), L.ptr(scratch), scratch.numel(), L.stream_ptr(x.device)))
        else:
            L.check(L.lib().imw_debug_conv3x3(L.ptr(x.contiguous()), L.ptr(w.contiguous()), L.ptr(bias), L.ptr(out), B, H, W_, Cin, Cout,
                                              int(relu), int(pool), L.stream_ptr(x.device)))
    return out


def debug_attention(q, k, v, counts, scale, cross=False, tensor_cores=True):
    """q,k,v [slots,4,cap,64] fp32 -> ctx [slots,cap,256]; counts [slots] int32 (unit-test hook)."""
    L.require_cuda(q, "debug_attention(q)")
    S, Hh, cap, hd = q.shape
    ctx = torch.zeros(S, cap, 256, device=q.device)
    scratch = torch.empty(int(q.numel() * 4 * 6 + 8192), dtype=torch.uint8, device=q.device)
    with torch.cuda.device(q.device):
        L.check(L.lib().imw_debug_attention(L.ptr(q.contiguous()), L.ptr(k.contiguous()), L.ptr(v.contiguous()), L.ptr(counts), S, cap,
                                            float(scale), int(cross), int(tensor_cores), L.ptr(ctx), L.ptr(scratch), scratch.numel(),
                                            L.stream_ptr(q.device)))
    return ctx
