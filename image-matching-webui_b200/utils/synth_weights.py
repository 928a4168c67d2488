"""Deterministic synthetic model parameters for every network the engine runs (SuperPoint, LightGlue, SuperGlue, LoFTR,
ALIKED) -- synthetic-data utilities like utils/synth.py: used by bench tooling, by tools/make_golden.py (which loads
the very same tensors into the unmodified reference modules) and, through oracle/, by the tests.  Pure torch, generated
key by key from a CPU torch.Generator so that every machine reproduces them bit for bit."""
import math

import torch


def loftr_random_weights(seed=0):
    """Deterministic random LoFTR parameters (no standard checkpoint exists offline).  Generated key by key from a CPU
    torch.Generator so that the GPU box reproduces them without shipping a 46 MB file; tools/make_golden.py loads the
    very same dict into the reference module.  BatchNorm statistics / affine terms are randomised (not the identity
    defaults) so that BN folding is exercised."""
    g = torch.Generator().manual_seed(1234 + seed)
    w = {}

    def conv(name, co, ci, k):
        w[name] = torch.randn(co, ci, k, k, generator=g) * math.sqrt(2.0 / (k * k * co))

    def bn(p, c):
        w[p + "weight"] = 0.9 + 0.2 * torch.rand(c, generator=g)
        w[p + "bias"] = 0.02 * torch.randn(c, generator=g)
        w[p + "running_mean"] = 0.02 * torch.randn(c, generator=g)
        w[p + "running_var"] = 0.9 + 0.2 * torch.rand(c, generator=g)

    def lin(name, o, i, bias=False):
        w[name + ".weight"] = torch.randn(o, i, generator=g) * math.sqrt(2.0 / (o + i))
        if bias:
            w[name + ".bias"] = 0.05 * torch.randn(o, generator=g)

    conv("backbone.conv1.weight", 128, 1, 7); bn("backbone.bn1.", 128)
    dims = [(128, 128), (128, 196), (196, 256)]
    for li, (ci, co) in enumerate(dims, 1):
        for bi in range(2):
            p = f"backbone.layer{li}.{bi}."
            cin = ci if bi == 0 else co
            conv(p + "conv1.weight", co, cin, 3); conv(p + "conv2.weight", co, co, 3)
            bn(p + "bn1.", co); bn(p + "bn2.", co)
            if bi == 0 and li > 1:
                conv(p + "downsample.0.weight", co, cin, 1); bn(p + "downsample.1.", co)
    conv("backbone.layer3_outconv.weight", 256, 256, 1)
    conv("backbone.layer2_outconv.weight", 256, 196, 1)
    conv("backbone.layer2_outconv2.0.weight", 256, 256, 3); bn("backbone.layer2_outconv2.1.", 256)
    conv("backbone.layer2_outconv2.3.weight", 196, 256, 3)
    conv("backbone.layer1_outconv.weight", 196, 128, 1)
    conv("backbone.layer1_outconv2.0.weight", 196, 196, 3); bn("backbone.layer1_outconv2.1.", 196)
    conv("backbone.layer1_outconv2.3.weight", 128, 196, 3)
    for prefix, n, d in (("loftr_coarse.", 8, 256), ("loftr_fine.", 2, 128)):
        for i in range(n):
            p = f"{prefix}layers.{i}."
            for nm in ("q_proj", "k_proj", "v_proj", "merge"):
                lin(p + nm, d, d)
            lin(p + "mlp.0", 2 * d, 2 * d); lin(p + "mlp.2", d, 2 * d)
            for nm in ("norm1", "norm2"):
                w[p + nm + ".weight"] = 1.0 + 0.05 * torch.randn(d, generator=g)
                w[p + nm + ".bias"] = 0.02 * torch.randn(d, generator=g)
    lin("fine_preprocess.down_proj", 128, 256, bias=True)
    lin("fine_preprocess.merge_feat", 128, 256, bias=True)
    return w


def aliked_random_weights(seed=0):
    """Deterministic random aliked-n16 parameters (reference key names), generated key by key from a CPU Generator."""
    g = torch.Generator().manual_seed(4321 + seed)
    w = {}
    c1, c2, c3, c4 = 16, 32, 64, 128   # aliked-n16 (aliked.py:627)
    dim, K, M = 128, 3, 16

    def conv(name, co, ci, k, bias=False, gain=1.0):
        w[name + ".weight"] = torch.randn(co, ci, k, k, generator=g) * (gain * math.sqrt(1.0 / (k * k * ci)))
        if bias:
            w[name + ".bias"] = 0.1 * torch.randn(co, generator=g)

    def bn(p, c):
        w[p + "weight"] = 0.9 + 0.2 * torch.rand(c, generator=g)
        w[p + "bias"] = 0.05 * torch.randn(c, generator=g)
        w[p + "running_mean"] = 0.05 * torch.randn(c, generator=g)
        w[p + "running_var"] = 0.9 + 0.2 * torch.rand(c, generator=g)
        w[p + "num_batches_tracked"] = torch.tensor(0)

    conv("block1.conv1", c1, 3, 3, gain=3.0); bn("block1.bn1.", c1); conv("block1.conv2", c1, c1, 3); bn("block1.bn2.", c1)
    for name, ci, co, dcn in (("block2", c1, c2, False), ("block3", c2, c3, True), ("block4", c3, c4, True)):
        for j, cin in ((1, ci), (2, co)):
            if dcn:
                conv(f"{name}.conv{j}.offset_conv", 18, cin, 3, bias=True, gain=2.0)
                conv(f"{name}.conv{j}.regular_conv", co, cin, 3)
            else:
                conv(f"{name}.conv{j}", co, cin, 3)
            bn(f"{name}.bn{j}.", co)
        conv(f"{name}.downsample", co, ci, 1, bias=True)
    conv("conv1", dim // 4, c1, 1); conv("conv2", dim // 4, c2, 1); conv("conv3", dim // 4, c3, 1); conv("conv4", dim // 4, dim, 1)
    conv("score_head.0", 8, dim, 1); conv("score_head.2", 4, 8, 3); conv("score_head.4", 4, 4, 3)
    conv("score_head.6", 1, 4, 3, gain=-1.0)   # sign chosen so that the score map is sparse (mean ~0.09, a few hundred maxima > 0.2)
    conv("desc_head.offset_conv.0", 2 * M, dim, K, bias=True, gain=6.0); conv("desc_head.offset_conv.2", 2 * M, 2 * M, 1, bias=True, gain=4.0)
    conv("desc_head.sf_conv", dim, dim, 1, gain=3.0)
    w["desc_head.agg_weights"] = torch.rand(M, dim, dim, generator=g)
    return w


def superpoint_random_weights(seed=0):
    """Deterministic random SuperPoint parameters (superpoint_v1 key names and shapes).  The detector head is scaled so
    that the 65-way softmax is peaked (a few hundred keypoints above 0.005 per 480x640 image), which keeps the keypoint
    set and top-k order well separated from fp32 rounding."""
    g = torch.Generator().manual_seed(2024 + seed)
    w = {}

    def conv(name, co, ci, k, gain=1.0):
        w[name + ".weight"] = torch.randn(co, ci, k, k, generator=g) * (gain * math.sqrt(2.0 / (k * k * ci)))
        w[name + ".bias"] = 0.01 * torch.randn(co, generator=g)

    c1, c2, c3, c4, c5, d1 = 64, 64, 128, 128, 256, 256   # superpoint.py:117-130
    conv("conv1a", c1, 1, 3, gain=4.0); conv("conv1b", c1, c1, 3)
    conv("conv2a", c2, c1, 3); conv("conv2b", c2, c2, 3)
    conv("conv3a", c3, c2, 3); conv("conv3b", c3, c3, 3)
    conv("conv4a", c4, c3, 3); conv("conv4b", c4, c4, 3)
    conv("convPa", c5, c4, 3); conv("convPb", 65, c5, 1, gain=2.0)
    w["convPb.bias"][64] = 6.0                                  # dustbin: most cells hold no keypoint
    conv("convDa", c5, c4, 3); conv("convDb", d1, c5, 1)
    # The random encoder maps every patch to nearly the same direction (non-negative ReLU features share a large mean), so
    # descriptors would all be alike.  convDb's bias removes that mean, measured on a fixed seeded texture and rounded to
    # 2^-10 so that every machine derives the same bits.
    F = torch.nn.functional
    x = F.interpolate(torch.rand(1, 1, 30, 40, generator=g), size=(240, 320), mode="bilinear", align_corners=False)
    for name in ("conv1a", "conv1b", None, "conv2a", "conv2b", None, "conv3a", "conv3b", None, "conv4a", "conv4b", "convDa"):
        x = F.max_pool2d(x, 2, 2) if name is None else F.relu(F.conv2d(x, w[name + ".weight"], w[name + ".bias"], padding=1))
    mean = F.conv2d(x, w["convDb.weight"], w["convDb.bias"]).mean((0, 2, 3))
    w["convDb.bias"] -= torch.round(mean * 1024.0) / 1024.0
    return w


def lightglue_random_weights(seed=0, n_layers=9, d=256, heads=4):
    """Deterministic random SuperPoint-LightGlue parameters (reference key names and shapes).  The transformer updates are
    small and final_proj is a scaled identity, so the assignment follows descriptor similarity and real correspondences
    are matched; token confidences rise with depth (early stop within the 9 layers) and matchability is spread widely
    (some tokens are pruned)."""
    g = torch.Generator().manual_seed(99 + seed)
    w = {"posenc.Wr.weight": torch.randn(d // heads // 2, 2, generator=g) * 2.0}

    def lin(name, o, i, gain=1.0, bias=0.02):
        w[name + ".weight"] = torch.randn(o, i, generator=g) * (gain / math.sqrt(i))
        w[name + ".bias"] = bias * torch.randn(o, generator=g)

    for i in range(n_layers):
        p = f"transformers.{i}.self_attn."
        lin(p + "Wqkv", 3 * d, d); lin(p + "out_proj", d, d)
        c = f"transformers.{i}.cross_attn."
        lin(c + "to_qk", d, d); lin(c + "to_v", d, d); lin(c + "to_out", d, d)
        for pre in (p, c):
            lin(pre + "ffn.0", 2 * d, 2 * d)
            w[pre + "ffn.1.weight"] = 1.0 + 0.05 * torch.randn(2 * d, generator=g)
            w[pre + "ffn.1.bias"] = 0.02 * torch.randn(2 * d, generator=g)
            lin(pre + "ffn.3", d, 2 * d, gain=0.005, bias=0.0)
        a = f"log_assignment.{i}."
        w[a + "final_proj.weight"] = 30.0 * torch.eye(d) + 0.05 * torch.randn(d, d, generator=g) / math.sqrt(d)
        w[a + "final_proj.bias"] = torch.zeros(d)
        lin(a + "matchability", 1, d, gain=60.0, bias=0.0)
        w[a + "matchability.bias"] += 3.0
        if i < n_layers - 1:
            lin(f"token_confidence.{i}.token.0", 1, d, gain=8.0, bias=0.0)
            w[f"token_confidence.{i}.token.0.bias"] += -1.0 + 0.8 * i
    return w


def superglue_random_weights(seed=0, d=256, layers=18, heads=4):
    """Deterministic random SuperGlue parameters (superglue_outdoor key names and shapes).  As for LightGlue, the
    message-passing updates are small and final_proj is a scaled identity, so Sinkhorn matches similar descriptors."""
    g = torch.Generator().manual_seed(777 + seed)
    w = {}

    def conv(name, o, i, gain=1.0, bias=0.02):
        w[name + ".weight"] = torch.randn(o, i, 1, generator=g) * (gain / math.sqrt(i))
        w[name + ".bias"] = bias * torch.randn(o, generator=g)

    def bn(p, c):
        w[p + "weight"] = 0.9 + 0.2 * torch.rand(c, generator=g)
        w[p + "bias"] = 0.05 * torch.randn(c, generator=g)
        w[p + "running_mean"] = 0.05 * torch.randn(c, generator=g)
        w[p + "running_var"] = 0.9 + 0.2 * torch.rand(c, generator=g)
        w[p + "num_batches_tracked"] = torch.tensor(0)

    chans = [3, 32, 64, 128, 256, d]                            # superglue.py:75-84 (keypoint_encoder 32-64-128-256)
    for l in range(5):
        conv(f"kenc.encoder.{3 * l}", chans[l + 1], chans[l], gain=0.05 if l == 4 else 1.0, bias=0.0 if l == 4 else 0.02)
        if l < 4:
            bn(f"kenc.encoder.{3 * l + 1}.", chans[l + 1])
    for i in range(layers):
        p = f"gnn.layers.{i}."
        for j in range(3):
            conv(p + f"attn.proj.{j}", d, d)
        conv(p + "attn.merge", d, d)
        conv(p + "mlp.0", 2 * d, 2 * d); bn(p + "mlp.1.", 2 * d)
        conv(p + "mlp.3", d, 2 * d, gain=0.005, bias=0.0)
    w["final_proj.weight"] = (18.0 * torch.eye(d) + 0.05 * torch.randn(d, d, generator=g) / math.sqrt(d))[:, :, None]
    w["final_proj.bias"] = torch.zeros(d)
    w["bin_score"] = torch.tensor(2.0)
    return w
