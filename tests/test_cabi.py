"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol include/imw_b200.h
declares; the plugin registry resolves like the reference's dynamic_load; host-side weight re-layout."""
import ctypes
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    from imcui_b200 import _lib
    header = (ROOT / "include" / "imw_b200.h").read_text()
    names = set(re.findall(r"\b(imw_[a-z0-9_]+)\s*\(", header))
    assert {"imw_superpoint_forward", "imw_lightglue_forward", "imw_nearest_neighbor", "imw_dual_softmax"} <= names
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for n in names:
        assert hasattr(lib, n), f"{n} declared in imw_b200.h but not exported"
    assert _lib.lib().imw_version() >= 100


def test_struct_sizes_match_header(tmp_path):
    """Every ctypes mirror has the size gcc gives the C struct of include/imw_b200.h."""
    import subprocess
    from imcui_b200 import _lib
    pairs = {"imw_sp_weights": _lib.SPWeights, "imw_sp_conf": _lib.SPConf, "imw_lg_block": _lib.LGBlock, "imw_lg_weights": _lib.LGWeights,
             "imw_lg_conf": _lib.LGConf, "imw_sg_layer": _lib.SGLayer, "imw_aliked_weights": _lib.AlikedWeights,
             "imw_aliked_conf": _lib.AlikedConf, "imw_loftr_conv": _lib.LoftrConv, "imw_loftr_backbone": _lib.LoftrBackbone,
             "imw_loftr_layer": _lib.LoftrLayer, "imw_loftr_weights": _lib.LoftrWeights, "imw_loftr_conf": _lib.LoftrConf}
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "imw_b200.h"\nint main(void){' +
                   "".join(f'printf("{n} %zu\\n", sizeof({n}));' for n in pairs) + "return 0;}")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for n, cls in pairs.items():
        assert ctypes.sizeof(cls) == int(out[n]), n


def test_superglue_packing_is_a_relabelling():
    """BN folding + head permutation reproduce the reference's first attention projection / keypoint encoder."""
    import oracle
    from oracle import superglue as osg
    from imcui_b200 import ops
    import ctypes
    from imcui_b200 import _lib
    assert ctypes.sizeof(_lib.SGLayer) == 8 * 8 + 8
    sd = oracle.synthetic_weights("superglue")
    pk = ops.sg_pack_weights(sd)
    x = torch.randn(1, 256, 7)
    ref = torch.nn.functional.conv1d(x, sd["gnn.layers.0.attn.proj.0.weight"], sd["gnn.layers.0.attn.proj.0.bias"]).view(1, 64, 4, 7)
    mine = (x[0].t() @ pk["l0.qkv_w"][:256].t() + pk["l0.qkv_b"][:256]).view(7, 4, 64)   # [token][head][dim]
    assert torch.allclose(ref[0].permute(2, 1, 0), mine, atol=1e-5)
    kin = torch.randn(1, 3, 5)
    ref = osg._mlp(sd, "kenc.encoder", kin, 5)
    h = torch.cat([kin[0].t(), torch.zeros(5, 13)], 1)
    for l in range(5):
        h = h @ pk[f"kenc_w{l}"].t() + pk[f"kenc_b{l}"]
        if l < 4:
            h = h.relu()
    assert torch.allclose(ref[0].t(), h, atol=1e-4)


def test_dynamic_load_registry():
    from imcui_b200.hloc import extractors, matchers
    from imcui_b200.hloc.utils.base_model import BaseModel, dynamic_load
    for root, name in ((extractors, "superpoint"), (matchers, "lightglue"), (matchers, "superglue"), (matchers, "nearest_neighbor"),
                       (matchers, "dual_softmax")):
        cls = dynamic_load(root, name)
        assert issubclass(cls, BaseModel) and isinstance(cls.default_conf, dict)
    m = dynamic_load(matchers, "nearest_neighbor")({})
    with pytest.raises(AssertionError):
        m({"descriptors0": torch.zeros(1, 4, 0)})


def test_no_cpu_fallback():
    """The product path refuses CPU tensors instead of silently computing elsewhere."""
    from imcui_b200.hloc import matchers
    from imcui_b200.hloc.utils.base_model import dynamic_load
    m = dynamic_load(matchers, "nearest_neighbor")({})
    with pytest.raises(RuntimeError):
        m({"descriptors0": torch.randn(1, 8, 3), "descriptors1": torch.randn(1, 8, 4)})


def test_qkv_permutation_is_a_relabelling():
    from imcui_b200 import ops
    import oracle
    sd = oracle.synthetic_weights("lightglue")
    packed = ops.lg_pack_weights(sd)
    w = sd["transformers.0.self_attn.Wqkv.weight"]
    x = torch.randn(5, 256)
    ref = (x @ w.t()).unflatten(-1, (4, 64, 3))          # lightglue.py:166
    assert packed["l0.self.qkv_w"].shape == (2 * 768, 256)            # weights followed by their split-fp16 planes (same bytes)
    w = packed["l0.self.qkv_w"][:768]
    planes = packed["l0.self.qkv_w"][768:].contiguous().view(torch.float16).reshape(2, 768, 256)
    assert torch.equal(planes[0], w.half()) and torch.equal(planes[1], ((w - w.half().float()) * 2048.0).half())
    assert float((planes[0].double() + planes[1].double() / 2048.0 - w.double()).abs().max()) < 2.0 ** -22 * float(w.abs().max())
    mine = (x @ packed["l0.self.qkv_w"][:768].t()).view(5, 3, 4, 64)
    for which in range(3):
        assert torch.allclose(ref[..., which], mine[:, which], atol=1e-5)
