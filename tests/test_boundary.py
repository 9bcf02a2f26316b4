"""CPU-side checks of the drop-in boundary: state-dict contract, C-ABI exports, index closed forms, loud failure
without a GPU."""
import ctypes
import os
import re

import pytest
import torch

from oracle import synth


def test_state_dict_contract_matches_reference_keys(golden):
    from vit_grid_model_b200 import MetNet3
    f = golden("metnet3_12hr_b1.pt")
    cfg = synth.GridConfig(**f["cfg"])
    m = MetNet3(**cfg.metnet3_kwargs())
    assert list(m.state_dict().keys()) == f["keys"]            # same names, same order as the reference module
    sd = synth.make_state_dict(synth.metnet3_spec(cfg))
    for k, v in m.state_dict().items():
        assert tuple(v.shape) == tuple(sd[k].shape), k
    m.load_state_dict(sd, strict=True)
    m.load_state_dict({"module." + k: v for k, v in sd.items()}, strict=True)     # evaluation_vit.py:107-109
    assert sum(p.numel() for p in m.parameters()) == f["n_params"]
    # rel_pos_indices is a non-persistent buffer (maxvit.py:168)
    assert not any("rel_pos_indices" in k for k in m.state_dict())
    assert m.vit.layers[0][1].rel_pos_indices.shape == (53, 53)


def test_depth2_uses_fn_prefix():
    from vit_grid_model_b200 import MaxViT
    m = MaxViT(dim=128, depth=2, cond_dim=2, vit_window_size=7)
    keys = set(m.state_dict().keys())
    assert "layers.0.0.0.weight" in keys and "layers.1.0.fn.0.weight" in keys and "register_tokens.1" in keys
    assert keys == set(synth.maxvit_spec(128, 2, 2, 32, 32, 7, 4, 0.25, 4).keys())


def test_rel_pos_indices_closed_form(golden):
    from vit_grid_model_b200.maxvit import rel_pos_indices
    g = golden("index_golden.pt")
    for (w, r) in ((7, 4), (8, 1), (4, 2)):
        assert torch.equal(rel_pos_indices(w, r), g[f"rel_pos_w{w}_r{r}"])


def test_constructor_errors():
    from vit_grid_model_b200 import MetNet3
    kw = synth.CFG_SMALL128.metnet3_kwargs()
    with pytest.raises(ValueError):
        MetNet3(**{**kw, "pm25_boundaries": None})
    with pytest.raises(NotImplementedError):
        MetNet3(**{**kw, "pm10": True})
    with pytest.raises(AssertionError):
        MetNet3(**{**kw, "ignore_backbone": True})


def test_library_exports_every_declared_symbol():
    from vit_grid_model_b200 import _lib, build
    protos = _lib.parse_header()
    hdr = open(_lib.HEADER).read()
    declared = set(re.findall(r"\b(vg_\w+)\s*\(", re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)))
    assert declared == set(protos) and len(declared) >= 20
    lib = ctypes.CDLL(build.build_library())
    for name in declared:
        assert hasattr(lib, name), name
    lib.vg_version.restype = ctypes.c_int
    assert lib.vg_version() >= 100
    lib.vg_pg_pixels.restype = ctypes.c_longlong
    assert lib.vg_pg_pixels(2, 84, 70) == (2 * 85 + 1) * 71


def test_library_reads_no_environment_variable():
    """Every code path of a library call is selected by its arguments or by what the library observes (the device, the
    shapes), never by an environment variable: the CUDA sources call no getenv, and INTEGRATION.md documents no switch."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    csrc = os.path.join(root, "vit-grid-model_b200", "csrc")
    for fn in os.listdir(csrc):
        src = open(os.path.join(csrc, fn)).read()
        assert not re.search(r"getenv\s*\(", src), fn
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    assert not re.search(r"^\| `VG_\w+=", doc, flags=re.M)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from vit_grid_model_b200 import MetNet3, VitGridError, focal_r_loss
    cfg = synth.CFG_SMALL128
    m = MetNet3(**cfg.metnet3_kwargs()).eval()
    x, ts, t = synth.make_inputs(cfg, 1)
    with pytest.raises(VitGridError):
        m(x, timestamps=ts)
    with pytest.raises(VitGridError):
        focal_r_loss(t, t)


def test_product_never_imports_oracle():
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "vit-grid-model_b200")
    for dirpath, _, files in os.walk(root):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn


def test_attention_logit_bound_dominates_the_logits():
    """ops.attn_logit_bound (host logic behind vg_attn_fused2_fwd's logit_bound): for random weights and inputs the bound must
    dominate |q.k + bias| * log2(e) of maxvit.py:26-30,203 -- it is what allows the fused kernel to drop the softmax's running
    maximum -- and the 3xTF32 operand split must reproduce its input exactly (hi + lo == x, hi has 13 zero low bits)."""
    import math
    import torch.nn.functional as F
    from vit_grid_model_b200 import ops
    g = torch.Generator().manual_seed(0)
    heads, dh, S, w = 4, 32, 53, 7
    for trial in range(5):
        qg = 0.5 + torch.rand(heads, dh, generator=g) * (1 + trial)
        kg = 0.5 + torch.rand(heads, dh, generator=g)
        table = torch.randn((2 * w - 1) ** 2 + 1, heads, generator=g) * (1 + trial)
        q = torch.randn(3, heads, S, dh, generator=g) * 10 ** (trial - 2)
        k = torch.randn(3, heads, S, dh, generator=g)
        qn = F.normalize(q, dim=-1) * math.sqrt(dh) * qg[None, :, None, :]
        kn = F.normalize(k, dim=-1) * math.sqrt(dh) * kg[None, :, None, :]
        sim = qn @ kn.transpose(-1, -2)
        worst = (sim.abs().max() + table.abs().max()).item() * 1.4426950408889634
        bound = ops.attn_logit_bound(table, qg.reshape(-1), kg.reshape(-1), dh)
        assert worst <= bound, (trial, worst, bound)
    x = torch.randn(1000, generator=g) * torch.logspace(-20, 20, 1000)
    hi = (x.view(torch.int32) & -8192).view(torch.float32)
    assert torch.equal(hi + (x - hi), x) and ((x - hi).abs() <= x.abs() * 2.0 ** -10).all()
