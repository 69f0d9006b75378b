"""CPU oracle helpers: seeded synthetic weights and inputs (SURVEY.md 8d).
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

There are no pretrained weights in this environment, so parity is checked on
architecture-exact modules with torch default inits under a fixed seed; LoRA ``up``
matrices are re-initialised non-zero (the default zero init would hide the LoRA path) and
``to_k_ip/to_v_ip`` start from ``to_k/to_v`` plus a perturbation (mirrors train.py:169-174).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .processors_ref import install_ref_processors
from .unet_ref import UNet2DConditionRef, UNetConfig, Attention


def build_ref_unet(cfg: UNetConfig, seed=1234, rank=128, dtype=torch.float32):
    torch.manual_seed(seed)
    unet = UNet2DConditionRef(cfg)
    procs = install_ref_processors(unet, rank=rank)
    g = torch.Generator().manual_seed(seed + 1)
    attn_by_name = {f"{n}.processor": m for n, m in unet.named_modules() if isinstance(m, Attention)}
    for name, p in procs.items():
        for lora in (p.to_q_lora, p.to_k_lora, p.to_v_lora, p.to_out_lora):
            lora.up.weight.data.normal_(0, 0.02, generator=g)
        if hasattr(p, "to_k_ip"):
            a = attn_by_name[name]
            p.to_k_ip.weight.data.copy_(a.to_k.weight.data + 0.02 * torch.randn(a.to_k.weight.shape, generator=g))
            p.to_v_ip.weight.data.copy_(a.to_v.weight.data + 0.02 * torch.randn(a.to_v.weight.shape, generator=g))
    # torch's default affine init (weight 1, bias 0) would hide every gamma / beta path (the engine folds LayerNorm into the neighbouring GEMMs and
    # GroupNorm into a per-channel affine): perturb them
    for m in unet.modules():
        if isinstance(m, (torch.nn.LayerNorm, torch.nn.GroupNorm)) and m.weight is not None:
            m.weight.data.add_(0.1 * torch.randn(m.weight.shape, generator=g))
            m.bias.data.add_(0.1 * torch.randn(m.bias.shape, generator=g))
    unet = unet.to(dtype).eval()
    for p in procs.values():
        p.to(dtype)
    for p in unet.parameters():
        p.requires_grad_(False)
    return unet


def adapter_state_dict(unet):
    """``adapter_modules`` part of the ConsistentID checkpoint: positional keys
    ``{i}.to_q_lora.down.weight`` ... (pipline_StableDiffusion_ConsistentID.py:143-144)."""
    ml = torch.nn.ModuleList(unet.attn_processors.values())
    return {k: v.detach().clone() for k, v in ml.state_dict().items()}


def synth_prompts(cad, seed=1, n_text=77, n_id=4, dtype=torch.float32):
    """null / augmented / text_only prompt tensors, each [1, 81, cad]: 77 CLIP-like rows + 4 LayerNorm-ed id rows."""
    out = []
    gid = torch.Generator().manual_seed(seed + 3)
    id_rows = F.layer_norm(torch.randn(1, n_id, cad, generator=gid), (cad,))
    gid0 = torch.Generator().manual_seed(seed + 4)
    id_rows_uncond = F.layer_norm(torch.randn(1, n_id, cad, generator=gid0), (cad,))
    for k in range(3):
        g = torch.Generator().manual_seed(seed + k)
        text = torch.randn(1, n_text, cad, generator=g)
        out.append(torch.cat([text, id_rows_uncond if k == 0 else id_rows], dim=1).to(dtype))
    return out  # null, augmented, text_only


def synth_latents(b, h, w, seed=0, dtype=torch.float32, init_noise_sigma=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(b, 4, h, w, generator=g) * init_noise_sigma).to(dtype)


def seeded_params(shapes, seed):
    """Seeded fp32 weights for a ``[(name, shape), ...]`` state-dict layout: matrices N(0, 1/fan_in), 1-D ``*weight`` entries (LayerNorm
    gains) 1 + 0.1 N(0, 1), other 1-D entries (biases) 0.1 N(0, 1).  Lets a golden fixture pin a module whose weights are too large to
    store: it keeps the layout and the seed, and the test rebuilds the same weights."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape in shapes:
        if len(shape) > 1:
            out[name] = torch.randn(shape, generator=g) * (shape[-1] ** -0.5)
        elif name.endswith("weight"):
            out[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            out[name] = 0.1 * torch.randn(shape, generator=g)
    return out
