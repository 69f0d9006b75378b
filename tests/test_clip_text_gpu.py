"""GPU checks of the CLIP text encoder path: the three kernels it adds (cid_attn_self_causal, the QuickGELU GEMM epilogue, cid_embed_tokens)
against fp32 torch, and consistentid_b200.clip.B200CLIPTextEncoder against tests/clip_text_ref.text_hidden_states (pinned on the installed
transformers, tests/test_clip_text_cpu.py) at reduced widths and at the two geometries the pipelines load: SD1.5 / SDXL ``text_encoder``
(OpenAI ViT-L/14: 768 wide, 12 layers, 12 heads of 64, MLP 3072, quick_gelu) and SDXL ``text_encoder_2`` (OpenCLIP ViT-bigG/14: 1280 wide,
32 layers, 20 heads of 64, MLP 5120, gelu, projection 1280), 77 tokens, vocabulary 49408."""
import warnings

import pytest
import torch
import torch.nn.functional as F

from tests import clip_text_ref
from tests.test_unet_gpu import _cmp

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rand(shape, dtype, seed, scale=1.0):
    return (torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale).to(dtype).to(DEV)


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("d", [40, 64, 128])
@pytest.mark.parametrize("N", [80, 128, 136, 384, 1000])
def test_attn_self_causal(N, d, dtype):
    from consistentid_b200 import ops
    B, H = 2, 3
    C = H * d
    qk = _rand((B * N, 2 * C), dtype, 0)
    v = _rand((B, N, H, d), dtype, 1)
    vt = v.permute(0, 2, 3, 1).reshape(B * H, d, N).contiguous()
    out = torch.full((B * N, C), float("nan"), dtype=dtype, device=DEV)
    ops.attn_self_causal(qk[:, :C], qk[:, C:], vt, out, B, H, N, d)
    torch.cuda.synchronize()
    sp = lambda t: t.float().reshape(B, N, H, d).transpose(1, 2)
    ref = F.scaled_dot_product_attention(sp(qk[:, :C]), sp(qk[:, C:]), v.float().transpose(1, 2), is_causal=True)
    ref = ref.transpose(1, 2).reshape(B * N, C)
    err = (out.float() - ref).abs().max().item()
    assert torch.isfinite(out.float()).all() and err <= 1e-2 * ref.abs().max().item(), err


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("path", ["tma_store", "fallback_store", "split_k"])
def test_gemm_quick_gelu(path, dtype):
    """fc1 of the ViT-L/14 text MLP on 3 padded sequences: M = 3 * 80, N = 3072, K = 768."""
    from consistentid_b200 import lib, ops
    M, N, K = 240, 3072, 768
    a, w, b = _rand((M, K), dtype, 0), _rand((N, K), dtype, 1, K ** -0.5), _rand((N,), dtype, 2)
    ld = N + 5 if path == "fallback_store" else N                   # a row pitch that is not a multiple of 8 rules out the TMA store
    buf = torch.full((M, ld), float("nan"), dtype=dtype, device=DEV)
    out = buf[:, :N]
    if path == "split_k":
        lib.set_splitk(4, 1)
    try:
        ops.gemm(a, w, out, bias=b, epi=lib.EPI_QUICK_GELU)
        torch.cuda.synchronize()
    finally:
        lib.set_splitk()
    y = a.float() @ w.float().T + b.float()
    ref = y * torch.sigmoid(1.702 * y)
    err = (out.float() - ref).abs().max().item()
    assert torch.isfinite(out.float()).all() and err <= 8e-3 * ref.abs().max().item(), err
    if path == "fallback_store":
        assert torch.isnan(buf[:, N:].float()).all()                 # nothing written past N


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_embed_tokens(dtype):
    from consistentid_b200 import ops
    B, L, Lp, V, C = 3, 77, 80, 1000, 768
    tok, pos = _rand((V, C), dtype, 0), _rand((77, C), dtype, 1, 0.1)
    ids = torch.randint(0, V, (B, L), generator=torch.Generator().manual_seed(2))
    ids_dev = ids.to(DEV)
    ids_dev[1, 5], ids_dev[2, 76] = V + 7, -3                       # out of range on the device: zero token rows, no out-of-bounds read
    out = torch.full((B * Lp, C), float("nan"), dtype=dtype, device=DEV)
    ops.embed_tokens(ids_dev, tok, pos, out, Lp)
    torch.cuda.synchronize()
    ref = tok[ids.to(DEV)] + pos[None, :L]                          # the 16-bit add torch does
    ref[1, 5], ref[2, 76] = pos[5], pos[76]
    got = out.view(B, Lp, C)
    assert torch.equal(got[:, :L], ref)
    assert (got[:, L:] == 0).all()


# ------------------------------------------------------------------------------------------------ encoder parity
def _weights(C, heads, layers, inter, vocab=49408, n_pos=77, proj=None, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s, std=1.0: torch.randn(*s, generator=g) * std
    sd = {"text_model.embeddings.token_embedding.weight": r(vocab, C, std=0.5),
          "text_model.embeddings.position_embedding.weight": r(n_pos, C, std=0.1),
          "text_model.final_layer_norm.weight": 1 + r(C, std=0.1), "text_model.final_layer_norm.bias": r(C, std=0.1)}
    for i in range(layers):
        b = f"text_model.encoder.layers.{i}."
        for ln in ("layer_norm1", "layer_norm2"):
            sd[b + ln + ".weight"], sd[b + ln + ".bias"] = 1 + r(C, std=0.1), r(C, std=0.1)
        for q in ("q_proj", "k_proj", "v_proj", "out_proj"):
            sd[b + f"self_attn.{q}.weight"], sd[b + f"self_attn.{q}.bias"] = r(C, C, std=C ** -0.5), r(C, std=0.1)
        sd[b + "mlp.fc1.weight"], sd[b + "mlp.fc1.bias"] = r(inter, C, std=C ** -0.5), r(inter, std=0.1)
        sd[b + "mlp.fc2.weight"], sd[b + "mlp.fc2.bias"] = r(C, inter, std=inter ** -0.5), r(C, std=0.1)
    if proj:
        sd["text_projection.weight"] = r(proj, C, std=C ** -0.5)
    return sd


def _ids(B, L, vocab, pad_with_eos, seed=3):
    """BOS, a prompt of 5..60 tokens, EOS (the two largest ids, as in the CLIP tokenizers), then padding: EOS (SD1.5 tokenizer) or 0
    (SDXL tokenizer_2 pads with "!")."""
    g = torch.Generator().manual_seed(seed)
    bos, eos = vocab - 2, vocab - 1
    ids = torch.full((B, L), eos if pad_with_eos else 0, dtype=torch.int64)
    for b in range(B):
        n = min(5 + 23 * b, L - 2)
        ids[b, 0], ids[b, 1:1 + n], ids[b, 1 + n] = bos, torch.randint(1, bos, (n,), generator=g), eos
    return ids


def _truth_and_eager(sd, ids, heads, act, eos, dtype):
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        sd32 = {k: v.cuda() for k, v in sd.items()}                 # fp32 truth evaluated on the GPU (TF32 off)
        truth = [t.cpu() if torch.is_tensor(t) else (None if t is None else [h.cpu() for h in t])
                 for t in clip_text_ref.text_hidden_states(sd32, ids.cuda(), heads, act, eos)]
        del sd32
        sd16 = {k: v.cuda().to(dtype) for k, v in sd.items()}
        eager = clip_text_ref.text_hidden_states(sd16, ids.cuda(), heads, act, eos)
        del sd16
    return truth, eager


def _check(name, enc, sd, ids, heads, act, eos, dtype):
    truth, eager = _truth_and_eager(sd, ids, heads, act, eos, dtype)
    (hs_t, last_t, pooled_t, te_t), (hs_e, last_e, pooled_e, te_e) = truth, eager
    ids_dev = ids.cuda()
    with warnings.catch_warnings():                                  # ("prototype feature" notice)
        warnings.simplefilter("ignore", UserWarning)
        torch.cuda.set_sync_debug_mode("error")                      # device-resident ids: the call never waits on the device
    try:
        out = enc(ids_dev, output_hidden_states=True)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    B, L = ids.shape
    assert out.last_hidden_state.shape == (B, L, enc.C) and len(out.hidden_states) == enc.n_layers + 1
    _cmp(f"{name} last_hidden_state", out.last_hidden_state, last_t, last_e)
    _cmp(f"{name} hidden_states[-2]", out.hidden_states[-2], hs_t[-2], hs_e[-2])
    _cmp(f"{name} pooler_output", out.pooler_output, pooled_t, pooled_e)
    if te_t is not None:
        _cmp(f"{name} text_embeds", out.text_embeds, te_t, te_e)
    # the pipelines' call patterns: text_encoder(ids)[0], _encode_prompt's (ids, attention_mask=None)[0], SDXL's hidden_states[-2]
    first = out.text_embeds if te_t is not None else out.last_hidden_state
    for got in (enc(ids_dev)[0], enc(ids, attention_mask=None)[0]):
        assert got.shape == first.shape and (got.float() - first.float()).abs().max().item() <= 1e-3 * first.float().abs().max().item()
    hs2 = enc(ids_dev, output_hidden_states=True).hidden_states[-2]
    assert (hs2.float() - out.hidden_states[-2].float()).abs().max().item() <= 1e-3 * hs2.float().abs().max().item()
    return out, truth, eager


@pytest.mark.parametrize("C,heads,layers,inter,act,eos,pad_eos,L,proj,dtype", [
    (128, 2, 3, 256, "quick_gelu", 2, True, 77, None, torch.float16),
    (192, 3, 4, 640, "gelu", 49407, False, 77, 128, torch.bfloat16),
    (128, 2, 2, 256, "quick_gelu", 49407, True, 20, 64, torch.bfloat16)])
def test_clip_text_encoder_parity_reduced(C, heads, layers, inter, act, eos, pad_eos, L, proj, dtype):
    from consistentid_b200.clip import B200CLIPTextEncoder
    sd = _weights(C, heads, layers, inter, proj=proj)
    ids = _ids(3, L, 49408, pad_eos)
    enc = B200CLIPTextEncoder(sd, num_attention_heads=heads, hidden_act=act, eos_token_id=eos, dtype=dtype)
    _check(f"clip text C={C} L={L} {act} {dtype}", enc, sd, ids, heads, act, eos, dtype)


@pytest.mark.parametrize("B", [1, 3])
def test_clip_text_encoder_parity_vit_l(B):
    """SD1.5 text_encoder / SDXL text_encoder: OpenAI ViT-L/14 text tower, legacy eos_token_id 2, padded with EOS."""
    from consistentid_b200.clip import B200CLIPTextEncoder
    sd = _weights(768, 12, 12, 3072)
    enc = B200CLIPTextEncoder(sd, num_attention_heads=12, hidden_act="quick_gelu", eos_token_id=2, dtype=torch.float16)
    _check(f"ViT-L/14 text B={B}", enc, sd, _ids(B, 77, 49408, True), 12, "quick_gelu", 2, torch.float16)


@pytest.mark.parametrize("B", [1, 2])
def test_clip_text_encoder_parity_vit_bigg(B):
    """SDXL text_encoder_2: OpenCLIP ViT-bigG/14 text tower with projection, first-EOS pooling, padded with 0."""
    from consistentid_b200.clip import B200CLIPTextEncoder
    sd = _weights(1280, 20, 32, 5120, proj=1280)
    enc = B200CLIPTextEncoder(sd, num_attention_heads=20, hidden_act="gelu", eos_token_id=49407, dtype=torch.float16)
    out, _, _ = _check(f"ViT-bigG/14 text B={B}", enc, sd, _ids(B, 77, 49408, False), 20, "gelu", 49407, torch.float16)
    assert out[0] is out.text_embeds and out.text_embeds.shape == (B, 1280)


def test_sdxl_prompt_embeds_concat():
    """pipline_StableDiffusionXL_ConsistentID.py:514-524: prompt_embeds = cat([text_encoder(ids).hidden_states[-2],
    text_encoder_2(ids2).hidden_states[-2]], -1) -> [B, 77, 2048], pooled_prompt_embeds = text_encoder_2(ids2)[0].  Full widths, 2 layers."""
    from consistentid_b200.clip import B200CLIPTextEncoder
    B = 2
    sd1, sd2 = _weights(768, 12, 2, 3072, seed=1), _weights(1280, 20, 2, 5120, proj=1280, seed=2)
    ids1, ids2 = _ids(B, 77, 49408, True), _ids(B, 77, 49408, False)
    enc1 = B200CLIPTextEncoder(sd1, num_attention_heads=12, hidden_act="quick_gelu", eos_token_id=2, dtype=torch.float16)
    enc2 = B200CLIPTextEncoder(sd2, num_attention_heads=20, hidden_act="gelu", eos_token_id=49407, dtype=torch.float16)
    o1, o2 = enc1(ids1.cuda(), output_hidden_states=True), enc2(ids2.cuda(), output_hidden_states=True)
    prompt_embeds = torch.concat([o1.hidden_states[-2], o2.hidden_states[-2]], dim=-1)
    torch.cuda.synchronize()
    assert prompt_embeds.shape == (B, 77, 2048) and o2[0].shape == (B, 1280)
    (t1, _, _, _), (e1, _, _, _) = _truth_and_eager(sd1, ids1, 12, "quick_gelu", 2, torch.float16)
    (t2, _, _, te2), (e2, _, _, tee2) = _truth_and_eager(sd2, ids2, 20, "gelu", 49407, torch.float16)
    _cmp("SDXL prompt_embeds", prompt_embeds, torch.cat([t1[-2], t2[-2]], -1), torch.cat([e1[-2], e2[-2]], -1))
    _cmp("SDXL pooled_prompt_embeds", o2[0], te2, tee2)
