"""CLIP text encoder (SD1.5 ``text_encoder`` ViT-L/14, SDXL ``text_encoder_2`` ViT-bigG/14) on the CPU: tests/clip_text_ref.text_hidden_states
pinned against the installed transformers ``CLIPTextModel`` / ``CLIPTextModelWithProjection``, and the host logic of
consistentid_b200.clip.B200CLIPTextEncoder (weight packing, padded layout, EOS pooling, output structure) on emulated kernels."""
import pytest
import torch
import torch.nn.functional as F

from oracle import clip_ref
from tests import clip_text_ref, emulated_ops

transformers = pytest.importorskip("transformers")

VOCAB = 100
BOS, EOS_MAX = 98, 99        # the real tokenizers' bos / eos are the two largest ids (49406 / 49407)


def _ids(B, L, eos_tok, pad_tok, seed=0):
    """Tokenizer-shaped sequences: BOS, a prompt of varying length, EOS, then padding (EOS for the SD1.5 tokenizer, 0 for SDXL's
    tokenizer_2).  Prompt tokens avoid eos_tok, so the pooled row tells the argmax rule from the first-EOS rule."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.full((B, L), pad_tok, dtype=torch.int64)
    for b in range(B):
        n = 1 + (b * 7 + 3) % (L - 2)
        body = torch.randint(3, 97, (n,), generator=g)
        body[body == eos_tok] = 3
        ids[b, 0], ids[b, 1:1 + n], ids[b, 1 + n] = BOS, body, eos_tok
    return ids


def _model(act, eos_cfg, proj, layers=2, C=64, heads=4, inter=128, n_pos=77):
    from transformers import CLIPTextConfig, CLIPTextModel, CLIPTextModelWithProjection
    torch.manual_seed(0)
    cfg = CLIPTextConfig(vocab_size=VOCAB, hidden_size=C, intermediate_size=inter, num_hidden_layers=layers, num_attention_heads=heads,
                         max_position_embeddings=n_pos, hidden_act=act, projection_dim=32, bos_token_id=BOS, eos_token_id=eos_cfg, pad_token_id=1)
    m = (CLIPTextModelWithProjection if proj else CLIPTextModel)(cfg).eval()
    for p in m.parameters():                                   # default init leaves biases at zero: make every term count
        if p.ndim == 1:
            p.data += 0.1 * torch.randn_like(p)
    return m


CASES = [  # act, eos_token_id in the config, eos token of the sequences, pad token, L, projection
    ("quick_gelu", 2, EOS_MAX, EOS_MAX, 77, False),            # SD1.5: legacy eos id, pad with EOS
    ("quick_gelu", 2, EOS_MAX, 0, 20, True),
    ("gelu", 50, 50, 0, 77, True),                             # SDXL text_encoder_2: first-EOS rule, pad with "!"
    ("gelu", 50, 50, 50, 13, False),
]


@pytest.mark.parametrize("act,eos_cfg,eos_tok,pad_tok,L,proj", CASES)
def test_clip_text_oracle_matches_transformers(act, eos_cfg, eos_tok, pad_tok, L, proj):
    m = _model(act, eos_cfg, proj)
    ids = _ids(3, L, eos_tok, pad_tok)
    with torch.no_grad():
        want = m(ids, output_hidden_states=True)
    hs, last, pooled, text_embeds = clip_text_ref.text_hidden_states(m.state_dict(), ids, 4, act, eos_cfg)
    assert len(hs) == len(want.hidden_states) == 3 and last.shape == (3, L, 64)
    close = lambda g, w: torch.allclose(g, w, atol=2e-5, rtol=2e-5)
    for g, w in zip(hs, want.hidden_states):
        assert close(g, w), (g - w).abs().max()
    assert close(last, want.last_hidden_state)
    if proj:
        assert close(text_embeds, want.text_embeds)
        with torch.no_grad():                                   # the projection variant reports no pooler_output: compare with the base model
            assert close(pooled, m.text_model(ids).pooler_output)
    else:
        assert text_embeds is None and close(pooled, want.pooler_output)


@pytest.mark.parametrize("act", ["gelu", "quick_gelu"])
def test_causal_layer_last_row_matches_the_unmasked_layer(act):
    """The last query sees every key, so it matches oracle/clip_ref.encoder_layer (the vision encoder's unmasked layer); the first does not."""
    m = _model(act, 50, False, layers=1)
    x = torch.randn(2, 9, 64)
    sd = m.state_dict()
    p = "text_model.encoder.layers.0"
    a, c = clip_ref.encoder_layer(sd, p, x, 4, act), clip_text_ref.causal_encoder_layer(sd, p, x, 4, act)
    assert torch.allclose(a[:, -1], c[:, -1], atol=1e-5) and not torch.allclose(a[:, 0], c[:, 0], atol=1e-3)


# ---- the engine's host logic on emulated kernels (fp32, device="cpu")
def _gemm(a, w, out, *args, epi=0, **kw):
    from consistentid_b200.lib import EPI_QUICK_GELU
    if epi != EPI_QUICK_GELU:
        return emulated_ops.gemm(a, w, out, *args, epi=epi, **kw)
    emulated_ops.gemm(a, w, out, *args, **kw)                   # the store epilogue, then q(x) = x sigmoid(1.702 x) on it
    out.copy_(out * torch.sigmoid(1.702 * out))
    return out


def _attn_self_causal(q, k, vt, out, B, H, N, d):
    v = vt.float().view(B, H, d, N).transpose(2, 3)
    o = F.scaled_dot_product_attention(emulated_ops._heads(q, B, N, H, d), emulated_ops._heads(k, B, N, H, d), v, is_causal=True)
    out.copy_(o.transpose(1, 2).reshape(B * N, H * d))
    return out


def _embed_tokens(ids, tok, pos, out, Lp):
    B, L = ids.shape
    V = tok.shape[0]
    ok = (ids >= 0) & (ids < V)
    rows = torch.where(ok[..., None], tok[ids.clamp(0, V - 1)], torch.zeros(())) + pos[:L]
    o = out.view(B, Lp, -1)
    o.zero_()
    o[:, :L] = rows
    return out


@pytest.fixture
def emulated(monkeypatch):
    from consistentid_b200 import ops
    emulated_ops.install(monkeypatch)
    monkeypatch.setattr(ops, "gemm", _gemm)
    monkeypatch.setattr(ops, "attn_self_causal", _attn_self_causal)
    monkeypatch.setattr(ops, "embed_tokens", _embed_tokens)


@pytest.mark.parametrize("act,eos_cfg,eos_tok,pad_tok,L,proj", CASES)
def test_text_encoder_host_logic_on_emulated_kernels(emulated, act, eos_cfg, eos_tok, pad_tok, L, proj):
    from consistentid_b200.clip import B200CLIPTextEncoder
    m = _model(act, eos_cfg, proj)
    sd = m.state_dict()
    ids = _ids(2, L, eos_tok, pad_tok, seed=1)
    hs, last, pooled, text_embeds = clip_text_ref.text_hidden_states(sd, ids, 4, act, eos_cfg)
    enc = B200CLIPTextEncoder(sd, num_attention_heads=4, hidden_act=act, eos_token_id=eos_cfg, dtype=torch.float32, device="cpu")
    assert enc.config.use_attention_mask is False and enc.config.hidden_size == 64 and enc.config.num_hidden_layers == 2
    assert enc.config.projection_dim == (32 if proj else None)
    out = enc(ids, output_hidden_states=True)
    close = lambda g, w: g.shape == w.shape and torch.allclose(g, w, atol=1e-4, rtol=1e-4)
    assert len(out.hidden_states) == len(hs)
    for g, w in zip(out.hidden_states, hs):
        assert close(g, w), (g - w).abs().max()
    assert close(out.last_hidden_state, last) and close(out.pooler_output, pooled)
    if proj:
        assert close(out.text_embeds, text_embeds) and out[0] is out.text_embeds and out[1] is out.last_hidden_state
    else:
        assert out.text_embeds is None and out[0] is out.last_hidden_state and out[1] is out.pooler_output
    assert out[-1] is out.hidden_states
    plain = enc(ids, attention_mask=None)                        # diffusers _encode_prompt: no hidden states
    assert plain.hidden_states is None and len(plain.to_tuple()) == 2 and close(plain[0], out[0])


def test_text_encoder_rejects_attention_mask_and_bad_ids(emulated):
    from consistentid_b200.clip import B200CLIPTextEncoder
    enc = B200CLIPTextEncoder(_model("quick_gelu", 2, False, layers=1).state_dict(), num_attention_heads=4, dtype=torch.float32, device="cpu")
    ids = _ids(1, 77, EOS_MAX, EOS_MAX)
    with pytest.raises(NotImplementedError):
        enc(ids, attention_mask=torch.ones_like(ids))
    with pytest.raises(ValueError):
        enc(torch.zeros(1, 78, dtype=torch.int64))              # more tokens than positions
    with pytest.raises(TypeError):
        enc(ids.float())


def test_embed_tokens_rejects_out_of_range_host_ids():
    """The wrapper range-checks host ids before anything reaches the device (on-device ids read a zero token row instead)."""
    from consistentid_b200 import ops
    tok, pos = torch.zeros(10, 8, dtype=torch.float16), torch.zeros(77, 8, dtype=torch.float16)
    out = torch.empty(8, 8, dtype=torch.float16)
    for bad in (10, -1):
        with pytest.raises(ValueError):
            ops.embed_tokens(torch.tensor([[1, bad]]), tok, pos, out, 8)
    with pytest.raises(TypeError):
        ops.embed_tokens(torch.tensor([[1, 2]], dtype=torch.int32), tok, pos, out, 8)
