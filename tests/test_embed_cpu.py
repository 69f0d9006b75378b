"""oracle/embed_ref.py (restated embedding producers, SURVEY.md 8f-1) against golden vectors generated from the reference's own
ProjPlusModel / AttentionMLP / FuseModule / FacialEncoder classes (tests/golden/make_embed_golden.py)."""
import os

import pytest
import torch

from oracle import embed_ref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "embed_golden.pt")
PINNED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pinned_golden.pt")


@pytest.fixture(scope="module")
def golden():
    return torch.load(GOLD, map_location="cpu", weights_only=True)


def _close(a, b, tol=2e-5):
    assert a.shape == b.shape
    assert (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item()), (a - b).abs().max().item()


def test_proj_plus_model_matches_reference(golden):
    n = 0
    for c in golden:
        if c["kind"] != "proj_plus":
            continue
        _close(embed_ref.proj_plus_model(c["sd"], c["id_embeds"], c["clip_embeds"]), c["y"])
        _close(embed_ref.proj_plus_model(c["sd"], c["id_embeds"], c["clip_embeds"], shortcut=True, scale=c["shortcut_scale"]), c["y_shortcut"])
        n += 1
    assert n >= 2


def test_facial_encoder_matches_reference(golden):
    n = 0
    for c in golden:
        if c["kind"] != "facial_encoder":
            continue
        bs, k, tl, idim = c["multi_image_embeds"].shape
        _close(embed_ref.attention_mlp(c["sd"], c["multi_image_embeds"].reshape(bs * k, tl, idim)), c["visual_projection"])
        for case in c["cases"]:
            y = embed_ref.facial_encoder(c["sd"], c["prompt_embeds"], c["multi_image_embeds"], case["class_tokens_mask"], case["valid_id_mask"])
            _close(y, case["y"])
            untouched = ~case["class_tokens_mask"]
            assert torch.equal(y[untouched], c["prompt_embeds"][untouched])      # only the <|facial|> rows change
            n += 1
    assert n >= 4


def test_facial_encoder_mask_mismatch_raises(golden):
    c = next(c for c in golden if c["kind"] == "facial_encoder")
    cm = c["cases"][0]["class_tokens_mask"].clone()
    cm[0, 70] = True                                                               # one more token than valid ids (attention.py:44 assert)
    with pytest.raises(AssertionError):
        embed_ref.facial_encoder(c["sd"], c["prompt_embeds"], c["multi_image_embeds"], cm, c["cases"][0]["valid_id_mask"])


def test_assemble_prompts_layout():
    D = 8
    f, uf, t = torch.ones(1, 77, D), 2 * torch.ones(1, 77, D), 3 * torch.ones(1, 77, D)
    idt, uidt = 4 * torch.ones(1, 4, D), 5 * torch.ones(1, 4, D)
    null, aug, txt = embed_ref.assemble_prompts(f, uf, t, idt, uidt)
    assert null.shape == aug.shape == txt.shape == (1, 81, D)
    assert (null[:, :77] == 2).all() and (null[:, 77:] == 5).all()
    assert (aug[:, :77] == 1).all() and (aug[:, 77:] == 4).all()
    assert (txt[:, :77] == 3).all() and (txt[:, 77:] == 4).all()


def test_full_width_against_verbatim_reference():
    """Full-width ProjPlusModel (cad 768, CLIP 1280, 257 patches) against the reference class's output on the same seeded weights and
    inputs (tests/golden/make_pinned_golden.py; the weights are rebuilt from their layout and seed, too large to store)."""
    from oracle import synth
    c = torch.load(PINNED, map_location="cpu", weights_only=True)["proj_plus"]
    sd = synth.seeded_params([(k, tuple(s)) for k, s in c["shapes"]], c["weight_seed"])
    g = torch.Generator().manual_seed(c["input_seed"])
    idv, clip = torch.randn(1, 512, generator=g), torch.randn(1, 257, 1280, generator=g)
    _close(embed_ref.proj_plus_model(sd, idv, clip), c["y"])
