"""CPU: pin the oracle's restatement of the reference processors against (a) golden vectors generated from the verbatim
reference (tests/golden/make_golden.py) and (b) the whole tiny UNet run with the verbatim reference processors (tests/golden/make_pinned_golden.py)."""
import os

import pytest
import torch

from oracle.processors_ref import ConsistentAttnRef, ConsistentIPAttnRef
from oracle.unet_ref import Attention

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "processors_golden.pt")
PINNED = os.path.join(os.path.dirname(__file__), "golden", "pinned_golden.pt")


@pytest.fixture(scope="module")
def pinned():
    return torch.load(PINNED, map_location="cpu", weights_only=True)


def _build(case):
    m = case["meta"]
    a1, a2 = Attention(m["C"], None, m["heads"], m["C"] // m["heads"]), Attention(m["C"], m["cad"], m["heads"], m["C"] // m["heads"])
    a1.load_state_dict(case["attn1"]); a2.load_state_dict(case["attn2"])
    p1 = ConsistentAttnRef(hidden_size=m["C"], cross_attention_dim=None, rank=m["rank"])
    p2 = ConsistentIPAttnRef(hidden_size=m["C"], cross_attention_dim=m["cad"], rank=m["rank"], scale=m["scale"], num_tokens=4)
    p1.load_state_dict(case["proc1"], strict=True)      # same parameter names as the reference processors
    p2.load_state_dict(case["proc2"], strict=True)
    return a1, a2, p1, p2


@pytest.mark.parametrize("idx", [0, 1, 2])
def test_oracle_matches_reference_golden(idx):
    case = torch.load(GOLDEN)[idx]
    a1, a2, p1, p2 = _build(case)
    with torch.no_grad():
        y1 = p1(a1, case["x"])
        y2 = p2(a2, case["x"], encoder_hidden_states=case["ehs"])
    assert torch.allclose(y1, case["y_self"], rtol=1e-5, atol=1e-5)
    assert torch.allclose(y2, case["y_cross"], rtol=1e-5, atol=1e-5)


def test_oracle_4d_input_path():
    case = torch.load(GOLDEN)[0]
    a1, a2, p1, p2 = _build(case)
    B, N, C = case["x"].shape
    x4 = case["x"].transpose(1, 2).reshape(B, C, 8, N // 8)
    with torch.no_grad():
        y = p2(a2, x4, encoder_hidden_states=case["ehs"])
    assert torch.allclose(y.reshape(B, C, N).transpose(1, 2), case["y_cross"], rtol=1e-5, atol=1e-5)


def test_oracle_matches_verbatim_reference_full_unet(pinned):
    """The tiny UNet with the oracle's processors against the same UNet with the original processors (tests/golden/make_pinned_golden.py):
    same parameter layout per processor, same output."""
    from oracle import synth
    from oracle.unet_ref import tiny_config
    cfg = tiny_config("sd15")
    cfg.sample_size = 16
    unet = synth.build_ref_unet(cfg, rank=8)
    mine = unet.attn_processors
    assert sorted(mine) == sorted(pinned["unet"]["layout"])
    for name, p in mine.items():
        assert [(k, tuple(v.shape)) for k, v in p.state_dict().items()] == [tuple(e) for e in pinned["unet"]["layout"][name]], name
    null, aug, _ = synth.synth_prompts(cfg.cross_attention_dim)
    x = synth.synth_latents(2, 16, 16)
    ehs = torch.cat([null, aug])
    with torch.no_grad():
        y_mine = unet(x, torch.tensor(500), ehs).sample
    assert torch.allclose(y_mine, pinned["unet"]["y"], rtol=1e-4, atol=1e-5)


# ---- independent cross-check of the (otherwise unpinned) diffusers restatement: TVM's relax port of diffusers' get_timestep_embedding,
# evaluated by tests/golden/make_pinned_golden.py
@pytest.mark.parametrize("dim,flip,shift", [(320, True, 0.0), (256, True, 0.0), (320, False, 1.0)])
def test_timestep_embedding_matches_the_tvm_port_of_diffusers(pinned, dim, flip, shift):
    """unet_ref.get_timestep_embedding (diffusers 0.23 restated, parity otherwise unpinned) against an independent port of the same function."""
    from oracle.unet_ref import get_timestep_embedding
    c = next(c for c in pinned["timestep_embedding"] if (c["dim"], c["flip_sin_to_cos"], c["downscale_freq_shift"]) == (dim, flip, shift))
    ours = get_timestep_embedding(c["timesteps"], dim, flip_sin_to_cos=flip, downscale_freq_shift=shift)
    theirs = c["y"]
    assert ours.shape == theirs.shape
    assert (ours - theirs).abs().max().item() < 2e-4      # fp32 sin/cos of arguments up to ~1e3 rad: ulp-level differences of the product; a layout or formula mismatch would be O(1)
