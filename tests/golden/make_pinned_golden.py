"""Generate ``pinned_golden.pt``: what three CPU tests compare the oracle with, recorded once from code outside this repository so
that the tests run anywhere.

* ``unet`` (tests/test_oracle_cpu.py): the tiny SD1.5 UNet of ``oracle.synth`` (sample 16, LoRA rank 8) with every attention
  processor replaced by the original project's ``Consistent_AttProcessor`` / ``Consistent_IPAttProcessor`` (its ``attention.py``
  imported verbatim through the 2-symbol ``oracle/diffusers_shim``), carrying the oracle processors' weights: the output, and the
  state-dict layout of every original processor.
* ``proj_plus`` (tests/test_embed_cpu.py): the original ``ProjPlusModel`` at full width (cross-attention 768, ID 512, CLIP 1280,
  257 patches) on weights from ``oracle.synth.seeded_params`` (too large to store): the layout, the seeds and the output.
* ``timestep_embedding`` (tests/test_oracle_cpu.py): TVM's relax port of diffusers' ``get_timestep_embedding``
  (``tvm/relax/frontend/nn/op.py``), its source executed with the relax ops bound to numpy, no TVM runtime needed.

    python tests/golden/make_pinned_golden.py --reference <ConsistentID checkout> --tvm-op <tvm>/python/tvm/relax/frontend/nn/op.py
"""
import argparse
import ast
import math
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import synth  # noqa: E402
from oracle.processors_ref import ConsistentIPAttnRef  # noqa: E402
from oracle.unet_ref import tiny_config  # noqa: E402

TIMESTEPS = [0, 1, 33, 500, 961, 999]
EMBED_CASES = [(320, True, 0.0), (256, True, 0.0), (320, False, 1.0)]   # (dim, flip_sin_to_cos, downscale_freq_shift)


def unet_case(ref_attention):
    cfg = tiny_config("sd15")
    cfg.sample_size = 16
    unet = synth.build_ref_unet(cfg, rank=8)
    theirs, layout = {}, {}
    for name, p in unet.attn_processors.items():
        if isinstance(p, ConsistentIPAttnRef):
            rp = ref_attention.Consistent_IPAttProcessor(p.hidden_size, p.cross_attention_dim, rank=8, num_tokens=4)
        else:
            rp = ref_attention.Consistent_AttProcessor(p.to_q_lora.down.in_features, None, rank=8)
        rp.load_state_dict(p.state_dict(), strict=True)
        theirs[name] = rp
        layout[name] = [(k, tuple(v.shape)) for k, v in rp.state_dict().items()]
    null, aug, _ = synth.synth_prompts(cfg.cross_attention_dim)
    x = synth.synth_latents(2, 16, 16)
    unet.set_attn_processor(theirs)
    with torch.no_grad():
        y = unet(x, torch.tensor(500), torch.cat([null, aug])).sample
    return dict(layout=layout, y=y)


def proj_plus_case(ref_functions, seed=5):
    m = ref_functions.ProjPlusModel(cross_attention_dim=768, id_embeddings_dim=512, clip_embeddings_dim=1280, num_tokens=4).eval()
    shapes = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    m.load_state_dict(synth.seeded_params(shapes, seed), strict=True)
    g = torch.Generator().manual_seed(seed + 1)
    idv, clip = torch.randn(1, 512, generator=g), torch.randn(1, 257, 1280, generator=g)
    with torch.no_grad():
        y = m(idv, clip)
    return dict(shapes=shapes, weight_seed=seed, input_seed=seed + 1, y=y)


def tvm_timestep_embedding(tvm_op, timesteps, dim, **kw):
    """Execute the SOURCE of tvm.relax.frontend.nn.op.get_timestep_embedding (a third-party port of the diffusers function, SURVEY
    Appendix A) with its relax ops bound to numpy: the port's own arithmetic graph, evaluated without a TVM runtime."""
    src = open(tvm_op).read()
    node = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "get_timestep_embedding")
    node.returns = None
    for a in node.args.args:
        a.annotation = None
    code = compile(ast.Module(body=[node], type_ignores=[]), tvm_op, "exec")
    f32 = lambda x: np.asarray(x, dtype=np.float32)
    op = types.SimpleNamespace(
        astype=lambda x, dt: f32(x), arange=lambda start, end, dtype: np.arange(start, end, dtype=np.float32), exp=lambda x: np.exp(f32(x)),
        expand_dims=lambda x, ax: np.expand_dims(x, ax), concat=lambda xs, axis: np.concatenate(xs, axis=axis), cos=lambda x: np.cos(f32(x)),
        sin=lambda x: np.sin(f32(x)), nn=types.SimpleNamespace(pad=lambda x, p: np.pad(x, ((p[2], p[3]), (p[0], p[1])))))
    ns = dict(math=math, _op=op, rx=types.SimpleNamespace(const=lambda v, dt: np.float32(v)), get_default_dtype=lambda: "float32",
              wrap_nested=lambda e, name: e, Tensor=object)
    exec(code, ns)
    return ns["get_timestep_embedding"](types.SimpleNamespace(_expr=np.asarray(timesteps)), dim, **kw)


def embedding_cases(tvm_op):
    t = np.asarray(TIMESTEPS)
    return [dict(dim=dim, flip_sin_to_cos=flip, downscale_freq_shift=shift, timesteps=torch.tensor(TIMESTEPS),
                 y=torch.from_numpy(np.asarray(tvm_timestep_embedding(tvm_op, t, dim, flip_sin_to_cos=flip, downscale_freq_shift=shift),
                                               dtype=np.float32)))
            for dim, flip, shift in EMBED_CASES]


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of the original ConsistentID project (attention.py, functions.py)")
    ap.add_argument("--tvm-op", required=True, help="tvm/relax/frontend/nn/op.py of a TVM source tree")
    args = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "oracle", "diffusers_shim"))
    sys.path.insert(0, os.path.abspath(args.reference))
    import attention as ref_attention  # noqa: E402  (the original, verbatim)
    import functions as ref_functions  # noqa: E402  (the original, verbatim)
    golden = dict(unet=unet_case(ref_attention), proj_plus=proj_plus_case(ref_functions), timestep_embedding=embedding_cases(args.tvm_op))
    out = os.path.join(HERE, "pinned_golden.pt")
    torch.save(golden, out)
    print("wrote", out, os.path.getsize(out) // 1024, "KiB")
