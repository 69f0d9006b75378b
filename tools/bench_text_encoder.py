"""Per-call time of the CLIP text encoders on one GPU: consistentid_b200.clip.B200CLIPTextEncoder against the 16-bit eager oracle
(tests/clip_text_ref.text_hidden_states: stock PyTorch kernels, no graph), each with its max error against the fp32 oracle (TF32 off) on the same
seeded weights and token ids.  SD1.5 / SDXL ``text_encoder`` = OpenAI ViT-L/14 (B = 1, 3), SDXL ``text_encoder_2`` = OpenCLIP ViT-bigG/14
(B = 1, 2), fp16 and bf16, 77 tokens, called as SDXL calls them: ``enc(ids, output_hidden_states=True)`` with the ids on the device.
Times are CUDA-event means over warmed calls; the weights (0.25 GB / 1.39 GB in 16 bit) exceed the 126 MB L2.  Prints one JSON line with
the GPU name, power limit and max SM clock read in the same run.
    python tools/bench_text_encoder.py [--calls 20] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from consistentid_b200.clip import B200CLIPTextEncoder  # noqa: E402
from tests.clip_text_ref import text_hidden_states  # noqa: E402
from tests.test_clip_text_gpu import _ids, _weights  # noqa: E402

MODELS = {  # C, heads, layers, MLP, act, eos_token_id, pad with EOS, projection, batches
    "vit_l14": (768, 12, 12, 3072, "quick_gelu", 2, True, None, (1, 3)),
    "vit_bigg14": (1280, 20, 32, 5120, "gelu", 49407, False, 1280, (1, 2)),
}


def _time(fn, calls):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def _err(a, b):
    return (a.float().cpu() - b.float().cpu()).abs().max().item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_text_encoder: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"tool": "tools/bench_text_encoder.py", "gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip().splitlines()[:1],
           "calls_timed": args.calls, "unit": "ms per call", "rows": []}
    for name, (C, heads, layers, inter, act, eos, pad_eos, proj, batches) in MODELS.items():
        sd = _weights(C, heads, layers, inter, proj=proj)
        sd32 = {k: v.cuda() for k, v in sd.items()}
        for dtype in (torch.float16, torch.bfloat16):
            enc = B200CLIPTextEncoder(sd, num_attention_heads=heads, hidden_act=act, eos_token_id=eos, dtype=dtype)
            sd16 = {k: v.cuda().to(dtype) for k, v in sd.items()}
            for B in batches:
                ids = _ids(B, 77, 49408, pad_eos).cuda()
                with torch.no_grad():
                    hs_t, _, pooled_t, te_t = text_hidden_states(sd32, ids, heads, act, eos)
                    eager = lambda: text_hidden_states(sd16, ids, heads, act, eos)
                    hs_e, _, pooled_e, te_e = eager()
                out = enc(ids, output_hidden_states=True)
                pooled_ours, pooled_truth, pooled_eager = (out.text_embeds, te_t, te_e) if proj else (out.pooler_output, pooled_t, pooled_e)
                with torch.no_grad():
                    ms_eager = _time(eager, args.calls)
                ms_ours = _time(lambda: enc(ids, output_hidden_states=True), args.calls)
                row = {"model": name, "batch": B, "dtype": str(dtype)[6:], "ms_b200": round(ms_ours, 3), "ms_eager16": round(ms_eager, 3),
                       "max_err_hidden_states[-2]": {"b200": _err(out.hidden_states[-2], hs_t[-2]), "eager16": _err(hs_e[-2], hs_t[-2])},
                       "max_err_" + ("text_embeds" if proj else "pooler_output"): {"b200": _err(pooled_ours, pooled_truth),
                                                                                  "eager16": _err(pooled_eager, pooled_truth)},
                       "max_abs_truth_hidden_states[-2]": hs_t[-2].abs().max().item()}
                res["rows"].append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
            del enc, sd16
        del sd32
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
