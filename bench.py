#!/usr/bin/env python
"""bench.py - images/sec of the ConsistentID denoising hot path (BASELINE.json metric) on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload sd15|sdxl] [--impl ours|reference] [--dump-outputs DIR]
  torchrun launches it once per GPU for N > 1 (RANK / LOCAL_RANK / WORLD_SIZE from the environment).

A bench "step" = ONE pass of the hot path over one batch: the full denoising loop (UNet x 2B with the ConsistentID
attention processors + CFG combine + scheduler step, `denoise_steps` iterations) for `per_gpu_batch` images per GPU.
  value  images/s with inputs resident in HBM, timed with CUDA events around K steps, max over ranks
  e2e    same metric through the public API (B200Denoiser.__call__) from PINNED HOST buffers: H2D of latents + prompt
         embeddings and D2H of the final latents inside the timed region, every step
  roofline / cpu_baseline / clocks / gpu_launches: see DESIGN.md "Measurement"
Weights are random-init tensors of the exact architecture, inputs synthetic (no network for checkpoints/datasets).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: SD1.5 ConsistentID 512x512 batch=8, 30 steps, fp16, 1xB200
    "sd15": dict(model="sd15", res=512, batch=8, denoise_steps=30, dtype="fp16", scheduler="ddim", guidance=5.0, start_merge_step=0,
                 tflop_per_sample_forward=0.8036),
    # BASELINE.json configs[2]: SDXL ConsistentID 1024x1024 batch=4, 30 steps, bf16, 1xB200
    "sdxl": dict(model="sdxl", res=1024, batch=4, denoise_steps=30, dtype="bf16", scheduler="euler", guidance=7.5, start_merge_step=0,
                 tflop_per_sample_forward=6.7657),
    # north_star target config: SDXL 1024x1024 batch 8 on 1xB200 (">= 5x the reference diffusers-CUDA pipeline")
    "sdxl_b8": dict(model="sdxl", res=1024, batch=8, denoise_steps=30, dtype="bf16", scheduler="euler", guidance=7.5, start_merge_step=0,
                    tflop_per_sample_forward=6.7657),
    # BASELINE.json configs[4]: SD1.5 ControlNet+Inpaint ConsistentID 512x512 batch=8, 50 steps, dual-network path (blend variant, 4-ch UNet)
    "sd15_cn": dict(model="sd15", res=512, batch=8, denoise_steps=50, dtype="fp16", scheduler="ddim", guidance=5.0, start_merge_step=0,
                    tflop_per_sample_forward=0.8036, controlnet=True, controlnet_tflop_per_image_step=0.283),
    # reduced-width variants for quick functional runs (NOT a bench result)
    "tiny": dict(model="tiny_sd15", res=256, batch=2, denoise_steps=4, dtype="fp16", scheduler="ddim", guidance=5.0, start_merge_step=0,
                 tflop_per_sample_forward=None),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            self.path = tempfile.mktemp(suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 9:
                rows.append(f)
        if rows:
            sm = sorted(float(r[1]) for r in rows if r[1].replace(".", "").isdigit())
            out["samples"] = len(rows)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
            try:
                out["sm_max_mhz"] = float(rows[0][2])
                out["power_w_max"] = max(float(r[3]) for r in rows)
            except Exception:
                pass
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for k, nm in enumerate(names):
                if any(r[5 + k].lower().startswith("active") for r in rows):
                    out["reasons"].append(nm)
        try:
            os.unlink(self.path)
        except Exception:
            pass
        return out


def synth_inputs(spec, B, h, w, seed, sdxl):
    """Synthetic inputs of SURVEY.md 8d on the HOST (pinned): latents + three [1,81,cad] prompt tensors (+ pooled / time ids)."""
    import torch
    import torch.nn.functional as F
    cad = spec.cross_attention_dim
    g = lambda s: torch.Generator().manual_seed(s)
    lat = torch.randn(B, 4, h, w, generator=g(seed))
    id_rows = F.layer_norm(torch.randn(1, 4, cad, generator=g(4)), (cad,))
    prompts = [torch.cat([torch.randn(1, 77, cad, generator=g(1 + k)), id_rows], 1) for k in range(3)]
    extra = {}
    if sdxl:
        extra = dict(neg_pooled=torch.randn(1, 1280, generator=g(5)), pooled_text_only=torch.randn(1, 1280, generator=g(6)),
                     pooled_facial=torch.randn(1, 1280, generator=g(7)), add_time_ids=torch.tensor([[1024., 1024., 0., 0., 1024., 1024.]]))
    return lat, prompts, extra


def _physical_cores_one_socket():
    """CPU ids of the physical cores (one hardware thread each) of ONE socket, restricted to this process's affinity mask: the thread
    count of the CPU arms.  os.cpu_count() threads on a 2-socket SMT host oversubscribes torch's intra-op pool and made the same arm
    swing 10x between boxes (VERDICT r1 weak #7)."""
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    try:
        cores, cur = {}, {}
        for line in open("/proc/cpuinfo"):
            if ":" not in line:
                if "processor" in cur:
                    cores.setdefault((cur.get("physical id", "0"), cur.get("core id", cur["processor"])), int(cur["processor"]))
                cur = {}
                continue
            k, v = line.split(":", 1)
            cur[k.strip()] = v.strip()
        if "processor" in cur:
            cores.setdefault((cur.get("physical id", "0"), cur.get("core id", cur["processor"])), int(cur["processor"]))
        by_socket = {}
        for (sock, _), cpu in cores.items():
            if cpu in allowed:
                by_socket.setdefault(sock, []).append(cpu)
        if by_socket:
            best = max(by_socket.values(), key=len)
            return sorted(best)
    except Exception:
        pass
    return allowed


def _build_controlnet(spec, dev, dtype, rankN, wl, B, h):
    import torch
    from consistentid_b200.arch import synth_state_dicts
    from consistentid_b200.controlnet import B200ControlNet
    gcn = torch.Generator(device=dev).manual_seed(4321)
    cn_sd = {k: v for k, v in synth_state_dicts(spec, dev, dtype, seed=99, rank=rankN)[0].items()
             if k.startswith(("conv_in", "time_embedding", "down_blocks", "mid_block"))}

    def rw(*shape):
        fan = 1
        for x_ in shape[1:]:
            fan *= x_
        return (torch.randn(shape, generator=gcn, device=dev) * fan ** -0.5).to(dtype)
    ch = (16, 32, 96, 256)
    cn_sd["controlnet_cond_embedding.conv_in.weight"], cn_sd["controlnet_cond_embedding.conv_in.bias"] = rw(ch[0], 3, 3, 3), rw(ch[0])
    for i in range(3):
        cn_sd[f"controlnet_cond_embedding.blocks.{2*i}.weight"], cn_sd[f"controlnet_cond_embedding.blocks.{2*i}.bias"] = rw(ch[i], ch[i], 3, 3), rw(ch[i])
        cn_sd[f"controlnet_cond_embedding.blocks.{2*i+1}.weight"], cn_sd[f"controlnet_cond_embedding.blocks.{2*i+1}.bias"] = rw(ch[i + 1], ch[i], 3, 3), rw(ch[i + 1])
    c0 = spec.block_out_channels[0]
    cn_sd["controlnet_cond_embedding.conv_out.weight"], cn_sd["controlnet_cond_embedding.conv_out.bias"] = rw(c0, ch[3], 3, 3), rw(c0)
    zc = [c0] + [c for i, c in enumerate(spec.block_out_channels) for _ in range(spec.layers_per_block + (0 if i == len(spec.block_out_channels) - 1 else 1))]
    for j, c in enumerate(zc):
        cn_sd[f"controlnet_down_blocks.{j}.weight"], cn_sd[f"controlnet_down_blocks.{j}.bias"] = rw(c, c, 1, 1), rw(c)
    cn_sd["controlnet_mid_block.weight"], cn_sd["controlnet_mid_block.bias"] = rw(zc[-1], zc[-1], 1, 1), rw(zc[-1])
    cnet = B200ControlNet(spec, cn_sd, dtype=dtype, device=dev)
    gh = torch.Generator().manual_seed(7)
    ctrl_h = torch.rand(B, 3, wl["res"], wl["res"], generator=gh).to(dtype).pin_memory()
    img_h = torch.randn(B, 4, h, h, generator=gh).pin_memory(); noise_h = torch.randn(B, 4, h, h, generator=gh).pin_memory()
    mask_h = torch.zeros(B, 1, h, h); mask_h[:, :, h // 4: 3 * h // 4, h // 4: 3 * h // 4] = 1; mask_h = mask_h.pin_memory()
    return cnet, ctrl_h, img_h, noise_h, mask_h


def bench_workload(args, name, steps, warmup, rank, local, world):
    """Time ONE workload (see WORKLOADS) on this rank's GPU: device-resident `value`, host-buffer `e2e`, per-launch roofline pass.
    Returns the result block (same keys as the headline line)."""
    import torch
    from consistentid_b200 import dist as cdist, lib
    from consistentid_b200.arch import sd15_spec, sdxl_spec, synth_state_dicts, UNetSpec
    from consistentid_b200.pipeline import B200Denoiser
    from consistentid_b200.scheduler import B200Scheduler
    from consistentid_b200.unet import B200UNet

    dev = torch.device("cuda", local)
    wl = WORKLOADS[name]
    dtype = torch.float16 if wl["dtype"] == "fp16" else torch.bfloat16
    if wl["model"] == "sd15":
        spec = sd15_spec()
    elif wl["model"] == "sdxl":
        spec = sdxl_spec()
    else:
        spec = UNetSpec(block_out_channels=(64, 128, 256, 256), num_attention_heads=(2, 2, 4, 4), cross_attention_dim=128, sample_size=32, name="tiny_sd15")
    sdxl = spec.addition_embed_type == "text_time"
    B, h = wl["batch"], wl["res"] // 8
    n_steps = wl["denoise_steps"]
    rankN = 16 if wl["model"].startswith("tiny") else 128

    # weights: every rank builds the layout, rank 0's packed arena is broadcast ONCE (the only collective of the run)
    t0 = time.time()
    usd, asd = synth_state_dicts(spec, dev, dtype, seed=1234, rank=rankN)
    unet = B200UNet(spec, usd, asd, dtype=dtype, device=dev, rank=rankN)
    del usd, asd
    if world > 1:
        if rank != 0:
            unet.params.arena.zero_()
        cdist.broadcast_arena(unet.params.arena, src=0)
        # every rank must now hold rank 0's bytes: compare an integer checksum of the arena across ranks
        chk = unet.params.arena.view(torch.int16).to(torch.int64).sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN); torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
        weights_identical = bool((lo == hi).item())
    else:
        weights_identical = True
    torch.cuda.synchronize()
    t_build = time.time() - t0

    sched = B200Scheduler(wl["scheduler"])
    sched.set_timesteps(n_steps)
    den = B200Denoiser(unet, sched, use_cuda_graph=not args.no_graph)
    lat_h, prompts_h, extra_h = synth_inputs(spec, B, h, h, seed=rank, sdxl=sdxl)
    lat_h = (lat_h * sched.init_noise_sigma).to(dtype)
    pin = lambda t: t.to(dtype if t.is_floating_point() and t.shape[-1] != 6 else t.dtype).pin_memory()
    lat_h, prompts_h = pin(lat_h), [pin(p) for p in prompts_h]
    extra_h = {k: pin(v) for k, v in extra_h.items()}
    out_h = torch.empty((B, 4, h, h), dtype=dtype).pin_memory()
    kw = dict(num_inference_steps=n_steps, guidance_scale=wl["guidance"], start_merge_step=wl["start_merge_step"])

    use_cn = bool(wl.get("controlnet"))
    if use_cn:
        cnet, ctrl_h, img_h, noise_h, mask_h = _build_controlnet(spec, dev, dtype, rankN, wl, B, h)

    def job_resident(lat_d, prompts_d, extra_d):
        if use_cn:
            return den.controlnet_inpaint(cnet, lat_d, prompts_d[0], prompts_d[1], prompts_d[2], ctrl_d, img_d, noise_d, mask_d,
                                          conditioning_scale=0.5, **kw)
        return den(lat_d, prompts_d[0], prompts_d[1], prompts_d[2], **kw, **extra_d)

    def job_e2e():
        lat_d = lat_h.to(dev, non_blocking=True)
        pd = [p.to(dev, non_blocking=True) for p in prompts_h]
        ed = {k: v.to(dev, non_blocking=True) for k, v in extra_h.items()}
        if use_cn:
            out = den.controlnet_inpaint(cnet, lat_d, pd[0], pd[1], pd[2], ctrl_h.to(dev, non_blocking=True), img_h.to(dev, non_blocking=True),
                                         noise_h.to(dev, non_blocking=True), mask_h.to(dev, non_blocking=True), conditioning_scale=0.5, **kw)
        else:
            out = den(lat_d, pd[0], pd[1], pd[2], **kw, **ed)
        out_h.copy_(out, non_blocking=True)
        return out_h

    lat_d = lat_h.to(dev); prompts_d = [p.to(dev) for p in prompts_h]; extra_d = {k: v.to(dev) for k, v in extra_h.items()}
    if use_cn:
        ctrl_d, img_d, noise_d, mask_d = ctrl_h.to(dev), img_h.to(dev), noise_h.to(dev), mask_h.to(dev)
    # ---- warm-up (also captures the CUDA graphs)
    for _ in range(max(warmup, 1)):
        job_resident(lat_d, prompts_d, extra_d)
    torch.cuda.synchronize()
    launches0 = lib.LAUNCHES

    def timed(fn, k):
        """k steps of fn between CUDA events: (max over ranks of the elapsed ms, what the last step returned)."""
        cdist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        torch.cuda.synchronize(); cdist.barrier()
        return cdist.max_over_ranks(e0.elapsed_time(e1), dev), out

    clocks = ClockSampler(local)
    clocks.start()
    try:
        ms_total, out_resident = timed(lambda: job_resident(lat_d, prompts_d, extra_d), steps)
    finally:
        clk = clocks.stop()
    eager_calls = lib.LAUNCHES - launches0      # host-issued (non-graph) launches during the timed region
    ms_e2e, out_e2e = timed(job_e2e, steps)
    final = out_e2e.float()
    finite = bool(torch.isfinite(final).all())
    if args.dump_outputs and rank == 0:
        # final latents of the last timed step of each path, as its caller receives them (the e2e path's land in pinned host memory)
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, f"{name}_latents.npy"), out_resident.float().cpu().numpy())
        np.save(os.path.join(args.dump_outputs, f"{name}_e2e_latents.npy"), final.numpy())

    # ---- launches: kernels inside the captured per-step graphs x replays + eager launches
    per_step = None
    if den.use_cuda_graph and not use_cn:
        c0 = lib.LAUNCHES
        den_e = B200Denoiser(unet, sched, use_cuda_graph=False)
        den_e(lat_d, prompts_d[0], prompts_d[1], prompts_d[2], **dict(kw, num_inference_steps=n_steps), **extra_d)
        torch.cuda.synchronize()
        per_job = lib.LAUNCHES - c0
        gpu_launches = per_job * steps
        per_step = per_job // n_steps
    else:
        gpu_launches = eager_calls

    img_per_s = world * B * steps / (ms_total / 1e3)
    e2e_img_per_s = world * B * steps / (ms_e2e / 1e3)
    pk = peaks()
    res = {
        "metric": "images_per_sec", "value": round(img_per_s, 4), "unit": "images/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(ms_total / steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": wl["dtype"], "data": "synthetic (random-init weights of the exact architecture, randn latents/embeddings)",
        "config": {"workload": f"{wl['model']} ConsistentID {wl['res']}x{wl['res']} batch={B}/GPU, {n_steps} {wl['scheduler']} steps, CFG {wl['guidance']}, LoRA r128 folded, 77+4 tokens",
                   "per_gpu_batch": B, "global_batch": B * world, "denoise_steps": n_steps, "scheduler": wl["scheduler"],
                   "parallelism": f"dp{world} (batch sharded, one weight-arena broadcast at init, no per-step collective)",
                   "cuda_graph": den.use_cuda_graph, "l2_policy": "working set >> L2: weights + per-step activations exceed 126 MB, no flush needed"},
        "clocks": clk,
        "e2e": {"value": round(e2e_img_per_s, 4), "unit": "images/s",
                "h2d_bytes_per_step": int(lat_h.numel() * 2 + sum(p.numel() * 2 for p in prompts_h) + sum(v.numel() * v.element_size() for v in extra_h.values())
                                          + ((ctrl_h.numel() * 2 + (img_h.numel() + noise_h.numel() + mask_h.numel()) * 4) if use_cn else 0)),
                "d2h_bytes_per_step": int(out_h.numel() * 2), "ms_per_step": round(ms_e2e / steps, 3)},
        "gpu_launches": int(gpu_launches), "launches_per_denoise_step": per_step, "finite_output": finite,
        "weights_identical_after_broadcast": weights_identical,
        "build_s": round(t_build, 1),
    }
    if wl["tflop_per_sample_forward"]:
        tf_job = (wl["tflop_per_sample_forward"] * 2 + wl.get("controlnet_tflop_per_image_step", 0.0)) * B * n_steps
        res["step_tflops"] = {"algorithmic_tflop_per_step": round(tf_job, 2), "achieved_tflops_per_gpu": round(tf_job / (ms_total / steps / 1e3), 1),
                              "frac_of_sustained_peak": round(tf_job / (ms_total / steps / 1e3) / pk["tf_sustained"], 4), "peak_src": pk["src"]}

    # ---- roofline of the dominant kernel: every tensor-core launch of ONE eager denoising step bracketed by CUDA events
    if rank == 0 and not args.no_profile and not use_cn:
        try:
            den_p = B200Denoiser(unet, sched, use_cuda_graph=False)
            den_p(lat_d, prompts_d[0], prompts_d[1], prompts_d[2], **dict(kw, num_inference_steps=2, start_merge_step=-1), **extra_d)  # warm
            den_p(lat_d, prompts_d[0], prompts_d[1], prompts_d[2], **dict(kw, num_inference_steps=1, start_merge_step=-1), **extra_d, profile=True)
            rec = den_p.last_profile
            agg = {}
            for r in rec:
                a = agg.setdefault(r["kind"], dict(launches=0, flops=0.0, bytes=0.0, ms=0.0))
                a["launches"] += 1; a["flops"] += r["flops"]; a["bytes"] += r["bytes"]; a["ms"] += r["ms"]
            tc = dict(launches=0, flops=0.0, ms=0.0)
            for k in ("gemm", "conv3x3"):
                if k in agg:
                    for f in tc:
                        tc[f] += agg[k][f]
            kern = {}
            for k, v in agg.items():
                d_ = dict(launches=v["launches"], ms=round(v["ms"], 3))
                if v["flops"] > 0:
                    d_["tflops"] = round(v["flops"] / max(v["ms"], 1e-9) / 1e9, 1)
                if v["bytes"] > 0 and k not in ("gemm", "conv3x3", "attn_self"):      # HBM-bound kernels: algorithmic GB/s vs the measured copy bandwidth
                    gbs = v["bytes"] / max(v["ms"], 1e-9) / 1e6
                    d_["gbs"] = round(gbs, 1); d_["frac_of_hbm"] = round(gbs / pk["hbm_gbs"], 3)
                kern[k] = d_
            res["kernels"] = kern
            achieved = tc["flops"] / max(tc["ms"], 1e-9) / 1e9
            # ncu dram__bytes capture of the same eager step (tools/summarize_dram.py), bytes per launch: a committed measurement, not taken in this run
            traffic, traffic_src = None, None
            for rnd in ("r02", "r01"):
                tpath = os.path.join(ROOT, "profiles", f"{rnd}_dram_traffic_{wl['model']}.json")
                if os.path.exists(tpath):
                    traffic = round(json.load(open(tpath))["tensor_core_kernels"]["bytes_per_launch"])
                    traffic_src = os.path.relpath(tpath, ROOT) + " (committed ncu capture of the same eager step, not measured in this run)"
                    break
            res["roofline"] = {"kernel": "gemm_tc2_kernel (persistent tcgen05 GEMM + implicit-GEMM conv3x3)", "bound": "tensor", "achieved": round(achieved, 1),
                               "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": round(achieved / pk["tf_sustained"], 4),
                               "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram read+write)", "traffic_src": traffic_src,
                               "peak_src": pk["src"] + " (sustained bf16 GEMM)", "launches_timed": tc["launches"],
                               "avg_launch_ms": round(tc["ms"] / max(tc["launches"], 1), 4),
                               "alg_flops_per_launch": round(tc["flops"] / max(tc["launches"], 1) / 1e9, 2), "alg_flops_unit": "GFLOP"}
            if "attn_self" in agg:
                a = agg["attn_self"]
                res["attention"] = {"tflops": round(a["flops"] / max(a["ms"], 1e-9) / 1e9, 1), "frac_of_peak": round(a["flops"] / max(a["ms"], 1e-9) / 1e9 / pk["tf_sustained"], 4),
                                    "launches": a["launches"], "ms": round(a["ms"], 3), "flops": "4*N*N*d per (sample, head), head dim NOT padded"}
            tot_ms = sum(v["ms"] for v in agg.values())
            res["iteration_ms_eager_sum"] = round(tot_ms, 3)
        except Exception as e:  # never lose the headline number to the profiling pass
            res["roofline"] = {"error": repr(e)}
    del den, unet
    torch.cuda.empty_cache()
    return res


def gpu_eager_baseline(workload, iters=4):
    """SURVEY 8d-(ii): the "reference diffusers-CUDA pipeline" stand-in (oracle modules eager 16-bit on the same GPU, stock cuBLAS/cuDNN
    kernels, LoRA unfolded, naive self-attention as attention.py:157-158, no graph) timed by tools/bench_eager_gpu.py in a SUBPROCESS, so the
    product process never imports oracle/.  A reported baseline (the denominator of north_star's ">= 5x"), not part of the product path."""
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_eager_gpu.py"), workload, str(iters)], capture_output=True, text=True,
                           timeout=900)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": (r.stderr or r.stdout)[-400:]}
        return json.loads(lines[-1])
    except Exception as e:
        return {"error": repr(e)}


def run_ours(args):
    """One JSON line.  Headline fields = BASELINE.json configs[1] (SD1.5 512^2 batch 8, fp16); the other half of the metric rides in the same line:
    "sdxl" = configs[2] (SDXL 1024^2 batch 4/GPU, bf16 - at --gpus 8 this IS configs[3], 32 images over 8 GPUs) and "sdxl_b8" = the north-star
    batch-8 config, each with its own value / e2e / roofline / attention / clocks.  --workload X times only X."""
    import torch
    from consistentid_b200 import dist as cdist

    rank, local, world = cdist.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (the product has no CPU path)"
    torch.cuda.set_device(local)
    names = ["sd15", "sdxl", "sdxl_b8"] if args.workload == "all" else [args.workload]
    res = None
    for i, name in enumerate(names):
        # every workload times the requested K steps (the riders --rider-steps if given); the riders' warm-up is bounded so that the default run
        # stays within minutes
        k = args.steps if i == 0 or args.rider_steps is None else max(1, args.rider_steps)
        w = args.warmup if i == 0 else max(1, min(args.warmup, 3))
        blk = bench_workload(args, name, k, w, rank, local, world)
        if i == 0:
            res = blk
        else:
            res[name] = blk
            res["gpu_launches"] += blk["gpu_launches"]
    # ---- baselines (rank 0, N = 1 only): eager-GPU stand-in of the reference CUDA pipeline, CPU oracle port
    if rank == 0 and world == 1 and not args.no_eager:
        for i, name in enumerate(names):
            if WORKLOADS[name].get("controlnet") or WORKLOADS[name]["model"].startswith("tiny"):
                continue
            eb = gpu_eager_baseline(name)
            blk = res if i == 0 else res[name]
            blk["gpu_eager_baseline"] = eb
            key = [k_ for k_ in eb if k_.startswith("images_per_sec")]
            if key:
                blk["speedup_vs_gpu_eager"] = round(blk["value"] / eb[key[0]], 3)
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            res["cpu_baseline"] = cpu_baseline(names[0], steps=2, warmup=1)
        except Exception as e:
            res["cpu_baseline"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(res), flush=True)
    if world > 1:
        cdist.barrier()
        torch.distributed.destroy_process_group()


def cpu_baseline(workload, steps=1, warmup=0, budget_s=None):
    """Oracle (CPU restatement of the reference path) timed on the host cores: B=1, `steps` denoising iterations of the same model after
    `warmup` untimed ones.  Threads = the physical cores of one socket (pinned), so that two boxes of the same model agree."""
    import torch
    from oracle import synth
    from oracle.loop_ref import denoise_sd15, denoise_sdxl
    from oracle.schedulers_ref import make_scheduler
    from oracle.unet_ref import sd15_config, sdxl_config, tiny_config
    wl = WORKLOADS[workload]
    cpus = _physical_cores_one_socket()
    cores = max(1, len(cpus))
    try:
        os.sched_setaffinity(0, set(cpus))
    except Exception:
        pass
    torch.set_num_threads(cores)
    cfg = {"sd15": sd15_config, "sdxl": sdxl_config}.get(wl["model"], lambda: tiny_config("sd15"))()
    rank = 16 if wl["model"].startswith("tiny") else 128
    unet = synth.build_ref_unet(cfg, rank=rank)
    h = wl["res"] // 8
    null, aug, txt = synth.synth_prompts(cfg.cross_attention_dim)
    sch = make_scheduler(wl["scheduler"])
    sch.set_timesteps(wl["denoise_steps"])
    lat = synth.synth_latents(1, h, h, init_noise_sigma=float(sch.init_noise_sigma))
    sdxl = wl["model"] == "sdxl"

    def run(n, callback=None):
        # n leading iterations of the full schedule (timesteps of a `denoise_steps` run)
        class _Trunc:
            def __getattr__(s, k):
                return getattr(sch, k)
            def set_timesteps(s, *_a, **_k):
                sch.set_timesteps(wl["denoise_steps"]); s.timesteps = sch.timesteps[:n]
        tr = _Trunc()
        if sdxl:
            pooled = [torch.randn(1, 1280) for _ in range(3)]
            return denoise_sdxl(unet, tr, lat, null, txt, null, aug, pooled[0], pooled[1], pooled[2],
                                torch.tensor([[1024., 1024., 0., 0., 1024., 1024.]]), n, guidance_scale=wl["guidance"], callback=callback)
        return denoise_sd15(unet, tr, lat, null, aug, txt, n, guidance_scale=wl["guidance"], callback=callback)

    # bounded sample: `warmup` + `steps` iterations, cut short once the wall budget is spent
    if budget_s is None:
        budget_s = float(os.environ.get("CID_CPU_BUDGET_S", "150"))
    n_total = min(max(warmup, 0) + max(steps, 1), wl["denoise_steps"])

    class _Stop(Exception):
        pass

    stamps = [time.time()]

    def on_iter(i, t, latents):
        stamps.append(time.time())
        if stamps[-1] - stamps[0] > budget_s and i + 1 < n_total:
            raise _Stop

    try:
        run(n_total, on_iter)
    except _Stop:
        pass
    done = len(stamps) - 1
    skip = min(max(warmup, 0), done - 1)
    timed = done - skip
    per_iter = (stamps[-1] - stamps[skip]) / timed
    return {"value": round(1.0 / (per_iter * wl["denoise_steps"]), 6), "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{timed} of {wl['denoise_steps']} denoising iterations (after {skip} warm-up; wall budget {budget_s:.0f} s) of {wl['model']} "
                      f"{wl['res']}x{wl['res']} at batch 1 (CFG pair), fp32 torch CPU on {cores} threads (physical cores of one socket, pinned), "
                      f"{per_iter:.2f} s/iteration; images/s = 1 / (s_per_iteration * {wl['denoise_steps']})",
            "s_per_iteration": round(per_iter, 3), "iterations_timed": timed, "iterations_warmup": skip}


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path = the oracle port (diffusers/insightface/weights are not
    installable here, see DESIGN.md) on the physical cores of one socket.  A bench step = ONE denoising iteration of the headline
    workload at batch 1 (a bounded sample of the job: 1/30 of an image); `steps` / `warmup` in the line are the iterations actually
    timed / skipped (the wall budget can cut a slow host short).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = "sd15" if args.workload == "all" else args.workload
    wl = WORKLOADS[name]
    t0 = time.time()
    cb = cpu_baseline(name, steps=max(args.steps, 1), warmup=max(args.warmup, 0), budget_s=float(os.environ.get("CID_CPU_BUDGET_S", "200")))
    res = {"impl": "reference", "metric": "images_per_sec", "value": cb["value"], "unit": "images/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
           "steps": cb["iterations_timed"], "warmup": cb["iterations_warmup"], "steps_requested": args.steps, "warmup_requested": args.warmup,
           "ms_per_step": round(cb["s_per_iteration"] * 1e3, 1), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
           "config": {"workload": f"{wl['model']} ConsistentID {wl['res']}x{wl['res']}, {wl['denoise_steps']} {wl['scheduler']} steps; each bench step = 1 denoising iteration at batch 1 on the host CPU "
                                  f"(images/s = 1 / (s_per_iteration * {wl['denoise_steps']}))"},
           "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": round(time.time() - t0, 1)}
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + list(WORKLOADS),
                    help="all = SD1.5 configs[1] headline + SDXL configs[2] + SDXL batch 8 riders in one line")
    ap.add_argument("--rider-steps", type=int, default=None, help="timed jobs of the non-headline workloads (default: --steps)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the eager-GPU stand-in baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write each workload's final latents of the last timed step as DIR/<workload>_latents.npy "
                         "(device-resident path) and DIR/<workload>_e2e_latents.npy (host-buffer path), float32; inputs and weights are seeded")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
