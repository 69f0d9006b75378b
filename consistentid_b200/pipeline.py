"""The ConsistentID denoising loop on the B200 engine.

Same control flow as the reference loop bodies
(pipline_StableDiffusion_ConsistentID.py:533-579, pipline_StableDiffusionXL_ConsistentID.py:608-667): per step
``cat([latents]*2)`` -> ``scale_model_input`` -> prompt switch at ``i <= start_merge_step`` -> UNet -> CFG combine ->
``scheduler.step``.  Here one step is ONE CUDA-graph replay: the UNet launch program followed by the fused
CFG + scheduler-step kernel, which also writes the next step's scaled, batch-duplicated NHWC UNet input, and a
1-thread bookkeeping kernel that advances the device-side step index / timestep.  No host sync inside the loop.

Batch semantics (SURVEY.md 8a): B independent latents sharing one identity's prompt embeddings
== B batch-1 runs of the reference.
"""
from __future__ import annotations

import torch

from . import ops
from .scheduler import B200Scheduler
from .unet import B200UNet, CIN_PAD


class B200Denoiser:
    def __init__(self, unet: B200UNet, scheduler: B200Scheduler, use_cuda_graph=True):
        self.unet, self.scheduler, self.use_cuda_graph = unet, scheduler, use_cuda_graph
        self._graphs = {}
        self._graph_sig = None
        self.launches_per_step = None

    # ------------------------------------------------------------------ helpers
    def _dev16(self, t):
        return t.to(device=self.unet.device, dtype=self.unet.dtype, non_blocking=True)

    def _persist(self, name, t, dtype=None):
        """``t`` copied into the engine buffer ``name``.  A captured step graph reads the addresses it was captured with, so every per-call
        tensor it reads (scheduler tables, which ``set_timesteps`` re-allocates, and caller inputs) must live at a fixed address: a fresh
        tensor per call would leave the graph reading freed memory that the allocator hands to something else."""
        b = self.unet._buf(name, tuple(t.shape), dtype or t.dtype)
        b.copy_(t)
        return b

    def _pair(self, neg, pos, B):
        """[2B, L, cad]: uncond rows first, then cond rows (``torch.cat([null, cond])``, :542-549)."""
        neg, pos = self._dev16(neg), self._dev16(pos)
        return torch.cat([neg.expand(B, *neg.shape[1:]), pos.expand(B, *pos.shape[1:])], dim=0).contiguous()

    def _step_eager(self, key, st):
        u = self.unet
        B, HW = st["B"], st["HW"]
        eps = u.forward(key)
        ops.cfg_sched_step(eps, 4, st["x"], st["x0"], st["x16"], u._buf("x_in", (2 * B * HW, CIN_PAD)), CIN_PAD, B, HW,
                           st["guidance"], st["coef"], st["step"])
        ops.advance_step(st["step"], u._buf("t_dev", (1,), torch.float32), st["ts"], st["n"])

    def _step(self, phase, key, st):
        if not self.use_cuda_graph:
            return self._step_eager(key, st)
        g = self._graphs.get(phase)
        if g is None:
            # warm-up once eagerly on a side stream (allocates every buffer, sets kernel attributes), restore state, capture
            snap = {k: st[k].clone() for k in ("x", "x0", "step")}
            t_dev = self.unet._buf("t_dev", (1,), torch.float32)
            x_in = self.unet._buf("x_in", (2 * st["B"] * st["HW"], CIN_PAD))
            t_snap, in_snap = t_dev.clone(), x_in.clone()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._step_eager(key, st)
            torch.cuda.current_stream().wait_stream(s)
            for k, v in snap.items():
                st[k].copy_(v)
            t_dev.copy_(t_snap); x_in.copy_(in_snap)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step_eager(key, st)
            for k, v in snap.items():       # capture does not execute, but keep state explicit
                st[k].copy_(v)
            t_dev.copy_(t_snap); x_in.copy_(in_snap)
            self._graphs[phase] = g
        g.replay()

    # ------------------------------------------------------------------ ControlNet + inpaint variant (config 5)
    @torch.no_grad()
    def controlnet_inpaint(self, controlnet, latents, null_embeds, augmented_embeds, text_embeds, control_image, image_latents,
                           noise, mask, num_inference_steps=50, guidance_scale=5.0, start_merge_step=0, conditioning_scale=1.0,
                           masked_image_latents=None):
        """``controlnet`` None = the plain inpaint loop (pipelines/StableDIffusionInpaint_ConsistentID.py:305-359): same steps without the
        ControlNet residuals; see ``inpaint``.
        The reference's ControlNet + inpaint loop (pipelines/StableDIffusionControlNetInpaint_ConsistentID.py:375-449, strength 1):
        per step ControlNet on the cond half -> residuals into the UNet (both CFG halves) -> CFG + scheduler step -> for the
        4-channel UNet the latent blend with the re-noised original; a 9-channel UNet instead sees [latents | mask | masked latents].
        One CUDA-graph replay per step, like ``__call__``.  mask [B,1,h,w]: 1 = repaint."""
        import numpy as np
        u, sch = self.unet, self.scheduler
        dev = u.device
        B, _, h, w = latents.shape
        HW, NB = h * w, 2 * B
        n = num_inference_steps
        nine = u.spec.in_channels == 9
        u.plan(NB, h, w)
        if controlnet is not None:
            controlnet.plan(B, h, w)
            controlnet.share_timestep(u)
        # a captured graph bakes in buffer addresses (valid for one plan epoch of each engine), the key-row split and the dtype
        sig = ("cn", B, h, w, n, float(guidance_scale), sch.kind, u.ip_scale, float(conditioning_scale), nine, u.plan_epoch,
               None if controlnet is None else (id(controlnet), controlnet.plan_epoch),
               tuple(null_embeds.shape), tuple(text_embeds.shape), u.num_tokens, str(u.dtype))
        if sig != self._graph_sig:
            self._graphs.clear()
            self._graph_sig = sig
        sch.set_timesteps(n, device=dev)
        coef, ts = (self._persist("sched_" + k, t) for k, t in zip(("coef", "ts"), sch.device_tables(dev)))
        if controlnet is not None:
            controlnet.set_control_image(control_image)
        phases, cn_phases = {}, {}
        for name, pos in (("text", text_embeds), ("aug", augmented_embeds)):
            if (name == "text" and start_merge_step >= 0) or (name == "aug" and start_merge_step < n - 1):
                phases[name] = u.set_prompt(self._pair(null_embeds, pos, B), None, key="phase:" + name)
                if controlnet is not None:
                    pos16 = self._dev16(pos)
                    cn_phases[name] = controlnet.set_prompt(pos16.expand(B, *pos16.shape[1:]).contiguous(), None, key="phase:" + name)
        # add_noise coefficients of the NEXT timestep for the blend ((1, 0) after the last step)
        acp = sch.acp
        blend = np.zeros((n, 2), dtype=np.float32)
        for i in range(n):
            if i < n - 1:
                a = acp[int(sch._ts_host[i + 1])]
                blend[i] = (np.sqrt(a), np.sqrt(1 - a))
            else:
                blend[i] = (1.0, 0.0)
        st = {"B": B, "HW": HW, "n": n, "guidance": float(guidance_scale), "coef": coef, "ts": ts,
              "x": u._buf("lat32", (B, 4, HW), torch.float32), "x0": u._buf("lat_x0", (B, 4, HW), torch.float32),
              "x16": u._buf("lat16", (B, 4, HW)), "step": u._buf("step_dev", (1,), torch.int32),
              "blend": self._persist("blend", torch.from_numpy(blend)), "img": self._persist("img", image_latents.reshape(B, 4, HW), torch.float32),
              "noise": self._persist("noise", noise.reshape(B, 4, HW), torch.float32),
              "mask": self._persist("mask", mask.reshape(B, 1, HW), torch.float32)}
        st["x"].copy_(latents.reshape(B, 4, HW).to(dev, non_blocking=True))
        st["x0"].zero_(); st["step"].zero_()
        u._buf("t_dev", (1,), torch.float32).copy_(ts[:1])
        x_in = u._buf("x_in", (NB * HW, CIN_PAD))
        if nine:   # static channels 4..8 of the UNet input: mask, masked-image latents (both CFG halves)
            extra = torch.cat([mask.reshape(B, 1, HW), masked_image_latents.reshape(B, 4, HW)], 1).to(dev, u.dtype)
            x_in.zero_()
            x_in.view(2, B, HW, CIN_PAD)[:, :, :, 4:9] = extra.permute(0, 2, 1)[None]
        ops.latents_to_input(st["x"], x_in, CIN_PAD, B, HW, coef, st["step"], n, keep_ch4_up=nine)

        def step_eager(phase):
            if controlnet is not None:
                down, mid = controlnet.forward(x_in[:B * HW], cn_phases[phase], conditioning_scale)
                eps = u.forward(phases[phase], residuals=(down, mid))
            else:
                eps = u.forward(phases[phase])
            ops.cfg_sched_step(eps, 4, st["x"], st["x0"], st["x16"], None, CIN_PAD, B, HW, st["guidance"], coef, st["step"])
            if not nine:
                ops.inpaint_blend(st["x"], st["x16"], st["img"], st["noise"], st["mask"], B, HW, st["blend"], st["step"])
            ops.advance_step(st["step"], u._buf("t_dev", (1,), torch.float32), ts, n)
            ops.latents_to_input(st["x"], x_in, CIN_PAD, B, HW, coef, st["step"], n, keep_ch4_up=nine)

        def run(phase):
            if not self.use_cuda_graph:
                return step_eager(phase)
            g = self._graphs.get(phase)
            if g is None:
                keys = ("x", "x0", "step")
                snap = {k: st[k].clone() for k in keys}
                t_dev = u._buf("t_dev", (1,), torch.float32)
                t_snap, in_snap = t_dev.clone(), x_in.clone()
                s_ = torch.cuda.Stream()
                s_.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s_):
                    step_eager(phase)
                torch.cuda.current_stream().wait_stream(s_)

                def restore():
                    for k in keys:
                        st[k].copy_(snap[k])
                    t_dev.copy_(t_snap); x_in.copy_(in_snap)
                restore()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    step_eager(phase)
                restore()
                self._graphs[phase] = g
            g.replay()

        for i in range(n):
            run("text" if i <= start_merge_step else "aug")
        return st["x16"].reshape(B, 4, h, w).clone()

    @torch.no_grad()
    def inpaint(self, latents, null_embeds, augmented_embeds, text_embeds, image_latents, noise, mask, num_inference_steps=50,
                guidance_scale=5.0, start_merge_step=0, masked_image_latents=None):
        """The reference's plain inpaint loop (pipelines/StableDIffusionInpaint_ConsistentID.py:305-359, strength 1): UNet x 2B -> CFG ->
        scheduler step -> for the 4-channel UNet ``latents = (1 - mask) * add_noise(image_latents, noise, t_next) + mask * latents``
        (:340-352); a 9-channel inpaint UNet instead sees ``cat([latents, mask, masked_image_latents])`` every step (:320-321).
        One CUDA-graph replay per step.  mask [B,1,h,w]: 1 = repaint."""
        return self.controlnet_inpaint(None, latents, null_embeds, augmented_embeds, text_embeds, None, image_latents, noise, mask,
                                       num_inference_steps=num_inference_steps, guidance_scale=guidance_scale, start_merge_step=start_merge_step,
                                       masked_image_latents=masked_image_latents)

    # ------------------------------------------------------------------ public API
    @torch.no_grad()
    def __call__(self, latents, null_embeds, augmented_embeds, text_embeds, num_inference_steps=30, guidance_scale=5.0,
                 start_merge_step=0, neg_pooled=None, pooled_text_only=None, pooled_facial=None, add_time_ids=None,
                 null_embeds_facial=None, output_device=None, profile=False):
        """latents [B,4,h,w] already multiplied by ``scheduler.init_noise_sigma`` (host or device, any float dtype).
        SD1.5: (null, augmented, text_only) each [1,81,cad] (chunk(3) of prompt_embeds, :527-531).
        SDXL: additionally pooled embeds [1,1280] x3 and add_time_ids [1,6]; ``null_embeds_facial`` is the uncond prompt of
        the facial phase (pipline_StableDiffusionXL_ConsistentID.py:578-587) and defaults to ``null_embeds``.
        Returns final latents [B,4,h,w] in the engine dtype (on ``output_device`` if given)."""
        u, sch = self.unet, self.scheduler
        dev = u.device
        B, _, h, w = latents.shape
        HW, NB = h * w, 2 * B
        n = num_inference_steps
        sdxl = u.spec.addition_embed_type == "text_time"
        u.plan(NB, h, w)
        # a captured graph bakes in buffer addresses (valid for one plan epoch of the engine), the key-row split (n_text / n_ip) and the dtype
        sig = (B, h, w, n, float(guidance_scale), sch.kind, u.ip_scale, u.plan_epoch, tuple(null_embeds.shape), tuple(text_embeds.shape),
               tuple(augmented_embeds.shape), u.num_tokens, str(u.dtype))
        if sig != self._graph_sig:
            self._graphs.clear()
            self._graph_sig = sig
        sch.set_timesteps(n, device=dev)
        coef, ts = (self._persist("sched_" + k, t) for k, t in zip(("coef", "ts"), sch.device_tables(dev)))
        # ---- prompt phases (K/V caches + SDXL added-cond embedding), computed once per call
        null_f = null_embeds if null_embeds_facial is None else null_embeds_facial
        phases = {}
        need_text = start_merge_step >= 0
        need_aug = start_merge_step < n - 1
        def added(pos_pooled):
            if not sdxl:
                return None
            te = torch.cat([self._dev16(neg_pooled).expand(B, -1), self._dev16(pos_pooled).expand(B, -1)], 0).contiguous()
            ti = torch.cat([add_time_ids.to(dev, torch.float32).expand(B, -1)] * 2, 0).contiguous()
            return {"text_embeds": te, "time_ids": ti}
        if need_text:
            phases["text"] = u.set_prompt(self._pair(null_embeds, text_embeds, B), added(pooled_text_only), key="phase:text")
        if need_aug:
            phases["aug"] = u.set_prompt(self._pair(null_f, augmented_embeds, B), added(pooled_facial), key="phase:aug")
        # ---- per-run state
        st = {"B": B, "HW": HW, "n": n, "guidance": float(guidance_scale), "coef": coef, "ts": ts,
              "x": u._buf("lat32", (B, 4, HW), torch.float32), "x0": u._buf("lat_x0", (B, 4, HW), torch.float32),
              "x16": u._buf("lat16", (B, 4, HW)), "step": u._buf("step_dev", (1,), torch.int32)}
        st["x"].copy_(latents.reshape(B, 4, HW).to(dev, non_blocking=True))
        st["x0"].zero_()
        st["step"].zero_()
        u._buf("t_dev", (1,), torch.float32).copy_(ts[:1])
        ops.latents_to_input(st["x"], u._buf("x_in", (NB * HW, CIN_PAD)), CIN_PAD, B, HW, coef)
        if profile:                       # bench.py roofline pass: event-bracket every tensor-core launch of the step loop only
            ops.profile_begin()
        for i in range(n):
            phase = "text" if i <= start_merge_step else "aug"
            self._step(phase, phases[phase], st)
        if profile:
            self.last_profile = ops.profile_end()
        out = st["x16"].reshape(B, 4, h, w)
        if output_device is not None:
            return out.to(output_device)
        return out.clone()
