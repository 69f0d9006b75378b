"""B200ControlNet - diffusers 0.23 ``ControlNetModel`` (SD1.5 topology) on the B200 engine, as driven by the reference's
ControlNet + inpaint loop (pipelines/StableDIffusionControlNetInpaint_ConsistentID.py:389-412): UNet encoder copy with
diffusers' DEFAULT attention processors (plain attention over all 81 encoder rows - no LoRA, no id branch), a conditioning
embedding (8 small 3x3 convs + SiLU on the control image, computed once per control image), and 13 1x1 "zero" convs whose
outputs, times ``conditioning_scale``, are the residuals injected into the UNet (NHWC rows, consumed directly by
``B200UNet.forward(residuals=...)``)."""
from __future__ import annotations

import torch

from . import ops
from .arch import UNetSpec, walk
from .unet import B200UNet, CIN_PAD, _Params
from .weights import pack_conv3x3


def _pad64(c):
    return (c + 63) // 64 * 64


class B200ControlNet(B200UNet):
    def __init__(self, spec, state_dict, dtype=torch.float16, device="cuda", cond_block_out_channels=(16, 32, 96, 256)):
        if not isinstance(spec, UNetSpec):
            spec = UNetSpec.from_config(spec)
        self.spec, self.dtype, self.device = spec, dtype, torch.device(device)
        self.in_channels = spec.in_channels
        self.num_tokens, self.ip_scale = 0, 0.0          # default processors: every encoder row is a text row
        sd = state_dict
        ops.ensure_workspace(self.device)
        P = _Params(spec, sd, None, dtype, self.device, rank=1, kinds=("down", "mid"), finalize=False)
        U = lambda n: sd[n].to(device=self.device, dtype=dtype)
        # conditioning embedding: channels zero-padded to multiples of 64 so the same implicit-GEMM conv kernel applies
        chans = [3] + [cond_block_out_channels[0]]
        self._cond_layers = []                           # (name, cin_pad, cout, stride2)
        names = ["controlnet_cond_embedding.conv_in"] + [f"controlnet_cond_embedding.blocks.{i}" for i in range(2 * (len(cond_block_out_channels) - 1))] \
            + ["controlnet_cond_embedding.conv_out"]
        for n in names:
            w = U(n + ".weight")
            cout, cin = w.shape[:2]
            stride2 = n.split(".")[-1].isdigit() and int(n.split(".")[-1]) % 2 == 1
            P._put(n + ".w", pack_conv3x3(w, _pad64(cin))); P._put(n + ".b", U(n + ".bias"))
            self._cond_layers.append((n, _pad64(cin), cout, stride2))
        self._zero = []
        n_down = 0
        for kind, i, layers, has_sampler in walk(spec):
            if kind == "down":
                n_down += len(layers) + (1 if has_sampler else 0)
        for j in range(n_down + 1):
            w = U(f"controlnet_down_blocks.{j}.weight")
            P._put(f"zero.{j}.w", w.reshape(w.shape[0], w.shape[1]).contiguous()); P._put(f"zero.{j}.b", U(f"controlnet_down_blocks.{j}.bias"))
        w = U("controlnet_mid_block.weight")
        P._put("zero.mid.w", w.reshape(w.shape[0], w.shape[1]).contiguous()); P._put("zero.mid.b", U("controlnet_mid_block.bias"))
        P._finalize()
        self.params = P
        self._bufs, self._plan = {}, None
        self._kv, self._aug, self._graphs = {}, {}, {}
        self._active_key = None
        self._slots, self._ident, self._auto_next = {}, {}, 0
        self._procs = {}
        self._cond = None
        self.plan_epoch = 0

    # ------------------------------------------------------------------ control image (once per generation)
    def set_control_image(self, control_image):
        """control_image [B,3,Himg,Wimg] (the pipeline's prepared ``control_image``) -> conditioning embedding rows
        [B*h*w, C0] at latent resolution (diffusers ControlNetConditioningEmbedding: conv, SiLU, ..., conv)."""
        B, c, Hi, Wi = control_image.shape
        P = self.params
        img = control_image.to(self.device, self.dtype).contiguous()
        x = torch.zeros((B * Hi * Wi, 64), dtype=self.dtype, device=self.device)
        ops.nchw_to_nhwc_pad(img, x, B, c, Hi * Wi, 64)
        h, w = Hi, Wi
        last = len(self._cond_layers) - 1
        for li, (n, cin_pad, cout, stride2) in enumerate(self._cond_layers):
            assert x.shape[1] == cin_pad, (n, x.shape, cin_pad)
            if stride2:
                ps = torch.empty_like(x)
                ops.phase_split(x, ps, B, h, w, cin_pad)
                h, w = h // 2, w // 2
                x = ps
            y = torch.zeros((B * h * w, _pad64(cout) if li != last else cout), dtype=self.dtype, device=self.device)
            ops.conv3x3(x, P[n + ".w"], y, B, h, w, cin_pad, cout, bias=P[n + ".b"], stride2=stride2)
            if li != last:
                ops.silu_inplace(y)
            x = y
        # into a persistent buffer: a captured denoising step keeps reading the address it was captured with
        cond = self._buf("cond", tuple(x.shape))
        cond.copy_(x)
        self._cond = (cond, B, h, w)
        return cond

    def plan(self, NB, H, W):
        if self._plan != (NB, H, W):
            self._plan = (NB, H, W)
            self.plan_epoch = getattr(self, "plan_epoch", 0) + 1
            self._kv.clear(); self._aug.clear(); self._slots.clear(); self._ident.clear()
            keep = {k: v for k, v in self._bufs.items() if k[0] == "t_dev"}
            self._bufs = keep
            if ("t_dev", (1,), torch.float32) not in self._bufs:
                self._buf("t_dev", (1,), torch.float32, zero=True)

    def share_timestep(self, unet: B200UNet):
        """Alias the UNet's device-side timestep so one ``advance_step`` drives both networks."""
        self._bufs[("t_dev", (1,), torch.float32)] = unet._buf("t_dev", (1,), torch.float32)

    # ------------------------------------------------------------------ per-step program
    def forward(self, x_in_rows, key=None, conditioning_scale=1.0):
        """x_in_rows: NHWC rows [B*H*W, 64] of the scaled latents (channels >= in_channels are ignored: zero weights).
        Returns (list of 12 down residual row tensors, mid residual rows), already multiplied by ``conditioning_scale``."""
        key = key if key is not None else self._active_key
        NB, H, W = self._plan
        spec, P, buf = self.spec, self.params, self._buf
        kv = self._kv[key]
        self._gn_k = 0
        self._stats_begin()
        cond, cb, ch, cw = self._cond
        assert (cb, ch, cw) == (NB, H, W), ("control image does not match the latent batch/resolution", (cb, ch, cw), (NB, H, W))
        emb, temb_all = self._time_embedding(key)
        c0 = spec.block_out_channels[0]
        x = buf("h.conv_in", (NB * H * W, c0))
        ops.conv3x3(x_in_rows, P["conv_in.w"], x, NB, H, W, CIN_PAD, c0, bias=P["conv_in.b"], residual=cond,
                    chan_stats=self._stats_slot(x, H * W, c0))
        skips = [(x, c0)]
        h, w = H, W
        for kind, i, layers, has_sampler in walk(spec):
            if kind == "up":
                continue
            for r, tf in layers:
                x = self._resnet(r, x, None, h, w, f"h.{r.name}", temb_all)
                if tf is not None:
                    x = self._transformer(tf, x, h, w, f"h.{tf.name}", kv)
                if kind == "down":
                    skips.append((x, r.cout))
            if has_sampler and kind == "down":
                c = layers[-1][0].cout
                x = self._downsample(x, i, h, w, c)
                h, w = h // 2, w // 2
                skips.append((x, c))
        down = []
        for j, (sk, c) in enumerate(skips):
            o = buf(f"zero_out.{j}", tuple(sk.shape))
            ops.gemm(sk, P[f"zero.{j}.w"], o, bias=P[f"zero.{j}.b"], out_scale=conditioning_scale)
            down.append(o)
        mid = buf("zero_out.mid", tuple(x.shape))
        ops.gemm(x, P["zero.mid.w"], mid, bias=P["zero.mid.b"], out_scale=conditioning_scale)
        self._stats_used = self._stats_off
        return down, mid

    def __call__(self, sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale=1.0, return_dict=False, **_):
        """diffusers call surface (pipelines/StableDIffusionControlNetInpaint_ConsistentID.py:405-412): NCHW in, NCHW residuals out."""
        NB, Cin, H, W = sample.shape
        self.plan(NB, H, W)
        if self._cond is None or self._cond[1:] != (NB, H, W) or getattr(self, "_cond_src", None) is not controlnet_cond:
            self.set_control_image(controlnet_cond)
            self._cond_src = controlnet_cond
        key = self.set_prompt(encoder_hidden_states)
        t = torch.as_tensor(timestep, device=self.device).to(torch.float32).reshape(-1)[:1]
        self._buf("t_dev", (1,), torch.float32).copy_(t)
        xin = self._buf("x_in", (NB * H * W, CIN_PAD))
        ops.nchw_to_nhwc_pad(sample.contiguous(), xin, NB, Cin, H * W, CIN_PAD)
        down, mid = self.forward(xin, key, conditioning_scale)

        def nchw(rows, hh, ww):
            c = rows.shape[1]
            return rows.reshape(NB, hh, ww, c).permute(0, 3, 1, 2).contiguous()
        sizes = []
        hh, ww = H, W
        sizes.append((hh, ww))
        for kind, i, layers, has_sampler in walk(self.spec):
            if kind != "down":
                continue
            sizes += [(hh, ww)] * len(layers)
            if has_sampler:
                hh, ww = hh // 2, ww // 2
                sizes.append((hh, ww))
        return [nchw(d, *s) for d, s in zip(down, sizes)], nchw(mid, hh, ww)
