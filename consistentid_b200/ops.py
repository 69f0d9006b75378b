"""Thin torch-tensor wrappers over the C ABI (device memory + current stream come from PyTorch; the arithmetic
is libcidb200.so).  Activations: 16-bit, row-major [rows, C] (== NHWC).  Every op launches on
``torch.cuda.current_stream()`` and is CUDA-graph capturable."""
from __future__ import annotations

import torch

from . import lib
from .lib import EPI_GEGLU, EPI_GELU, EPI_QKV, EPI_STORE, call


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float16:
        return lib.F16
    if t.dtype == torch.bfloat16:
        return lib.BF16
    raise TypeError(f"cidb200 kernels compute in fp16/bf16, got {t.dtype}")


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ---- GEMM tail-balancing workspace: one zero-filled buffer per DEVICE, owned here and passed to cid_gemm / cid_conv3x3 on every call
# (the library keeps no pointer; include/cidb200.h "Workspace convention")
_WORKSPACES = {}
WORKSPACE_BYTES = 24 << 20


def ensure_workspace(device=None):
    """The split-K scratch tensor of ``device`` (allocated and zero-filled once; never under CUDA-graph capture: the engines call this at
    construction)."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    ws = _WORKSPACES.get(dev.index)
    if ws is None:
        ws = _WORKSPACES[dev.index] = torch.zeros(WORKSPACE_BYTES, dtype=torch.uint8, device=dev)
    return ws


# ---- optional per-launch profiling (bench.py roofline pass): each tensor-core launch bracketed by CUDA events on the
# launching (= torch current) stream, with its algorithmic FLOPs / bytes
_PROFILE = None


def profile_begin():
    global _PROFILE
    _PROFILE = []


def profile_end():
    """-> list of dicts {kind, flops, bytes, ms}"""
    global _PROFILE
    rec, _PROFILE = _PROFILE, None
    torch.cuda.synchronize()
    return [dict(kind=k, flops=f, bytes=b, ms=e0.elapsed_time(e1), shape=sh) for k, f, b, e0, e1, sh in rec]


class _prof:
    def __init__(self, kind, flops, nbytes, shape=None):
        self.kind, self.flops, self.nbytes, self.shape = kind, flops, nbytes, shape

    def __enter__(self):
        if _PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True); self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *a):
        if _PROFILE is not None:
            self.e1.record()
            _PROFILE.append((self.kind, self.flops, self.nbytes, self.e0, self.e1, self.shape))


def _chk(t, name):
    if t is not None and not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")


def gemm(a, w, out, bias=None, residual=None, rowbias=None, rows_per_group=1, a2=None, epi=EPI_STORE, vt=None,
         n_split=0, heads=0, hdim=0, ntok=0, out_scale=1.0, chan_stats=None, stats_rows=0, row_stats=None, ln=None):
    """out[M, :] = epi([a | a2] @ w.T + bias + rowbias[row // rows_per_group] + residual) * out_scale.
    a: [M, K1] (last-dim contiguous, row pitch a.stride(0)); w: [N, K1+K2] contiguous.
    chan_stats: fp32 [M / stats_rows, N, 2] (zeroed by the caller) += per (sample, column) sum / sum of squares of ``out``.
    row_stats: fp32 [M, 2] (zeroed by the caller) += per-row sum / sum of squares of ``out`` (the LayerNorm statistics of the next block).
    ln = (stats [M, 2] fp32, colsum [N] fp32, eps): ``a`` is un-normalised, ``w`` / ``bias`` carry gamma / beta (weights.fold_layernorm): the
    epilogue applies rstd * (acc - mean * colsum) + bias, i.e. LayerNorm(a) @ W.T + b without a LayerNorm pass."""
    _chk(a, "a")
    M, K1 = a.shape
    K2 = 0 if a2 is None else a2.shape[1]
    N = w.shape[0]
    assert w.shape[1] == K1 + K2 and w.is_contiguous()
    assert a.stride(1) == 1 and out.stride(1) == 1
    for nm, t in (("w", w), ("out", out), ("a2", a2), ("bias", bias), ("residual", residual), ("rowbias", rowbias), ("vt", vt)):
        if t is not None and t.dtype != a.dtype:      # the kernels read raw 16-bit words: a dtype mismatch would be silent garbage
            raise TypeError(f"cid_gemm: {nm} is {t.dtype} but a is {a.dtype}")
    ws = ensure_workspace(a.device)
    with _prof("gemm", 2.0 * M * N * (K1 + K2), 2.0 * (M * (K1 + K2) + N * (K1 + K2) + M * N), (M, N, K1 + K2, epi)):
        call("cid_gemm", _p(a), a.stride(0), _p(a2), 0 if a2 is None else a2.stride(0), K1, K2, _p(w), _p(out), out.stride(0),
             M, N, _p(bias), _p(residual), 0 if residual is None else residual.stride(0), _p(rowbias), rows_per_group,
             0 if rowbias is None else rowbias.stride(0), epi, _p(vt), n_split, heads, hdim, ntok, float(out_scale), _dt(a),
             ws.data_ptr(), WORKSPACE_BYTES, _p(chan_stats), stats_rows, _p(row_stats),
             None if ln is None else ln[0].data_ptr(), None if ln is None else ln[1].data_ptr(), 0.0 if ln is None else float(ln[2]), _stream())
    return out


def conv3x3(x, w, out, NB, H, W, Cin, Cout, bias=None, residual=None, rowbias=None, stride2=False, out_scale=1.0, chan_stats=None):
    """x: NHWC [NB,H,W,Cin] (or phase-split [NB,4,H,W,Cin] when stride2; H,W = output dims); w: [Cout, 9*Cin];
    out: [NB*H*W, >=Cout] rows."""
    M = NB * H * W
    ws = ensure_workspace(x.device)
    with _prof("conv3x3", 2.0 * M * Cout * 9 * Cin, 2.0 * (M * Cin * (4 if stride2 else 1) + 9 * Cin * Cout + M * Cout), (M, Cout, 9 * Cin, 0)):
        call("cid_conv3x3", _p(x), _p(w), _p(out), out.stride(0), NB, H, W, Cin, Cout, 1 if stride2 else 0, _p(bias), _p(residual),
             0 if residual is None else residual.stride(0), _p(rowbias), 0 if rowbias is None else rowbias.stride(0),
             float(out_scale), _dt(x), ws.data_ptr(), WORKSPACE_BYTES, _p(chan_stats), _stream())
    return out


def attn_self(q, k, vt, out, B, H, N, d, n_valid=None):
    """q,k: views [B*N, >=H*d] (row pitch = stride(0)); vt: [B*H, d, N]; out: [B*N, H*d].  n_valid < N: keys >= n_valid are masked."""
    nv = N if n_valid is None else n_valid
    with _prof("attn_self", 4.0 * B * H * N * nv * d, 2.0 * 4 * B * N * H * d, ("B%d" % B, "H%d" % H, "N%d" % N, "d%d" % d)):
        if nv == N:
            call("cid_attn_self", _p(q), q.stride(0), _p(k), k.stride(0), _p(vt), _p(out), out.stride(0), B, H, N, d, _dt(q), _stream())
        else:
            call("cid_attn_self_ragged", _p(q), q.stride(0), _p(k), k.stride(0), _p(vt), _p(out), out.stride(0), B, H, N, nv, d, _dt(q), _stream())
    return out


def attn_self_causal(q, k, vt, out, B, H, N, d):
    """attn_self under the causal mask of the CLIP text transformer: query row i attends to keys 0..i (same layouts as attn_self)."""
    with _prof("attn_self", 2.0 * B * H * N * (N + 1) * d, 2.0 * 4 * B * N * H * d, ("B%d" % B, "H%d" % H, "N%d" % N, "d%d" % d)):
        call("cid_attn_self_causal", _p(q), q.stride(0), _p(k), k.stride(0), _p(vt), _p(out), out.stride(0), B, H, N, d, _dt(q), _stream())
    return out


def embed_tokens(ids, tok, pos, out, Lp):
    """out[b*Lp + i] = tok[ids[b, i]] + pos[i] for i < L, zero rows up to Lp.  ids: int64 [B, L]; tok [V, C], pos [>= L, C], out [B*Lp, C].
    Host ids are range-checked (ValueError) and copied to out's device; on-device ids outside [0, V) read as zero token rows."""
    if ids.ndim != 2 or ids.dtype != torch.int64:
        raise TypeError(f"embed_tokens: ids must be int64 [B, L], got {ids.dtype} {tuple(ids.shape)}")
    B, L = ids.shape
    V, C = tok.shape
    if L > pos.shape[0] or L > Lp:
        raise ValueError(f"embed_tokens: {L} tokens but {pos.shape[0]} positions / {Lp} rows")
    if ids.device.type == "cpu":
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= V):
            raise ValueError(f"embed_tokens: token ids must lie in [0, {V}), got [{int(ids.min())}, {int(ids.max())}]")
        ids = ids.to(out.device)
    ids = ids.contiguous()
    _chk(ids, "ids")
    if tok.dtype != out.dtype or pos.dtype != out.dtype:
        raise TypeError(f"embed_tokens: tok {tok.dtype} / pos {pos.dtype} / out {out.dtype} must match")
    assert tok.is_contiguous() and pos.is_contiguous() and out.is_contiguous() and out.shape == (B * Lp, C)
    call("cid_embed_tokens", _p(ids), B, L, Lp, _p(tok), V, _p(pos), _p(out), C, _dt(out), _stream())
    return out


def attn_cross(q, k_cat, vt_cat, out, B, H, N, d, n_text, n_ip, ip_scale):
    with _prof("attn_cross", 4.0 * B * H * N * (n_text + n_ip) * d, 2.0 * 2 * B * N * H * d, ("B%d" % B, "H%d" % H, "N%d" % N, "d%d" % d)):
        call("cid_attn_cross", _p(q), q.stride(0), _p(k_cat), _p(vt_cat), _p(out), out.stride(0), B, H, N, d, n_text, n_ip,
             float(ip_scale), _dt(q), _stream())
    return out


def pack_cross_kv(k_text, v_text, k_ip, v_ip, k_cat, vt_cat, B, C, heads, n_text, n_ip):
    call("cid_pack_cross_kv", _p(k_text), _p(v_text), _p(k_ip), _p(v_ip), _p(k_cat), _p(vt_cat), B, C, heads, n_text, n_ip, _stream())


def gn_stats(x1, C1, x2, C2, NB, HW, groups, sums, zero_sums=True):
    with _prof("gn_stats", 0.0, 2.0 * NB * HW * (C1 + C2), (NB * HW, C1 + C2)):                     # one read of the tensor
        call("cid_gn_stats", _p(x1), C1, _p(x2), C2, NB, HW, groups, _p(sums), 1 if zero_sums else 0, _dt(x1), _stream())


def gn_apply(x1, C1, x2, C2, NB, HW, groups, sums, gamma, beta, eps, silu, out, zero_next=None):
    with _prof("gn_apply", 0.0, 4.0 * NB * HW * (C1 + C2), (NB * HW, C1 + C2)):                     # one read + one write
        call("cid_gn_apply", _p(x1), C1, _p(x2), C2, NB, HW, groups, _p(sums), _p(gamma), _p(beta), float(eps), 1 if silu else 0,
             _p(out), _p(zero_next), _dt(x1), _stream())
    return out


def gn_apply_ch(x1, C1, sums1, x2, C2, sums2, NB, HW, groups, gamma, beta, eps, silu, out):
    """GroupNorm apply with per-(sample, channel) statistics from the producers' epilogues (``chan_stats`` of gemm / conv3x3)."""
    with _prof("gn_apply", 0.0, 4.0 * NB * HW * (C1 + C2), (NB * HW, C1 + C2)):
        call("cid_gn_apply_ch", _p(x1), C1, _p(sums1), _p(x2), C2, _p(sums2), NB, HW, groups, _p(gamma), _p(beta), float(eps), 1 if silu else 0,
             _p(out), _dt(x1), _stream())
    return out


GN_SMALL_MAX_ELEMS = 32768          # HW * C/groups a CTA of cid_gn_small holds in registers


def gn_small_ok(C1, C2, HW, groups):
    """True when cid_gn_small applies: 8-channel vectors inside groups, groups inside one source of the virtual concat, slab small enough."""
    C = C1 + C2
    if C % groups:
        return False
    cpg = C // groups
    return cpg % 8 == 0 and C1 % cpg == 0 and HW * cpg <= GN_SMALL_MAX_ELEMS


def gn_small(x1, C1, x2, C2, NB, HW, groups, gamma, beta, eps, silu, out):
    """One-pass GroupNorm(+SiLU) of a small tensor (statistics and apply in one launch)."""
    with _prof("gn_apply", 0.0, 4.0 * NB * HW * (C1 + C2), (NB * HW, C1 + C2)):
        call("cid_gn_small", _p(x1), C1, _p(x2), C2, NB, HW, groups, _p(gamma), _p(beta), float(eps), 1 if silu else 0, _p(out), _dt(x1), _stream())
    return out


def layernorm(x, gamma, beta, out, rows, C, eps=1e-5):
    with _prof("layernorm", 0.0, 4.0 * rows * C, (rows, C)):
        call("cid_layernorm", _p(x), _p(gamma), _p(beta), _p(out), rows, C, float(eps), _dt(x), _stream())
    return out


def upsample2x(x, out, NB, H, W, C):
    with _prof("upsample2x", 0.0, 2.0 * NB * H * W * C * 5):                    # read 1x, write 4x
        call("cid_upsample2x", _p(x), _p(out), NB, H, W, C, _stream())
    return out


def phase_split(x, out, NB, H, W, C):
    with _prof("phase_split", 0.0, 4.0 * NB * H * W * C):
        call("cid_phase_split", _p(x), _p(out), NB, H, W, C, _stream())
    return out


def nchw_to_nhwc_pad(x, out, NB, Cin, HW, CP, scale_dev=None):
    call("cid_nchw_to_nhwc_pad", _p(x), _p(out), NB, Cin, HW, CP, _p(scale_dev), _dt(x), _stream())
    return out


def rows_to_nchw(x, ld, out, NB, Cout, HW):
    call("cid_rows_to_nchw", _p(x), ld, _p(out), NB, Cout, HW, _stream())
    return out


def add_inplace(y, x):
    call("cid_add_inplace", _p(y), _p(x), y.numel(), _dt(y), _stream())
    return y


def timestep_embed(t_dev, t_stride, rows, dim, out, ld, col0=0):
    call("cid_timestep_embed", _p(t_dev), t_stride, rows, dim, _p(out), ld, col0, _dt(out), _stream())
    return out


def skinny_linear(x, w, bias, out, M, N, K, silu_in=False, accumulate=False, act_in=None):
    """out[M,N] (+)= act(x) @ w.T + bias; act_in: None -> SiLU if silu_in else identity; "silu" | "gelu" | "none"."""
    act = {None: 1 if silu_in else 0, "none": 0, "silu": 1, "gelu": 2}[act_in]
    call("cid_skinny_linear", _p(x), x.stride(0), _p(w), _p(bias), _p(out), out.stride(0), M, N, K, act,
         1 if accumulate else 0, _dt(x), _stream())
    return out


def layernorm_rows(x, gamma, beta, out, rows, C, eps=1e-5, rows_per_group=None, x_group_rows=None, x_row0=0, y_group_rows=None, y_row0=0):
    """LayerNorm over ``rows`` logical rows of width C with the grouped row mapping of cid_layernorm_rows (x, out: 2-D row views)."""
    rpg = rows if rows_per_group is None else rows_per_group
    call("cid_layernorm_rows", _p(x), x.stride(0), rpg if x_group_rows is None else x_group_rows, x_row0, _p(gamma), _p(beta), _p(out),
         out.stride(0), rpg if y_group_rows is None else y_group_rows, y_row0, rows, max(rpg, 1), C, float(eps), _dt(x), _stream())
    return out


def softmax_rows(x, rows, cols):
    """In-place fp32-math softmax over the rows of the 16-bit matrix x[rows, cols] (row pitch x.stride(0))."""
    call("cid_softmax_rows", _p(x), x.stride(0), rows, cols, _dt(x), _stream())
    return x


def perceiver_attn(q, kv, out, B, L, n_kv, heads, dim_head=64):
    """q [B*L, heads*64], kv [B*n_kv, 2*heads*64] (K | V), out [B*L, heads*64] (functions.py:446-453)."""
    call("cid_perceiver_attn", _p(q), q.stride(0), _p(kv), kv.stride(0), _p(out), out.stride(0), B, L, n_kv, heads, dim_head, _dt(q), _stream())
    return out


def cfg_sched_step(eps, ld_eps, x, x0_prev, x16, next_in, CP, B, HW, guidance, coef_table, step_dev):
    # eps 2 x 4 ch x 2 B read (a 16-byte sector per pixel is touched), x / x0 fp32 read + write, x16 write, next input 2 x 16 B write
    with _prof("cfg_sched_step", 0.0, B * HW * (2 * 8 + 4 * 4 * 4 + 4 * 2 + (32 if next_in is not None else 0))):
        return _cfg_sched_step(eps, ld_eps, x, x0_prev, x16, next_in, CP, B, HW, guidance, coef_table, step_dev)


def _cfg_sched_step(eps, ld_eps, x, x0_prev, x16, next_in, CP, B, HW, guidance, coef_table, step_dev):
    call("cid_cfg_sched_step", _p(eps), ld_eps, _p(x), _p(x0_prev), _p(x16), _p(next_in), CP, B, HW, float(guidance),
         _p(coef_table), _p(step_dev), _dt(eps), _stream())


def latents_to_input(x, next_in, CP, B, HW, coef_table, step_dev=None, nsteps=1, keep_ch4_up=False):
    call("cid_latents_to_input", _p(x), _p(next_in), CP, B, HW, _p(coef_table), _p(step_dev), nsteps, 1 if keep_ch4_up else 0,
         _dt(next_in), _stream())


def silu_inplace(y):
    call("cid_silu_inplace", _p(y), y.numel(), _dt(y), _stream())
    return y


def inpaint_blend(x, x16, image_latents, noise, mask, B, HW, blend_table, step_dev):
    call("cid_inpaint_blend", _p(x), _p(x16), _p(image_latents), _p(noise), _p(mask), B, HW, _p(blend_table), _p(step_dev),
         _dt(x16), _stream())


def advance_step(step_dev, t_dev, ts_table, n):
    call("cid_advance_step", _p(step_dev), _p(t_dev), _p(ts_table), n, _stream())
