"""Python operators over the C ABI (include/motionclone_b200.h): tensors in, tensors out, autograd where the
reference's torch.autograd.grad (utils/motionclone_functions.py:236) must keep working. CUDA fp16 only — anything
else raises; there is no eager fallback."""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import TemporalLayout

Tensor = torch.Tensor


class KernelTimer:
    """CUDA-event timing of this package's launches on the launching stream (bench.py's roofline leg). Installed with
    `ops.TIMER = KernelTimer()`; `summary()` synchronises and returns {kernel: (launches, algorithmic_bytes, ms)}."""

    def __init__(self):
        self.records = []

    def start(self):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream())
        return ev

    def stop(self, name: str, nbytes: int, ev0):
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record(torch.cuda.current_stream())
        self.records.append((name, nbytes, ev0, ev1))

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, nbytes, e0, e1 in self.records:
            n, b, ms = out.get(name, (0, 0, 0.0))
            out[name] = (n + 1, b + nbytes, ms + e0.elapsed_time(e1))
        return out


TIMER: Optional[KernelTimer] = None


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _require(t: Tensor, name: str, dtype=torch.float16) -> None:
    if not t.is_cuda or t.dtype != dtype:
        raise TypeError(f"{name}: expected a CUDA {dtype} tensor, got {t.device} {t.dtype} "
                        "(motionclone_b200 kernels have no CPU / fp32 path)")


def _layout_bfpc(t: Tensor) -> TemporalLayout:
    """t is a [B, F, P, C] view (any strides, C contiguous)."""
    if t.dim() != 4 or t.stride(3) != 1:
        raise ValueError("temporal tensor must be a [B, F, P, C] view with contiguous channels")
    return TemporalLayout(t.stride(0), t.stride(1), t.stride(2))


# ----------------------------------------------------------------------------------------------------------------
# temporal attention
# ----------------------------------------------------------------------------------------------------------------
def temporal_attention_forward(q: Tensor, k: Tensor, v: Optional[Tensor], heads: int, scale: float, *,
                               want_o: bool = True, want_probs: bool = False, want_top1: bool = False,
                               gather_idx: Optional[Tensor] = None):
    """q, k, v: [B, F, P, C] views sharing one stride pattern (e.g. slices of a fused QKV buffer).

    Returns (o [B,F,P,C] contiguous | None, probs [B*P,H,F,F] | None, (top_val, top_idx) [B*P,H,F,1] | None,
             gathered [B*P,H,F,1] | None) — per-row outputs in the reference's order (motionclone_functions.py:280).
    """
    _require(q, "q"), _require(k, "k")
    B, F, P, C = q.shape
    if C % heads:
        raise ValueError("channels not divisible by heads")
    lay = _layout_bfpc(q)
    for name, t in (("k", k), ("v", v)):
        if t is not None and (t.shape != q.shape or t.stride() != q.stride()):
            raise ValueError(f"{name} must share q's shape and strides")
    o = torch.empty((B, F, P, C), dtype=q.dtype, device=q.device) if want_o else None
    if want_o:
        _require(v, "v")
    rows = (B * P, heads, F)
    probs = torch.empty(rows + (F,), dtype=q.dtype, device=q.device) if want_probs else None
    tv = torch.empty(rows + (1,), dtype=q.dtype, device=q.device) if want_top1 else None
    ti = torch.empty(rows + (1,), dtype=torch.uint8, device=q.device) if want_top1 else None
    gathered = None
    if gather_idx is not None:
        _require(gather_idx, "gather_idx", torch.uint8)
        if gather_idx.numel() != B * P * heads * F or not gather_idx.is_contiguous():
            raise ValueError("gather_idx must be a contiguous uint8 [B*P, H, F, 1] tensor")
        gathered = torch.zeros(rows + (1,), dtype=q.dtype, device=q.device)
    ev0 = TIMER.start() if TIMER is not None else None
    st = _lib.lib().mc_temporal_attn_fwd(_ptr(q), _ptr(k), _ptr(v if want_o else None), lay,
                                         _ptr(o), _layout_bfpc(o) if want_o else TemporalLayout(0, 0, 0),
                                         _ptr(probs), _ptr(tv), _ptr(ti), _ptr(gather_idx), _ptr(gathered),
                                         B, P, F, heads, C // heads, float(scale), _stream())
    _lib.check(st, "mc_temporal_attn_fwd")
    if ev0 is not None:  # algorithmic bytes: Q, K, V read + O written (SURVEY.md §8d); by-products are not counted
        TIMER.stop("temporal_attn_fwd", (4 if want_o else 2) * B * F * P * C * 2, ev0)
    return o, probs, ((tv, ti) if want_top1 else None), gathered


def _is_fused_qkv(q: Tensor, k: Tensor, v: Optional[Tensor]) -> bool:
    c = q.shape[-1]
    return (v is not None and q.stride(2) == 3 * c and k.data_ptr() == q.data_ptr() + 2 * c
            and v.data_ptr() == q.data_ptr() + 4 * c)


def temporal_attention_backward(q: Tensor, k: Tensor, v: Optional[Tensor], heads: int, scale: float,
                                d_o: Optional[Tensor], d_probs: Optional[Tensor], gather_idx: Optional[Tensor],
                                d_gathered: Optional[Tensor], need_dv: bool = True, return_fused: bool = False):
    """-> (dq, dk, dv). When q, k, v are the column blocks of one fused [B, F, P, 3C] buffer the gradients are written
    as the column blocks of one [B, F, P, 3C] buffer too (`return_fused=True` returns that buffer instead)."""
    B, F, P, C = q.shape
    lay = _layout_bfpc(q)
    if d_o is not None:
        _require(d_o, "d_o")
        if d_o.stride(3) != 1:
            d_o = d_o.contiguous()
    if d_probs is not None:
        d_probs = d_probs.contiguous()
    if d_gathered is not None:
        d_gathered = d_gathered.contiguous()
    want_dv = need_dv and d_o is not None
    fused = _is_fused_qkv(q, k, v)
    if fused:
        dqkv = torch.empty((B, F, P, 3 * C), dtype=q.dtype, device=q.device)
        dq, dk, dv = dqkv[..., :C], dqkv[..., C:2 * C], dqkv[..., 2 * C:]
        if not want_dv:
            dv.zero_()
    else:
        dqkv = None
        dq = torch.empty((B, F, P, C), dtype=q.dtype, device=q.device)
        dk = torch.empty_like(dq)
        dv = torch.empty_like(dq) if want_dv else None
    ev0 = TIMER.start() if TIMER is not None else None
    st = _lib.lib().mc_temporal_attn_bwd(_ptr(q), _ptr(k), _ptr(v), lay,
                                         _ptr(d_o), _layout_bfpc(d_o) if d_o is not None else TemporalLayout(0, 0, 0),
                                         _ptr(d_probs), _ptr(gather_idx), _ptr(d_gathered),
                                         _ptr(dq), _ptr(dk), _ptr(dv if want_dv else None), _layout_bfpc(dq),
                                         B, P, F, heads, C // heads, float(scale), _stream())
    _lib.check(st, "mc_temporal_attn_bwd")
    if ev0 is not None:  # Q, K (V, dO) read; dQ, dK (dV) written
        TIMER.stop("temporal_attn_bwd", (7 if d_o is not None else 4) * B * F * P * C * 2, ev0)
    if return_fused:
        if not fused:
            raise ValueError("return_fused needs q, k, v to be column blocks of one [.., 3C] buffer")
        return dqkv
    return dq, dk, (dv if (want_dv or fused) else None)


class TemporalAttention(torch.autograd.Function):
    """o, probs, gathered = f(qkv) with qkv = [B, F, P, 3C] (one fused projection; q | k | v column blocks); probs and
    gathered can be switched off.

    Backward recomputes the probabilities in-kernel, sums the three incoming gradient branches before the softmax
    backward (the reference builds them as separate autograd branches off the same q, k: models/attention.py:461-490
    for o and :564-611 via utils/motionclone_functions.py:279 for the probabilities) and writes ONE [B, F, P, 3C]
    gradient, so autograd sees a single edge instead of three slice-backward zero-fills.
    """

    @staticmethod
    def forward(ctx, qkv, heads: int, scale: float, want_probs: bool, gather_idx):
        c = qkv.shape[-1] // 3
        q, k, v = qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:]
        o, probs, _, gathered = temporal_attention_forward(q, k, v, heads, scale, want_o=True, want_probs=want_probs,
                                                           gather_idx=gather_idx)
        ctx.save_for_backward(qkv, gather_idx)
        ctx.heads, ctx.scale = heads, scale
        outs = (o, probs if probs is not None else qkv.new_empty(0),
                gathered if gathered is not None else qkv.new_empty(0))
        ctx.mark_non_differentiable(*[t for t, used in ((outs[1], want_probs), (outs[2], gather_idx is not None))
                                      if not used])
        return outs

    @staticmethod
    def backward(ctx, d_o, d_probs, d_gathered):
        qkv, gather_idx = ctx.saved_tensors
        c = qkv.shape[-1] // 3
        q, k, v = qkv[..., :c], qkv[..., c:2 * c], qkv[..., 2 * c:]
        if d_probs is not None and d_probs.numel() == 0:
            d_probs = None
        if d_gathered is not None and d_gathered.numel() == 0:
            d_gathered = None
        dqkv = temporal_attention_backward(q, k, v, ctx.heads, ctx.scale, d_o, d_probs,
                                           gather_idx if d_gathered is not None else None, d_gathered,
                                           need_dv=True, return_fused=True)
        return dqkv, None, None, None, None


class TemporalProbs(torch.autograd.Function):
    """probs = softmax(scale q k^T) only (get_attention_scores, models/attention.py:564-611), differentiable."""

    @staticmethod
    def forward(ctx, q, k, heads: int, scale: float):
        _, probs, _, _ = temporal_attention_forward(q, k, None, heads, scale, want_o=False, want_probs=True)
        ctx.save_for_backward(q, k)
        ctx.heads, ctx.scale = heads, scale
        return probs

    @staticmethod
    def backward(ctx, d_probs):
        q, k = ctx.saved_tensors
        dq, dk, _ = temporal_attention_backward(q, k, None, ctx.heads, ctx.scale, None, d_probs, None, None)
        return dq, dk, None, None


def top1_rows(probs: Tensor) -> Tuple[Tensor, Tensor]:
    """torch.topk(probs, k=1, dim=-1) -> (values, uint8 indices), lowest index on ties (motionclone_functions.py:79)."""
    _require(probs, "probs")
    probs = probs.contiguous()
    L = probs.shape[-1]
    rows = probs.numel() // L
    val = torch.empty(probs.shape[:-1] + (1,), dtype=probs.dtype, device=probs.device)
    idx = torch.empty(probs.shape[:-1] + (1,), dtype=torch.uint8, device=probs.device)
    _lib.check(_lib.lib().mc_top1_rows(_ptr(probs), rows, L, _ptr(val), _ptr(idx), _stream()), "mc_top1_rows")
    return val, idx


# ----------------------------------------------------------------------------------------------------------------
# motion loss on gathered probabilities
# ----------------------------------------------------------------------------------------------------------------
def _ptr_array(ts: Sequence[Tensor]):
    arr = (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    return arr


class MotionLoss(torch.autograd.Function):
    """sum_m mse(cur_m, ref_m) with F.mse_loss's fp16 rounding sequence (utils/motionclone_functions.py:96-100)."""

    @staticmethod
    def forward(ctx, n_modules: int, *tensors):
        cur = [t.contiguous() for t in tensors[:n_modules]]
        ref = [t.contiguous() for t in tensors[n_modules:]]
        for t in cur + ref:
            _require(t, "motion loss operand")
        n = (ctypes.c_int64 * n_modules)(*[t.numel() for t in cur])
        per = torch.empty(n_modules, dtype=torch.float16, device=cur[0].device)
        total = torch.empty((), dtype=torch.float16, device=cur[0].device)
        st = _lib.lib().mc_motion_loss_fwd(n_modules, _ptr_array(cur), _ptr_array(ref), n, _ptr(per), _ptr(total),
                                           _stream())
        _lib.check(st, "mc_motion_loss_fwd")
        ctx.save_for_backward(*cur, *ref)
        ctx.n_modules = n_modules
        ctx.shapes = [t.shape for t in tensors[:n_modules]]
        return total

    @staticmethod
    def backward(ctx, g):
        M = ctx.n_modules
        saved = ctx.saved_tensors
        cur, ref = list(saved[:M]), list(saved[M:])
        d = [torch.empty_like(t) for t in cur]
        n = (ctypes.c_int64 * M)(*[t.numel() for t in cur])
        g = g.to(torch.float16).contiguous()
        st = _lib.lib().mc_motion_loss_bwd(M, _ptr_array(cur), _ptr_array(ref), n, _ptr(g), _ptr_array(d), _stream())
        _lib.check(st, "mc_motion_loss_bwd")
        return (None, *[x.view(s) for x, s in zip(d, ctx.shapes)], *([None] * M))


def motion_loss(cur: List[Tensor], ref: List[Tensor]) -> Tensor:
    return MotionLoss.apply(len(cur), *cur, *ref)


# ----------------------------------------------------------------------------------------------------------------
# CFG + DDIM, add_noise
# ----------------------------------------------------------------------------------------------------------------
def cfg_ddim_step(eps_cond: Tensor, eps_uncond: Optional[Tensor], x: Tensor, score: Optional[Tensor], cfg_scale: float,
                  alpha_t: Tensor, alpha_prev: Tensor, guidance_scale: float = 1.0) -> Tensor:
    """One fused launch for motionclone_functions.py:239 + :339-389. alpha_* are 0-dim fp32 CPU tensors taken from
    alphas_cumprod on the host (no device sync); the scalar algebra is done in fp32 torch ops exactly as the
    reference does it (`beta_prod_t ** 0.5` etc.), so the coefficients are bit-identical."""
    for name, t in (("eps_cond", eps_cond), ("x", x)):
        _require(t, name)
    eps_cond, x = eps_cond.contiguous(), x.contiguous()
    if eps_uncond is not None:
        _require(eps_uncond, "eps_uncond")
        eps_uncond = eps_uncond.contiguous()
    if score is not None:
        _require(score, "score")
        score = score.contiguous()
    a_t = alpha_t.detach().to(torch.float32).cpu()
    a_p = alpha_prev.detach().to(torch.float32).cpu()
    sb = float((1 - a_t) ** 0.5)
    inv_sa = float(1.0 / (a_t ** 0.5))
    sap = float(a_p ** 0.5)
    c = float((1 - a_p - 0.0) ** 0.5)
    sc = float(guidance_scale * (1 - a_t) ** 0.5)
    out = torch.empty_like(x)
    st = _lib.lib().mc_cfg_ddim_step(_ptr(eps_cond), _ptr(eps_uncond), _ptr(x), _ptr(score), _ptr(out), x.numel(),
                                     float(cfg_scale), sb, inv_sa, sap, c, sc, _stream())
    _lib.check(st, "mc_cfg_ddim_step")
    return out


def add_noise(x0: Tensor, noise: Tensor, alpha_t: Tensor) -> Tensor:
    """motionclone_functions.py:19-23."""
    _require(x0, "x0"), _require(noise, "noise")
    x0, noise = x0.contiguous(), noise.contiguous()
    a = alpha_t.detach().to(torch.float32).cpu()
    out = torch.empty_like(x0)
    st = _lib.lib().mc_add_noise(_ptr(x0), _ptr(noise), _ptr(out), x0.numel(), float(a ** 0.5), float((1 - a) ** 0.5),
                                 _stream())
    _lib.check(st, "mc_add_noise")
    return out


# ----------------------------------------------------------------------------------------------------------------
# NHWC GroupNorm(+SiLU), LayerNorm, GEGLU (inference passes)
# ----------------------------------------------------------------------------------------------------------------
_gn_workspace = {}


def glue_kernels_ok(x: Tensor) -> bool:
    """CUDA fp16 activations: the only thing the kernels of this package accept."""
    return x.is_cuda and x.dtype == torch.float16


def _require_param(t: Tensor, name: str, like: Tensor, numel: int) -> Tensor:
    """Norm gains / biases are read as raw fp16 pointers by the kernels: same device, fp16, contiguous, right length."""
    _require(t, name)
    if t.device != like.device or t.numel() != numel:
        raise ValueError(f"{name}: expected {numel} fp16 values on {like.device}, got {t.numel()} on {t.device}")
    return t.contiguous()


def _workspace(x: Tensor, need: int, role: str = "fwd") -> Tensor:
    """Per (device, stream, role) scratch for the GroupNorm kernels. Zero-initialised: its first 4 KB are the per-frame
    tickets of the last-CTA reduction, which the kernels leave at zero (include/motionclone_b200.h). Forward and backward
    use different buffers (the forward's finalised statistics are copied out for the backward)."""
    key = (x.device, torch.cuda.current_stream().cuda_stream, role)
    ws = _gn_workspace.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=x.device)
        _gn_workspace[key] = ws
    return ws


def _check_chan_bias(x: Tensor, chan_bias: Optional[Tensor]):
    if chan_bias is None:
        return None, 0
    _require(chan_bias, "chan_bias")
    chan_bias = chan_bias.contiguous()
    if chan_bias.dim() != 2 or chan_bias.shape[1] != x.shape[1] or x.shape[0] % chan_bias.shape[0]:
        raise ValueError("chan_bias must be [NB, C] with N divisible by NB")
    return chan_bias, x.shape[0] // chan_bias.shape[0]


def groupnorm_nhwc(x: Tensor, weight: Tensor, bias: Tensor, groups: int, eps: float, silu: bool = False,
                   chan_bias: Optional[Tensor] = None, want_stats: bool = False):
    """x: [N, C, h, w] in channels_last (physically [N, h, w, C]); returns the same format. `chan_bias` [NB, C]
    (N % NB == 0) is added to x first, row n // (N // NB) — the resnet's time-embedding add folded in.
    `want_stats` also returns (mean, rstd) [N, groups, 2] fp32 for the backward."""
    _require(x, "x")
    if x.dim() != 4 or not x.is_contiguous(memory_format=torch.channels_last):
        raise ValueError("groupnorm_nhwc expects a 4-D channels_last tensor")
    chan_bias, fpr = _check_chan_bias(x, chan_bias)
    N, C, H, W = x.shape
    weight, bias = _require_param(weight, "groupnorm weight", x, C), _require_param(bias, "groupnorm bias", x, C)
    y = torch.empty_like(x)  # preserves channels_last
    ws = _workspace(x, int(_lib.lib().mc_groupnorm_workspace_bytes(N, groups)))
    st = _lib.lib().mc_groupnorm_nhwc(_ptr(x), _ptr(chan_bias), fpr, _ptr(y), _ptr(weight), _ptr(bias), _ptr(ws),
                                      ws.numel(), N, H * W, C, groups, float(eps), int(silu), _stream())
    _lib.check(st, "mc_groupnorm_nhwc")
    if not want_stats:
        return y
    stats = torch.empty(N, groups, 2, dtype=torch.float32, device=x.device)
    _lib.check(_lib.lib().mc_groupnorm_nhwc_stats(_ptr(ws), _ptr(stats), N, H * W, groups, float(eps), _stream()),
               "mc_groupnorm_nhwc_stats")
    return y, stats


class GroupNormNHWCFn(torch.autograd.Function):
    """GroupNorm(+chan_bias)(+SiLU) on channels_last with the input gradient from csrc/norm_act.cu (weights frozen)."""

    @staticmethod
    def forward(ctx, x, weight, bias, chan_bias, groups: int, eps: float, silu: bool):
        y, stats = groupnorm_nhwc(x, weight, bias, groups, eps, silu, chan_bias, want_stats=True)
        ctx.save_for_backward(x, weight, bias, chan_bias, stats)
        ctx.groups, ctx.silu = groups, silu
        return y

    @staticmethod
    def backward(ctx, dz):
        x, weight, bias, chan_bias, stats = ctx.saved_tensors
        _require(dz, "dz")
        dz = dz.contiguous(memory_format=torch.channels_last)
        chan_bias, fpr = _check_chan_bias(x, chan_bias)
        N, C, H, W = x.shape
        weight, bias = _require_param(weight, "groupnorm weight", x, C), _require_param(bias, "groupnorm bias", x, C)
        dx = torch.empty_like(x)
        ws = _workspace(x, int(_lib.lib().mc_groupnorm_workspace_bytes(N, ctx.groups)), "bwd")
        st = _lib.lib().mc_groupnorm_nhwc_bwd(_ptr(x), _ptr(chan_bias), fpr, _ptr(dz), _ptr(dx), _ptr(stats), _ptr(weight),
                                              _ptr(bias), _ptr(ws), ws.numel(), N, H * W, C, ctx.groups, int(ctx.silu),
                                              _stream())
        _lib.check(st, "mc_groupnorm_nhwc_bwd")
        return dx, None, None, None, None, None, None


def layernorm(x: Tensor, weight: Tensor, bias: Tensor, eps: float, post_add: Optional[Tensor] = None,
              rows_per_frame: int = 0, pre_bias: Optional[Tensor] = None) -> Tensor:
    """LayerNorm over the last dim of (x + pre_bias); `post_add` [F, C] is added to row r at frame
    (r // rows_per_frame) % F (the temporal positional encoding on (b f)-major tokens)."""
    _require(x, "x")
    x = x.contiguous()
    C = x.shape[-1]
    weight, bias = _require_param(weight, "layernorm weight", x, C), _require_param(bias, "layernorm bias", x, C)
    if pre_bias is not None:
        pre_bias = _require_param(pre_bias, "layernorm pre_bias", x, C)
    y = torch.empty_like(x)
    frames = 0
    if post_add is not None:
        _require(post_add, "post_add")
        post_add = post_add.contiguous()
        frames = post_add.shape[0]
    st = _lib.lib().mc_layernorm(_ptr(x), _ptr(y), _ptr(weight), _ptr(bias), _ptr(post_add), _ptr(pre_bias),
                                 int(rows_per_frame), frames, x.numel() // C, C, float(eps), _stream())
    _lib.check(st, "mc_layernorm")
    return y


class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps: float, post_add, rows_per_frame: int, pre_bias=None):
        x = x.contiguous()
        ctx.save_for_backward(x, weight, pre_bias)
        ctx.eps = eps
        return layernorm(x, weight, bias, eps, post_add, rows_per_frame, pre_bias)

    @staticmethod
    def backward(ctx, dy):
        x, weight, pre_bias = ctx.saved_tensors
        _require(dy, "dy")
        dy = dy.contiguous()
        C = x.shape[-1]
        weight = _require_param(weight, "layernorm weight", x, C)
        dx = torch.empty_like(x)
        st = _lib.lib().mc_layernorm_bwd(_ptr(x), _ptr(dy), _ptr(dx), _ptr(weight), _ptr(pre_bias), x.numel() // C, C,
                                         float(ctx.eps), _stream())
        _lib.check(st, "mc_layernorm_bwd")
        return dx, None, None, None, None, None, None


def geglu(x: Tensor) -> Tensor:
    """x [..., 2I] = [h | gate] -> h * gelu_erf(gate) [..., I]."""
    _require(x, "x")
    x = x.contiguous()
    I = x.shape[-1] // 2
    out = torch.empty(x.shape[:-1] + (I,), dtype=x.dtype, device=x.device)
    st = _lib.lib().mc_geglu(_ptr(x), _ptr(out), x.numel() // (2 * I), I, _stream())
    _lib.check(st, "mc_geglu")
    return out


class GEGLUFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous()
        ctx.save_for_backward(x)
        return geglu(x)

    @staticmethod
    def backward(ctx, dout):
        (x,) = ctx.saved_tensors
        dout = dout.contiguous()
        I = x.shape[-1] // 2
        din = torch.empty_like(x)
        st = _lib.lib().mc_geglu_bwd(_ptr(x), _ptr(dout), _ptr(din), x.numel() // (2 * I), I, _stream())
        _lib.check(st, "mc_geglu_bwd")
        return din


def bias_residual_add(a: Tensor, b: Tensor, bias: Tensor) -> Tensor:
    """a + bias[c] + b for channels_last 4-D (or channel-last N-D) tensors with identical strides."""
    _require(a, "a"), _require(b, "b"), _require(bias, "bias")
    if a.shape != b.shape or a.stride() != b.stride():
        raise ValueError("bias_residual_add: a and b must share shape and strides")
    if a.dim() == 4:
        if not a.is_contiguous(memory_format=torch.channels_last):
            raise ValueError("bias_residual_add: 4-D inputs must be channels_last")
        C = a.shape[1]
    else:
        if not a.is_contiguous():
            raise ValueError("bias_residual_add: N-D inputs must be contiguous with channels last")
        C = a.shape[-1]
    out = torch.empty_like(a)
    st = _lib.lib().mc_bias_residual_add(_ptr(a), _ptr(b), _ptr(bias.contiguous()), _ptr(out), a.numel(), C, _stream())
    _lib.check(st, "mc_bias_residual_add")
    return out


class BiasResidualAddFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, bias):
        return bias_residual_add(a, b, bias)

    @staticmethod
    def backward(ctx, g):
        return g, g, None


def _check_xattn(q: Tensor, k: Tensor, v: Tensor) -> None:
    for name, t in (("q", q), ("k", k), ("v", v)):
        _require(t, name)
        if t.dim() != 3 or t.stride(2) != 1:
            raise ValueError(f"{name} must be [B, N, C] with contiguous channels")
    if k.shape != v.shape or k.stride() != v.stride():
        raise ValueError("k and v must share shape and strides")


def cross_attention_forward(q: Tensor, k: Tensor, v: Tensor, heads: int, scale: float) -> Tensor:
    """tcgen05 text cross-attention (csrc/cross_attn_fwd_tc.cu, csrc/cross_attn_bwd_tc.cu): q [B, Nq, C], k / v [B, Nk <= 80, C] -> [B, Nq, C]."""
    _check_xattn(q, k, v)
    B, Nq, C = q.shape
    o = torch.empty((B, Nq, C), dtype=q.dtype, device=q.device)
    ev0 = TIMER.start() if TIMER is not None else None
    st = _lib.lib().mc_cross_attn_fwd(_ptr(q), _ptr(k), _ptr(v), _ptr(o), B, Nq, k.shape[1], heads, C // heads,
                                      q.stride(0), q.stride(1), k.stride(0), k.stride(1), o.stride(0), o.stride(1),
                                      float(scale), _stream())
    _lib.check(st, "mc_cross_attn_fwd")
    if ev0 is not None:  # algorithmic bytes: Q read + O written (K, V are 77 rows)
        TIMER.stop("cross_attn_fwd", 2 * B * Nq * C * 2, ev0)
    return o


def cross_attention_backward(q: Tensor, k: Tensor, v: Tensor, d_o: Tensor, heads: int, scale: float) -> Tensor:
    """dQ of the text cross-attention (the text K / V carry no gradient on this path): q, d_o [B, Nq, C] -> dq."""
    _check_xattn(q, k, v)
    _require(d_o, "d_o")
    if d_o.shape != q.shape:
        raise ValueError("d_o must have q's shape")
    if d_o.stride(2) != 1:
        d_o = d_o.contiguous()
    B, Nq, C = q.shape
    dq = torch.empty((B, Nq, C), dtype=q.dtype, device=q.device)
    ev0 = TIMER.start() if TIMER is not None else None
    st = _lib.lib().mc_cross_attn_bwd_dq(_ptr(q), _ptr(k), _ptr(v), _ptr(d_o), _ptr(dq), B, Nq, k.shape[1], heads,
                                         C // heads, q.stride(0), q.stride(1), k.stride(0), k.stride(1), d_o.stride(0),
                                         d_o.stride(1), dq.stride(0), dq.stride(1), float(scale), _stream())
    _lib.check(st, "mc_cross_attn_bwd_dq")
    if ev0 is not None:  # Q, dO read + dQ written
        TIMER.stop("cross_attn_bwd", 3 * B * Nq * C * 2, ev0)
    return dq


class CrossAttentionTC(torch.autograd.Function):
    """o = softmax(scale q k^T) v on the tcgen05 kernels, differentiable w.r.t. q only (see mc_cross_attn_bwd_dq)."""

    @staticmethod
    def forward(ctx, q, k, v, heads: int, scale: float):
        ctx.save_for_backward(q, k, v)
        ctx.heads, ctx.scale = heads, scale
        return cross_attention_forward(q, k, v, heads, scale)

    @staticmethod
    def backward(ctx, d_o):
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            raise NotImplementedError("cross-attention gradients w.r.t. the text K / V are not on the MotionClone path "
                                      "(frozen projections of a constant prompt embedding)")
        q, k, v = ctx.saved_tensors
        return cross_attention_backward(q, k, v, d_o, ctx.heads, ctx.scale), None, None, None, None


# ----------------------------------------------------------------------------------------------------------------
# spatial self-attention (tcgen05 + tensor-map TMA flash kernel, csrc/spatial_attn_tc.cu)
# ----------------------------------------------------------------------------------------------------------------
# head dims the attention kernels are instantiated for: spatial self-attention and text cross-attention alike
ATTN_HEAD_DIMS = (8, 16, 32, 40, 64, 80, 160)


def _check_bnc(name: str, t: Tensor) -> None:
    _require(t, name)
    if t.dim() != 3 or t.stride(2) != 1 or t.stride(0) % 8 or t.stride(1) % 8 or t.data_ptr() % 16:
        raise ValueError(f"{name} must be a [B, N, C] view with contiguous channels, strides that are multiples of 8 "
                         "elements and a 16-byte aligned base")


def spatial_attention_forward(q: Tensor, k: Tensor, v: Tensor, heads: int, scale: float, want_lse: bool = False):
    """q, k, v: [B, N, C] views (any frame / token strides, e.g. column blocks of a fused QKV projection).
    -> (o [B, N, C] contiguous, lse [B, H, N] fp32 | None). attention.py:535-542 semantics."""
    for name, t in (("q", q), ("k", k), ("v", v)):
        _check_bnc(name, t)
        if t.shape != q.shape:
            raise ValueError("q, k, v must share one shape")
    B, N, C = q.shape
    if C % heads or (C // heads) not in ATTN_HEAD_DIMS:
        raise NotImplementedError(f"spatial attention: head dim {C // heads if C % heads == 0 else '?'} not in "
                                  f"{ATTN_HEAD_DIMS}")
    o = torch.empty((B, N, C), dtype=q.dtype, device=q.device)
    lse = torch.empty((B, heads, N), dtype=torch.float32, device=q.device) if want_lse else None
    ev0 = TIMER.start() if TIMER is not None else None
    st = _lib.lib().mc_spatial_attn_fwd(_ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(lse), B, N, heads, C // heads,
                                        q.stride(0), q.stride(1), k.stride(0), k.stride(1), v.stride(0), v.stride(1),
                                        o.stride(0), o.stride(1), float(scale), _stream())
    _lib.check(st, "mc_spatial_attn_fwd")
    if ev0 is not None:  # flops: 4 B N^2 C (QK^T + PV); reported as the tensor-bound kernel of the path
        TIMER.stop("spatial_attn_fwd", 4 * B * N * N * C, ev0)
    return o, lse


def spatial_attention_backward(q: Tensor, k: Tensor, v: Tensor, o: Tensor, lse: Tensor, d_o: Tensor, heads: int,
                               scale: float) -> Tensor:
    """-> dqkv [B, N, 3C]: the gradients w.r.t. q, k, v as the column blocks of ONE buffer (the gradient of the fused
    QKV projection output, no concatenation)."""
    for name, t in (("q", q), ("k", k), ("v", v), ("o", o)):
        _check_bnc(name, t)
    _require(d_o, "d_o")
    if d_o.dim() != 3 or d_o.stride(2) != 1 or d_o.stride(0) % 8 or d_o.stride(1) % 8 or d_o.data_ptr() % 16:
        d_o = d_o.contiguous()
    _require(lse, "lse", torch.float32)
    B, N, C = q.shape
    dqkv = torch.empty((B, N, 3 * C), dtype=q.dtype, device=q.device)
    ws = torch.empty(int(_lib.lib().mc_spatial_attn_bwd_workspace_bytes(B, N, heads)), dtype=torch.uint8, device=q.device)
    ev0 = TIMER.start() if TIMER is not None else None
    st = _lib.lib().mc_spatial_attn_bwd(_ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(d_o), _ptr(lse),
                                        ctypes.c_void_p(dqkv.data_ptr()), ctypes.c_void_p(dqkv.data_ptr() + 2 * C),
                                        ctypes.c_void_p(dqkv.data_ptr() + 4 * C), _ptr(ws), B, N, heads, C // heads,
                                        q.stride(0), q.stride(1), k.stride(0), k.stride(1), v.stride(0), v.stride(1),
                                        o.stride(0), o.stride(1), d_o.stride(0), d_o.stride(1), dqkv.stride(0),
                                        dqkv.stride(1), float(scale), _stream())
    _lib.check(st, "mc_spatial_attn_bwd")
    if ev0 is not None:  # flops as launched: 7 GEMMs of 2 B N^2 C (S and dP are computed in both kernels)
        TIMER.stop("spatial_attn_bwd", 14 * B * N * N * C, ev0)
    return dqkv


class SpatialAttentionTC(torch.autograd.Function):
    """O = softmax(scale Q K^T) V per (frame, head) on the tcgen05 kernels, forward and backward.
    q, k, v: [B, N, C] views; when they are the column blocks of one fused [B, N, 3C] tensor autograd accumulates the
    three returned gradient views into that tensor's gradient."""

    @staticmethod
    def forward(ctx, q, k, v, heads, scale):
        o, lse = spatial_attention_forward(q, k, v, heads, scale, want_lse=True)
        ctx.save_for_backward(q, k, v, o, lse)
        ctx.heads, ctx.scale = heads, scale
        return o

    @staticmethod
    def backward(ctx, d_o):
        q, k, v, o, lse = ctx.saved_tensors
        C = q.shape[-1]
        dqkv = spatial_attention_backward(q, k, v, o, lse, d_o, ctx.heads, ctx.scale)
        return dqkv[..., :C], dqkv[..., C:2 * C], dqkv[..., 2 * C:], None, None


class SpatialAttentionFusedTC(torch.autograd.Function):
    """Same, on a fused projection output qkv [B, N, 3C]: one gradient tensor comes back (no view accumulation)."""

    @staticmethod
    def forward(ctx, qkv, heads, scale):
        C = qkv.shape[-1] // 3
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        o, lse = spatial_attention_forward(q, k, v, heads, scale, want_lse=True)
        ctx.save_for_backward(qkv, o, lse)
        ctx.heads, ctx.scale = heads, scale
        return o

    @staticmethod
    def backward(ctx, d_o):
        qkv, o, lse = ctx.saved_tensors
        C = qkv.shape[-1] // 3
        return spatial_attention_backward(qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:], o, lse, d_o, ctx.heads,
                                          ctx.scale), None, None
