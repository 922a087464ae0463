"""Per-frame spatial transformer (self-attention + text cross-attention + GEGLU feed-forward), token-major.

Interface and state-dict keys follow the reference's motionclone/models/attention.py: Transformer3DModel (:31),
BasicTransformerBlock (:145), CrossAttention (:302), plus diffusers-0.16's FeedForward/GEGLU that the reference
imports (:14; keys ff.net.0.proj.*, ff.net.2.*).

Design differences (B200-first):
* tokens `[(b f), h*w, C]` are a zero-copy view of the channels_last activation; proj_in/proj_out (1x1 convs in the
  checkpoint, `use_linear_projection=False`) run as GEMMs on that view;
* self-attention projects q,k,v with one GEMM; cross-attention projects the text K/V ONCE per prompt, not once per
  frame (the reference repeats the text f times, attention.py:100, and re-projects it for every frame);
* text cross-attention (`attn2`) runs on this package's tcgen05 / TMEM kernels (csrc/cross_attn_fwd_tc.cu, csrc/cross_attn_bwd_tc.cu), forward and
  the gradient w.r.t. the queries (the text K / V carry no gradient on the MotionClone path);
* spatial SELF-attention at the reference's xformers seam (`_memory_efficient_attention_xformers`, :535-542) runs on this
  package's tcgen05 + tensor-map TMA flash kernels (csrc/spatial_attn_tc.cu), forward and backward (dQ, dK, dV);
* there is no ATen / library fallback on this path: CPU tensors, fp32 activations, trainable norm weights or shapes
  outside the compiled instantiations raise (DESIGN.md §4).
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F
from torch import nn

from . import ops


def _need_kernels(x, what: str) -> None:
    if not ops.glue_kernels_ok(x):
        raise TypeError(f"{what}: expected CUDA fp16 activations, got {x.device} {x.dtype} "
                        "(motionclone_b200 has no CPU / fp32 / eager path)")


def _frozen(*params) -> bool:
    return not any(p is not None and p.requires_grad for p in params)


class LayerNorm(nn.LayerNorm):
    """nn.LayerNorm (same parameters / state-dict keys) on csrc/norm_act.cu's warp-per-row kernels (forward, and the
    input gradient when the guided pass runs under autograd with frozen weights)."""

    def forward(self, x, post_add=None, rows_per_frame: int = 0, pre_bias=None):
        """post_add [F, C]: added after the norm to the rows of frame (r // rows_per_frame) % F (temporal PE).
        pre_bias [C]: LayerNorm(x + pre_bias) - see `fold_residual_biases`."""
        c = x.shape[-1]
        _need_kernels(x, "LayerNorm")
        if not (self.elementwise_affine and c % 8 == 0 and c <= 1280 and _frozen(self.weight, self.bias)):
            raise NotImplementedError("LayerNorm kernel: affine, frozen weights, C % 8 == 0, C <= 1280")
        if torch.is_grad_enabled() and x.requires_grad:
            return ops.LayerNormFn.apply(x, self.weight, self.bias, self.eps, post_add, rows_per_frame, pre_bias)
        return ops.layernorm(x, self.weight, self.bias, self.eps, post_add, rows_per_frame, pre_bias)


def linear_into_residual(x, linear: nn.Linear, residual):
    """residual + x @ W^T as ONE GEMM (beta = 1 epilogue) - the projection's bias is NOT added here: the caller carries it
    inside the residual stream (fold_residual_biases)."""
    c_out = linear.out_features
    r2, x2 = residual.reshape(-1, c_out), x.reshape(-1, x.shape[-1])
    if not torch.is_grad_enabled() or not (residual.requires_grad or x.requires_grad):
        # no-grad forwards (plain steps, the unconditional half of guided steps): accumulate INTO the residual stream.
        # Out of place, ATen first copies `residual` into the result (a memcpy of the whole activation per projection:
        # 108 per UNet forward, 3 % of a plain step in the round-2 profile) and then runs the same beta = 1 GEMM on it, so
        # the values are identical. The stream tensor is owned by the transformer (the output of its proj_in GEMM) and
        # its previous value is dead after this add.
        return r2.addmm_(x2, linear.weight.t()).view(residual.shape)
    return torch.addmm(r2, x2, linear.weight.t()).view(residual.shape)


def fold_residual_biases(biases):
    """A transformer block computes  t1 = t + f1(t) + b1,  t2 = t1 + f2(t1) + b2,  t3 = t2 + f3(t2) + b3  (b_i: the output
    biases of its projections; attention.py:271-300, motion_module.py:213-225). With the stream shifted by the constant
    B = b1 + b2 + b3 up front (folded into the bias of the proj_in GEMM that produces t) every residual add becomes the
    beta = 1 epilogue of its GEMM:  t' = t + B;  t1' = t' + f1(LN(t' - B));  t2' = t1' + f2(LN(t1' - b2 - b3));
    t3 = t2' + f3(LN(t2' - b3))  - identical algebra, three elementwise passes fewer. Returns (B, [-B, -(b2+b3), -b3])
    as fp16 tensors: the shift and the `pre_bias` of the three LayerNorms."""
    zero = torch.zeros_like(biases[0])
    bs = [b if b is not None else zero for b in biases]
    suffix = [None] * len(bs)
    acc = zero
    for i in range(len(bs) - 1, -1, -1):
        acc = acc + bs[i]
        suffix[i] = acc
    return suffix[0].contiguous(), [(-sfx).contiguous() for sfx in suffix]


class GroupNormNHWC(nn.GroupNorm):
    """nn.GroupNorm (same parameters / state-dict keys) that reads channels_last activations directly, optionally
    fusing the time-embedding add before it and the SiLU after it (resnet blocks). ATen's CUDA GroupNorm converts a
    channels_last input to NCHW first (a copy) and hands NCHW to the next cuDNN conv (another copy)."""

    def forward(self, x, silu: bool = False, chan_bias=None):
        """chan_bias [NB, C]: per-(batch row, channel) bias added to x first (the resnet's `+ temb`)."""
        _need_kernels(x, "GroupNorm")
        if not (x.dim() == 4 and x.shape[1] % 8 == 0 and x.shape[1] <= 4096
                and x.is_contiguous(memory_format=torch.channels_last) and _frozen(self.weight, self.bias, chan_bias)):
            raise NotImplementedError("GroupNorm kernel: 4-D channels_last input, C % 8 == 0, C <= 4096, frozen weights")
        if torch.is_grad_enabled() and x.requires_grad:
            return ops.GroupNormNHWCFn.apply(x, self.weight, self.bias, chan_bias, self.num_groups, self.eps, silu)
        return ops.groupnorm_nhwc(x, self.weight, self.bias, self.num_groups, self.eps, silu, chan_bias)


class GEGLU(nn.Module):
    """diffusers 0.16 GEGLU: Linear(d, 2*inner) -> h * gelu_erf(gate)."""

    def __init__(self, dim_in: int, dim_out: int):
        super().__init__()
        self.proj = nn.Linear(dim_in, dim_out * 2)

    def forward(self, x):
        y = self.proj(x)
        _need_kernels(y, "GEGLU")
        if y.shape[-1] % 16:
            raise NotImplementedError("GEGLU kernel: inner dim must be a multiple of 8")
        if torch.is_grad_enabled() and y.requires_grad:
            return ops.GEGLUFn.apply(y)
        return ops.geglu(y)  # one pass instead of chunk -> gelu -> mul (csrc/norm_act.cu)


class FeedForward(nn.Module):
    """diffusers 0.16 FeedForward(activation_fn='geglu'): net = [GEGLU, Dropout, Linear]."""

    def __init__(self, dim: int, dim_out: Optional[int] = None, mult: int = 4, dropout: float = 0.0,
                 activation_fn: str = "geglu"):
        super().__init__()
        if activation_fn != "geglu":
            raise NotImplementedError("the reference only instantiates geglu (attention.py:211, motion_module.py:209)")
        inner = int(dim * mult)
        self.net = nn.ModuleList([GEGLU(dim, inner), nn.Dropout(dropout), nn.Linear(inner, dim_out or dim)])

    def forward(self, x, residual=None):
        """residual given: returns residual + net(x) WITHOUT net[2]'s bias (carried by the caller, fold_residual_biases)."""
        if residual is None:
            for m in self.net:
                x = m(x)
            return x
        return linear_into_residual(self.net[0](x), self.net[2], residual)


class CrossAttention(nn.Module):
    """attention.py:302-611. Same parameters / attributes; `forward` keeps the reference signature."""

    def __init__(self, query_dim: int, cross_attention_dim: Optional[int] = None, heads: int = 8, dim_head: int = 64,
                 dropout: float = 0.0, bias=False, upcast_attention: bool = False, upcast_softmax: bool = False,
                 added_kv_proj_dim: Optional[int] = None, norm_num_groups: Optional[int] = None):
        super().__init__()
        inner_dim = dim_head * heads
        self.is_self = cross_attention_dim is None
        cross_attention_dim = cross_attention_dim if cross_attention_dim is not None else query_dim
        if upcast_attention or upcast_softmax or added_kv_proj_dim is not None or norm_num_groups is not None:
            raise NotImplementedError("upcast / added_kv / group_norm variants are dead in every shipped config")
        self.upcast_attention, self.upcast_softmax = upcast_attention, upcast_softmax
        self.scale = dim_head ** -0.5
        self.heads = heads
        self.sliceable_head_dim = heads
        self._slice_size = None
        self._use_memory_efficient_attention_xformers = True  # the fused core is always on; flag kept for API parity
        self.added_kv_proj_dim = added_kv_proj_dim
        self.processor = None
        self.group_norm = None
        self.to_q = nn.Linear(query_dim, inner_dim, bias=bias)
        self.to_k = nn.Linear(cross_attention_dim, inner_dim, bias=bias)
        self.to_v = nn.Linear(cross_attention_dim, inner_dim, bias=bias)
        self.to_out = nn.ModuleList([nn.Linear(inner_dim, query_dim), nn.Dropout(dropout)])
        self._fused = None
        self._fused_kv = None

    # ---- reference helpers kept for drop-in use (attention.py:367-385, :544-562) ----
    def reshape_heads_to_batch_dim(self, tensor):
        b, s, d = tensor.shape
        h = self.heads
        return tensor.reshape(b, s, h, d // h).permute(0, 2, 1, 3).reshape(b * h, s, d // h)

    def reshape_batch_dim_to_heads(self, tensor):
        b, s, d = tensor.shape
        h = self.heads
        return tensor.reshape(b // h, h, s, d).permute(0, 2, 1, 3).reshape(b // h, s, d * h)

    def set_attention_slice(self, slice_size):
        if slice_size is not None and slice_size > self.sliceable_head_dim:
            raise ValueError(f"slice_size {slice_size} has to be smaller or equal to {self.sliceable_head_dim}.")
        self._slice_size = slice_size  # accepted, unused: the fused cores never materialise the score matrix

    def set_processor(self, processor) -> None:
        self.processor = processor

    def invalidate_fused_weights(self) -> None:
        """Drop the cached [3C, C] / [2C, c] concatenations. Called automatically by load_state_dict and by
        .to() / .half() / .cuda(); call it by hand after editing to_q / to_k / to_v through `.data` (a LoRA merge as in
        the reference's convert_lora_safetensor_to_diffusers.py does not bump the tensors' version counters)."""
        self._fused = None
        self._fused_kv = None

    def _load_from_state_dict(self, *args, **kwargs):
        super()._load_from_state_dict(*args, **kwargs)
        self.invalidate_fused_weights()

    def _apply(self, fn, *args, **kwargs):
        self.invalidate_fused_weights()
        return super()._apply(fn, *args, **kwargs)

    def fused_qkv_weight(self) -> torch.Tensor:
        """[3C, C] concatenation of to_q/to_k/to_v, rebuilt if any of them was replaced or moved (weights are frozen
        on this path: t2v_video_sample.py:67-68)."""
        ws = (self.to_q.weight, self.to_k.weight, self.to_v.weight)
        key = tuple((w.data_ptr(), w._version, w.dtype, w.device) for w in ws)
        if self._fused is None or self._fused[0] != key:
            self._fused = (key, torch.cat([w.detach() for w in ws], dim=0).contiguous())
        return self._fused[1]

    def fused_kv_weight(self) -> torch.Tensor:
        """[2C, c_text] concatenation of to_k/to_v (cross-attention: one GEMM projects the text K | V)."""
        ws = (self.to_k.weight, self.to_v.weight)
        key = tuple((w.data_ptr(), w._version, w.dtype, w.device) for w in ws)
        if self._fused_kv is None or self._fused_kv[0] != key:
            self._fused_kv = (key, torch.cat([w.detach() for w in ws], dim=0).contiguous())
        return self._fused_kv[1]

    def get_attention_scores(self, query, key, attention_mask=None):
        """attention.py:564-611: query/key `[B*heads, S, dh]` -> probabilities in the input dtype. Only the temporal
        use (S = frames, motionclone_functions.py:279) exists on this path; it runs on the fused kernel."""
        if attention_mask is not None:
            raise NotImplementedError
        bh, s, dh = query.shape
        if s not in (8, 16, 32) or key.shape[1] != s:
            raise NotImplementedError("get_attention_scores: temporal shapes only (S = key length in {8, 16, 32}); "
                                      "spatial probabilities are never materialised on this path")
        h = self.heads
        to_bfpc = lambda t: t.reshape(bh // h, h, s, dh).permute(0, 2, 1, 3).reshape(1, bh // h, s, h * dh) \
            .permute(0, 2, 1, 3)  # noqa: E731  [(B h), S, dh] -> [1, S(frames), B(positions), C]
        probs = ops.TemporalProbs.apply(to_bfpc(query).contiguous(), to_bfpc(key).contiguous(), h, self.scale)
        return probs.reshape(bh, s, s)

    def _memory_efficient_attention_xformers(self, query, key, value, attention_mask=None):
        """attention.py:535-542 seam with the reference's calling convention: `[B*heads, S, dh]` in,
        `[B, S, heads*dh]` out (the head split is undone into the kernels' `[B, S, C]` views first)."""
        if attention_mask is not None:
            raise NotImplementedError
        h = self.heads
        bh, s, dh = query.shape
        merge = lambda t: t.reshape(bh // h, h, t.shape[1], dh).permute(0, 2, 1, 3).reshape(bh // h, t.shape[1], h * dh)  # noqa: E731
        q, k, v = merge(query), merge(key), merge(value)
        if key.shape[1] == s:
            if torch.is_grad_enabled() and (q.requires_grad or k.requires_grad or v.requires_grad):
                return ops.SpatialAttentionTC.apply(q, k, v, h, self.scale)
            return ops.spatial_attention_forward(q, k, v, h, self.scale)[0]
        if torch.is_grad_enabled() and (k.requires_grad or v.requires_grad):
            raise NotImplementedError("cross-attention with trainable K / V is not on the MotionClone path")
        if torch.is_grad_enabled() and q.requires_grad:
            return ops.CrossAttentionTC.apply(q, k, v, h, self.scale)
        return ops.cross_attention_forward(q, k, v, h, self.scale)

    def forward(self, hidden_states, encoder_hidden_states=None, attention_mask=None, text_batch: Optional[int] = None,
                residual=None):
        """hidden_states `[(b f), N, C]`. encoder_hidden_states: `[(b f), n, c]` as in the reference, or `[b, n, c]`
        with `text_batch=b` so the text K/V are projected once per prompt. `residual` given: returns
        residual + to_out(attention) WITHOUT to_out's bias, as one GEMM (fold_residual_biases)."""
        if attention_mask is not None:
            raise NotImplementedError("no mask reaches attention on the live path (SURVEY appendix)")
        _need_kernels(hidden_states, "CrossAttention")
        bf, n, c = hidden_states.shape
        h = self.heads
        inner = self.to_q.out_features
        dh = inner // h
        if encoder_hidden_states is None:
            # spatial self-attention: one fused QKV GEMM, then the tcgen05 + TMA flash kernels on its column blocks
            qkv = F.linear(hidden_states, self.fused_qkv_weight())  # [(b f), N, 3C]
            if self.processor is not None:
                self.processor.record_qkv(self, hidden_states, qkv[..., :inner], qkv[..., inner:2 * inner],
                                          qkv[..., 2 * inner:], None)
            if torch.is_grad_enabled() and qkv.requires_grad:
                o = ops.SpatialAttentionFusedTC.apply(qkv, h, self.scale)
            else:
                o, _ = ops.spatial_attention_forward(qkv[..., :inner], qkv[..., inner:2 * inner], qkv[..., 2 * inner:],
                                                     h, self.scale)
        else:
            ctx = encoder_hidden_states
            b = ctx.shape[0]
            if bf % b:
                raise ValueError("encoder_hidden_states batch must divide the frame batch")
            f = bf // b
            q = self.to_q(hidden_states).view(b, f * n, inner)                        # frames of one prompt share K/V
            kv = F.linear(ctx, self.fused_kv_weight())                                # [b, 77, 2C]: K | V column blocks
            k, v = kv[..., :inner], kv[..., inner:]
            if ctx.shape[1] > 80 or dh not in ops.ATTN_HEAD_DIMS or (torch.is_grad_enabled() and kv.requires_grad):
                raise NotImplementedError("text cross-attention kernel: <= 80 context tokens, head dim in "
                                          f"{ops.ATTN_HEAD_DIMS}, frozen K / V projections of a constant prompt")
            # tcgen05 / TMEM kernels (csrc/cross_attn_{fwd,bwd}_tc.cu); dQ only: the text K / V carry no gradient here
            if torch.is_grad_enabled() and q.requires_grad:
                o = ops.CrossAttentionTC.apply(q, k, v, h, self.scale)
            else:
                o = ops.cross_attention_forward(q, k, v, h, self.scale)
            o = o.view(bf, n, inner)
        if residual is not None:
            return linear_into_residual(o, self.to_out[0], residual)
        return self.to_out[1](self.to_out[0](o))


class BasicTransformerBlock(nn.Module):
    """attention.py:145-300 with unet_use_cross_frame_attention = unet_use_temporal_attention = False (live config)."""

    def __init__(self, dim: int, num_attention_heads: int, attention_head_dim: int, dropout=0.0,
                 cross_attention_dim: Optional[int] = None, activation_fn: str = "geglu",
                 num_embeds_ada_norm: Optional[int] = None, attention_bias: bool = False,
                 only_cross_attention: bool = False, upcast_attention: bool = False,
                 unet_use_cross_frame_attention=None, unet_use_temporal_attention=None):
        super().__init__()
        if num_embeds_ada_norm is not None or unet_use_cross_frame_attention or unet_use_temporal_attention \
                or only_cross_attention:
            raise NotImplementedError("AdaLayerNorm / SC-attention / attn_temp are never configured by the reference")
        self.only_cross_attention = only_cross_attention
        self.use_ada_layer_norm = False
        self.unet_use_cross_frame_attention = unet_use_cross_frame_attention
        self.unet_use_temporal_attention = unet_use_temporal_attention
        self.attn1 = CrossAttention(query_dim=dim, heads=num_attention_heads, dim_head=attention_head_dim,
                                    dropout=dropout, bias=attention_bias, upcast_attention=upcast_attention)
        self.norm1 = LayerNorm(dim)
        if cross_attention_dim is not None:
            self.attn2 = CrossAttention(query_dim=dim, cross_attention_dim=cross_attention_dim,
                                        heads=num_attention_heads, dim_head=attention_head_dim, dropout=dropout,
                                        bias=attention_bias, upcast_attention=upcast_attention)
            self.norm2 = LayerNorm(dim)
        else:
            self.attn2 = self.norm2 = None
        self.ff = FeedForward(dim, dropout=dropout, activation_fn=activation_fn)
        self.norm3 = LayerNorm(dim)

    def set_use_memory_efficient_attention_xformers(self, use: bool, op=None):
        self.attn1._use_memory_efficient_attention_xformers = use
        if self.attn2 is not None:
            self.attn2._use_memory_efficient_attention_xformers = use

    def residual_biases(self):
        """Output biases of the three residual branches, in order (attention.py:271-300)."""
        return [self.attn1.to_out[0].bias, self.attn2.to_out[0].bias if self.attn2 is not None else None,
                self.ff.net[2].bias]

    def forward(self, hidden_states, encoder_hidden_states=None, timestep=None, attention_mask=None, video_length=None,
                folded=None):
        """`folded` = the pre-bias list of fold_residual_biases: `hidden_states` then is the stream shifted by the sum of
        this block's output biases and the result is the TRUE block output (see fold_residual_biases)."""
        if folded is not None:
            h = self.attn1(self.norm1(hidden_states, pre_bias=folded[0]), attention_mask=attention_mask,
                           residual=hidden_states)
            if self.attn2 is not None:
                h = self.attn2(self.norm2(h, pre_bias=folded[1]), encoder_hidden_states=encoder_hidden_states,
                               attention_mask=attention_mask, residual=h)
            return self.ff(self.norm3(h, pre_bias=folded[2]), residual=h)
        hidden_states = self.attn1(self.norm1(hidden_states), attention_mask=attention_mask) + hidden_states
        if self.attn2 is not None:
            hidden_states = self.attn2(self.norm2(hidden_states), encoder_hidden_states=encoder_hidden_states,
                                       attention_mask=attention_mask) + hidden_states
        return self.ff(self.norm3(hidden_states)) + hidden_states


class Transformer3DModelOutput:
    def __init__(self, sample):
        self.sample = sample


class Transformer3DModel(nn.Module):
    """attention.py:31-142. 5-D `[b, c, f, h, w]` (reference convention) or internal 4-D NHWC `[(b f), c, h, w]`."""

    def __init__(self, num_attention_heads: int = 16, attention_head_dim: int = 88, in_channels: Optional[int] = None,
                 num_layers: int = 1, dropout: float = 0.0, norm_num_groups: int = 32,
                 cross_attention_dim: Optional[int] = None, attention_bias: bool = False, activation_fn: str = "geglu",
                 num_embeds_ada_norm: Optional[int] = None, use_linear_projection: bool = False,
                 only_cross_attention: bool = False, upcast_attention: bool = False,
                 unet_use_cross_frame_attention=None, unet_use_temporal_attention=None):
        super().__init__()
        self.use_linear_projection = use_linear_projection
        self.num_attention_heads = num_attention_heads
        self.attention_head_dim = attention_head_dim
        inner_dim = num_attention_heads * attention_head_dim
        self.in_channels = in_channels
        self.norm = GroupNormNHWC(num_groups=norm_num_groups, num_channels=in_channels, eps=1e-6, affine=True)
        if use_linear_projection:
            self.proj_in = nn.Linear(in_channels, inner_dim)
            self.proj_out = nn.Linear(in_channels, inner_dim)
        else:
            self.proj_in = nn.Conv2d(in_channels, inner_dim, kernel_size=1, stride=1, padding=0)
            self.proj_out = nn.Conv2d(inner_dim, in_channels, kernel_size=1, stride=1, padding=0)
        self.transformer_blocks = nn.ModuleList([
            BasicTransformerBlock(inner_dim, num_attention_heads, attention_head_dim, dropout=dropout,
                                  cross_attention_dim=cross_attention_dim, activation_fn=activation_fn,
                                  num_embeds_ada_norm=num_embeds_ada_norm, attention_bias=attention_bias,
                                  only_cross_attention=only_cross_attention, upcast_attention=upcast_attention,
                                  unet_use_cross_frame_attention=unet_use_cross_frame_attention,
                                  unet_use_temporal_attention=unet_use_temporal_attention)
            for _ in range(num_layers)])

    def _folded(self):
        """(proj_in bias + sum of the block's output biases, pre-biases of its three LayerNorms); rebuilt when a bias
        tensor was replaced, moved or cast (weights are frozen on this path)."""
        bs = [self.proj_in.bias] + [b for b in self.transformer_blocks[0].residual_biases() if b is not None]
        key = tuple((b.data_ptr(), b._version, b.dtype, b.device) for b in bs)
        if getattr(self, "_fold_cache", None) is None or self._fold_cache[0] != key:
            with torch.no_grad():
                shift, pre = fold_residual_biases([b.detach() for b in self.transformer_blocks[0].residual_biases()])
                self._fold_cache = (key, ((self.proj_in.bias.detach() + shift).contiguous(), pre))
        return self._fold_cache[1]

    @staticmethod
    def _as_linear(conv_or_linear, t):
        w = conv_or_linear.weight
        return F.linear(t, w.reshape(w.shape[0], w.shape[1]), conv_or_linear.bias)

    def forward(self, hidden_states, encoder_hidden_states=None, timestep=None, return_dict: bool = True,
                video_length: Optional[int] = None):
        five_d = hidden_states.dim() == 5
        if five_d:
            b, c, f, h, w = hidden_states.shape
            video_length = f
            hidden_states = hidden_states.permute(0, 2, 1, 3, 4).reshape(b * f, c, h, w)
        n, c, h, w = hidden_states.shape
        residual = hidden_states.permute(0, 2, 3, 1).reshape(n, h * w, c)  # token view (zero-copy when channels_last)
        t = self.norm(hidden_states).permute(0, 2, 3, 1).reshape(n, h * w, c)
        if len(self.transformer_blocks) == 1 and self.proj_in.bias is not None:
            # the block's three residual adds ride in their GEMMs' epilogues: its output biases are pre-added to the stream
            # through proj_in's bias and taken back out inside the LayerNorms (fold_residual_biases)
            shift, pre = self._folded()
            w_in = self.proj_in.weight
            t = F.linear(t, w_in.reshape(w_in.shape[0], w_in.shape[1]), shift)
            t = self.transformer_blocks[0](t, encoder_hidden_states=encoder_hidden_states, timestep=timestep,
                                           video_length=video_length, folded=pre)
        else:
            t = self._as_linear(self.proj_in, t)
            for block in self.transformer_blocks:
                # encoder_hidden_states stays [b, 77, c]: K/V are projected once per prompt, not per frame
                t = block(t, encoder_hidden_states=encoder_hidden_states, timestep=timestep, video_length=video_length)
        t = self._as_linear(self.proj_out, t) + residual  # contiguous + contiguous: vectorised add
        out = t.reshape(n, h, w, -1).permute(0, 3, 1, 2)
        if five_d:
            out = out.reshape(b, f, c, h, w).permute(0, 2, 1, 3, 4)
        return Transformer3DModelOutput(out) if return_dict else (out,)
