"""PyTorch-facing operators over the C ABI (`include/guided_attn.h`): `torch.autograd.Function` wrappers whose forward and
backward are single launches of the hand-written sm_100a kernels.  PyTorch is plumbing here (device memory, streams,
autograd graph); no op in this file has a PyTorch or CPU implementation -- a missing library or a CPU tensor is an
error.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _cabi as abi

# Every launch made through this module is counted (bench.py reports it as `gpu_launches`).
launch_counts = {}


def _count(name, n=1):
    launch_counts[name] = launch_counts.get(name, 0) + n


def total_launches() -> int:
    return sum(launch_counts.values())


def reset_launch_counts():
    launch_counts.clear()


class LaunchProfiler:
    """Optional per-launch CUDA-event timing on the launching stream (bench.py's roofline leg).  Off by default."""

    def __init__(self):
        self.records = []   # (kernel, shape key, algorithmic bytes, start event, end event)

    class _Span:
        def __init__(self, prof, name, key, nbytes, device):
            self.prof, self.name, self.key, self.nbytes, self.device = prof, name, key, nbytes, device

        def __enter__(self):
            self.start = torch.cuda.Event(enable_timing=True)
            self.end = torch.cuda.Event(enable_timing=True)
            self.start.record(torch.cuda.current_stream(self.device))
            return self

        def __exit__(self, *exc):
            self.end.record(torch.cuda.current_stream(self.device))
            self.prof.records.append((self.name, self.key, self.nbytes, self.start, self.end))
            return False

    def span(self, name, key, nbytes, device):
        return LaunchProfiler._Span(self, name, key, nbytes, device)

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, key, nbytes, s, e in self.records:
            d = out.setdefault((name, key), {"launches": 0, "ms": 0.0, "bytes_per_launch": nbytes})
            d["launches"] += 1
            d["ms"] += s.elapsed_time(e)
        return out


class _NoSpan:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


profiler: Optional[LaunchProfiler] = None
_NOSPAN = _NoSpan()

# NVTX ranges (SURVEY section 5, tracing): with GA_NVTX=1 every launch made through this module sits in a range named
# "ga::<kernel> <shape key>", and the pipeline adds "ga::denoise_step i" / "ga::image" ranges around them, so
# `ncu --nvtx --nvtx-include "ga::cross_attn_fwd*/"` (or any NVTX-aware tool) can select one kernel or one denoising step
# of a whole image.  Off by default: a range push/pop per launch is host time the eager path would pay for nothing.
nvtx_enabled = os.environ.get("GA_NVTX", "0") == "1"


class _NvtxSpan:
    def __init__(self, label, inner):
        self.label, self.inner = label, inner

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.label)
        self.inner.__enter__()
        return self

    def __exit__(self, *exc):
        self.inner.__exit__(*exc)
        torch.cuda.nvtx.range_pop()
        return False


def nvtx_range(label):
    """Context manager: an NVTX range when GA_NVTX=1, nothing otherwise (used by the pipeline around steps / images)."""
    return _NvtxSpan("ga::" + label, _NOSPAN) if nvtx_enabled else _NOSPAN


def nvtx_push(label):
    if nvtx_enabled:
        torch.cuda.nvtx.range_push("ga::" + label)


def nvtx_pop():
    if nvtx_enabled:
        torch.cuda.nvtx.range_pop()


def _span(name, key, nbytes, device):
    inner = profiler.span(name, key, nbytes, device) if profiler is not None else _NOSPAN
    if nvtx_enabled:
        return _NvtxSpan("ga::%s %s" % (name, "x".join(str(k) for k in key) if isinstance(key, (tuple, list)) else key),
                         inner)
    return inner


def attn_fwd_bytes(B, H, N, T, d, esize, with_acc):
    """Algorithmic HBM bytes of one K1 launch (DESIGN.md): read Q, K, V, write O, row LSE, optional accumulator."""
    D = H * d
    return 2 * B * N * D * esize + 2 * B * T * D * esize + B * H * N * 4 + (B * N * T * 4 if with_acc else 0)


def attn_bwd_bytes(B, H, N, T, d, esize, with_dacc):
    """One K2 launch: read Q, dO, K, V, LSE (+ the (N, T) map gradient), write dQ."""
    D = H * d
    return 3 * B * N * D * esize + 2 * B * T * D * esize + B * H * N * 4 + (N * T * 4 if with_dacc else 0)


_DTYPES = {torch.float32: abi.GA_F32, torch.float16: abi.GA_F16, torch.bfloat16: abi.GA_BF16}
default_impl = abi.GA_IMPL_AUTO       # forward kernel variant (tests force SIMT / TCGEN05 through `impl=`)
default_bwd_impl = abi.GA_IMPL_AUTO   # backward kernel variant


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise abi.GuidedAttnLibraryError(
                "guided_attention_b200 ops run on CUDA tensors only (no CPU fallback); got a tensor on " + str(t.device))


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


# ======================================================================================== K1 / K2 cross-attention
class ScoreBias:
    """Optional additive score bias of the cross-attention kernels (`ga_score_bias_t`).

    mask      attention_mask of the processor call (reference utils/ptp_utils.py:135-136): fp32, broadcastable to
              (B*H, N, T); kept as a stride-0 expanded view, never materialised.
    pww_*     paint-with-words (reference utils/ptp_utils.py:113-138): `pww_masks` (n, N) uint8 = the BOX tokens' masks at
              this layer's resolution, `pww_columns` their token indices, `pww_coef` a 1-element fp32 DEVICE tensor
              holding w * 0.4 * ln(1 + sigma_t) (0 = off).  `smax` (1-element int64 device tensor) receives the packed
              global score max from `ga_cross_attn_smax`; the backward reads the argmax from it."""

    def __init__(self, mask=None, pww_masks=None, pww_columns=(), pww_coef=None):
        self.mask, self.pww_masks, self.pww_columns, self.pww_coef = mask, pww_masks, list(pww_columns), pww_coef
        self.smax = None

    def struct(self, B, H, N, T, device):
        sb = abi.GaScoreBias()
        if self.mask is not None:
            m = self.mask
            if m.dtype != torch.float32:
                m = m.float()
            m = torch.broadcast_to(m, (B * H, N, T))         # raises like the reference's `scores + mask` would
            if m.stride(2) != 1:
                m = m.contiguous()
            self._mask_view = m
            sb.mask, sb.mask_stride_bh, sb.mask_stride_n = m.data_ptr(), m.stride(0), m.stride(1)
        n = len(self.pww_columns)
        if n:
            if n > abi.GA_MAX_TOKENS:
                raise ValueError(f"at most {abi.GA_MAX_TOKENS} paint-with-words tokens")
            if self.pww_masks.shape != (n, N) or self.pww_masks.dtype != torch.uint8:
                raise ValueError(f"pww_masks must be ({n}, {N}) uint8, got {tuple(self.pww_masks.shape)}")
            if self.smax is None:
                self.smax = torch.zeros(1, dtype=torch.int64, device=device)
            sb.pww_masks, sb.pww_coef = self.pww_masks.data_ptr(), self.pww_coef.data_ptr()
            sb.pww_smax, sb.pww_count = self.smax.data_ptr(), n
            for i, c in enumerate(self.pww_columns):
                sb.pww_column[i] = int(c)
        return sb

    @property
    def has_pww(self):
        return len(self.pww_columns) > 0


def score_max(q, k, heads: int, scale: float, bias: "ScoreBias"):
    """Launches `ga_cross_attn_smax` into `bias.smax` (paint-with-words pre-pass: the launch-wide max of the scores,
    reference utils/ptp_utils.py:138 `attention_scores.max()`).  Returns the float value as a 0-dim tensor view."""
    lib = abi.load()
    B, N, Cdim = q.shape
    T = k.shape[1]
    sb = bias.struct(B, heads, N, T, q.device)
    with torch.cuda.device(q.device):
        abi.check(lib.ga_cross_attn_smax(_ptr(q), _ptr(k), _ptr(bias.smax), C.byref(sb), B, heads, N, T, Cdim // heads,
                                         float(scale), _DTYPES[q.dtype], _stream(q)), "ga_cross_attn_smax")
    _count("cross_attn_smax")
    return bias.smax


class _CrossAttnFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, heads: int, scale: float, want_acc: bool, impl: int, bias=None):
        _need_cuda(q, k, v)
        lib = abi.load()
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        B, N, Cdim = q.shape
        T = k.shape[1]
        d = Cdim // heads
        if k.shape[0] != B or k.shape[2] != Cdim or v.shape != k.shape:
            raise ValueError(f"shape mismatch q {tuple(q.shape)} k {tuple(k.shape)} v {tuple(v.shape)}")
        o = torch.empty_like(q)
        lse = torch.empty((B, heads, N), dtype=torch.float32, device=q.device)
        acc = torch.empty((B, N, T), dtype=torch.float32, device=q.device) if want_acc else None
        nbytes = attn_fwd_bytes(B, heads, N, T, d, q.element_size(), want_acc)
        if bias is not None:
            if bias.has_pww:
                score_max(q, k, heads, scale, bias)
            sb = bias.struct(B, heads, N, T, q.device)
            with torch.cuda.device(q.device):
                abi.check(lib.ga_cross_attn_fwd_ex(_ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(lse), _ptr(acc),
                                                   C.byref(sb), B, heads, N, T, d, float(scale), _DTYPES[q.dtype],
                                                   abi.GA_IMPL_AUTO, _stream(q)), "ga_cross_attn_fwd_ex")
        else:
            with torch.cuda.device(q.device), _span("cross_attn_fwd", (B, heads, N, T, d, str(q.dtype), want_acc),
                                                    nbytes, q.device):
                abi.check(lib.ga_cross_attn_fwd(_ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(lse), _ptr(acc), B, heads, N, T,
                                                d, float(scale), _DTYPES[q.dtype], impl, _stream(q)),
                          "ga_cross_attn_fwd")
        _count("cross_attn_fwd")
        ctx.save_for_backward(q, k, v, lse)
        ctx.meta = (heads, float(scale), impl)
        ctx.bias = bias
        # layers whose maps do not feed the loss (32^2 and 8^2 at attention_res 16) get d_acc = None, not a
        # materialised all-zero (B, N, 77) tensor that K2 would still read
        ctx.set_materialize_grads(False)
        if acc is None:
            return o, None
        return o, acc

    @staticmethod
    def backward(ctx, d_o, d_acc):
        q, k, v, lse = ctx.saved_tensors
        heads, scale, _ = ctx.meta
        impl = default_bwd_impl
        lib = abi.load()
        B, N, Cdim = q.shape
        T = k.shape[1]
        d = Cdim // heads
        d_o = torch.zeros_like(q) if d_o is None else d_o.contiguous()
        bstride, rstride = 0, T
        if d_acc is not None:
            if d_acc.dtype != torch.float32:
                d_acc = d_acc.float()
            if d_acc.dim() == 3 and d_acc.stride(0) == 0 and d_acc.stride(1) >= T and d_acc.stride(2) == 1:
                # one (N, T) slice broadcast over the batch, rows possibly padded (what the tail backward returns)
                bstride, rstride = 0, d_acc.stride(1)
            else:
                d_acc = d_acc.contiguous()
                bstride, rstride = N * T, T
        d_q = torch.empty_like(q)
        need_k, need_v = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        d_k = torch.zeros(k.shape, dtype=torch.float32, device=q.device) if need_k else None
        d_v = torch.zeros(v.shape, dtype=torch.float32, device=q.device) if need_v else None
        nbytes = attn_bwd_bytes(B, heads, N, T, d, q.element_size(), d_acc is not None)
        bias = ctx.bias
        if bias is not None:
            sb = bias.struct(B, heads, N, T, q.device)
            partials = torch.empty(B * heads * ((N + 63) // 64), dtype=torch.float32, device=q.device) \
                if bias.has_pww else None
            with torch.cuda.device(q.device):
                abi.check(lib.ga_cross_attn_bwd_ex(_ptr(q), _ptr(k), _ptr(v), _ptr(lse), _ptr(d_o), _ptr(d_acc),
                                                   bstride, rstride, _ptr(d_q), _ptr(d_k), _ptr(d_v), C.byref(sb),
                                                   _ptr(partials), B, heads, N, T, d, scale, _DTYPES[q.dtype],
                                                   abi.GA_IMPL_AUTO, _stream(q)), "ga_cross_attn_bwd_ex")
        else:
            with torch.cuda.device(q.device), _span("cross_attn_bwd",
                                                    (B, heads, N, T, d, str(q.dtype), d_acc is not None), nbytes,
                                                    q.device):
                abi.check(lib.ga_cross_attn_bwd(_ptr(q), _ptr(k), _ptr(v), _ptr(lse), _ptr(d_o), _ptr(d_acc), bstride,
                                                rstride, _ptr(d_q), _ptr(d_k), _ptr(d_v), B, heads, N, T, d, scale,
                                                _DTYPES[q.dtype], impl, _stream(q)), "ga_cross_attn_bwd")
        _count("cross_attn_bwd")
        return (d_q, d_k.to(k.dtype) if need_k else None, d_v.to(v.dtype) if need_v else None, None, None, None, None,
                None)


def cross_attention(q, k, v, heads: int, scale: float, want_acc: bool = False, impl: Optional[int] = None,
                    bias: Optional[ScoreBias] = None):
    """O = softmax(scale Q K^T [+ bias]) V per head, q (B, N, H*d), k/v (B, T, H*d).  Returns (o, acc) with
    acc (B, N, T) fp32 = sum over heads of the probabilities (None unless `want_acc`).  Differentiable in q (and k, v
    when they require grad) through BOTH outputs; with a paint-with-words bias also through the global score max."""
    return _CrossAttnFn.apply(q, k, v, heads, scale, want_acc, default_impl if impl is None else impl, bias)


def self_attn_flops(B, H, N, d, direction="fwd"):
    """Tensor-core FLOPs one launch pair issues: the forward runs the algorithm's 2 GEMMs; the backward runs 7 for the
    algorithm's 5."""
    return (2 if direction == "fwd" else 7) * 2 * B * H * N * N * d


def self_attention_forward(q, k, v, heads: int, scale: float):
    """Fused exact self-attention forward (no autograd): returns (o, lse)."""
    _need_cuda(q, k, v)
    lib = abi.load()
    q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
    B, N, Cdim = q.shape
    o = torch.empty_like(q)
    lse = torch.empty((B, heads, N), dtype=torch.float32, device=q.device)
    d = Cdim // heads
    with torch.cuda.device(q.device), _span("self_attn_fwd", (B, heads, N, d, str(q.dtype)),
                                            self_attn_flops(B, heads, N, d, "fwd"), q.device):
        abi.check(lib.ga_self_attn_fwd(_ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(lse), B, heads, N, d,
                                       float(scale), _DTYPES[q.dtype], _stream(q)), "ga_self_attn_fwd")
    _count("self_attn_fwd")
    return o, lse


class _SelfAttnFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, heads: int, scale: float):
        o, lse = self_attention_forward(q, k, v, heads, scale)
        ctx.save_for_backward(q.contiguous(), k.contiguous(), v.contiguous(), o, lse)
        ctx.meta = (heads, float(scale))
        return o

    @staticmethod
    def backward(ctx, d_o):
        q, k, v, o, lse = ctx.saved_tensors
        heads, scale = ctx.meta
        lib = abi.load()
        B, N, Cdim = q.shape
        d = Cdim // heads
        d_o = d_o.contiguous()
        d_q, d_k, d_v = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        dvec = torch.empty((B, heads, N), dtype=torch.float32, device=q.device)
        with torch.cuda.device(q.device), _span("self_attn_bwd", (B, heads, N, d, str(q.dtype)),
                                                self_attn_flops(B, heads, N, d, "bwd"), q.device):
            abi.check(lib.ga_self_attn_bwd(_ptr(q), _ptr(k), _ptr(v), _ptr(o), _ptr(lse), _ptr(d_o), _ptr(d_q),
                                           _ptr(d_k), _ptr(d_v), _ptr(dvec), B, heads, N, d, scale,
                                           _DTYPES[q.dtype], _stream(q)), "ga_self_attn_bwd")
        _count("self_attn_bwd", 2)
        return d_q, d_k, d_v, None, None


def self_attention(q, k, v, heads: int, scale: float):
    """O = softmax(scale Q K^T) V per head over the same N tokens; q, k, v (B, N, H*d) fp16/bf16.  Differentiable in
    q, k and v; the (B*H, N, N) probabilities are never materialised (forward: one launch, backward: two)."""
    return _SelfAttnFn.apply(q, k, v, heads, scale)


def self_attention_supported(dtype, head_dim: int) -> bool:
    return dtype in (torch.float16, torch.bfloat16) and head_dim % 8 == 0 and 8 <= head_dim <= 160


def attention_probs(q, k, heads: int, scale: float, bias=None):
    """Materialised P (B*H, N, T), rows ordered b*H + h like the reference's stored maps.  Not differentiable; exists for
    API compatibility (`AttentionStore.get_average_attention`) and for tests."""
    _need_cuda(q, k)
    lib = abi.load()
    q, k = q.contiguous(), k.contiguous()
    B, N, Cdim = q.shape
    T = k.shape[1]
    p = torch.empty((B * heads, N, T), dtype=q.dtype, device=q.device)
    with torch.cuda.device(q.device):
        if bias is not None:
            if bias.has_pww and bias.smax is None:
                score_max(q, k, heads, scale, bias)
            sb = bias.struct(B, heads, N, T, q.device)
            abi.check(lib.ga_attn_probs_ex(_ptr(q), _ptr(k), _ptr(p), C.byref(sb), B, heads, N, T, Cdim // heads,
                                           float(scale), _DTYPES[q.dtype], _stream(q)), "ga_attn_probs_ex")
        else:
            abi.check(lib.ga_attn_probs(_ptr(q), _ptr(k), _ptr(p), B, heads, N, T, Cdim // heads, float(scale),
                                        _DTYPES[q.dtype], _stream(q)), "ga_attn_probs")
    _count("attn_probs")
    return p


# ================================================================================= GroupNorm (+ SiLU) of the UNet
_gn_plan_cache = {}   # (n, hw, c, groups) -> workspace bytes (-1: unsupported shape)


def group_norm_ws_bytes(n: int, hw: int, c: int, groups: int) -> int:
    key = (n, hw, c, groups)
    if key not in _gn_plan_cache:
        _gn_plan_cache[key] = int(abi.load().ga_group_norm_ws_bytes(n, hw, c, groups))
    return _gn_plan_cache[key]


def group_norm_supported(x: torch.Tensor, weight, bias, groups: int) -> bool:
    """The fused kernels take channels-last-able 4-D CUDA activations in fp16 / bf16 with frozen affine parameters."""
    if not (x.is_cuda and x.dim() == 4 and x.dtype in (torch.float16, torch.bfloat16)):
        return False
    if weight is None or bias is None or weight.requires_grad or bias.requires_grad:
        return False
    n, c, h, w = x.shape
    return group_norm_ws_bytes(n, h * w, c, groups) >= 0


class _GroupNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, shift, groups: int, eps: float, silu: bool):
        _need_cuda(x, weight, bias, shift)
        lib = abi.load()
        x = x.contiguous(memory_format=torch.channels_last)
        n, c, h, w = x.shape
        if weight.dtype != x.dtype:
            weight, bias = weight.to(x.dtype), bias.to(x.dtype)
        weight, bias = weight.contiguous(), bias.contiguous()
        if shift is not None:
            # rows of c values, any row stride that keeps 16-byte alignment (a column slice of a wider matrix is fine)
            shift = shift.to(x.dtype).reshape(n, c)
            if shift.stride(1) != 1 or shift.stride(0) % 8 != 0 or shift.stride(0) < c or shift.data_ptr() % 16 != 0:
                shift = shift.contiguous()
        y = torch.empty_like(x)                       # keeps the channels-last strides
        stats = torch.empty(n, groups, 2, dtype=torch.float32, device=x.device)
        ws = torch.empty(max(group_norm_ws_bytes(n, h * w, c, groups), 8) // 4, dtype=torch.float32, device=x.device)
        nbytes = 3 * x.numel() * x.element_size()     # x read twice (the second time from L2), y written
        with torch.cuda.device(x.device), _span("group_norm_fwd", (n, h * w, c, groups, int(silu)), nbytes, x.device):
            abi.check(lib.ga_group_norm_fwd(_ptr(x), _ptr(shift), shift.stride(0) if shift is not None else 0,
                                            _ptr(weight), _ptr(bias), _ptr(y), _ptr(stats),
                                            _ptr(ws), n, h * w, c, groups, float(eps), int(silu), _DTYPES[x.dtype],
                                            _stream(x)), "ga_group_norm_fwd")
        _count("group_norm_fwd", 2)
        ctx.save_for_backward(x, weight, bias, stats, shift)
        ctx.meta = (groups, bool(silu))
        return y

    @staticmethod
    def backward(ctx, d_y):
        x, weight, bias, stats, shift = ctx.saved_tensors
        groups, silu = ctx.meta
        lib = abi.load()
        n, c, h, w = x.shape
        d_y = d_y.contiguous(memory_format=torch.channels_last)
        d_x = torch.empty_like(x)
        ws = torch.empty(max(group_norm_ws_bytes(n, h * w, c, groups), 8) // 4, dtype=torch.float32, device=x.device)
        nbytes = 5 * x.numel() * x.element_size()
        with torch.cuda.device(x.device), _span("group_norm_bwd", (n, h * w, c, groups, int(silu)), nbytes, x.device):
            abi.check(lib.ga_group_norm_bwd(_ptr(x), _ptr(shift), shift.stride(0) if shift is not None else 0,
                                            _ptr(d_y), _ptr(weight), _ptr(bias), _ptr(stats),
                                            _ptr(d_x), _ptr(ws), n, h * w, c, groups, int(silu), _DTYPES[x.dtype],
                                            _stream(x)), "ga_group_norm_bwd")
        _count("group_norm_bwd", 2)
        return d_x, None, None, None, None, None, None


def group_norm(x, weight, bias, groups: int, eps: float = 1e-5, silu: bool = False, shift=None):
    """`silu(GroupNorm(x + shift))` (SiLU and the per-(sample, channel) `shift` optional) on a (n, C, h, w) fp16 / bf16
    CUDA tensor, computed on its channels-last layout (a channels-first input is converted once): two launches forward,
    two backward, differentiable in x only (`shift` -- a conv bias plus the time-embedding projection -- does not depend
    on the latents).  Replaces `torch.nn.GroupNorm` (+ `F.silu`, + the broadcast adds in front of it) inside the UNet
    the guidance path runs forward and backward."""
    if shift is not None and shift.requires_grad:
        raise ValueError("group_norm: `shift` must not require a gradient (only x is differentiated)")
    return _GroupNormFn.apply(x, weight, bias, shift, int(groups), float(eps), bool(silu))


class _AddBiasResidualFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, bias, b):
        _need_cuda(a, bias, b)
        lib = abi.load()
        a = a.contiguous(memory_format=torch.channels_last)
        n, c, h, w = a.shape
        if b is not None:
            b = b.contiguous(memory_format=torch.channels_last)
        bias = bias.to(a.dtype).contiguous()
        out = torch.empty_like(a)
        nbytes = (3 if b is not None else 2) * a.numel() * a.element_size()
        with torch.cuda.device(a.device), _span("add_bias_residual", (n, h * w, c, int(b is not None)), nbytes, a.device):
            abi.check(lib.ga_add_bias_residual(_ptr(a), _ptr(b), _ptr(bias), _ptr(out), n * h * w, c, _DTYPES[a.dtype],
                                               _stream(a)), "ga_add_bias_residual")
        _count("add_bias_residual")
        ctx.has_b = b is not None
        return out

    @staticmethod
    def backward(ctx, g):
        return g, None, (g if ctx.has_b else None)


def add_bias_residual(a, bias, b=None):
    """`a + bias[None, :, None, None] (+ b)` on (n, C, h, w) fp16 / bf16 CUDA tensors in one vectorised channels-last
    pass: a convolution's bias and, with `b`, the block's residual connection.  Differentiable in a and b."""
    if bias.requires_grad:
        raise ValueError("add_bias_residual: `bias` must not require a gradient")
    return _AddBiasResidualFn.apply(a, bias, b)


class _GegluFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, proj):
        _need_cuda(proj)
        lib = abi.load()
        proj = proj.contiguous()
        inner = proj.shape[-1] // 2
        rows = proj.numel() // (2 * inner)
        out = torch.empty(proj.shape[:-1] + (inner,), dtype=proj.dtype, device=proj.device)
        with torch.cuda.device(proj.device), _span("geglu_fwd", (rows, inner), 3 * rows * inner * proj.element_size(),
                                                   proj.device):
            abi.check(lib.ga_geglu_fwd(_ptr(proj), _ptr(out), rows, inner, _DTYPES[proj.dtype], _stream(proj)),
                      "ga_geglu_fwd")
        _count("geglu_fwd")
        ctx.save_for_backward(proj)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (proj,) = ctx.saved_tensors
        lib = abi.load()
        inner = proj.shape[-1] // 2
        rows = proj.numel() // (2 * inner)
        d_out = d_out.contiguous()
        d_proj = torch.empty_like(proj)
        with torch.cuda.device(proj.device), _span("geglu_bwd", (rows, inner), 5 * rows * inner * proj.element_size(),
                                                   proj.device):
            abi.check(lib.ga_geglu_bwd(_ptr(proj), _ptr(d_out), _ptr(d_proj), rows, inner, _DTYPES[proj.dtype],
                                       _stream(proj)), "ga_geglu_bwd")
        _count("geglu_bwd")
        return d_proj


def geglu(proj: torch.Tensor) -> torch.Tensor:
    """`h * gelu(gate)` with `h, gate = proj.chunk(2, dim=-1)` (exact erf GELU) on a 16-bit CUDA tensor (..., 2 * inner):
    one vectorised launch per direction.  The gate of the transformer blocks' feed-forward (diffusers `GEGLU`)."""
    return _GegluFn.apply(proj)


def geglu_supported(proj: torch.Tensor) -> bool:
    return (proj.is_cuda and proj.dtype in (torch.float16, torch.bfloat16) and proj.shape[-1] % 16 == 0
            and proj.numel() > 0)


class _LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps: float):
        _need_cuda(x, weight, bias)
        lib = abi.load()
        x = x.contiguous()
        c = x.shape[-1]
        rows = x.numel() // c
        if weight.dtype != x.dtype:
            weight, bias = weight.to(x.dtype), bias.to(x.dtype)
        weight, bias = weight.contiguous(), bias.contiguous()
        y = torch.empty_like(x)
        stat_shape = x.shape[:-1] + (1,)
        mean = torch.empty(stat_shape, dtype=torch.float32, device=x.device)
        rstd = torch.empty(stat_shape, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device), _span("layer_norm_fwd", (rows, c), 2 * x.numel() * x.element_size(), x.device):
            abi.check(lib.ga_layer_norm_fwd(_ptr(x), _ptr(weight), _ptr(bias), _ptr(y), _ptr(mean), _ptr(rstd), rows, c,
                                            float(eps), _DTYPES[x.dtype], _stream(x)), "ga_layer_norm_fwd")
        _count("layer_norm_fwd")
        ctx.save_for_backward(x, weight, bias, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, d_y):
        x, weight, bias, mean, rstd = ctx.saved_tensors
        # the input gradient stays PyTorch's kernel (one launch, already vectorised); gamma / beta are frozen
        d_x = torch.ops.aten.native_layer_norm_backward(d_y.contiguous(), x, [x.shape[-1]], mean, rstd, weight, bias,
                                                        [True, False, False])[0]
        return d_x, None, None, None


def layer_norm(x, weight, bias, eps: float = 1e-5):
    """`F.layer_norm(x, (C,), weight, bias, eps)` over the last dimension of a 16-bit CUDA tensor: one warp per row, the
    row in registers (forward).  The three norms of every transformer block."""
    return _LayerNormFn.apply(x, weight, bias, float(eps))


def layer_norm_supported(x, weight, bias) -> bool:
    return (x.is_cuda and x.dtype in (torch.float16, torch.bfloat16) and weight is not None and bias is not None
            and not weight.requires_grad and not bias.requires_grad and x.shape[-1] % 8 == 0 and 8 <= x.shape[-1] <= 2048
            and x.numel() > 0)


# ============================================================================================== K5 rasteriser
def rasterize_boxes(boxes: Sequence[Sequence[float]], res: int, shrink: float, device) -> torch.Tensor:
    """(n, res, res) uint8 masks of `helpers.inside_box` for unit-square boxes (x, y, w, h); bit-exact vs the host."""
    lib = abi.load()
    n = len(boxes)
    masks = torch.empty((n, res, res), dtype=torch.uint8, device=device)
    _need_cuda(masks)
    if n == 0:
        return masks
    arr = (C.c_double * (4 * n))(*[float(c) for b in boxes for c in b])
    with torch.cuda.device(masks.device):
        abi.check(lib.ga_rasterize_boxes(arr, n, res, float(shrink), _ptr(masks), _stream(masks)), "ga_rasterize_boxes")
    _count("rasterize_boxes", (n + abi.GA_MAX_BOXES - 1) // abi.GA_MAX_BOXES)
    return masks


# ================================================================================================ guidance tail
def gaussian_taps(kernel_size: int = 3, sigma: float = 0.5) -> List[float]:
    """Separable taps equivalent to the reference's normalised 2-D kernel (utils/gaussian_smoothing.py:37-43): the 2-D
    kernel is outer(g, g) / sum, i.e. outer(w, w) with w = g / sum(g); g uses the reference's exponent
    exp(-((k - mean) / (2 sigma))^2) evaluated in fp32 like the reference."""
    if kernel_size != 3:
        raise NotImplementedError("the reference pads by one pixel (pipeline_guided_attention.py:253): only "
                                  "kernel_size=3 keeps the map size")
    ax = torch.arange(kernel_size, dtype=torch.float32)
    mean = (kernel_size - 1) / 2
    g = 1 / (sigma * math.sqrt(2 * math.pi)) * torch.exp(-((ax - mean) / (2 * sigma)) ** 2)
    w = g.double() / g.double().sum()
    return [float(x) for x in w]


@dataclass
class TailSpec:
    """Everything the tail kernels need besides the accumulators: built once per (prompt, res) on the host."""
    res: int
    n_ctx: int
    first: int
    last: int
    token_indices: List[int]
    kinds: List[int]
    groups: List[object]                 # sub-prompt of each token
    tokens: object = None                # (GaToken * n)
    params: abi.GaTailParams = None
    masks: Optional[torch.Tensor] = None   # (n_boxes, res, res) uint8, device
    weights: Optional[torch.Tensor] = None  # (n_boxes, res, res) fp32, device (strict only)
    n_inside: List[int] = field(default_factory=list)


_tickets = {}


def _ticket(device, n=1) -> torch.Tensor:
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _tickets or _tickets[key].numel() < n:
        _tickets[key] = torch.zeros(max(n, 64), dtype=torch.int32, device=device)
    return _tickets[key]


class _GuidanceTailFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, spec: TailSpec, n_maps: int, n_samples: int, *accs):
        _need_cuda(*accs)
        lib = abi.load()
        n = len(accs)
        if n == 0:
            raise ValueError("no attention accumulators to aggregate")   # reference: torch.cat([]) error
        accs = [a.contiguous() for a in accs]
        dev = accs[0].device
        npix, T, S = spec.res * spec.res, spec.n_ctx, int(n_samples)
        ptrs = (C.c_void_p * n)()
        slices = (C.c_int32 * n)()
        for i, a in enumerate(accs):
            if a.dtype != torch.float32 or a.dim() != 3 or a.shape[1] != npix or a.shape[2] != T or a.shape[0] % S:
                raise ValueError(f"accumulator {i}: expected ({S}*k, {npix}, {T}) fp32, got {tuple(a.shape)} {a.dtype}")
            ptrs[i] = a.data_ptr()
            slices[i] = a.shape[0] // S
        p = abi.GaTailParams.from_buffer_copy(spec.params)
        p.inv_count = 1.0 / float(n_maps)
        p.n_samples = S
        nt, tp = p.n_tokens, spec.last - spec.first
        lead = () if S == 1 else (S,)
        attn_text = torch.empty(lead + (spec.res, spec.res, tp), dtype=torch.float32, device=dev)
        smoothed = torch.empty(lead + (nt, spec.res, spec.res), dtype=torch.float32, device=dev)
        stats = torch.empty(lead + (nt, abi.GA_STATS), dtype=torch.float32, device=dev)
        argmax = torch.empty(lead + (nt,), dtype=torch.int32, device=dev)
        total = torch.empty((S,), dtype=torch.float32, device=dev)
        nbytes = (sum(a.numel() for a in accs) + attn_text.numel() + smoothed.numel()) * 4 + S * nt * npix
        with torch.cuda.device(dev), _span("guidance_tail_fwd", (spec.res, T, n, nt, S), nbytes, dev):
            abi.check(lib.ga_guidance_tail_fwd(ptrs, slices, n, C.byref(p), spec.tokens, _ptr(spec.masks),
                                               _ptr(spec.weights), _ptr(attn_text), _ptr(smoothed), _ptr(stats),
                                               _ptr(argmax), _ptr(total), _ptr(_ticket(dev, S)), _stream(attn_text)),
                      "ga_guidance_tail_fwd")
        _count("guidance_tail_fwd")
        ctx.save_for_backward(attn_text, smoothed, stats, argmax)
        ctx.spec, ctx.params, ctx.batches = spec, p, [a.shape[0] for a in accs]
        ctx.mark_non_differentiable(smoothed, argmax)
        # outputs that do not feed the loss hand back None, not zeros: with g_attn_text = NULL the backward takes the
        # sparse fast path (the built-in losses never differentiate attn_text directly)
        ctx.set_materialize_grads(False)
        return attn_text, smoothed, stats, argmax, total

    @staticmethod
    def backward(ctx, g_attn_text, g_smoothed, g_stats, g_argmax, g_total):
        attn_text, smoothed, stats, argmax = ctx.saved_tensors
        spec, p = ctx.spec, ctx.params
        lib = abi.load()
        dev = attn_text.device
        npix, T, S = spec.res * spec.res, spec.n_ctx, p.n_samples

        def prep(g):
            return None if g is None else g.contiguous().float()
        g_attn_text, g_stats, g_total = prep(g_attn_text), prep(g_stats), prep(g_total)
        pitch = (T + 3) // 4 * 4      # rows padded to 16 bytes: K2 reads them with 128-bit loads
        d_abar = torch.empty((S, npix, pitch), dtype=torch.float32, device=dev)
        nbytes = (attn_text.numel() + d_abar.numel()) * 4
        with torch.cuda.device(dev), _span("guidance_tail_bwd", (spec.res, T, p.n_tokens, S), nbytes, dev):
            abi.check(lib.ga_guidance_tail_bwd(C.byref(p), spec.tokens, _ptr(spec.masks), _ptr(spec.weights),
                                               _ptr(attn_text), _ptr(smoothed), _ptr(stats), _ptr(argmax),
                                               _ptr(g_total), _ptr(g_stats), _ptr(g_attn_text), _ptr(d_abar), pitch,
                                               _stream(d_abar)), "ga_guidance_tail_bwd")
        _count("guidance_tail_bwd")
        # every accumulator slice of a sample receives the same gradient: hand out stride-0 views (K2 reads a broadcast)
        if S == 1:
            grads = tuple(d_abar[0, :, :T].unsqueeze(0).expand(b, npix, T) for b in ctx.batches)
        else:
            grads = tuple(d_abar[:, None, :, :T].expand(S, b // S, npix, T).reshape(b, npix, T) for b in ctx.batches)
        return (None, None, None) + grads


def guidance_tail(spec: TailSpec, accs: Sequence[torch.Tensor], n_maps: int, n_samples: int = 1):
    """(attn_text (res,res,T'), smoothed (n,res,res), stats (n, GA_STATS), argmax (n), total (1)) -- one launch.
    With `n_samples` S > 1 (extension, not in the reference: independent samples, e.g. seeds, evaluated by one launch)
    every accumulator is (S*k, res^2, T), sample-major, `n_maps` counts the maps of ONE sample and every output gains a
    leading S dimension.
    `accs`: K1 accumulators (B_l, res^2, T), each slice a sum over that layer's heads; `n_maps` = total number of
    head-maps they hold (sum over layers of B_l * heads_l), the divisor of the reference's mean
    (utils/ptp_utils.py:288)."""
    return _GuidanceTailFn.apply(spec, int(n_maps), int(n_samples), *accs)


# ===================================================================================== stand-alone stage operators
class _SmoothFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, maps, taps):
        _need_cuda(maps)
        lib = abi.load()
        x = maps.contiguous().float()
        n, res = x.shape[0], x.shape[-1]
        out = torch.empty_like(x)
        w = (C.c_float * 3)(*taps)
        with torch.cuda.device(x.device):
            abi.check(lib.ga_smooth_fwd(_ptr(x), _ptr(out), n, res, w, _stream(x)), "ga_smooth_fwd")
        _count("smooth_fwd")
        ctx.taps = taps
        return out

    @staticmethod
    def backward(ctx, g):
        lib = abi.load()
        g = g.contiguous().float()
        n, res = g.shape[0], g.shape[-1]
        out = torch.empty_like(g)
        w = (C.c_float * 3)(*ctx.taps)
        with torch.cuda.device(g.device):
            abi.check(lib.ga_smooth_bwd(_ptr(g), _ptr(out), n, res, w, _stream(g)), "ga_smooth_bwd")
        _count("smooth_bwd")
        return out, None


def smooth(maps: torch.Tensor, kernel_size: int = 3, sigma: float = 0.5) -> torch.Tensor:
    """reflect-pad + 3x3 Gaussian on (n, res, res) maps (reference pipeline :253-254 + GaussianSmoothing.forward)."""
    squeeze = maps.dim() == 2
    x = maps[None] if squeeze else maps
    out = _SmoothFn.apply(x, tuple(gaussian_taps(kernel_size, sigma)))
    out = out.to(maps.dtype)
    return out[0] if squeeze else out


class _BoxLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, mask, weights, strict):
        _need_cuda(p, mask)
        lib = abi.load()
        x = p.contiguous().float()
        res = x.shape[-1]
        out = torch.empty(2, dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            abi.check(lib.ga_box_loss_fwd(_ptr(x), _ptr(mask), _ptr(weights), res, int(strict), _ptr(out), _stream(x)),
                      "ga_box_loss_fwd")
        _count("box_loss_fwd")
        ctx.save_for_backward(x, mask, weights if weights is not None else torch.empty(0, device=x.device))
        ctx.strict, ctx.has_w = int(strict), weights is not None
        return out

    @staticmethod
    def backward(ctx, g):
        x, mask, weights = ctx.saved_tensors
        lib = abi.load()
        g = g.contiguous().float()
        gp = torch.empty_like(x)
        with torch.cuda.device(x.device):
            abi.check(lib.ga_box_loss_bwd(_ptr(x), _ptr(mask), _ptr(weights if ctx.has_w else None), x.shape[-1],
                                          ctx.strict, _ptr(g), _ptr(gp), _stream(x)), "ga_box_loss_bwd")
        _count("box_loss_bwd")
        return gp, None, None, None


def box_losses(image_softmax: torch.Tensor, rect, shrink: float, strict: bool):
    """(loss_inside, loss_outside) as 1-element tensors; `rect` is a helpers.Rect already scaled to the map size."""
    from . import helpers
    res = image_softmax.shape[-1]
    unit = (rect.x / rect.size, rect.y / rect.size, rect.width / rect.size, rect.height / rect.size)
    # the rect arrives pre-scaled (reference call site pipeline :279): rasterise it as a size-`res` box on the host
    # grid -- one multiplication by 1.0 keeps the doubles bit-identical
    mask_np = helpers.box_mask_host(rect, res)
    if int(mask_np.sum()) == 0:
        raise ZeroDivisionError("float division by zero")   # reference: at_most = 1.0 / num_inside
    dev = image_softmax.device
    mask = torch.from_numpy(mask_np).to(dev)
    weights = torch.from_numpy(helpers.strict_weights_host(rect, res)).to(dev) if strict else None
    out = _BoxLossFn.apply(image_softmax, mask, weights, strict)
    return out[0:1].to(image_softmax.dtype), out[1:2].to(image_softmax.dtype)
