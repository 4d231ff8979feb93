"""Differentiable ops of the engine.

Every op is a ``torch.autograd.Function`` with a hand-written backward that calls the *same
primitive set* on both back-ends: ``cuda_kernels`` (sm_100a, tcgen05/TMA) for CUDA tensors and
``torch_kernels`` (ATen oracle) for CPU tensors.  Weights are read through the live
``Parameter.data`` in backward (never through autograd-saved views) because the sharded runtime
re-points parameters at a freshly gathered buffer between forward and backward; weight
gradients are written straight into the runtime's flat gradient buffer when the parameter
carries ``_grad_buf`` (no autograd accumulation pass).
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from fms_fsdp_b200.ops import _ext, torch_kernels

_KERNEL_PATH = os.environ.get("FMS_B200_KERNEL_PATH", "auto")  # auto | fused | torch


def set_kernel_path(path: str):
    global _KERNEL_PATH
    if path not in ("auto", "fused", "torch"):
        raise ValueError(f"kernel_path must be auto|fused|torch, got {path}")
    _KERNEL_PATH = path


def get_kernel_path() -> str:
    return _KERNEL_PATH


def kernels_for(t: torch.Tensor):
    """Primitive namespace for tensor ``t``: CUDA tensors *require* the sm_100a extension."""
    if t.is_cuda and _KERNEL_PATH != "torch":
        if not _ext.available():
            if _ext.allow_torch_fallback():
                return torch_kernels
            _ext.require()
        from fms_fsdp_b200.ops import cuda_kernels
        return cuda_kernels
    return torch_kernels


def _wdata(w):
    return w.data if isinstance(w, torch.nn.Parameter) else w


def _deliver_wgrad(w, compute):
    """Run ``compute(out, accumulate)`` into the runtime grad buffer if present, else return a grad."""
    push = getattr(w, "_grad_push", None)
    if push is not None:   # experimental fused GEMM -> reduce-scatter: the wgrad goes straight to the owning ranks
        if getattr(w, "_grad_ready", False):
            raise RuntimeError("push reduce-scatter: a second gradient contribution to the same weight is not supported")
        compute(push, False)
        w._grad_ready = True
        return None
    buf = getattr(w, "_grad_buf", None)
    if buf is not None:
        acc = bool(getattr(w, "_grad_ready", False))
        compute(buf, acc)
        w._grad_ready = True
        return None
    out = torch.empty_like(_wdata(w))
    compute(out, False)
    return out


# ------------------------------------------------------------------------------------------ linear
class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, residual, bias=None):
        K = kernels_for(x)
        x2 = x.reshape(-1, x.shape[-1])
        r2 = None if residual is None else residual.reshape(-1, residual.shape[-1])
        wd = _wdata(w)
        # allocate in the caller's shape: returning a view from a custom Function would forbid the
        # in-place RoPE that follows the QKV projection
        y = torch.empty(*x.shape[:-1], wd.shape[0], dtype=x.dtype, device=x.device)
        K.gemm(x2, wd, "nt", out=y.view(-1, wd.shape[0]), residual=r2, bias=None if bias is None else _wdata(bias))
        ctx.K, ctx.w, ctx.b, ctx.has_res = K, w, bias, residual is not None
        ctx.save_for_backward(x)
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        K, w = ctx.K, ctx.w
        dy2 = dy.reshape(-1, dy.shape[-1])
        if not dy2.is_contiguous():
            dy2 = dy2.contiguous()
        x2 = x.reshape(-1, x.shape[-1])
        dx = None
        if ctx.needs_input_grad[0]:
            dx = K.gemm(dy2, _wdata(w), "nn").view_as(x)
        dw = None
        if ctx.needs_input_grad[1]:
            dw = _deliver_wgrad(w, lambda out, acc: K.gemm(dy2, x2, "tn", out=out, accumulate=acc))
        db = None
        if ctx.b is not None and ctx.needs_input_grad[3]:
            db = _deliver_wgrad(ctx.b, lambda out, acc: K.bias_grad(dy2, out, acc))
        return dx, dw, (dy if ctx.has_res else None), db


# ---- optional reduced-precision forward GEMMs (default "bf16"; "fp8" is opt-in and never used for the headline metric)
_GEMM_PRECISION = os.environ.get("FMS_B200_PRECISION", "bf16")


def set_gemm_precision(p: str):
    global _GEMM_PRECISION
    if p not in ("bf16", "fp8"):
        raise ValueError(f"precision must be bf16|fp8, got {p}")
    _GEMM_PRECISION = p


def get_gemm_precision() -> str:
    return _GEMM_PRECISION


class _LinearFP8(torch.autograd.Function):
    """y = x @ w^T with BOTH operands quantised row-wise to e4m3 on the fly (scale = row amax / 448) and multiplied on the
    fp8 tensor cores with fp32 accumulation; the backward is the bf16 backward of ``_Linear`` (fp8 forward / bf16
    backward recipe).  Activations and weights stay bf16 in memory."""

    @staticmethod
    def forward(ctx, x, w, residual, bias=None):
        K = kernels_for(x)
        x2 = x.reshape(-1, x.shape[-1])
        wd = _wdata(w)
        xq, sx = K.quant_rowwise_e4m3(x2 if x2.is_contiguous() else x2.contiguous())
        wq, sw = K.quant_rowwise_e4m3(wd if wd.is_contiguous() else wd.contiguous())
        y = torch.empty(*x.shape[:-1], wd.shape[0], dtype=x.dtype, device=x.device)
        K.gemm_fp8(xq, wq, sx, sw, out=y.view(-1, wd.shape[0]))
        if bias is not None:   # unfused: the fp8 path is opt-in and its epilogue carries the scales
            y += _wdata(bias)
        if residual is not None:
            y += residual
        ctx.K, ctx.w, ctx.b, ctx.has_res = K, w, bias, residual is not None
        ctx.save_for_backward(x)
        return y

    backward = _Linear.backward


def linear(x, w, residual: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None):
    """y = x @ w^T (+ bias [N]) (+ residual), bias and residual fused in the GEMM epilogue."""
    if _GEMM_PRECISION == "fp8" and x.dtype == torch.bfloat16 and x.shape[-1] % 16 == 0:
        return _LinearFP8.apply(x, w, residual, bias)
    return _Linear.apply(x, w, residual, bias)


# ----------------------------------------------------------------------------------------- rmsnorm
class _RMSNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, eps):
        K = kernels_for(x)
        x2 = x.reshape(-1, x.shape[-1])
        y, rstd = K.rmsnorm_fwd(x2, _wdata(w), eps)
        ctx.K, ctx.w = K, w
        ctx.save_for_backward(x, rstd)
        return y.view_as(x)

    @staticmethod
    def backward(ctx, dy):
        x, rstd = ctx.saved_tensors
        K, w = ctx.K, ctx.w
        D = x.shape[-1]
        dx, dw32 = K.rmsnorm_bwd(dy.reshape(-1, D).contiguous(), x.reshape(-1, D), _wdata(w), rstd)
        dw = None
        if ctx.needs_input_grad[1]:
            def put(out, acc):
                if acc:
                    out.add_(dw32.to(out.dtype))
                else:
                    out.copy_(dw32)
            dw = _deliver_wgrad(w, put)
        return dx.view_as(x), dw, None


def rmsnorm(x, w, eps=1e-5):
    return _RMSNorm.apply(x, w, eps)


class _RMSNormFork(torch.autograd.Function):
    """(rmsnorm(x), x): the pre-norm residual fork as ONE node, so the gradient of the residual branch is summed into
    the norm's dx inside the backward kernel instead of by a separate autograd accumulate."""

    @staticmethod
    def forward(ctx, x, w, eps):
        K = kernels_for(x)
        y, rstd = K.rmsnorm_fwd(x.reshape(-1, x.shape[-1]), _wdata(w), eps)
        ctx.K, ctx.w = K, w
        ctx.save_for_backward(x, rstd)
        return y.view_as(x), x.view_as(x)

    @staticmethod
    def backward(ctx, dy, dres):
        x, rstd = ctx.saved_tensors
        K, w = ctx.K, ctx.w
        D = x.shape[-1]
        if dy is None:
            return dres, None, None
        dx, dw32 = K.rmsnorm_bwd(dy.reshape(-1, D).contiguous(), x.reshape(-1, D), _wdata(w), rstd,
                                 None if dres is None else dres.reshape(-1, D))
        dw = None
        if ctx.needs_input_grad[1]:
            def put(out, acc):
                if acc:
                    out.add_(dw32.to(out.dtype))
                else:
                    out.copy_(dw32)
            dw = _deliver_wgrad(w, put)
        return dx.view_as(x), dw, None


def rmsnorm_fork(x, w, eps=1e-5):
    """Returns ``(rmsnorm(x) * w, x)``; use the second output as the residual."""
    return _RMSNormFork.apply(x, w, eps)


class _RMSNormGated(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, z, w, eps, group_size):
        K = kernels_for(x)
        y, rstd = K.rmsnorm_gated_fwd(x, z, _wdata(w), eps, group_size)
        ctx.K, ctx.w, ctx.gs = K, w, group_size
        ctx.save_for_backward(x, z, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, z, rstd = ctx.saved_tensors
        dx, dz, dw32 = ctx.K.rmsnorm_gated_bwd(dy.contiguous(), x, z, _wdata(ctx.w), rstd, ctx.gs)
        def put(out, acc):
            if acc:
                out.add_(dw32.to(out.dtype))
            else:
                out.copy_(dw32)
        dw = _deliver_wgrad(ctx.w, put) if ctx.needs_input_grad[2] else None
        return dx, dz, dw, None, None


def rmsnorm_gated(x, z, w, eps=1e-5, group_size=None):
    return _RMSNormGated.apply(x, z, w, eps, group_size or x.shape[-1])


# -------------------------------------------------------------------------------------------- rope
class _Rope(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkv, table, seq_len, nheads, kvheads, head_dim, rot_dim, interleaved):
        K = kernels_for(qkv)
        ctx.K, ctx.args = K, (seq_len, nheads, kvheads, head_dim, rot_dim, interleaved)
        ctx.save_for_backward(table)
        ctx.mark_dirty(qkv)
        K.rope_(qkv.view(-1, qkv.shape[-1]), table, seq_len, nheads, kvheads, head_dim, rot_dim, False, 0, interleaved)
        return qkv

    @staticmethod
    def backward(ctx, dqkv):
        (table,) = ctx.saved_tensors
        seq_len, nheads, kvheads, head_dim, rot_dim, interleaved = ctx.args
        # the roped projection feeds exactly one consumer (attention), so its incoming gradient is
        # exclusively ours: rotate it back in place instead of paying for a copy.
        d = dqkv.contiguous()
        ctx.K.rope_(d.view(-1, d.shape[-1]), table, seq_len, nheads, kvheads, head_dim, rot_dim, True, 0, interleaved)
        return d, None, None, None, None, None, None, None


def rope_(qkv, table, seq_len, nheads, kvheads, head_dim, rot_dim=None, interleaved=True):
    """Rotate the q,k sections of the fused projection in place.  ``interleaved=True`` is the FMS
    pair convention (2i, 2i+1); False is the half-split (i, i+rot/2) convention of mamba_ssm / HF."""
    return _Rope.apply(qkv, table, seq_len, nheads, kvheads, head_dim, rot_dim or head_dim, interleaved)


# --------------------------------------------------------------------------------------- attention
class _Attention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkv, B, S, H, KVH, hd, scale):
        K = kernels_for(qkv)
        q2 = qkv.view(B * S, -1)
        o, lse = K.attn_fwd(q2, B, S, H, KVH, hd, scale)
        ctx.K, ctx.args = K, (B, S, H, KVH, hd, scale)
        ctx.save_for_backward(qkv, o, lse)
        return o.view(B, S, H * hd)

    @staticmethod
    def backward(ctx, do):
        qkv, o, lse = ctx.saved_tensors
        B, S, H, KVH, hd, scale = ctx.args
        dqkv = ctx.K.attn_bwd(do.reshape(B * S, H * hd).contiguous(), qkv.view(B * S, -1), o, lse,
                              B, S, H, KVH, hd, scale)
        return dqkv.view_as(qkv), None, None, None, None, None, None


class _QKVAttention(torch.autograd.Function):
    """QKV projection + RoPE + causal attention as ONE autograd node: the rotary embedding is the epilogue of the
    projection GEMM in forward and of the dq / dk kernels in backward, so no standalone RoPE pass touches HBM
    (SURVEY.md K1-K3; reference path: fms MultiHeadAttention.in_proj -> RotaryEmbedding.adjusted_qk -> SDPA)."""

    @staticmethod
    def forward(ctx, h, w, table, S, H, KVH, hd, scale, bias=None):
        K = kernels_for(h)
        B = h.shape[0]
        h2 = h.reshape(-1, h.shape[-1])
        qkv = K.gemm(h2, _wdata(w), "nt", rope=(table, S, hd, H, KVH), bias=None if bias is None else _wdata(bias))
        o, lse = K.attn_fwd(qkv, B, S, H, KVH, hd, scale)
        ctx.K, ctx.w, ctx.b, ctx.args = K, w, bias, (B, S, H, KVH, hd, scale)
        ctx.save_for_backward(h, qkv, o, lse, table)
        return o.view(B, S, H * hd)

    @staticmethod
    def backward(ctx, do):
        h, qkv, o, lse, table = ctx.saved_tensors
        B, S, H, KVH, hd, scale = ctx.args
        K, w = ctx.K, ctx.w
        dqkv = K.attn_bwd(do.reshape(B * S, H * hd).contiguous(), qkv, o, lse, B, S, H, KVH, hd, scale,
                          rope_table=table)
        h2 = h.reshape(-1, h.shape[-1])
        dh = K.gemm(dqkv, _wdata(w), "nn").view_as(h) if ctx.needs_input_grad[0] else None
        dw = None
        if ctx.needs_input_grad[1]:
            dw = _deliver_wgrad(w, lambda out, acc: K.gemm(dqkv, h2, "tn", out=out, accumulate=acc))
        db = None
        if ctx.b is not None and ctx.needs_input_grad[8]:   # the bias sits before RoPE: dL/db = column sums of dqkv
            db = _deliver_wgrad(ctx.b, lambda out, acc: K.bias_grad(dqkv, out, acc))
        return dh, dw, None, None, None, None, None, None, db


def qkv_attention(h, w, table, nheads, kvheads, head_dim, scale=None, bias=None):
    """attention(rope(h @ w^T + bias)) for a fused [(H + 2 KVH) * hd, D] projection weight and optional [(H + 2 KVH) * hd]
    bias (Qwen2); h: [B, S, D]."""
    S = h.shape[1]
    scale = (head_dim ** -0.5) if scale is None else scale
    if _GEMM_PRECISION == "fp8":     # fp8 projection, then the stand-alone RoPE kernel and attention
        return attention(rope_(linear(h, w, bias=bias), table, S, nheads, kvheads, head_dim), nheads, kvheads, head_dim,
                         scale)
    return _QKVAttention.apply(h, w, table, S, nheads, kvheads, head_dim, scale, bias)


def attention(qkv, nheads, kvheads, head_dim, scale=None):
    """Causal GQA flash attention on a fused (roped) projection [B, S, (H+2KVH)*hd] -> [B, S, H*hd]."""
    B, S, _ = qkv.shape
    scale = (head_dim ** -0.5) if scale is None else scale
    return _Attention.apply(qkv, B, S, nheads, kvheads, head_dim, scale)


# ------------------------------------------------------------------------------------------ swiglu
class _SwiGLU(torch.autograd.Function):
    @staticmethod
    def forward(ctx, gu, gate_first):
        K = kernels_for(gu)
        ctx.K, ctx.gate_first = K, gate_first
        ctx.save_for_backward(gu)
        return K.swiglu_fwd(gu, gate_first)

    @staticmethod
    def backward(ctx, ds):
        (gu,) = ctx.saved_tensors
        return ctx.K.swiglu_bwd(ds.contiguous(), gu, ctx.gate_first), None


def swiglu(gu, gate_first=True):
    """silu(gate) * up on a fused projection; ``gate_first`` = FMS [gate | up], False = mamba_ssm [up | gate]."""
    return _SwiGLU.apply(gu, gate_first)


class _GatedMLP(torch.autograd.Function):
    """y = (silu(gate) * up) @ w2^T (+ residual) with [gate | up] = x @ wg1^T as ONE node, so that the activation can be
    the epilogue of the gate/up GEMM and its backward the epilogue of the down-projection dgrad GEMM (SURVEY.md K6-K8;
    reference op: fms GatedLinearUnit, weights ``ff_sub_layer.wg1_fused`` / ``w2``, ``fms_to_hf_llama.py:89-96``)."""

    @staticmethod
    def forward(ctx, x, wg1, w2, residual, gate_first):
        K = kernels_for(x)
        x2 = x.reshape(-1, x.shape[-1])
        gu, act = K.gated_up_fwd(x2, _wdata(wg1), gate_first)
        w2d = _wdata(w2)
        y = torch.empty(*x.shape[:-1], w2d.shape[0], dtype=x.dtype, device=x.device)
        r2 = None if residual is None else residual.reshape(-1, residual.shape[-1])
        K.gemm(act, w2d, "nt", out=y.view(-1, w2d.shape[0]), residual=r2)
        ctx.K, ctx.wg1, ctx.w2, ctx.gate_first, ctx.has_res = K, wg1, w2, gate_first, residual is not None
        ctx.save_for_backward(x, gu, act)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gu, act = ctx.saved_tensors
        K, wg1, w2 = ctx.K, ctx.wg1, ctx.w2
        dy2 = dy.reshape(-1, dy.shape[-1])
        if not dy2.is_contiguous():
            dy2 = dy2.contiguous()
        x2 = x.reshape(-1, x.shape[-1])
        dgu = K.gated_down_bwd(dy2, _wdata(w2), gu, ctx.gate_first)
        dw2 = _deliver_wgrad(w2, lambda out, acc: K.gemm(dy2, act, "tn", out=out, accumulate=acc)) \
            if ctx.needs_input_grad[2] else None
        dx = K.gemm(dgu, _wdata(wg1), "nn").view_as(x) if ctx.needs_input_grad[0] else None
        dwg1 = _deliver_wgrad(wg1, lambda out, acc: K.gemm(dgu, x2, "tn", out=out, accumulate=acc)) \
            if ctx.needs_input_grad[1] else None
        return dx, dwg1, dw2, (dy if ctx.has_res else None), None


def gated_mlp(x, wg1, w2, residual: Optional[torch.Tensor] = None, gate_first: bool = True):
    """SwiGLU MLP: ``(silu(g) * u) @ w2^T (+ residual)`` with ``[g | u] = x @ wg1^T`` (``gate_first=False``: ``[u | g]``,
    the mamba_ssm GatedMLP order)."""
    if _GEMM_PRECISION == "fp8":
        return linear(swiglu(linear(x, wg1), gate_first), w2, residual)
    return _GatedMLP.apply(x, wg1, w2, residual, gate_first)


class _AddRMSNorm(torch.autograd.Function):
    """residual_out = residual + x (kept in the residual stream dtype, fp32 for Mamba);
    y = rmsnorm(residual_out) in x.dtype.  (mamba_ssm fused_add_norm, SURVEY.md M6.)"""

    @staticmethod
    def forward(ctx, x, res, w, eps, res_fp32):
        K = kernels_for(x)
        D = x.shape[-1]
        y, res_out, rstd = K.add_rmsnorm_fwd(x.reshape(-1, D), res.reshape(-1, D), _wdata(w), eps)
        ctx.K, ctx.w, ctx.xdtype = K, w, x.dtype
        ctx.save_for_backward(res_out, rstd)
        return y.view(x.shape), res_out.view(res.shape)

    @staticmethod
    def backward(ctx, dy, dres_out):
        res_out, rstd = ctx.saved_tensors
        D = res_out.shape[-1]
        dn, dw32 = ctx.K.rmsnorm_bwd(dy.reshape(-1, D).contiguous(), res_out, _wdata(ctx.w), rstd)
        dres = dn.float()
        if dres_out is not None:
            dres = dres + dres_out.reshape(-1, D).float()
        def put(out, acc):
            if acc:
                out.add_(dw32.to(out.dtype))
            else:
                out.copy_(dw32)
        dw = _deliver_wgrad(ctx.w, put) if ctx.needs_input_grad[2] else None
        return dres.to(ctx.xdtype).view(dy.shape), dres.to(res_out.dtype).view(dy.shape), dw, None, None


def add_rmsnorm(x, residual, w, eps=1e-5, residual_in_fp32=True):
    return _AddRMSNorm.apply(x, residual, w, eps, residual_in_fp32)


# --------------------------------------------------------------------------------------- embedding
class _Embedding(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tokens, w):
        K = kernels_for(_wdata(w))
        ctx.K, ctx.w = K, w
        ctx.save_for_backward(tokens)
        y = K.embedding_fwd(tokens, _wdata(w))
        return y.view(*tokens.shape, y.shape[-1])

    @staticmethod
    def backward(ctx, dx):
        (tokens,) = ctx.saved_tensors
        D = dx.shape[-1]
        dw = _deliver_wgrad(ctx.w, lambda out, acc: ctx.K.embedding_bwd(
            dx.reshape(-1, D).contiguous(), tokens, out, accumulate=acc))
        return None, dw


def embedding(tokens, w):
    return _Embedding.apply(tokens, w)


# ------------------------------------------------------------------------- fused linear + CE loss
# The engine's own schedule always differentiates the loss with an upstream gradient of exactly 1 (``_backward(None)``);
# it says so here, and ``_LinearCE.backward`` then skips the multiplication.  Every other caller (``loss.backward()`` on a
# scaled loss, gradient accumulation with loss / k, ...) gets the upstream gradient applied ON DEVICE -- never a host
# read, never silently dropped.
_UNIT_UPSTREAM = False


def set_unit_upstream(flag: bool):
    global _UNIT_UPSTREAM
    _UNIT_UPSTREAM = bool(flag)


class _LinearCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, w, labels, ignore_index):
        K = kernels_for(h)
        h2 = h.reshape(-1, h.shape[-1])
        buf = getattr(w, "_grad_buf", None)
        ctx.buf = None
        if buf is not None:
            # the runtime bound the root unit's gradient buffer before the head: dW lands there directly (no [V, D]
            # temporary, no copy in collect_grads)
            acc = bool(getattr(w, "_grad_ready", False))
            loss, dh = K.linear_ce_fwd_bwd(h2, _wdata(w), labels, buf, ignore_index, accumulate=acc)
            w._grad_ready = True
            ctx.dw = None
            ctx.buf, ctx.buf_accumulated = buf, acc
        else:
            dw = torch.zeros_like(_wdata(w))
            loss, dh = K.linear_ce_fwd_bwd(h2, _wdata(w), labels, dw, ignore_index)
            ctx.dw = dw
        ctx.w = w
        ctx.save_for_backward(dh)
        ctx.shape = h.shape
        return loss

    @staticmethod
    def backward(ctx, dloss):
        (dh,) = ctx.saved_tensors
        # dh / dW were produced in forward for an upstream gradient of 1
        if not _UNIT_UPSTREAM:
            g = dloss.reshape(()).to(dh.device)
            dh = dh * g.to(dh.dtype)
            if ctx.dw is not None:
                ctx.dw.mul_(g.to(ctx.dw.dtype))
            elif ctx.buf is not None:
                if ctx.buf_accumulated:
                    raise RuntimeError("a scaled loss cannot be applied to a head gradient that was accumulated into "
                                       "an existing buffer; scale the loss before the fused linear-cross-entropy instead")
                ctx.buf.mul_(g.to(ctx.buf.dtype))
        return dh.view(ctx.shape), ctx.dw, None, None


def linear_cross_entropy(h, w, labels, ignore_index=-100):
    """mean CE( h @ w^T , labels ) without materialising the logits (fwd+bwd in one pass)."""
    return _LinearCE.apply(h, w, labels, ignore_index)


class _CE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, ignore_index):
        K = kernels_for(logits)
        loss, dlogits = K.cross_entropy_fwd_bwd(logits.reshape(-1, logits.shape[-1]), labels, ignore_index)
        ctx.save_for_backward(dlogits)
        ctx.shape = logits.shape
        return loss

    @staticmethod
    def backward(ctx, dloss):
        (dl,) = ctx.saved_tensors
        return (dl * dloss.to(dl.dtype)).view(ctx.shape), None, None


def cross_entropy(logits, labels, ignore_index=-100):
    return _CE.apply(logits, labels, ignore_index)


# ------------------------------------------------------------------------------------------- mamba
class _CausalConv1d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, seq_len, activation):
        K = kernels_for(x)
        ctx.K, ctx.w, ctx.b, ctx.args = K, w, b, (seq_len, activation)
        ctx.save_for_backward(x)
        return K.causal_conv1d_fwd(x, _wdata(w), None if b is None else _wdata(b), seq_len, activation)

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        seq_len, activation = ctx.args
        w, b = ctx.w, ctx.b
        dx, dw32, db32 = ctx.K.causal_conv1d_bwd(dy.contiguous(), x, _wdata(w),
                                                 None if b is None else _wdata(b), seq_len, activation)
        def putter(val):
            def put(out, acc):
                if acc:
                    out.add_(val.to(out.dtype))
                else:
                    out.copy_(val)
            return put
        dw = _deliver_wgrad(w, putter(dw32))
        db = None if b is None else _deliver_wgrad(b, putter(db32))
        return dx, dw, db, None, None


def causal_conv1d(x, w, b, seq_len, activation=True):
    return _CausalConv1d.apply(x, w, b, seq_len, activation)


class _SSDScan(torch.autograd.Function):
    """Mamba2 SSD scan. Backward recomputes through the primitive's own bwd (CUDA) or autograd of
    the sequential oracle (torch path)."""

    @staticmethod
    def forward(ctx, x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size):
        K = kernels_for(x)
        ctx.K, ctx.params, ctx.args = K, (A, D, dt_bias), (seq_len, chunk_size)
        ctx.save_for_backward(x, dt, Bm, Cm)
        return K.ssd_scan_fwd(x, dt, _wdata(A), Bm, Cm, None if D is None else _wdata(D),
                              None if dt_bias is None else _wdata(dt_bias), seq_len, chunk_size)

    @staticmethod
    def backward(ctx, dy):
        x, dt, Bm, Cm = ctx.saved_tensors
        A, D, dt_bias = ctx.params
        seq_len, chunk_size = ctx.args
        K = ctx.K
        native = None
        if hasattr(K, "ssd_scan_bwd"):
            native = K.ssd_scan_bwd(dy.contiguous(), x, dt, _wdata(A), Bm, Cm, None if D is None else _wdata(D),
                                    None if dt_bias is None else _wdata(dt_bias), seq_len, chunk_size)
        if native is not None:
            dx, ddt, dA, dB, dC, dD, ddtb = native
        else:
            with torch.enable_grad():
                leaves = [t.detach().float().requires_grad_() for t in (x, dt, _wdata(A), Bm, Cm)]
                Dl = None if D is None else _wdata(D).detach().float().requires_grad_()
                bl = None if dt_bias is None else _wdata(dt_bias).detach().float().requires_grad_()
                y = torch_kernels.ssd_scan_chunked(leaves[0], leaves[1], leaves[2], leaves[3], leaves[4], Dl, bl,
                                                   seq_len, chunk_size)
                ins = leaves + [t for t in (Dl, bl) if t is not None]
                gs = list(torch.autograd.grad(y, ins, dy.float()))
            dx, ddt, dA, dB, dC = gs[:5]
            rest = gs[5:]
            dD = rest.pop(0) if D is not None else None
            ddtb = rest.pop(0) if dt_bias is not None else None
        def putter(val):
            def put(out, acc):
                if acc:
                    out.add_(val.to(out.dtype))
                else:
                    out.copy_(val)
            return put
        gA = _deliver_wgrad(A, putter(dA))
        gD = None if D is None else _deliver_wgrad(D, putter(dD))
        gb = None if dt_bias is None else _deliver_wgrad(dt_bias, putter(ddtb))
        return (dx.to(x.dtype), ddt.to(dt.dtype), gA, dB.to(Bm.dtype), dC.to(Cm.dtype), gD, gb, None, None)


def ssd_scan(x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size=256):
    return _SSDScan.apply(x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size)


class _SelectiveScan(torch.autograd.Function):
    @staticmethod
    def forward(ctx, u, delta, A, Bm, Cm, D, z, delta_bias, seq_len):
        K = kernels_for(u)
        ctx.K, ctx.params, ctx.seq_len = K, (A, D, delta_bias), seq_len
        ctx.save_for_backward(u, delta, Bm, Cm, z)
        return K.selective_scan_fwd(u, delta, _wdata(A), Bm, Cm, None if D is None else _wdata(D), z,
                                    None if delta_bias is None else _wdata(delta_bias), seq_len)

    @staticmethod
    def backward(ctx, dy):
        u, delta, Bm, Cm, z = ctx.saved_tensors
        A, D, delta_bias = ctx.params
        K = ctx.K
        native = None
        if hasattr(K, "selective_scan_bwd"):
            native = K.selective_scan_bwd(dy.contiguous(), u, delta, _wdata(A), Bm, Cm, None if D is None else _wdata(D), z,
                                          None if delta_bias is None else _wdata(delta_bias), ctx.seq_len)
        if native is not None:
            du, dd, dA, dB, dC, dD, dz, ddb = native
        else:
            with torch.enable_grad():
                lv = [t.detach().float().requires_grad_() for t in (u, delta, _wdata(A), Bm, Cm)]
                Dl = None if D is None else _wdata(D).detach().float().requires_grad_()
                zl = None if z is None else z.detach().float().requires_grad_()
                bl = None if delta_bias is None else _wdata(delta_bias).detach().float().requires_grad_()
                y = torch_kernels.selective_scan_fwd(lv[0], lv[1], lv[2], lv[3], lv[4], Dl, zl, bl, ctx.seq_len)
                ins = lv + [t for t in (Dl, zl, bl) if t is not None]
                gs = list(torch.autograd.grad(y, ins, dy.float()))
            du, dd, dA, dB, dC = gs[:5]
            rest = gs[5:]
            dD = rest.pop(0) if D is not None else None
            dz = rest.pop(0) if z is not None else None
            ddb = rest.pop(0) if delta_bias is not None else None
        def putter(val):
            def put(out, acc):
                if acc:
                    out.add_(val.to(out.dtype))
                else:
                    out.copy_(val)
            return put
        gA = _deliver_wgrad(A, putter(dA))
        gD = None if D is None else _deliver_wgrad(D, putter(dD))
        gb = None if delta_bias is None else _deliver_wgrad(delta_bias, putter(ddb))
        return (du.to(u.dtype), dd.to(delta.dtype), gA, dB.to(Bm.dtype), dC.to(Cm.dtype), gD,
                None if z is None else dz.to(z.dtype), gb, None)


def selective_scan(u, delta, A, Bm, Cm, D=None, z=None, delta_bias=None, seq_len=None):
    return _SelectiveScan.apply(u, delta, A, Bm, Cm, D, z, delta_bias, seq_len or u.shape[0])
