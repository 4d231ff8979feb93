"""LLaMA for the B200 engine.

State-dict names, fused-weight layout, initialisation and numerics contract follow the
ibm-fms LLaMA that the reference trains (SURVEY.md §2.4 E2; names evidenced by reference
``fms_to_hf_llama.py:54-128``): ``shared.emb/head``, ``layers.N.{ln, attn.in_proj.qkv_fused,
attn.dense, ff_ln, ff_sub_layer.wg1_fused, ff_sub_layer.w2}``, ``dec_norm``; RoPE in the
interleaved-pair convention; RMSNorm in fp32; SwiGLU on ``[gate | up]``.

The architecture is *not* a module-per-op graph: each block is one straight-line sequence of
engine ops (``fms_fsdp_b200.ops``) that run as sm_100a kernels on GPU, and the model exposes
``engine_units()`` so the sharded runtime can schedule gather / compute / reduce per unit.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional

import torch
import torch.nn as nn

from fms_fsdp_b200 import ops
from fms_fsdp_b200.ops import torch_kernels


@dataclass
class LLaMAConfig:
    src_vocab_size: int = 32000
    emb_dim: int = 4096
    norm_eps: float = 1e-5
    nheads: int = 32
    kvheads: int = 0
    nlayers: int = 32
    pad_id: int = -1
    hidden_grow_factor: float = 8 / 3
    multiple_of: int = 256
    activation_fn: str = "swish"
    p_dropout: float = 0.0
    max_expected_seq_len: int = 4096
    ntk_scaling: bool = False
    attn_bias: bool = False
    mlp_bias: bool = False
    tie_heads: bool = False
    rope_theta: float = 10000.0
    linear_config: Optional[dict] = None
    fused_weights: bool = True
    # extension (not an fms field): HF-style frequency rescaling of long-context checkpoints, e.g. Llama 3.1
    # {"rope_type": "llama3", "factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0, "original_max_position_embeddings": 8192}
    rope_scaling: Optional[dict] = None
    # extension (not an fms field): a bias on the fused q, k, v projection, added before RoPE (Qwen2 / Qwen2.5).
    # State-dict key ``layers.N.attn.in_proj.qkv_fused.bias``; no bias on the output projection or the MLP.
    qkv_bias: bool = False

    @property
    def hidden_dim(self) -> int:
        return self.multiple_of * ((int(self.hidden_grow_factor * self.emb_dim) + self.multiple_of - 1)
                                   // self.multiple_of)

    @property
    def kv_heads(self) -> int:
        return self.nheads if self.kvheads == 0 else self.kvheads

    @property
    def head_dim(self) -> int:
        return self.emb_dim // self.nheads


class _Weight(nn.Module):
    """A linear weight holder: keeps FMS's ``<name>.weight`` (and, with ``bias=True``, ``<name>.bias``) state-dict keys."""

    def __init__(self, out_features: int, in_features: int, device=None, dtype=None, bias: bool = False):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        self.weight = nn.Parameter(torch.empty(out_features, in_features, device=device, dtype=dtype))
        self.bias = nn.Parameter(torch.empty(out_features, device=device, dtype=dtype)) if bias else None

    def forward(self, x, residual=None):
        return ops.linear(x, self.weight, residual, bias=self.bias)


class RMSNorm(nn.Module):
    """FMS LayerNormParameterized(use_mean=False, elementwise_scale=True, no shift)."""

    def __init__(self, dim: int, eps: float, device=None, dtype=None):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.empty(dim, device=device, dtype=dtype))

    def reset_parameters(self):
        nn.init.ones_(self.weight)

    def forward(self, x):
        return ops.rmsnorm(x, self.weight, self.eps)

    def fork(self, x):
        """(norm(x), x) with the residual-branch gradient folded into the norm's backward kernel."""
        return ops.rmsnorm_fork(x, self.weight, self.eps)


class RotaryEmbedding(nn.Module):
    """cos/sin table cache; attrs mirror what the reference exporter reads
    (``dim, ratio, max_seq_len, ntk_scaling, _alpha``: reference ``fms_to_hf_llama.py:43-51``)."""

    def __init__(self, dim: int, ratio: float = 10000.0, max_seq_len: int = 2048, ntk_scaling: bool = False, scaling=None):
        super().__init__()
        self.dim, self.ratio, self.max_seq_len, self.ntk_scaling = dim, ratio, max_seq_len, ntk_scaling
        self.scaling = dict(scaling) if scaling else None
        self._tables = {}

    def _alpha(self, seq_len) -> int:
        if not self.ntk_scaling:
            return 1
        return max(1, 2 ** math.ceil(math.log2(max(seq_len / self.max_seq_len, 1))))

    def compute_freqs_cis(self, device, max_seq_len: int = 2048):
        """Precompute (and cache per device) the [S, dim/2, 2] cos/sin table (reference
        ``main_training_llama.py:93-96`` calls this after wrapping)."""
        alpha = self._alpha(max_seq_len)
        key = (str(device), alpha)
        tab = self._tables.get(key)
        if tab is None or tab.shape[0] < max_seq_len:
            n = max(max_seq_len, self.max_seq_len * alpha)
            tab = torch_kernels.rope_table(n, self.dim, self.ratio, float(alpha), device=device, scaling=self.scaling)
            self._tables[key] = tab
        return tab

    def table(self, device, seq_len):
        return self.compute_freqs_cis(device, seq_len)


class _InProj(nn.Module):
    def __init__(self, cfg: LLaMAConfig, device=None, dtype=None):
        super().__init__()
        hd = cfg.head_dim
        self.splits = [cfg.nheads * hd, cfg.kv_heads * hd, cfg.kv_heads * hd]
        self.qkv_fused = _Weight(sum(self.splits), cfg.emb_dim, device, dtype, bias=getattr(cfg, "qkv_bias", False))


class MultiHeadAttention(nn.Module):
    def __init__(self, cfg: LLaMAConfig, device=None, dtype=None):
        super().__init__()
        self.nheads, self.kvheads, self.head_dim = cfg.nheads, cfg.kv_heads, cfg.head_dim
        self.emb_dim = cfg.emb_dim
        self.in_proj = _InProj(cfg, device, dtype)
        self.dense = _Weight(cfg.emb_dim, cfg.nheads * cfg.head_dim, device, dtype)

    def reset_parameters(self):
        for w in (self.in_proj.qkv_fused.weight, self.dense.weight):
            nn.init.trunc_normal_(w, mean=0.0, std=0.02)
        if self.in_proj.qkv_fused.bias is not None:
            nn.init.zeros_(self.in_proj.qkv_fused.bias)


class GatedLinearUnit(nn.Module):
    def __init__(self, cfg: LLaMAConfig, device=None, dtype=None):
        super().__init__()
        self.hidden_dim = cfg.hidden_dim
        self.wg1_fused = _Weight(2 * cfg.hidden_dim, cfg.emb_dim, device, dtype)
        self.w2 = _Weight(cfg.emb_dim, cfg.hidden_dim, device, dtype)

    def reset_parameters(self):
        for w in (self.wg1_fused.weight, self.w2.weight):
            nn.init.trunc_normal_(w, mean=0.0, std=0.02)


class WordEmbedding(nn.Module):
    """Embedding + reversible (untied unless tie_heads) output head: ``shared.emb`` / ``shared.head``."""

    def __init__(self, cfg: LLaMAConfig, device=None, dtype=None):
        super().__init__()
        self.vocab_size, self.emb_dim, self.tie_weights = cfg.src_vocab_size, cfg.emb_dim, cfg.tie_heads
        self.padding_idx = cfg.pad_id if cfg.pad_id >= 0 else None
        self.emb = nn.Embedding(cfg.src_vocab_size, cfg.emb_dim, device=device, dtype=dtype)
        self.head = _Weight(cfg.src_vocab_size, cfg.emb_dim, device, dtype)
        if self.tie_weights:
            self.head.weight = self.emb.weight

    def reset_parameters(self):
        nn.init.trunc_normal_(self.emb.weight, mean=0.0, std=self.emb_dim ** -0.5)
        if not self.tie_weights:
            nn.init.trunc_normal_(self.head.weight, mean=0.0, std=self.emb_dim ** -0.5)
        if self.padding_idx is not None:
            with torch.no_grad():
                self.emb.weight[self.padding_idx].zero_()

    def forward(self, x, reverse: bool = False):
        if reverse:
            return ops.linear(x, self.head.weight)
        return ops.embedding(x, self.emb.weight)


class LLaMABlock(nn.Module):
    """ln -> fused QKV -> RoPE -> causal flash attention -> dense(+res) -> ff_ln -> gate/up -> SwiGLU
    -> w2(+res).  Hot-op inventory K1-K8 of SURVEY.md §2.5(a)."""

    def __init__(self, cfg: LLaMAConfig, rot_emb: RotaryEmbedding, device=None, dtype=None):
        super().__init__()
        self.config = cfg
        self.ln = RMSNorm(cfg.emb_dim, cfg.norm_eps, device, dtype)
        self.ff_ln = RMSNorm(cfg.emb_dim, cfg.norm_eps, device, dtype)
        self.attn = MultiHeadAttention(cfg, device, dtype)
        self.ff_sub_layer = GatedLinearUnit(cfg, device, dtype)
        object.__setattr__(self, "_rot", rot_emb)  # shared, not a submodule (no params, not in state dict)

    def forward(self, x):
        a, cfg = self.attn, self.config
        B, S, _ = x.shape
        h, x = self.ln.fork(x)
        # projection + RoPE + attention: one node, RoPE fused into the GEMM / dq-dk epilogues
        ctx = ops.qkv_attention(h, a.in_proj.qkv_fused.weight, self._rot.table(x.device, S), a.nheads, a.kvheads,
                                a.head_dim, bias=a.in_proj.qkv_fused.bias)
        x = a.dense(ctx, residual=x)
        h, x = self.ff_ln.fork(x)
        ff = self.ff_sub_layer
        # gate/up GEMM with the SwiGLU epilogue, down projection with the residual epilogue: one autograd node
        return ops.gated_mlp(h, ff.wg1_fused.weight, ff.w2.weight, residual=x)


class LLaMA(nn.Module):
    def __init__(self, config: Optional[LLaMAConfig] = None, device=None, dtype=None, **kwargs):
        super().__init__()
        self.config = config if config is not None else LLaMAConfig()
        for k, v in kwargs.items():
            setattr(self.config, k, v)
        cfg = self.config
        self.width = cfg.emb_dim
        self.pad_id = cfg.pad_id
        self.max_expected_seq_len = cfg.max_expected_seq_len
        self.shared = WordEmbedding(cfg, device, dtype)
        self.rot_emb = RotaryEmbedding(cfg.head_dim, cfg.rope_theta, cfg.max_expected_seq_len, cfg.ntk_scaling,
                                       getattr(cfg, "rope_scaling", None))
        self.layers = nn.ModuleList([LLaMABlock(cfg, self.rot_emb, device, dtype) for _ in range(cfg.nlayers)])
        self.dec_norm = RMSNorm(cfg.emb_dim, cfg.norm_eps, device, dtype)

    def get_config(self) -> LLaMAConfig:
        return self.config

    def reset_parameters(self):
        self.shared.reset_parameters()
        self.dec_norm.reset_parameters()
        for blk in self.layers:
            blk.ln.reset_parameters()
            blk.ff_ln.reset_parameters()
            blk.attn.reset_parameters()
            blk.ff_sub_layer.reset_parameters()

    # ---- plain (unsharded) forward: logits, as the reference model returns
    def forward(self, x, labels=None, return_hidden: bool = False):
        h = self.shared(x)
        for blk in self.layers:
            h = blk(h)
        h = self.dec_norm(h)
        if return_hidden:
            return h
        if labels is not None:
            return ops.linear_cross_entropy(h, self.shared.head.weight, labels)
        return self.shared(h, reverse=True)

    # ---- sharded-runtime protocol -------------------------------------------------------------
    def engine_units(self):
        """(blocks, root_modules): one shard unit per block; embedding+head+final norm form the root
        unit (reference wrapping policy, ``policies/wrapping.py:6-14``)."""
        return list(self.layers), [self.shared, self.dec_norm]

    def engine_embed(self, tokens):
        return self.shared(tokens)

    def engine_head(self, h, labels=None, ignore_index=-100):
        h = self.dec_norm(h)
        if labels is None:
            return self.shared(h, reverse=True)
        return ops.linear_cross_entropy(h, self.shared.head.weight, labels, ignore_index)


def param_count(model: nn.Module) -> int:
    return sum(p.numel() for p in model.parameters())
