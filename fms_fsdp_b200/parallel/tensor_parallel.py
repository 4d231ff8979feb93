"""Tensor parallelism for the FROZEN base model of speculator training (the only place the reference uses TP:
``speculator/train_speculator.py:133-160``; SURVEY.md §2.2).  Megatron layout: column-parallel fused QKV and
gate/up (heads / hidden units split across ranks), row-parallel dense and down projection followed by an
all-reduce, vocab-parallel head followed by an all-gather.  Forward-only (no_grad).

``shard_for_tp`` covers the three base-model families of the speculator registry: Llama (``shard_llama_for_tp``), Mixtral
(Llama attention + every expert's hidden units split, the router replicated) and GPT-BigCode (query heads split, the single
shared K/V head replicated on every rank, biases of row-parallel layers kept on TP rank 0 only so the all-reduce adds them
once)."""
from __future__ import annotations

import torch
import torch.distributed as dist

from fms_fsdp_b200.models.llama import LLaMA


def _rows(t: torch.Tensor, r: int, n: int) -> torch.Tensor:
    """Rank r's block of n rows (dim 0), as its own storage."""
    return t[r * n:(r + 1) * n].clone()


def _cols(t: torch.Tensor, r: int, n: int) -> torch.Tensor:
    return t[..., r * n:(r + 1) * n].clone()


def _slice_llama_attention(blk, c, tp: int, r: int):
    hd = c.head_dim
    H, KV = c.nheads // tp, c.kv_heads // tp
    q, k, v = torch.split(blk.attn.in_proj.qkv_fused.weight.data, [c.nheads * hd, c.kv_heads * hd, c.kv_heads * hd], dim=0)
    blk.attn.in_proj.qkv_fused.weight.data = torch.cat([_rows(q, r, H * hd), _rows(k, r, KV * hd), _rows(v, r, KV * hd)])
    bias = blk.attn.in_proj.qkv_fused.bias
    if bias is not None:   # qkv_bias (Qwen2): sliced by heads exactly like the weight rows
        q, k, v = torch.split(bias.data, [c.nheads * hd, c.kv_heads * hd, c.kv_heads * hd])
        bias.data = torch.cat([_rows(q, r, H * hd), _rows(k, r, KV * hd), _rows(v, r, KV * hd)])
    blk.attn.dense.weight.data = _cols(blk.attn.dense.weight.data, r, H * hd)
    blk.attn.nheads, blk.attn.kvheads = H, KV


def _check_llama_divisible(c, tp: int):
    assert c.nheads % tp == 0 and c.kv_heads % tp == 0 and c.hidden_dim % tp == 0 and c.src_vocab_size % tp == 0, \
        "tp size must divide heads, kv heads, hidden dim and vocab"


def shard_llama_for_tp(model: LLaMA, group) -> LLaMA:
    """Slice the weights of a loaded LLaMA in place; afterwards every block computes on 1/tp of the heads and
    of the MLP hidden units.  The model is flagged so ``EmbedLLaMA.forward`` inserts the collectives."""
    tp, r = dist.get_world_size(group), dist.get_rank(group)
    c = model.config
    _check_llama_divisible(c, tp)
    F = c.hidden_dim // tp
    with torch.no_grad():
        for blk in model.layers:
            _slice_llama_attention(blk, c, tp, r)
            g, u = blk.ff_sub_layer.wg1_fused.weight.data.chunk(2, dim=0)
            blk.ff_sub_layer.wg1_fused.weight.data = torch.cat([_rows(g, r, F), _rows(u, r, F)])
            blk.ff_sub_layer.w2.weight.data = _cols(blk.ff_sub_layer.w2.weight.data, r, F)
        model.shared.head.weight.data = _rows(model.shared.head.weight.data, r, c.src_vocab_size // tp)
    model._tp_group, model._tp_size = group, tp
    return model


def shard_mixtral_for_tp(model, group):
    """Mixtral base (``EmbedMixtral``): attention as Llama; each expert keeps 1/tp of its hidden units (``moe.w1 [E, 2F, D]``
    = gate | up, ``moe.w2 [E, D, F]``), the router stays whole so every rank routes identically, and the block's MoE output is
    all-reduced like a row-parallel linear."""
    tp, r = dist.get_world_size(group), dist.get_rank(group)
    c = model.config
    _check_llama_divisible(c, tp)
    F = c.hidden_dim // tp
    with torch.no_grad():
        for blk in model.layers:
            _slice_llama_attention(blk, c, tp, r)
            g, u = blk.moe.w1.data.chunk(2, dim=1)
            blk.moe.w1.data = torch.cat([g[:, r * F:(r + 1) * F], u[:, r * F:(r + 1) * F]], dim=1).contiguous()
            blk.moe.w2.data = _cols(blk.moe.w2.data, r, F)
        model.shared.head.weight.data = _rows(model.shared.head.weight.data, r, c.src_vocab_size // tp)
    model._tp_group, model._tp_size = group, tp
    return model


def shard_gpt_bigcode_for_tp(model, group):
    """GPT-BigCode base (``EmbedGPTBigCode``, multi-query attention): query heads and MLP hidden units are split; the one
    K/V head is computed on every rank (it is 2/(nheads+2) of the QKV projection).  ``dense`` and ``w2`` are row-parallel:
    their bias survives on TP rank 0 only, so the all-reduce of the partial outputs adds it exactly once."""
    tp, r = dist.get_world_size(group), dist.get_rank(group)
    blk0 = model.layers[0]
    nheads, hd, hidden = blk0.nheads, blk0.hd, blk0.w1.out_features
    vocab = model.head.out_features
    assert nheads % tp == 0 and hidden % tp == 0 and vocab % tp == 0, "tp size must divide heads, MLP hidden dim and vocab"
    H, F, D = nheads // tp, hidden // tp, nheads * hd
    with torch.no_grad():
        for blk in model.layers:
            w, b = blk.qkv.weight.data, blk.qkv.bias.data
            blk.qkv.weight.data = torch.cat([_rows(w[:D], r, H * hd), w[D:].clone()])
            blk.qkv.bias.data = torch.cat([_rows(b[:D], r, H * hd), b[D:].clone()])
            blk.dense.weight.data = _cols(blk.dense.weight.data, r, H * hd)
            blk.w1.weight.data, blk.w1.bias.data = _rows(blk.w1.weight.data, r, F), _rows(blk.w1.bias.data, r, F)
            blk.w2.weight.data = _cols(blk.w2.weight.data, r, F)
            if r != 0:
                blk.dense.bias.data.zero_()
                blk.w2.bias.data.zero_()
            blk.nheads, blk.tp_group = H, group
        model.head.weight.data = _rows(model.head.weight.data, r, vocab // tp)
    model._tp_group, model._tp_size = group, tp
    return model


def shard_for_tp(model, group):
    """Dispatch on the base-model family (duck-typed so this module does not import the speculator package)."""
    if isinstance(model, LLaMA):
        if hasattr(model.layers[0], "moe"):
            return shard_mixtral_for_tp(model, group)
        return shard_llama_for_tp(model, group)
    if hasattr(model, "pos") and hasattr(model.layers[0], "qkv"):
        return shard_gpt_bigcode_for_tp(model, group)
    raise TypeError(f"no tensor-parallel plan for {type(model).__name__}")


def tp_all_reduce(x, group):
    dist.all_reduce(x, group=group)
    return x


def tp_all_gather_last(x, group):
    tp = dist.get_world_size(group)
    parts = [torch.empty_like(x) for _ in range(tp)]
    dist.all_gather(parts, x.contiguous(), group=group)
    return torch.cat(parts, dim=-1)
