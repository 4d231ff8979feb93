"""Load HuggingFace checkpoints (safetensors / .bin) into this repo's models (stand-in for
``fms.models.get_model(..., source="hf")``, SURVEY.md §2.4 E5; reference call ``speculator/train_speculator.py:150-160`` with
the adapters of ``train_speculator_utils.py:526-569``):

* Llama   -> ``LLaMA`` / ``EmbedLLaMA``: fuses q/k/v and gate/up, permutes q/k rows from HF's half-split RoPE layout back
  to the FMS interleaved-pair layout (the inverse of ``fms_to_hf_llama._interleaved_to_halfsplit``); Qwen2 / Qwen2.5 (a
  Llama block with q/k/v biases) loads the same way with ``qkv_bias=True``;
* GPT-BigCode (multi-query attention, learned positions) -> ``EmbedGPTBigCode``;
* Mixtral (Llama attention + top-k sparse MoE) -> ``EmbedMixtral``; both the hub format (``block_sparse_moe.experts.N.w1/w2/w3``)
  and the fused in-memory format of recent transformers (``mlp.experts.gate_up_proj / down_proj``)."""
from __future__ import annotations

import glob
import json
import os
from typing import Dict

import torch

from fms_fsdp_b200.models.llama import LLaMA, LLaMAConfig


def _halfsplit_to_interleaved(w: torch.Tensor, nheads: int) -> torch.Tensor:
    """q / k projection rows (2-D weight) or entries (1-D bias) of each head from (i, i + hd/2) to (2i, 2i + 1) order."""
    return w.view(nheads, 2, -1, *w.shape[1:]).transpose(1, 2).reshape(w.shape)


def is_qwen2(hf_cfg: dict) -> bool:
    """Qwen2 / Qwen2.5: Llama weight names and block, plus a bias on q, k and v (no ``attention_bias`` key says so)."""
    return hf_cfg.get("model_type") == "qwen2" or "Qwen2ForCausalLM" in (hf_cfg.get("architectures") or [])


def _sliding_window_in_use(hf_cfg: dict) -> bool:
    window = hf_cfg.get("sliding_window")
    if not window or window >= hf_cfg.get("max_position_embeddings", window):
        return False
    if hf_cfg.get("use_sliding_window") is False:          # Qwen2: the window is configured but switched off
        return False
    layer_types = hf_cfg.get("layer_types")
    if layer_types and all(t == "full_attention" for t in layer_types):
        return False
    return True


def _refuse_unsupported(hf_cfg: dict):
    """Features this repo's models do not implement must stop the load instead of silently changing the logits."""
    scaling = hf_cfg.get("rope_scaling") or {}
    params = hf_cfg.get("rope_parameters") or {}
    kind = scaling.get("rope_type") or scaling.get("type") or params.get("rope_type") or "default"
    if kind not in ("default", None, "llama3", "linear"):
        raise NotImplementedError(f"HF checkpoint uses rope scaling {kind!r}; plain RoPE, 'linear' and 'llama3' (Llama 3.1 / 3.2) "
                                  "are implemented, loading it would change the logits")
    if _sliding_window_in_use(hf_cfg):
        raise NotImplementedError(f"HF checkpoint uses sliding-window attention (window {hf_cfg['sliding_window']}); only full "
                                  "causal attention is implemented")
    if hf_cfg.get("attention_bias") or hf_cfg.get("mlp_bias"):
        raise NotImplementedError("HF checkpoint has attention-output / MLP biases; the LLaMA blocks here carry a bias on the "
                                  "q, k, v projection only (Qwen2)")


def config_from_hf(hf_cfg: dict) -> LLaMAConfig:
    _refuse_unsupported(hf_cfg)
    D, F = hf_cfg["hidden_size"], hf_cfg["intermediate_size"]
    rope = hf_cfg.get("rope_theta") or (hf_cfg.get("rope_parameters") or {}).get("rope_theta", 10000.0)
    scaling = hf_cfg.get("rope_scaling") or hf_cfg.get("rope_parameters") or {}
    kind = scaling.get("rope_type") or scaling.get("type")
    rope_scaling = {k: v for k, v in scaling.items() if k != "rope_theta"} if kind in ("llama3", "linear") else None
    return LLaMAConfig(
        src_vocab_size=hf_cfg["vocab_size"], emb_dim=D, norm_eps=hf_cfg.get("rms_norm_eps", 1e-5),
        nheads=hf_cfg["num_attention_heads"], kvheads=hf_cfg.get("num_key_value_heads", 0) or 0,
        nlayers=hf_cfg["num_hidden_layers"], hidden_grow_factor=F / D, multiple_of=1,
        max_expected_seq_len=hf_cfg.get("max_position_embeddings", 4096), rope_theta=float(rope),
        rope_scaling=rope_scaling, qkv_bias=is_qwen2(hf_cfg))


def _read_hf_tensors(model_path: str) -> Dict[str, torch.Tensor]:
    out: Dict[str, torch.Tensor] = {}
    st = sorted(glob.glob(os.path.join(model_path, "*.safetensors")))
    if st:
        from safetensors.torch import load_file
        for f in st:
            out.update(load_file(f))
        return out
    for f in sorted(glob.glob(os.path.join(model_path, "pytorch_model*.bin"))):
        out.update(torch.load(f, map_location="cpu", weights_only=True))
    if not out:
        raise FileNotFoundError(f"no safetensors / pytorch_model*.bin under {model_path}")
    return out


def _refuse_unaccounted_biases(hf: Dict[str, torch.Tensor], cfg: LLaMAConfig):
    """A bias tensor the config does not account for would be dropped and change the logits: stop instead."""
    allowed = (".self_attn.q_proj.bias", ".self_attn.k_proj.bias", ".self_attn.v_proj.bias") if cfg.qkv_bias else ()
    extra = sorted(k for k in hf if k.endswith(".bias") and not k.endswith(allowed))
    if extra:
        raise NotImplementedError(f"HF checkpoint carries bias tensors the model does not have ({', '.join(extra[:4])}"
                                  f"{', ...' if len(extra) > 4 else ''}); loading it would drop them and change the logits")


def convert_hf_state_dict(hf: Dict[str, torch.Tensor], cfg: LLaMAConfig) -> Dict[str, torch.Tensor]:
    _refuse_unaccounted_biases(hf, cfg)
    sd = {"shared.emb.weight": hf["model.embed_tokens.weight"],
          "shared.head.weight": hf.get("lm_head.weight", hf["model.embed_tokens.weight"]),
          "dec_norm.weight": hf["model.norm.weight"]}
    for i in range(cfg.nlayers):
        s, d = f"model.layers.{i}.", f"layers.{i}."
        q = _halfsplit_to_interleaved(hf[s + "self_attn.q_proj.weight"], cfg.nheads)
        k = _halfsplit_to_interleaved(hf[s + "self_attn.k_proj.weight"], cfg.kv_heads)
        sd[d + "attn.in_proj.qkv_fused.weight"] = torch.cat([q, k, hf[s + "self_attn.v_proj.weight"]], dim=0)
        if cfg.qkv_bias:
            sd[d + "attn.in_proj.qkv_fused.bias"] = torch.cat([
                _halfsplit_to_interleaved(hf[s + "self_attn.q_proj.bias"], cfg.nheads),
                _halfsplit_to_interleaved(hf[s + "self_attn.k_proj.bias"], cfg.kv_heads), hf[s + "self_attn.v_proj.bias"]])
        sd[d + "attn.dense.weight"] = hf[s + "self_attn.o_proj.weight"]
        sd[d + "ff_sub_layer.wg1_fused.weight"] = torch.cat([hf[s + "mlp.gate_proj.weight"], hf[s + "mlp.up_proj.weight"]], dim=0)
        sd[d + "ff_sub_layer.w2.weight"] = hf[s + "mlp.down_proj.weight"]
        sd[d + "ln.weight"] = hf[s + "input_layernorm.weight"]
        sd[d + "ff_ln.weight"] = hf[s + "post_attention_layernorm.weight"]
    return sd


def load_hf_llama(model_path: str, device="cpu", dtype=torch.bfloat16, model_cls=LLaMA) -> LLaMA:
    with open(os.path.join(model_path, "config.json")) as f:
        cfg = config_from_hf(json.load(f))
    with torch.device("meta"):
        model = model_cls(cfg)
    model.to_empty(device=device)
    sd = convert_hf_state_dict(_read_hf_tensors(model_path), cfg)
    model.load_state_dict({k: v.to(dtype) for k, v in sd.items()})
    return model.to(dtype)


# ------------------------------------------------------------------------------------------ GPT-BigCode
def load_hf_gpt_bigcode(model_path: str, model_cls, device="cpu", dtype=torch.bfloat16):
    """``model_cls`` = ``speculator.train_speculator_utils.EmbedGPTBigCode`` (kept out of this module's imports)."""
    with open(os.path.join(model_path, "config.json")) as f:
        c = json.load(f)
    if not c.get("multi_query", True):
        raise ValueError("only multi-query GPT-BigCode checkpoints are supported")
    act = c.get("activation_function", "gelu_pytorch_tanh")
    if act not in ("gelu_pytorch_tanh", "gelu_new", "gelu_fast"):     # all three are the tanh approximation the block computes
        raise NotImplementedError(f"GPT-BigCode activation {act!r}: the block implements tanh-approximated GELU only")
    if not c.get("scale_attn_weights", True):
        raise NotImplementedError("GPT-BigCode checkpoints with scale_attn_weights=False are not supported")
    D = c["n_embd"]
    hidden = c.get("n_inner") or 4 * D
    if hidden % D:
        raise ValueError(f"n_inner {hidden} is not a multiple of n_embd {D}")
    with torch.device("meta"):
        model = model_cls(vocab=c["vocab_size"], emb_dim=D, nheads=c["n_head"], nlayers=c["n_layer"], max_pos=c["n_positions"],
                          hidden_mult=hidden // D, eps=c.get("layer_norm_epsilon", 1e-5))
    model.to_empty(device=device)
    hf = _read_hf_tensors(model_path)
    sd = {"emb.weight": hf["transformer.wte.weight"], "pos.weight": hf["transformer.wpe.weight"],
          "dec_norm.weight": hf["transformer.ln_f.weight"], "dec_norm.bias": hf["transformer.ln_f.bias"],
          "head.weight": hf.get("lm_head.weight", hf["transformer.wte.weight"])}
    names = {"ln": "ln_1", "ff_ln": "ln_2", "qkv": "attn.c_attn", "dense": "attn.c_proj", "w1": "mlp.c_fc", "w2": "mlp.c_proj"}
    for i in range(c["n_layer"]):
        for ours, theirs in names.items():
            for part in ("weight", "bias"):
                sd[f"layers.{i}.{ours}.{part}"] = hf[f"transformer.h.{i}.{theirs}.{part}"]
    model.load_state_dict({k: v.to(dtype) for k, v in sd.items()})
    return model.to(dtype)


# ---------------------------------------------------------------------------------------------- Mixtral
def load_hf_mixtral(model_path: str, model_cls, device="cpu", dtype=torch.bfloat16):
    """``model_cls`` = ``EmbedMixtral``.  Attention weights follow the Llama conversion; expert weights are stacked to
    ``moe.w1 [E, 2F, D]`` (gate | up) and ``moe.w2 [E, D, F]``."""
    with open(os.path.join(model_path, "config.json")) as f:
        c = json.load(f)
    cfg = config_from_hf(c)
    hf = _read_hf_tensors(model_path)
    _refuse_unaccounted_biases(hf, cfg)
    E, top_k = c["num_local_experts"], c.get("num_experts_per_tok", 2)
    with torch.device("meta"):
        model = model_cls(cfg, n_experts=E, top_k=top_k)
    model.to_empty(device=device)
    sd = {"shared.emb.weight": hf["model.embed_tokens.weight"],
          "shared.head.weight": hf.get("lm_head.weight", hf["model.embed_tokens.weight"]),
          "dec_norm.weight": hf["model.norm.weight"]}
    for i in range(cfg.nlayers):
        s, d = f"model.layers.{i}.", f"layers.{i}."
        q = _halfsplit_to_interleaved(hf[s + "self_attn.q_proj.weight"], cfg.nheads)
        k = _halfsplit_to_interleaved(hf[s + "self_attn.k_proj.weight"], cfg.kv_heads)
        sd[d + "attn.in_proj.qkv_fused.weight"] = torch.cat([q, k, hf[s + "self_attn.v_proj.weight"]], dim=0)
        sd[d + "attn.dense.weight"] = hf[s + "self_attn.o_proj.weight"]
        sd[d + "ln.weight"] = hf[s + "input_layernorm.weight"]
        sd[d + "ff_ln.weight"] = hf[s + "post_attention_layernorm.weight"]
        if s + "mlp.experts.gate_up_proj" in hf:                       # fused in-memory layout of recent transformers
            sd[d + "moe.gate.weight"] = hf[s + "mlp.gate.weight"]
            sd[d + "moe.w1"] = hf[s + "mlp.experts.gate_up_proj"]
            sd[d + "moe.w2"] = hf[s + "mlp.experts.down_proj"]
        else:                                                          # hub layout: w1 = gate, w3 = up, w2 = down
            b = s + "block_sparse_moe."
            sd[d + "moe.gate.weight"] = hf[b + "gate.weight"]
            sd[d + "moe.w1"] = torch.stack([torch.cat([hf[f"{b}experts.{e}.w1.weight"], hf[f"{b}experts.{e}.w3.weight"]], 0)
                                            for e in range(E)])
            sd[d + "moe.w2"] = torch.stack([hf[f"{b}experts.{e}.w2.weight"] for e in range(E)])
    model.load_state_dict({k: v.to(dtype) for k, v in sd.items()})
    return model.to(dtype)
