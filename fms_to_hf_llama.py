"""Export a sharded training checkpoint to a HuggingFace ``LlamaForCausalLM`` directory (``Qwen2ForCausalLM`` for a model
with ``qkv_bias``)
(CLI parity with reference ``fms_to_hf_llama.py:133-171``):

    python fms_to_hf_llama.py --model_variant llama2_7b --nocompiled --load_path <step_N_ckp> \
        --save_path <out> --tokenizer_name_or_path <tok>

Reads the DCP checkpoint (``model_state.*`` keys, or ``model_state._orig_mod.*`` for checkpoints written under
torch.compile by the reference) without any process group, splits the fused QKV / gate-up weights, and permutes
q/k rows from the FMS interleaved-pair RoPE layout to HF's half-split layout.  Unlike the reference (SURVEY.md
Q17) the exported config carries the right ``rope_theta`` / ``max_position_embeddings``, so llama3 / 34b exports
round-trip (tests/test_exporters.py checks logits equality).
"""
import os

import torch

from fms_fsdp_b200.models.llama import LLaMA
from fms_fsdp_b200.utils.cli import run
from fms_fsdp_b200.utils.config_utils import get_model_config


def _interleaved_to_halfsplit(w: torch.Tensor, nheads: int) -> torch.Tensor:
    """rows [h, (pair, 2)] -> [h, (2, pair)]: (x0,x1,x2,x3,..) -> (x0,x2,..,x1,x3,..) per head (2-D weight or 1-D bias)."""
    return w.view(nheads, -1, 2, *w.shape[1:]).transpose(1, 2).reshape(w.shape)


def convert_to_hf(model: LLaMA, model_variant: str, is_old_fms: bool = False):
    """``is_old_fms`` is kept for the reference's signature; this repo's LLaMA is always fused, pre-fusion checkpoints are
    fused when they are read (``load_dcp_into``)."""
    from transformers import LlamaConfig, LlamaForCausalLM, Qwen2Config, Qwen2ForCausalLM

    c = model.config
    qwen2 = getattr(c, "qkv_bias", False)
    rope_theta = c.rope_theta
    if c.ntk_scaling:
        alpha = model.rot_emb._alpha(c.max_expected_seq_len)
        rope_theta = rope_theta * alpha ** (c.head_dim / (c.head_dim - 2))
    kw = dict(
        vocab_size=c.src_vocab_size, hidden_size=c.emb_dim, rms_norm_eps=c.norm_eps, num_attention_heads=c.nheads,
        num_key_value_heads=c.kv_heads, num_hidden_layers=c.nlayers, intermediate_size=c.hidden_dim,
        pad_token_id=None if c.pad_id == -1 else c.pad_id, max_position_embeddings=c.max_expected_seq_len,
        rope_theta=rope_theta, tie_word_embeddings=False,
    )
    if not qwen2:
        kw.update(attention_bias=False, mlp_bias=False)
    else:   # Qwen2: biased q/k/v, full attention (the window is configured but switched off)
        kw.update(use_sliding_window=False, sliding_window=None)
    if "llama3" in model_variant:
        kw.update(bos_token_id=128000, eos_token_id=128001)
    if getattr(c, "rope_scaling", None):          # long-context frequency rescaling travels with the export
        kw["rope_scaling"] = dict(c.rope_scaling)
    hf = Qwen2ForCausalLM(Qwen2Config(**kw)) if qwen2 else LlamaForCausalLM(LlamaConfig(**kw))
    sd = model.state_dict()
    hd = c.head_dim
    with torch.no_grad():
        hf.model.embed_tokens.weight.copy_(sd["shared.emb.weight"])
        for i, layer in enumerate(hf.model.layers):
            p = f"layers.{i}."
            q, k, v = torch.split(sd[p + "attn.in_proj.qkv_fused.weight"],
                                  [c.nheads * hd, c.kv_heads * hd, c.kv_heads * hd], dim=0)
            layer.self_attn.q_proj.weight.copy_(_interleaved_to_halfsplit(q, c.nheads))
            layer.self_attn.k_proj.weight.copy_(_interleaved_to_halfsplit(k, c.kv_heads))
            layer.self_attn.v_proj.weight.copy_(v)
            if qwen2:
                qb, kb, vb = torch.split(sd[p + "attn.in_proj.qkv_fused.bias"],
                                         [c.nheads * hd, c.kv_heads * hd, c.kv_heads * hd])
                layer.self_attn.q_proj.bias.copy_(_interleaved_to_halfsplit(qb, c.nheads))
                layer.self_attn.k_proj.bias.copy_(_interleaved_to_halfsplit(kb, c.kv_heads))
                layer.self_attn.v_proj.bias.copy_(vb)
            layer.self_attn.o_proj.weight.copy_(sd[p + "attn.dense.weight"])
            fused = sd[p + "ff_sub_layer.wg1_fused.weight"]
            wg, w1 = torch.split(fused, [fused.size(0) // 2, fused.size(0) // 2], dim=0)
            layer.mlp.gate_proj.weight.copy_(wg)
            layer.mlp.up_proj.weight.copy_(w1)
            layer.mlp.down_proj.weight.copy_(sd[p + "ff_sub_layer.w2.weight"])
            layer.input_layernorm.weight.copy_(sd[p + "ln.weight"])
            layer.post_attention_layernorm.weight.copy_(sd[p + "ff_ln.weight"])
        hf.model.norm.weight.copy_(sd["dec_norm.weight"])
        hf.lm_head.weight.copy_(sd["shared.head.weight"])
    return hf


def _unfused_template(model: LLaMA):
    """State-dict template in the layout of pre-fusion FMS releases: separate ``attn.query/key/value`` and
    ``ff_sub_layer.wg/w1`` instead of ``attn.in_proj.qkv_fused`` and ``ff_sub_layer.wg1_fused``."""
    c, hd, out = model.config, model.config.head_dim, {}
    for k, v in model.state_dict().items():
        if k.endswith("attn.in_proj.qkv_fused.weight"):
            base = k[:-len("in_proj.qkv_fused.weight")]
            for name, rows in (("query", c.nheads * hd), ("key", c.kv_heads * hd), ("value", c.kv_heads * hd)):
                out[base + name + ".weight"] = v.new_empty(rows, v.size(1))
        elif k.endswith("ff_sub_layer.wg1_fused.weight"):
            base = k[:-len("wg1_fused.weight")]
            out[base + "wg.weight"] = v.new_empty(v.size(0) // 2, v.size(1))
            out[base + "w1.weight"] = v.new_empty(v.size(0) // 2, v.size(1))
        else:
            out[k] = v
    return out


def _fuse_old_fms(sd):
    out = {}
    for k, v in sd.items():
        if k.endswith("attn.query.weight"):
            base = k[:-len("query.weight")]
            out[base + "in_proj.qkv_fused.weight"] = torch.cat([v, sd[base + "key.weight"], sd[base + "value.weight"]], dim=0)
        elif k.endswith("ff_sub_layer.wg.weight"):
            base = k[:-len("wg.weight")]
            out[base + "wg1_fused.weight"] = torch.cat([v, sd[base + "w1.weight"]], dim=0)
        elif not k.endswith(("attn.key.weight", "attn.value.weight", "ff_sub_layer.w1.weight")):
            out[k] = v
    return out


def load_dcp_into(model: torch.nn.Module, load_path: str, compiled: bool = False, is_old_fms: bool = False):
    """no_dist DCP read of ``model_state`` into a full CPU model.  Handles the ``_orig_mod`` level of checkpoints written
    under torch.compile and -- ``is_old_fms``, or detected from the keys -- checkpoints of pre-fusion FMS releases, whose
    separate q / k / v and gate / up matrices are fused on the way in (this repo's LLaMA is always fused)."""
    import torch.distributed.checkpoint as dcp
    from torch.distributed.checkpoint import FileSystemReader
    keys = set(FileSystemReader(load_path).read_metadata().state_dict_metadata.keys())
    unfused = is_old_fms or any(k.endswith("attn.query.weight") for k in keys)
    if unfused and any(k.endswith("attn.in_proj.qkv_fused.weight") for k in keys):
        unfused = False          # --is_old_fms given for a checkpoint that is already fused: nothing to do
    template = _unfused_template(model) if unfused else model.state_dict()
    nested = compiled or any(k.startswith("model_state._orig_mod.") for k in keys)
    prefix = "model_state._orig_mod." if nested else "model_state."
    # tied parameters (e.g. Mamba ``lm_head.weight`` = ``backbone.embedding.weight``) are stored once by this runtime: ask
    # only for what the checkpoint holds, and let the module's own tying supply the alias
    absent = [k for k in template if prefix + k not in keys]
    template = {k: v for k, v in template.items() if prefix + k in keys}
    state = {"model_state": {"_orig_mod": template} if nested else template}
    dcp.load(state, checkpoint_id=load_path, no_dist=True)
    sd = state["model_state"]
    sd = sd.get("_orig_mod", sd)
    sd = _fuse_old_fms(sd) if unfused else sd
    loaded_ptrs = {p.data_ptr() for n, p in model.state_dict().items() if n in sd}
    untied = [k for k in absent if model.state_dict()[k].data_ptr() not in loaded_ptrs] if not unfused else []
    if untied:
        raise RuntimeError(f"checkpoint {load_path} lacks {untied[:5]} (and they are not aliases of loaded parameters)")
    model.load_state_dict(sd, strict=not absent)
    return model


def main(model_variant, compiled=False, is_old_fms=False, load_path=None, save_path=None, tokenizer_name_or_path=None):
    """Parameter order of the reference (``fms_to_hf_llama.py:133-135``); ``--compiled`` / ``--is_old_fms`` default to False."""
    if load_path is None or save_path is None:
        raise SystemExit("usage: fms_to_hf_llama.py --model_variant V [--compiled] [--is_old_fms] --load_path CKPT --save_path OUT "
                         "[--tokenizer_name_or_path TOK]")
    print("Initializing model...")
    cfg = get_model_config(model_variant)
    with torch.device("meta"):
        model = LLaMA(cfg)
    model.to_empty(device="cpu")
    print(f"Reading state dict from {load_path}")
    load_dcp_into(model, load_path, compiled, is_old_fms)
    print("Converting to HF Qwen2..." if cfg.qkv_bias else "Converting to HF Llama...")
    hf = convert_to_hf(model, model_variant, is_old_fms)
    hf.save_pretrained(save_path)
    print(f"Model saving at {save_path}")
    if tokenizer_name_or_path:
        from transformers import AutoTokenizer
        AutoTokenizer.from_pretrained(tokenizer_name_or_path).save_pretrained(save_path)
    print("Done.")


if __name__ == "__main__":
    run(main)
