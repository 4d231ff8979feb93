"""Config overrides and the model zoo.

Parity: reference ``fms_fsdp/utils/config_utils.py:6-22`` (update_config) and
``:25-189`` (get_model_config).  The zoo is table-driven here; shapes are the
reference's (SURVEY.md App. A) plus the two BASELINE.json additions
``llama2_tiny`` and ``mamba_2.8b``.
"""
from __future__ import annotations

import copy
from typing import Any, Dict

from fms_fsdp_b200.config import train_config
from fms_fsdp_b200.models.llama import LLaMAConfig


def update_config(config, **kwargs):
    """Apply ``--key=value`` overrides. Unknown keys only warn (reference :21-22);
    ``ClassName.field`` addresses a specific config object (reference :14-20)."""
    if isinstance(config, (tuple, list)):
        for c in config:
            update_config(c, **kwargs)
        return
    for key, value in kwargs.items():
        if hasattr(config, key):
            setattr(config, key, value)
            continue
        if "." in key:
            owner, _, attr = key.partition(".")
            if type(config).__name__ == owner:
                if hasattr(config, attr):
                    setattr(config, attr, value)
                else:
                    print(f"Warning: {owner} does not accept parameter: {key}")
            continue
        if isinstance(config, train_config):
            print(f"Warning: unknown parameter {key}")


def _llama3(emb_dim, nheads, nlayers, grow, seq):
    return dict(src_vocab_size=128256, emb_dim=emb_dim, nheads=nheads, kvheads=8, nlayers=nlayers,
                hidden_grow_factor=grow, max_expected_seq_len=seq, rope_theta=500000.0)


_LLAMA_ZOO: Dict[str, Dict[str, Any]] = {
    "llama2_70b": dict(emb_dim=8192, multiple_of=4096, nheads=64, kvheads=8, nlayers=80,
                       hidden_grow_factor=28672 / 8192),
    "llama2_34b": dict(emb_dim=8192, nheads=64, kvheads=8, nlayers=48, hidden_grow_factor=22016 / 8192,
                       max_expected_seq_len=16384, rope_theta=1000000.0),
    "llama2_13b": dict(emb_dim=5120, nheads=40, nlayers=40, hidden_grow_factor=13824 / 5120),
    "llama2_7b": dict(hidden_grow_factor=11008 / 4096, kvheads=32),
    "llama2_1.4b": dict(emb_dim=2048, nheads=16, nlayers=24, hidden_grow_factor=3, kvheads=4),
    "llama3_8b": _llama3(4096, 32, 32, 3.5, 8192),
    "llama3_8b_4k": _llama3(4096, 32, 32, 3.5, 4096),
    "llama3_1.8b": _llama3(2048, 16, 24, 3.5, 8192),
    "llama3_1.8b_4k": _llama3(2048, 16, 24, 3.5, 4096),
    "llama3_3.2b": _llama3(3072, 24, 24, 8 / 3, 8192),
    "llama3_3.2b_4k": _llama3(3072, 24, 24, 8 / 3, 4096),
    "llama3_70b": _llama3(8192, 64, 80, 3.5, 8192),
    "llama3_70b_4k": _llama3(8192, 64, 80, 3.5, 4096),
    "llama3_194m_4k": dict(src_vocab_size=128256, emb_dim=1024, nheads=8, nlayers=10,
                           max_expected_seq_len=4096, rope_theta=500000.0),
    # --- extensions (BASELINE.json config #1; plumbing / CPU-gloo tests)
    "llama2_tiny": dict(src_vocab_size=1024, emb_dim=256, nheads=4, kvheads=4, nlayers=2,
                        hidden_grow_factor=8 / 3, multiple_of=64, max_expected_seq_len=512),
    # --- Qwen2 family: Llama block + q/k/v projection bias (HF Qwen2ForCausalLM).  qwen2.5_7b follows the published
    # config.json (not checked against a downloaded file; hf_to_fms_llama.py --model_variant compares on first use)
    "qwen2.5_7b": dict(src_vocab_size=152064, emb_dim=3584, nheads=28, kvheads=4, nlayers=28,
                       hidden_grow_factor=18944 / 3584, norm_eps=1e-6, max_expected_seq_len=32768,
                       rope_theta=1000000.0, qkv_bias=True),
    "qwen2_tiny": dict(src_vocab_size=1024, emb_dim=256, nheads=4, kvheads=2, nlayers=2, hidden_grow_factor=2,
                       multiple_of=64, norm_eps=1e-6, max_expected_seq_len=512, rope_theta=1000000.0, qkv_bias=True),
}

_MAMBA_ZOO: Dict[str, Dict[str, Any]] = {
    "mamba_9.8b": {
        "d_model": 4096, "d_intermediate": 14336, "n_layer": 32, "vocab_size": 128256,
        "ssm_cfg": {"layer": "Mamba2"},
        "attn_layer_idx": [9, 18, 27],
        "attn_cfg": {"causal": True, "d_conv": 0, "head_dim": 128, "num_heads": 32, "num_heads_kv": 8,
                     "out_proj_bias": False, "qkv_proj_bias": False, "rotary_emb_dim": 64},
        "rms_norm": True, "residual_in_fp32": True, "fused_add_norm": True,
        "pad_vocab_size_multiple": 16, "tie_embeddings": False,
    },
    # --- extension (BASELINE.json config #5): the standard Mamba2-2.7B shape, pure SSM stack
    "mamba_2.8b": {
        "d_model": 2560, "d_intermediate": 0, "n_layer": 64, "vocab_size": 50277,
        "ssm_cfg": {"layer": "Mamba2"}, "attn_layer_idx": [], "attn_cfg": {},
        "rms_norm": True, "residual_in_fp32": True, "fused_add_norm": True,
        "pad_vocab_size_multiple": 16, "tie_embeddings": True,
    },
    # Mamba (v1) stack: selective-scan mixers, no attention, no MLP (plumbing / CPU tests of the Mamba1 layer type)
    "mamba1_tiny": {
        "d_model": 128, "d_intermediate": 0, "n_layer": 3, "vocab_size": 512,
        "ssm_cfg": {"layer": "Mamba1", "d_state": 16}, "attn_layer_idx": [], "attn_cfg": {},
        "rms_norm": True, "residual_in_fp32": True, "fused_add_norm": True,
        "pad_vocab_size_multiple": 16, "tie_embeddings": True,
    },
    "mamba_tiny": {
        "d_model": 128, "d_intermediate": 256, "n_layer": 4, "vocab_size": 512,
        "ssm_cfg": {"layer": "Mamba2", "headdim": 32, "d_state": 32, "chunk_size": 32},
        "attn_layer_idx": [2],
        "attn_cfg": {"causal": True, "d_conv": 0, "head_dim": 32, "num_heads": 4, "num_heads_kv": 2,
                     "out_proj_bias": False, "qkv_proj_bias": False, "rotary_emb_dim": 16},
        "rms_norm": True, "residual_in_fp32": True, "fused_add_norm": True,
        "pad_vocab_size_multiple": 16, "tie_embeddings": False,
    },
}


def get_model_config(model_variant: str):
    """LLaMAConfig for llama* variants, plain dict for mamba* (reference :162-185)."""
    if model_variant in _LLAMA_ZOO:
        return LLaMAConfig(**_LLAMA_ZOO[model_variant])
    if model_variant in _MAMBA_ZOO:
        return copy.deepcopy(_MAMBA_ZOO[model_variant])
    raise ValueError(f"model variant {model_variant} not supported.  Known variants: {', '.join(sorted([*_LLAMA_ZOO, *_MAMBA_ZOO]))}")


def list_model_variants():
    return sorted(_LLAMA_ZOO) + sorted(_MAMBA_ZOO)
