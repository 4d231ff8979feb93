"""Import a HuggingFace ``LlamaForCausalLM`` (or ``Qwen2ForCausalLM``) directory as a single-file model checkpoint for this
trainer -- the inverse of ``fms_to_hf_llama.py`` (the reference has only the export direction; continued pre-training /
fine-tuning from public weights needs the way back):

    python hf_to_fms_llama.py --hf_path <hf dir> --save_path llama.pth [--model_variant llama2_7b]
    torchrun ... main_training_llama.py --model_variant=llama2_7b --ckpt_load_path=llama.pth ...

The file holds ``{"model_state": {<fms parameter name>: tensor}}`` -- the single-file format ``Checkpointer.load`` accepts
(weights only; step count, optimizer and data-loader state start fresh, as in reference ``checkpointing_utils.py:216-233``).
q/k rows are permuted from HF's half-split RoPE layout to the FMS interleaved-pair layout and q/k/v, gate/up are fused
(``models/hf_loader.convert_hf_state_dict``).  ``--model_variant`` is optional: when given, the HF config is checked against
that entry of the model zoo so that a mismatch is reported here and not as a shape error on 8 GPUs.
"""
import json
import os

import torch

from fms_fsdp_b200.models.hf_loader import _read_hf_tensors, config_from_hf, convert_hf_state_dict
from fms_fsdp_b200.utils.cli import run
from fms_fsdp_b200.utils.config_utils import get_model_config

_CHECKED = ("src_vocab_size", "emb_dim", "nheads", "kv_heads", "nlayers", "hidden_dim", "rope_theta", "rope_scaling",
            "qkv_bias")


def main(hf_path: str, save_path: str, model_variant: str = "", dtype: str = "bf16"):
    with open(os.path.join(hf_path, "config.json")) as f:
        cfg = config_from_hf(json.load(f))
    if model_variant:
        want = get_model_config(model_variant)
        bad = {k: (getattr(cfg, k), getattr(want, k)) for k in _CHECKED if getattr(cfg, k) != getattr(want, k)}
        if bad:
            raise ValueError(f"{hf_path} does not have the architecture of {model_variant}: (checkpoint, zoo) = {bad}")
    torch_dtype = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": torch.float32}[dtype]
    sd = {k: v.to(torch_dtype).contiguous() for k, v in convert_hf_state_dict(_read_hf_tensors(hf_path), cfg).items()}
    os.makedirs(os.path.dirname(os.path.abspath(save_path)), exist_ok=True)
    torch.save({"model_state": sd}, save_path)
    n = sum(v.numel() for v in sd.values())
    print(f"--> wrote {save_path}: {len(sd)} tensors, {n / 1e6:.1f} M parameters, {dtype}")


if __name__ == "__main__":
    run(main)
