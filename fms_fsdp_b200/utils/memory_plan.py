"""Per-GPU memory plan of a Llama run on this engine -- "does this configuration fit in 180 GB of HBM3e, and what should be
recomputed?" answered before a job is queued.

    python -m fms_fsdp_b200.utils.memory_plan --model_variant=llama2_13b --gpus=8 --sharding_strategy=fsdp \
        --batch_size=2 --seq_length=4096 --selective_checkpointing=1/2

The numbers follow what the runtime allocates (``parallel/engine.py``) and what the autograd nodes of ``ops/functional.py`` save:

* state, per parameter and divided by the shard-group size: fp32 master + bf16 shard + two fp32 AdamW moments (14 B) and the
  fp32 gradient shard (4 B); unsharded (1 GPU / ddp) the gradient stays in the bf16 reduce dtype (2 B);
* gathered parameters: ``prefetch + 1`` block-sized bf16 buffers and the root unit (embedding + head + final norm);
* gradient staging (sharded only): ``push_pool`` block-sized buffers the wgrad GEMMs of all ranks push into, plus the root
  unit's unsharded gradient (pull path);
* activations per block kept for backward (bf16; T = batch * seq tokens): block input, two normed inputs, rotated QKV,
  attention output, post-attention residual, gate|up and SwiGLU output = 2T(6D + 2*KV*hd + 3F) bytes, plus fp32 row
  statistics; a recomputed block keeps its input only, one block's worth of activations is live while it is recomputed;
* head: the final hidden states, their gradient and one [4096, V] logits chunk (+ its gradient in place).

Checked against the measured peak of the caching allocator: Llama2-7B, 1 GPU, no recomputation = 133.53 GiB
(``profiles/bench1_on8box_r2.log``), plan 133.0 GiB (``tests/test_config.py``).  Symmetric-memory buffers of the peer
collectives are not visible to the caching allocator; ``bench.py`` therefore also reports ``mem_device_gb``.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict

GiB = float(2 ** 30)
HBM_GIB_B200 = 180e9 / GiB      # 180 GB of HBM3e (the driver, context and NCCL take a few GiB of it)


@dataclass
class MemoryPlan:
    model_variant: str
    gpus: int
    shard_size: int
    parts_gib: Dict[str, float] = field(default_factory=dict)

    @property
    def total_gib(self) -> float:
        return sum(self.parts_gib.values())

    def fits(self, budget_gib: float = HBM_GIB_B200, headroom: float = 0.92) -> bool:
        """``headroom``: fraction of the device the plan may take (allocator fragmentation, CUDA context, NCCL buffers)."""
        return self.total_gib <= budget_gib * headroom

    def table(self) -> str:
        w = max(len(k) for k in self.parts_gib)
        rows = [f"{k:<{w}}  {v:8.2f} GiB" for k, v in self.parts_gib.items()]
        rows.append(f"{'total':<{w}}  {self.total_gib:8.2f} GiB   ({'fits' if self.fits() else 'DOES NOT FIT'} in "
                    f"{HBM_GIB_B200:.0f} GiB at 92 % usable)")
        return "\n".join(rows)


def _recomputed_blocks(nlayers: int, selective_checkpointing, enabled: bool) -> int:
    """Number of blocks whose activations are recomputed: the selection rule of ``policies/ac_handler.py`` itself."""
    if not enabled:
        return 0
    from fms_fsdp_b200.policies.ac_handler import selection_mask
    return sum(selection_mask(nlayers, selective_checkpointing))


def plan_llama(model_variant: str, gpus: int = 1, sharding_strategy: str = "fsdp", hsdp_shard_size: int = 0,
               batch_size: int = 2, seq_length: int = 4096, fsdp_activation_checkpointing: bool = False,
               selective_checkpointing="1", prefetch: int = 1, push_pool: int = 3, ce_chunk_rows: int = 4096) -> MemoryPlan:
    from fms_fsdp_b200.parallel.mesh import resolve_shard_size
    from fms_fsdp_b200.utils.config_utils import get_model_config

    c = get_model_config(model_variant)
    D, F, V, L, hd = c.emb_dim, c.hidden_dim, c.src_vocab_size, c.nlayers, c.head_dim
    kvd = c.kv_heads * hd
    S = resolve_shard_size(sharding_strategy, gpus, hsdp_shard_size, None)
    T = batch_size * seq_length

    block_params = (c.nheads * hd + 2 * kvd) * D + D * c.nheads * hd + 2 * F * D + D * F + 2 * D
    if c.qkv_bias:
        block_params += c.nheads * hd + 2 * kvd
    root_params = 2 * V * D + D
    n_params = L * block_params + root_params

    parts: Dict[str, float] = {}
    parts["master + bf16 shard + AdamW moments (14 B/param / shard)"] = 14.0 * n_params / S / GiB
    parts["gradient shard (fp32; bf16 when unsharded)"] = (4.0 if S > 1 else 2.0) * n_params / S / GiB
    if S > 1:
        parts[f"gathered parameters ({prefetch + 1} blocks + root, bf16)"] = 2.0 * ((prefetch + 1) * block_params + root_params) / GiB
        parts[f"gradient staging ({push_pool} block buffers + root, bf16)"] = 2.0 * (push_pool * block_params + root_params) / GiB

    per_block = 2.0 * T * (6 * D + 2 * kvd + 3 * F) + 4.0 * T * (2 + c.nheads)    # bf16 tensors + rstd x2 + lse
    n_re = _recomputed_blocks(L, selective_checkpointing, fsdp_activation_checkpointing)
    kept = (L - n_re) * per_block + n_re * 2.0 * T * D + (per_block if n_re else 0.0)
    parts[f"activations ({L - n_re} blocks kept, {n_re} recomputed)"] = kept / GiB
    rows = min(ce_chunk_rows, T)
    parts["head: hidden states + gradient + one logits chunk"] = (2 * 2.0 * T * D + 2.0 * rows * V + 2.0 * T * D) / GiB
    return MemoryPlan(model_variant, gpus, S, parts)


def main(**kw):
    p = plan_llama(**kw)
    print(f"{p.model_variant} on {p.gpus} GPU(s), shard group of {p.shard_size}:")
    print(p.table())
    return p


if __name__ == "__main__":
    from fms_fsdp_b200.utils.cli import run
    run(main)
