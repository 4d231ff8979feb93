import pytest

from fms_fsdp_b200.config import train_config
from fms_fsdp_b200.utils.cli import parse_argv
from fms_fsdp_b200.utils.config_utils import get_model_config, list_model_variants, update_config


def test_defaults_match_reference_surface():
    c = train_config()
    assert (c.seq_length, c.batch_size, c.sharding_strategy, c.learning_rate) == (4096, 2, "hsdp", 3e-4)
    assert c.selective_checkpointing == 1 and c.logical_shards == 1024 and c.eos_token == 0
    assert len(c.datasets.split(",")) == 13 == len(c.weights.split(","))


def test_update_config_known_unknown_dotted(capsys):
    c = train_config()
    update_config(c, batch_size=4, **{"train_config.seq_length": 128, "bogus": 1})
    assert c.batch_size == 4 and c.seq_length == 128
    assert "unknown parameter bogus" in capsys.readouterr().out


def test_cli_literal_typing():
    kw = parse_argv(["--batch_size=4", "--learning_rate", "3e-4", "--use_dummy_dataset", "--nolow_cpu_fsdp",
                     "--selective_checkpointing=1/3", "--tracker=None", "--model_variant=llama2_7b"])
    assert kw == dict(batch_size=4, learning_rate=3e-4, use_dummy_dataset=True, low_cpu_fsdp=False,
                      selective_checkpointing="1/3", tracker=None, model_variant="llama2_7b")


def test_model_zoo_shapes():
    c = get_model_config("llama2_7b")
    assert (c.emb_dim, c.nheads, c.kv_heads, c.nlayers, c.hidden_dim) == (4096, 32, 32, 32, 11008)
    c = get_model_config("llama2_70b")
    assert (c.hidden_dim, c.kv_heads) == (28672, 8)
    c = get_model_config("llama3_8b")
    assert (c.hidden_dim, c.src_vocab_size, c.rope_theta) == (14336, 128256, 500000.0)
    assert get_model_config("mamba_9.8b")["attn_layer_idx"] == [9, 18, 27]
    assert "mamba_2.8b" in list_model_variants() and "llama2_tiny" in list_model_variants()
    with pytest.raises(ValueError):
        get_model_config("7b")  # the reference's own default is not a valid key (SURVEY Q1)


def test_param_counts():
    import torch
    from fms_fsdp_b200.models.llama import LLaMA
    with torch.device("meta"):
        m = LLaMA(get_model_config("llama2_7b"))
    assert sum(p.numel() for p in m.parameters()) == 6738415616


def test_grad_dtype_and_precision_switches():
    import torch
    from fms_fsdp_b200.config import train_config
    from fms_fsdp_b200.models.llama import LLaMABlock
    from fms_fsdp_b200.utils.train_utils import get_policies
    cfg = train_config()
    assert get_policies(cfg, 1, LLaMABlock)[0].reduce_dtype == torch.bfloat16
    cfg.grad_dtype = "fp32"
    mp = get_policies(cfg, 1, LLaMABlock)[0]
    assert mp.reduce_dtype == torch.float32 and mp.param_dtype == torch.bfloat16
    cfg.precision = "mxfp8"
    import pytest
    with pytest.raises(NotImplementedError):
        get_policies(cfg, 1, LLaMABlock)


def test_every_llama_zoo_variant_meets_the_native_kernel_shape_rules():
    """The sm_100a kernels have shape preconditions (else a counted ATen fallback, ``ops/cuda_kernels.py``): attention head
    dim 64 / 128, RMSNorm width <= 8192 and % 8, SwiGLU-epilogue hidden dim % 128, LM-head vocab % 8, and every weight matrix
    must be eligible for the wgrad push epilogue.  All reference variants must take the native path."""
    from fms_fsdp_b200.ops.cuda_kernels import push_eligible_shape
    names = [n for n in list_model_variants() if n.startswith("llama") and n != "llama2_tiny"]
    assert len(names) >= 14
    for n in names:
        c = get_model_config(n)
        hd = c.head_dim
        assert hd in (64, 128), n
        assert c.emb_dim % 8 == 0 and c.emb_dim <= 8192, n
        assert c.hidden_dim % 128 == 0, n
        assert c.src_vocab_size % 8 == 0, n
        assert c.nheads % c.kv_heads == 0, n
        for shape in ((c.nheads * hd + 2 * c.kv_heads * hd, c.emb_dim), (c.emb_dim, c.nheads * hd),
                      (2 * c.hidden_dim, c.emb_dim), (c.emb_dim, c.hidden_dim), (c.src_vocab_size, c.emb_dim)):
            assert push_eligible_shape(shape), (n, shape)


def test_memory_plan_matches_the_measured_1gpu_peak_and_scales_with_sharding():
    """``utils/memory_plan.py`` against the one number that is directly comparable: the caching allocator's peak of the
    Llama2-7B 1-GPU bench (133.53 GiB, profiles/bench1_on8box_r2.log)."""
    from fms_fsdp_b200.utils.memory_plan import plan_llama
    p1 = plan_llama("llama2_7b", gpus=1)
    assert abs(p1.total_gib - 133.53) / 133.53 < 0.02, p1.table()
    p8 = plan_llama("llama2_7b", gpus=8)
    assert p8.shard_size == 8 and p8.fits() and p8.total_gib < 0.45 * p1.total_gib
    h = plan_llama("llama2_7b", gpus=8, sharding_strategy="hsdp", hsdp_shard_size=4)
    assert h.shard_size == 4 and h.total_gib > p8.total_gib
    # recomputation trades activations for nothing else; the block counts follow the ac_handler selection rule
    full = plan_llama("llama2_13b", gpus=8)
    half = plan_llama("llama2_13b", gpus=8, fsdp_activation_checkpointing=True, selective_checkpointing="1/2")
    assert any("20 blocks kept, 20 recomputed" in k for k in half.parts_gib) and half.total_gib < full.total_gib
    assert not plan_llama("llama2_70b", gpus=8, fsdp_activation_checkpointing=True).fits()
    assert plan_llama("llama2_70b", gpus=64, sharding_strategy="hsdp", hsdp_shard_size=8).shard_size == 8


def _reference_golden(name):
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", name)) as f:
        return json.load(f)


def test_model_zoo_equals_the_reference_installs_zoo():
    """Every variant the original's ``get_model_config`` knows (tests/golden/reference/model_zoo.json) has identical
    architecture numbers here."""
    theirs = _reference_golden("model_zoo.json")
    variants = sorted(theirs)
    assert len(variants) >= 15
    for v in variants:
        mine = get_model_config(v)
        if isinstance(mine, dict):      # mamba: a plain dict in both
            assert mine == theirs[v], v
            continue
        for k in ("src_vocab_size", "emb_dim", "nheads", "kvheads", "nlayers", "hidden_grow_factor", "multiple_of",
                  "max_expected_seq_len", "rope_theta", "norm_eps"):
            assert getattr(mine, k) == theirs[v][k], (v, k, getattr(mine, k), theirs[v][k])


def test_train_config_defaults_and_dummy_stream_equal_the_reference_install():
    """(1) every ``train_config`` field of the original exists here with the same default; (2) the synthetic
    ``get_dummy_loader`` stream is the same token for token (it is what both bench arms train on).  The original's values
    are in tests/golden/reference/train_config.json."""
    import dataclasses
    theirs = _reference_golden("train_config.json")
    mine = dataclasses.asdict(train_config())
    for k, v in theirs["cfg"].items():
        assert k in mine, f"missing train_config field {k}"
        assert mine[k] == v, (k, mine[k], v)
    from fms_fsdp_b200.utils.dataloader_utils import get_dummy_loader
    c = train_config()
    c.seq_length, c.batch_size, c.vocab_size = 16, 2, 50
    it = iter(get_dummy_loader(c, 1, 4))
    for want in theirs["batches"]:
        got = [t.tolist() for t in next(it)]
        assert got == want
