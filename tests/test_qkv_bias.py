"""Q/K/V projection biases (``LLaMAConfig.qkv_bias``, the Qwen2 / Qwen2.5 block) on the ATen path: HF loading and export,
gradients, the sharded engine (FSDP + DCP resharding), tensor-parallel speculator bases and the refusals that remain."""
import json
import os
import sys
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import free_port
from fms_fsdp_b200 import ops
from fms_fsdp_b200.models.llama import LLaMA
from fms_fsdp_b200.ops import torch_kernels as TK
from fms_fsdp_b200.parallel import ShardedAdamW, ShardedModel
from fms_fsdp_b200.policies import fp32_policy
from fms_fsdp_b200.utils.config_utils import get_model_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tiny_qwen2(tmp_path, seed=0, **over):
    """A 2-layer ``transformers`` Qwen2 with large random q/k/v biases, saved with ``save_pretrained``."""
    from transformers import Qwen2Config, Qwen2ForCausalLM
    torch.manual_seed(seed)
    kw = dict(vocab_size=512, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=4,
              num_key_value_heads=2, max_position_embeddings=256, sliding_window=256, use_sliding_window=False,
              tie_word_embeddings=False, rope_theta=1e6, rms_norm_eps=1e-6)
    kw.update(over)
    hf = Qwen2ForCausalLM(Qwen2Config(**kw)).eval()
    with torch.no_grad():
        for n, p in hf.named_parameters():
            if n.endswith("bias"):
                p.normal_(0, 0.5)
    d = str(tmp_path / "qwen2")
    hf.save_pretrained(d)
    return hf, d


def _as_hf(model, values):
    """``values`` (our parameter names -> tensors, e.g. gradients) in HF Qwen2 names and layouts: the q/k row / entry
    permutation of the export is linear, so it maps gradients exactly like weights."""
    import fms_to_hf_llama as ex
    twin = LLaMA(model.config)
    twin.load_state_dict(values)
    return dict(ex.convert_to_hf(twin, "qwen2").named_parameters())


def test_qwen2_checkpoint_loads_with_equal_logits_and_gradients(tmp_path):
    from fms_fsdp_b200.models.hf_loader import load_hf_llama
    hf, d = _tiny_qwen2(tmp_path)
    ours = load_hf_llama(d, "cpu", torch.float32).eval()
    assert ours.config.qkv_bias and ours.layers[0].attn.in_proj.qkv_fused.bias.shape == (128 + 2 * 64,)
    x = torch.randint(0, 512, (2, 40))
    want = hf(x).logits
    got = ours(x)
    assert torch.allclose(got, want, atol=3e-4, rtol=1e-3), (got - want).abs().max()
    # gradients of the same loss with respect to every parameter, biases included
    want_loss = torch.nn.functional.cross_entropy(want.view(-1, 512), x.view(-1))
    got_loss = torch.nn.functional.cross_entropy(got.view(-1, 512), x.view(-1))
    want_loss.backward()
    got_loss.backward()
    grads = _as_hf(ours, {n: p.grad for n, p in ours.named_parameters()})
    hf_params = dict(hf.named_parameters())
    assert {n for n in hf_params if n.endswith("bias")} <= set(grads)
    for n, p in hf_params.items():
        assert torch.allclose(grads[n], p.grad, atol=1e-5, rtol=1e-3), (n, (grads[n] - p.grad).abs().max())


def test_qwen2_export_round_trip_and_hf_to_fms_variant_check(tmp_path):
    import fms_to_hf_llama as ex
    import hf_to_fms_llama
    from fms_fsdp_b200.models.hf_loader import load_hf_llama
    hf, d = _tiny_qwen2(tmp_path, seed=1)
    ours = load_hf_llama(d, "cpu", torch.float32).eval()
    back = ex.convert_to_hf(ours, "qwen2").eval()
    assert type(back).__name__ == "Qwen2ForCausalLM" and back.config.use_sliding_window is False
    want_sd, got_sd = hf.state_dict(), back.state_dict()
    assert set(want_sd) == set(got_sd)
    for k, v in want_sd.items():
        assert torch.equal(got_sd[k], v), k
    x = torch.randint(0, 512, (1, 24))
    with torch.no_grad():
        assert torch.allclose(back(x).logits, hf(x).logits, atol=1e-5, rtol=1e-5)
    # the zoo's qwen2_tiny shape: hf_to_fms_llama checks the architecture (qkv_bias included) and writes a checkpoint
    c = get_model_config("qwen2_tiny")
    _, d2 = _tiny_qwen2(tmp_path / "zoo", seed=2, vocab_size=c.src_vocab_size, hidden_size=c.emb_dim,
                        intermediate_size=c.hidden_dim, num_attention_heads=c.nheads, num_key_value_heads=c.kv_heads,
                        max_position_embeddings=c.max_expected_seq_len, sliding_window=c.max_expected_seq_len)
    out = str(tmp_path / "qwen2_tiny.pth")
    hf_to_fms_llama.main(d2, out, model_variant="qwen2_tiny")
    sd = torch.load(out, weights_only=True)["model_state"]
    m = LLaMA(c)
    m.load_state_dict(sd)                     # strict: the biases are there and nothing else is missing
    assert "layers.1.attn.in_proj.qkv_fused.bias" in sd
    with pytest.raises(ValueError, match="qkv_bias"):
        hf_to_fms_llama.main(d2, str(tmp_path / "x.pth"), model_variant="llama2_tiny")


def _edit_config(d, **kv):
    p = os.path.join(d, "config.json")
    with open(p) as f:
        c = json.load(f)
    c.update(kv)
    with open(p, "w") as f:
        json.dump(c, f)


@pytest.mark.parametrize("edit,match", [
    (dict(mlp_bias=True), "MLP biases"),
    (dict(attention_bias=True), "MLP biases"),
    (dict(use_sliding_window=True, sliding_window=64, layer_types=["full_attention", "sliding_attention"]), "sliding-window"),
])
def test_qwen2_loader_still_refuses_what_it_cannot_reproduce(tmp_path, edit, match):
    from fms_fsdp_b200.models.hf_loader import load_hf_llama
    _, d = _tiny_qwen2(tmp_path)
    _edit_config(d, **edit)
    with pytest.raises(NotImplementedError, match=match):
        load_hf_llama(d, "cpu", torch.float32)


def test_full_attention_layer_types_are_not_a_sliding_window():
    from fms_fsdp_b200.models.hf_loader import config_from_hf
    base = dict(model_type="qwen2", hidden_size=64, intermediate_size=128, num_attention_heads=4, num_key_value_heads=2,
                num_hidden_layers=2, vocab_size=64, max_position_embeddings=256, sliding_window=64)
    assert config_from_hf({**base, "layer_types": ["full_attention"] * 2}).qkv_bias
    with pytest.raises(NotImplementedError, match="sliding-window"):
        config_from_hf({**base, "layer_types": ["sliding_attention", "full_attention"]})


def test_llama_typed_checkpoint_with_projection_biases_is_refused(tmp_path):
    """A Llama config with Qwen2 weights (biases present, nothing in the config says so) must not load without them."""
    from fms_fsdp_b200.models.hf_loader import load_hf_llama
    _, d = _tiny_qwen2(tmp_path)
    _edit_config(d, model_type="llama", architectures=["LlamaForCausalLM"])
    with pytest.raises(NotImplementedError, match="q_proj.bias"):
        load_hf_llama(d, "cpu", torch.float32)


def test_bias_ops_match_autograd_of_the_formula():
    torch.manual_seed(0)
    x = torch.randn(2, 6, 32, requires_grad=True)
    w = torch.nn.Parameter(torch.randn(48, 32) * 0.1)
    b = torch.nn.Parameter(torch.randn(48))
    y = ops.linear(x, w, bias=b)
    gy = torch.randn_like(y)
    y.backward(gy)
    x2, w2, b2 = (t.detach().clone().requires_grad_() for t in (x, w, b))
    ref = x2 @ w2.t() + b2
    ref.backward(gy)
    assert torch.allclose(y, ref, atol=1e-5)
    for got, want in ((x.grad, x2.grad), (w.grad, w2.grad), (b.grad, b2.grad)):
        assert torch.allclose(got, want, atol=1e-5)
    # the column sum into an existing bf16 / fp32 buffer
    dy = torch.randn(37, 16)
    for dt, tol in ((torch.float32, 1e-5), (torch.bfloat16, 0.1)):
        out = torch.ones(16, dtype=dt)
        TK.bias_grad(dy, out, accumulate=True)
        assert torch.allclose(out.float(), 1 + dy.sum(0), atol=tol)


def test_qkv_attention_bias_is_added_before_rope():
    torch.manual_seed(1)
    B, S, D, H, KVH, hd = 2, 16, 64, 4, 2, 16
    h = torch.randn(B, S, D, requires_grad=True)
    w = torch.nn.Parameter(torch.randn((H + 2 * KVH) * hd, D) * 0.1)
    b = torch.nn.Parameter(torch.randn((H + 2 * KVH) * hd))
    table = TK.rope_table(S, hd, 10000.0)
    out = ops.qkv_attention(h, w, table, H, KVH, hd, bias=b)
    g = torch.randn_like(out)
    out.backward(g)
    h2, w2, b2 = (t.detach().clone().requires_grad_() for t in (h, w, b))
    qkv = ops.rope_(h2 @ w2.t() + b2, table, S, H, KVH, hd)
    ref = ops.attention(qkv, H, KVH, hd)
    ref.backward(g)
    assert torch.allclose(out, ref, atol=1e-5)
    for got, want in ((h.grad, h2.grad), (w.grad, w2.grad), (b.grad, b2.grad)):
        assert torch.allclose(got, want, atol=1e-4), (got - want).abs().max()


def test_fp8_precision_adds_the_bias_after_the_fp8_gemm():
    from fms_fsdp_b200.ops.functional import set_gemm_precision
    torch.manual_seed(2)
    x = torch.randn(64, 32, dtype=torch.bfloat16)
    w = torch.nn.Parameter((torch.randn(48, 32) * 0.1).bfloat16())
    b = torch.nn.Parameter(torch.randn(48).bfloat16())
    set_gemm_precision("fp8")
    try:
        y8 = ops.linear(x, w, bias=b)
        y8.float().sum().backward()
    finally:
        set_gemm_precision("bf16")
    ref = (x.float() @ w.float().t() + b.float())
    assert (y8.float() - ref).abs().max() < 0.1 * ref.abs().max()
    assert torch.allclose(b.grad.float(), torch.full((48,), 64.0))


def test_reset_parameters_zeroes_the_bias_and_keys_follow_fms_naming():
    m = LLaMA(get_model_config("qwen2_tiny"))
    m.reset_parameters()
    sd = m.state_dict()
    assert [k for k in sd if k.endswith("bias")] == [f"layers.{i}.attn.in_proj.qkv_fused.bias" for i in range(2)]
    assert all(torch.count_nonzero(sd[f"layers.{i}.attn.in_proj.qkv_fused.bias"]) == 0 for i in range(2))
    assert not any(k.endswith("bias") for k in LLaMA(get_model_config("llama2_tiny")).state_dict())


def test_qwen25_7b_meets_the_native_kernel_shape_rules():
    from fms_fsdp_b200.ops.cuda_kernels import push_eligible_shape
    c = get_model_config("qwen2.5_7b")
    assert (c.emb_dim, c.nheads, c.kv_heads, c.nlayers, c.hidden_dim, c.src_vocab_size) == (3584, 28, 4, 28, 18944, 152064)
    assert c.qkv_bias and not c.tie_heads and c.rope_theta == 1e6 and c.norm_eps == 1e-6
    hd = c.head_dim
    assert hd in (64, 128) and c.emb_dim % 8 == 0 and c.emb_dim <= 8192 and c.hidden_dim % 128 == 0
    assert c.src_vocab_size % 8 == 0 and c.nheads % c.kv_heads == 0
    n_qkv = c.nheads * hd + 2 * c.kv_heads * hd
    assert n_qkv % 8 == 0                     # bias epilogue and bias_grad: N % 8
    for shape in ((n_qkv, c.emb_dim), (c.emb_dim, c.nheads * hd), (2 * c.hidden_dim, c.emb_dim), (c.emb_dim, c.hidden_dim),
                  (c.src_vocab_size, c.emb_dim)):
        assert push_eligible_shape(shape), shape


# ------------------------------------------------------------------------------------------ sharded engine (gloo)
STEPS, B, S = 3, 2, 32


def _batch(rank, step, V):
    g = torch.Generator().manual_seed(1000 * step + rank)
    return torch.randint(0, V, (B, S), generator=g)


def _init_model():
    torch.manual_seed(0)
    m = LLaMA(get_model_config("qwen2_tiny"))
    m.reset_parameters()
    with torch.no_grad():                     # a non-zero bias, so that it shapes the forward from the first step
        for blk in m.layers:
            blk.attn.in_proj.qkv_fused.bias.normal_(0, 0.3)
    return m


def _oracle(world):
    m = _init_model()
    V = m.config.src_vocab_size
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, betas=(0.9, 0.95), weight_decay=0.1)
    losses = []
    for st in range(STEPS):
        opt.zero_grad()
        tot = 0.0
        for r in range(world):
            x = _batch(r, st, V)
            l = m(x, labels=x) / world
            l.backward()
            tot += l.item()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
        opt.step()
        losses.append(tot)
    return losses, {k: v.detach().clone() for k, v in m.state_dict().items()}


def _worker(rank, world, port, outdir, ckpt_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from fms_fsdp_b200.utils.checkpointing_utils import Checkpointer
        m = _init_model()
        V = m.config.src_vocab_size
        eng = ShardedModel(m, sharding_strategy="fsdp", mixed_precision=fp32_policy, device="cpu", collective_impl="torch")
        opt = ShardedAdamW(eng, lr=1e-3)
        losses = []
        for st in range(STEPS):
            x = _batch(rank, st, V)
            loss = eng.forward_backward(x, x)
            eng.clip_grad_norm_(1.0)
            opt.step()
            t = loss.clone(); dist.all_reduce(t); losses.append(t.item() / world)
        sd = eng.full_state_dict()
        Checkpointer(ckpt_dir, 5, "fsdp", rank, rank).save(STEPS, eng, opt, None, tokens_seen=7)
        if rank == 0:
            torch.save(dict(losses=losses, sd=sd), os.path.join(outdir, "out.pt"))
    finally:
        dist.barrier()
        dist.destroy_process_group()


def _load_worker(rank, world, port, outdir, ckpt_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from fms_fsdp_b200.utils.checkpointing_utils import Checkpointer
        torch.manual_seed(5)
        m = LLaMA(get_model_config("qwen2_tiny")); m.reset_parameters()
        eng = ShardedModel(m, sharding_strategy="fsdp", mixed_precision=fp32_policy, device="cpu", collective_impl="torch")
        opt = ShardedAdamW(eng, lr=1e-3)
        _, _, _, step, ntok, resuming = Checkpointer(ckpt_dir, 5, "fsdp", rank, rank).load(eng, opt, None, path="")
        sd = eng.full_state_dict()
        if rank == 0:
            torch.save(dict(sd=sd, step=step, ntok=ntok, resuming=resuming), os.path.join(outdir, "loaded.pt"))
    finally:
        dist.barrier()
        dist.destroy_process_group()


def test_engine_trains_qwen2_tiny_like_the_unsharded_model_and_reshards_its_checkpoint_2_to_4():
    outdir, ck = tempfile.mkdtemp(), tempfile.mkdtemp()
    mp.spawn(_worker, args=(2, free_port(), outdir, ck), nprocs=2, join=True)
    out = torch.load(os.path.join(outdir, "out.pt"), weights_only=False)
    losses, sd = _oracle(2)
    assert out["losses"] == pytest.approx(losses, rel=2e-4, abs=2e-4)
    for k, v in sd.items():                   # the biases moved exactly as the unsharded AdamW moved them
        assert torch.allclose(out["sd"][k], v, atol=2e-5, rtol=1e-4), k
    mp.spawn(_load_worker, args=(4, free_port(), outdir, ck), nprocs=4, join=True)
    got = torch.load(os.path.join(outdir, "loaded.pt"), weights_only=False)
    assert (got["step"], got["ntok"], got["resuming"]) == (STEPS, 7, True)
    for k, v in out["sd"].items():
        assert torch.equal(got["sd"][k], v), k


@pytest.mark.parametrize("ac", [None, "1"])
def test_engine_bias_gradient_equals_unsharded_autograd(ac):
    from fms_fsdp_b200.models.llama import LLaMABlock
    from fms_fsdp_b200.policies import apply_fsdp_checkpointing
    m = _init_model()
    ref = _init_model()
    if ac:                                    # selective activation checkpointing: the block forward is recomputed
        apply_fsdp_checkpointing(m, LLaMABlock, ac)
    x = _batch(0, 0, m.config.src_vocab_size)
    eng = ShardedModel(m, mixed_precision=fp32_policy, device="cpu")
    eng.forward_backward(x, x)
    ref(x, labels=x).backward()
    ours = dict(m.named_parameters())
    grads = {}
    for u in eng.units:                       # one process: every unit's gradient "shard" is its whole flat gradient
        for (_, p), slot in zip(u.params, u.layout.slots):
            grads[id(p)] = u.grad_shard[slot.offset:slot.offset + slot.numel].view(slot.shape)
    for i in range(2):
        n = f"layers.{i}.attn.in_proj.qkv_fused.bias"
        want = dict(ref.named_parameters())[n].grad
        assert torch.count_nonzero(want) > 0
        assert torch.allclose(grads[id(ours[n])], want, atol=1e-6, rtol=1e-4), n


# ----------------------------------------------------------------------------------- tensor-parallel speculator base
def _tp_worker(rank, world, port, outdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sys.path.insert(0, os.path.join(ROOT, "speculator"))
        from train_speculator_utils import EmbedLLaMA
        from fms_fsdp_b200.parallel.tensor_parallel import shard_llama_for_tp
        torch.manual_seed(0)
        m = EmbedLLaMA(get_model_config("qwen2_tiny")); m.reset_parameters(); m.eval()
        with torch.no_grad():
            for blk in m.layers:
                blk.attn.in_proj.qkv_fused.bias.normal_(0, 0.5)
        x = torch.randint(0, m.config.src_vocab_size, (2, 12))
        with torch.no_grad():
            ref_logits = m(x)
            l0, cache = m(x[:, :-1], use_cache=True)
            l1, _ = m(x[:, -1:], past_key_value_states=cache, use_cache=True)
            shard_llama_for_tp(m, dist.group.WORLD)
            tp_logits = m(x)
            t0, tcache = m(x[:, :-1], use_cache=True)
            t1, _ = m(x[:, -1:], past_key_value_states=tcache, use_cache=True)
        if rank == 0:
            torch.save(dict(logits=(tp_logits - ref_logits).abs().max().item(), prefill=(t0 - l0).abs().max().item(),
                            decode=(t1 - l1).abs().max().item(), scale=ref_logits.abs().max().item(),
                            bias_len=m.layers[0].attn.in_proj.qkv_fused.bias.numel()), os.path.join(outdir, "out.pt"))
    finally:
        dist.barrier()
        dist.destroy_process_group()


def test_tp2_qwen2_base_model_matches_unsharded():
    outdir = tempfile.mkdtemp()
    mp.spawn(_tp_worker, args=(2, free_port(), outdir), nprocs=2, join=True)
    r = torch.load(os.path.join(outdir, "out.pt"), weights_only=False)
    tol = 1e-4 * max(1.0, r["scale"])
    assert r["logits"] < tol and r["prefill"] < tol and r["decode"] < tol, r
    assert r["bias_len"] == (4 + 2 * 2) * 64 // 2


def test_qwen2_greedy_generation_equals_transformers(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "speculator"))
    from train_speculator_utils import EmbedLLaMA
    from fms_fsdp_b200.models.hf_loader import load_hf_llama
    hf, d = _tiny_qwen2(tmp_path, seed=3)
    ours = load_hf_llama(d, "cpu", torch.float32, model_cls=EmbedLLaMA).eval()
    x = torch.randint(0, 512, (1, 8))
    with torch.no_grad():
        want = hf.generate(x, max_new_tokens=12, do_sample=False, pad_token_id=0)[0, 8:]
        toks = x
        logits, cache = ours(toks, use_cache=True)
        got = []
        for _ in range(12):
            nxt = logits[:, -1].argmax(-1, keepdim=True)
            got.append(nxt)
            logits, cache = ours(nxt, past_key_value_states=cache, use_cache=True)
    assert torch.equal(torch.cat(got, 1)[0], want)
