"""GPU tier of the q/k/v projection bias (``pytest -m gpu``): the bias epilogue of the CTA-pair GEMM (store and RoPE, plain
and with the fused all-gather), the deterministic bias-gradient reduction, ``qkv_attention`` with a bias at the Qwen2.5-7B
head layout (GQA group 7) and at group 5, and a few ``qwen2_tiny`` training steps on the native kernels only."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def K():
    from fms_fsdp_b200.ops import cuda_kernels as CK
    from fms_fsdp_b200.ops import torch_kernels as TK
    assert CK._C.__file__.endswith("_C.so")
    return CK, TK


def rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp(min=1e-6)).item()


def tile_rel(a, b, tile=256):
    """max over 256x256 tiles of (max |a-b| in the tile) / (max |b| in the tile): a wrong low-magnitude tile fails."""
    a, b = a.float(), b.float()
    M, N = b.shape
    worst = 0.0
    for i in range(0, M, tile):
        d = (a[i:i + tile] - b[i:i + tile]).abs()
        r = b[i:i + tile].abs()
        for j in range(0, N, tile):
            worst = max(worst, (d[:, j:j + tile].max() / r[:, j:j + tile].max().clamp(min=1e-6)).item())
    return worst


def table(tensors):
    return torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64, device=DEV)


@pytest.mark.parametrize("shape", [(1000, 520, 256), (8192, 4608, 3584)])
def test_bias_store_epilogue(K, shape):
    CK, TK = K
    M, N, Kd = shape
    torch.manual_seed(0)
    a = torch.randn(M, Kd, device=DEV).bfloat16()
    b = (torch.randn(N, Kd, device=DEV) * 0.05).bfloat16()
    bias = (torch.randn(N, device=DEV) * 2).bfloat16()
    n0, f0 = CK.launch_count(), CK.fallback_count()
    out = CK.gemm(a, b, "nt", bias=bias)
    assert CK.launch_count() == n0 + 1 and CK.fallback_count() == f0
    assert tile_rel(out, a.float() @ b.float().t() + bias.float()) < 1e-2


@pytest.mark.parametrize("heads", [(28, 4), (40, 8)])
def test_bias_rope_epilogue(K, heads):
    CK, TK = K
    H, KVH = heads
    B, S, D, hd = 2, 512, 1024, 128
    torch.manual_seed(1)
    tab = TK.rope_table(S, hd, 1e6, device=DEV)
    h = torch.randn(B * S, D, device=DEV).bfloat16()
    w = (torch.randn((H + 2 * KVH) * hd, D, device=DEV) * 0.05).bfloat16()
    bias = (torch.randn((H + 2 * KVH) * hd, device=DEV) * 2).bfloat16()
    n0, f0 = CK.launch_count(), CK.fallback_count()
    out = CK.gemm(h, w, "nt", rope=(tab, S, hd, H, KVH), bias=bias)
    assert CK.launch_count() == n0 + 1 and CK.fallback_count() == f0
    ref = TK.rope_(h.float() @ w.float().t() + bias.float(), tab, S, H, KVH, hd)
    assert tile_rel(out, ref) < 1e-2
    # the bias goes in before the rotation: adding it after would differ by far more than the rounding
    wrong = TK.rope_(h.float() @ w.float().t(), tab, S, H, KVH, hd) + bias.float()
    assert tile_rel(wrong, ref) > 10 * tile_rel(out, ref)


@pytest.mark.parametrize("rope", [False, True])
@pytest.mark.parametrize("dependent", [True, False])
def test_bias_epilogues_with_fused_all_gather(K, rope, dependent):
    """The all-gather-fused launch (the FSDP training forward): W 'peer' shards are local buffers of one GPU."""
    CK, TK = K
    C = CK._C
    torch.manual_seed(5)
    W, S, hd, H, KVH, Kd = 4, 512, 128, 28, 4, 1024
    N = (H + 2 * KVH) * hd
    M = 2 * S
    total = (N * Kd + 65536) // (W * 64) * (W * 64)
    n = total // W
    shards = [(torch.randn(n, device=DEV) * 0.05).bfloat16() for _ in range(W)]
    ref_full = torch.cat(shards)
    x = torch.randn(M, Kd, device=DEV).bfloat16()
    bias = (torch.randn(N, device=DEV) * 2).bfloat16()
    tab = TK.rope_table(S, hd, 1e6, device=DEV)
    yref = x.float() @ ref_full[:N * Kd].view(N, Kd).float().t() + bias.float()
    if rope:
        yref = TK.rope_(yref, tab, S, H, KVH, hd)
    for r in (0, W - 1):
        full = torch.zeros(total, dtype=torch.bfloat16, device=DEV)
        flags = torch.zeros((total * 2 + 65535) // 65536, dtype=torch.int32, device=DEV)
        Wm = (full if dependent else ref_full)[:N * Kd].view(N, Kd)
        y = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
        if rope:
            C.set_gemm_rope(tab, S, hd, (H + KVH) * hd)
        C.gemm_ag(x, Wm, y, 0, 3 if rope else 0, None, table(shards), full, n * 2, 0, total * 2, W, r, flags, 1, dependent,
                  bias=bias)
        torch.cuda.synchronize()
        assert torch.equal(full, ref_full)
        assert tile_rel(y, yref) < 1e-2


@pytest.mark.parametrize("N", [4608, 8])
@pytest.mark.parametrize("M", [8191, 1, 333])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_bias_grad_matches_fp64_column_sum_and_is_deterministic(K, M, N, out_dtype):
    CK, _ = K
    torch.manual_seed(M + N)
    dy = torch.randn(M, N, device=DEV).bfloat16()
    want = dy.double().sum(0)
    scale = dy.double().abs().sum(0).max().item()
    tol = (2e-6 if out_dtype == torch.float32 else 8e-3) * scale
    n0 = CK.launch_count()
    got = CK.bias_grad(dy, torch.empty(N, dtype=out_dtype, device=DEV))
    assert CK.launch_count() == n0 + 2                       # partial sums + fixed-order reduction, no fallback
    assert (got.double() - want).abs().max().item() <= tol
    again = CK.bias_grad(dy, torch.empty(N, dtype=out_dtype, device=DEV))
    assert torch.equal(got, again)
    base = torch.randn(N, device=DEV).to(out_dtype)
    acc = CK.bias_grad(dy, base.clone(), accumulate=True)
    assert (acc.double() - (want + base.double())).abs().max().item() <= tol + 8e-3 * base.abs().max().item()
    assert torch.equal(acc, CK.bias_grad(dy, base.clone(), accumulate=True))


@pytest.mark.parametrize("cfg", [(1, 4096, 28, 4, 128, 3584), (1, 1024, 40, 8, 128, 1024)])
def test_qkv_attention_with_bias_matches_aten_path(K, cfg):
    """Forward and backward of the one-node projection + RoPE + attention with a bias, against the ATen path on the same
    GPU.  GQA groups 7 (Qwen2.5-7B: 28 / 4) and 5 (40 / 8) are group sizes the other attention tests do not use."""
    from fms_fsdp_b200 import ops
    from fms_fsdp_b200.ops import set_kernel_path
    CK, TK = K
    B, S, H, KVH, hd, D = cfg
    torch.manual_seed(2)
    tab = TK.rope_table(S, hd, 1e6, device=DEV)
    h0 = (torch.randn(B, S, D, device=DEV) * 0.5).bfloat16()
    w0 = (torch.randn((H + 2 * KVH) * hd, D, device=DEV) * 0.03).bfloat16()
    b0 = (torch.randn((H + 2 * KVH) * hd, device=DEV) * 0.5).bfloat16()
    dy = torch.randn(B, S, H * hd, device=DEV).bfloat16()

    def run(path):
        set_kernel_path(path)
        try:
            h = h0.clone().requires_grad_()
            w, b = torch.nn.Parameter(w0.clone()), torch.nn.Parameter(b0.clone())
            y = ops.qkv_attention(h, w, tab, H, KVH, hd, bias=b)
            y.backward(dy)
            torch.cuda.synchronize()
            return y, h.grad, w.grad, b.grad
        finally:
            set_kernel_path("auto")

    f0 = CK.fallback_count()
    native = run("fused")
    assert CK.fallback_count() == f0
    aten = run("torch")
    names = ("out", "dh", "dw", "db")
    tols = (2e-2, 3e-2, 3e-2, 3e-2)
    for name, got, want, tol in zip(names, native, aten, tols):
        assert rel(got, want) < tol, (name, rel(got, want))


def test_qwen2_tiny_trains_on_native_kernels_like_the_aten_path():
    from fms_fsdp_b200.models.llama import LLaMA
    from fms_fsdp_b200.ops import cuda_kernels as CK
    from fms_fsdp_b200.ops import set_kernel_path
    from fms_fsdp_b200.parallel import ShardedAdamW, ShardedModel
    from fms_fsdp_b200.policies import bfSixteen
    from fms_fsdp_b200.utils.config_utils import get_model_config

    def run(path):
        set_kernel_path(path)
        try:
            torch.manual_seed(0); torch.cuda.manual_seed(0)
            m = LLaMA(get_model_config("qwen2_tiny"))
            m.reset_parameters()
            with torch.no_grad():
                for blk in m.layers:
                    blk.attn.in_proj.qkv_fused.bias.normal_(0, 0.3)
            eng = ShardedModel(m, mixed_precision=bfSixteen, device=torch.device("cuda", 0))
            opt = ShardedAdamW(eng, lr=1e-3)
            x = torch.randint(0, 1024, (2, 256), generator=torch.Generator().manual_seed(3)).cuda()
            out = []
            for _ in range(4):
                l = eng.forward_backward(x, x); g = eng.clip_grad_norm_(1.0); opt.step(); out.append((l.item(), g.item()))
            return out
        finally:
            set_kernel_path("auto")

    CK.reset_fallback_count()
    n0 = CK.launch_count()
    fused = run("fused")
    assert CK.fallback_count() == 0, CK.FALLBACKS
    assert CK.launch_count() - n0 > 50
    aten = run("torch")
    for (lf, gf), (la, ga) in zip(fused, aten):
        assert abs(lf - la) < 3e-2 * abs(la) and abs(gf - ga) < 6e-2 * abs(ga)
    assert fused[-1][0] < fused[0][0]
