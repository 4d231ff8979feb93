"""GPU tier (run on the B200 box with ``pytest -m gpu``): every sm_100a kernel against the plain-PyTorch
fp32 oracle of the same op (``ops/torch_kernels.py``), and the engine on the fused kernels against the ATen
kernel path.  These tests load ``fms_fsdp_b200/_C.so`` -- there is no silent eager fallback."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def K():
    from fms_fsdp_b200.ops import cuda_kernels as CK
    from fms_fsdp_b200.ops import torch_kernels as TK
    assert CK._C.__file__.endswith("_C.so")
    return CK, TK


def rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp(min=1e-6)).item()


DEV = "cuda"


@pytest.mark.parametrize("layout", ["nt", "nn", "tn"])
@pytest.mark.parametrize("shape", [(128, 256, 64), (384, 768, 192), (1000, 520, 72), (2048, 1024, 4096)])
def test_gemm_layouts(K, layout, shape):
    CK, TK = K
    M, N, Kd = shape
    torch.manual_seed(0)
    a = torch.randn((M, Kd) if layout != "tn" else (Kd, M), device=DEV).bfloat16()
    b = torch.randn((N, Kd) if layout == "nt" else (Kd, N), device=DEV).bfloat16()
    n0 = CK.launch_count()
    out = CK.gemm(a, b, layout)
    assert CK.launch_count() == n0 + 1  # our kernel ran, not a library fallback
    assert rel(out, TK.gemm(a.float(), b.float(), layout)) < 1e-2


def test_gemm_epilogues(K):
    CK, TK = K
    a = torch.randn(512, 256, device=DEV).bfloat16(); b = torch.randn(768, 256, device=DEV).bfloat16()
    r = torch.randn(512, 768, device=DEV).bfloat16()
    ref = a.float() @ b.float().t()
    assert rel(CK.gemm(a, b, "nt", residual=r), ref + r.float()) < 1e-2
    c = torch.randn(512, 768, device=DEV); c0 = c.clone()
    CK.gemm(a, b, "nt", out=c, accumulate=True)
    assert rel(c, ref + c0) < 1e-3
    c = torch.randn(512, 768, device=DEV).bfloat16(); c0 = c.clone()
    CK.gemm(a, b, "nt", out=c, accumulate=True)
    assert rel(c, ref + c0.float()) < 1e-2


def test_rmsnorm_rope_swiglu_embedding(K):
    CK, TK = K
    M, D = 512, 4096
    x = torch.randn(M, D, device=DEV).bfloat16(); w = (1 + 0.1 * torch.randn(D, device=DEV)).bfloat16()
    dy = torch.randn(M, D, device=DEV).bfloat16()
    y0, r0 = TK.rmsnorm_fwd(x, w, 1e-5); y1, r1 = CK.rmsnorm_fwd(x, w, 1e-5)
    assert rel(y1, y0) < 1e-2 and rel(r1, r0) < 1e-4
    dx0, dw0 = TK.rmsnorm_bwd(dy, x, w, r0); dx1, dw1 = CK.rmsnorm_bwd(dy, x, w, r1)
    assert rel(dx1, dx0) < 1e-2 and rel(dw1, dw0) < 1e-3
    dres = torch.randn(M, D, device=DEV).bfloat16()     # residual-branch gradient folded into the kernel
    dx2, _ = CK.rmsnorm_bwd(dy, x, w, r1, dres)
    assert rel(dx2, TK.rmsnorm_bwd(dy, x, w, r0, dres)[0]) < 1e-2
    for D2 in (1024, 5120, 8192):                       # other chunk-count instantiations
        x2 = torch.randn(64, D2, device=DEV).bfloat16(); w2 = (1 + 0.1 * torch.randn(D2, device=DEV)).bfloat16()
        d2 = torch.randn(64, D2, device=DEV).bfloat16()
        ya, ra = TK.rmsnorm_fwd(x2, w2, 1e-5); yb, rb = CK.rmsnorm_fwd(x2, w2, 1e-5)
        assert rel(yb, ya) < 1e-2 and rel(rb, ra) < 1e-4
        da, wa = TK.rmsnorm_bwd(d2, x2, w2, ra); db, wb = CK.rmsnorm_bwd(d2, x2, w2, rb)
        assert rel(db, da) < 1e-2 and rel(wb, wa) < 1e-3
    S, H, KVH, hd = 128, 8, 4, 128
    tab = TK.rope_table(S, hd, device=DEV)
    q = torch.randn(2 * S, (H + 2 * KVH) * hd, device=DEV).bfloat16()
    for inter in (True, False):
        assert rel(CK.rope_(q.clone(), tab, S, H, KVH, hd, interleaved=inter), TK.rope_(q.clone(), tab, S, H, KVH, hd, interleaved=inter)) < 1e-2
        rt = CK.rope_(CK.rope_(q.clone(), tab, S, H, KVH, hd, interleaved=inter), tab, S, H, KVH, hd, inverse=True, interleaved=inter)
        assert rel(rt, q) < 2e-2
    tab64 = TK.rope_table(S, 64, device=DEV)
    assert rel(CK.rope_(q.clone(), tab64, S, H, KVH, hd, 64, interleaved=False), TK.rope_(q.clone(), tab64, S, H, KVH, hd, 64, interleaved=False)) < 1e-2
    gu = torch.randn(M, 2 * 1024, device=DEV).bfloat16(); ds = torch.randn(M, 1024, device=DEV).bfloat16()
    for gf in (True, False):
        assert rel(CK.swiglu_fwd(gu, gf), TK.swiglu_fwd(gu, gf)) < 1e-2
        assert rel(CK.swiglu_bwd(ds, gu, gf), TK.swiglu_bwd(ds, gu, gf)) < 1e-2
    V = 4096
    wt = torch.randn(V, D, device=DEV).bfloat16(); tok = torch.randint(0, V, (M,), device=DEV, dtype=torch.int32)
    assert torch.equal(CK.embedding_fwd(tok, wt), TK.embedding_fwd(tok, wt))
    g0 = TK.embedding_bwd(dy, tok, torch.empty(V, D, device=DEV)); g1 = CK.embedding_bwd(dy, tok, torch.empty(V, D, device=DEV))
    assert rel(g1, g0) < 1e-3


def test_linear_cross_entropy(K):
    CK, TK = K
    V, D, M = 8192, 512, 1024
    h = (0.5 * torch.randn(M, D, device=DEV)).bfloat16(); w = (0.05 * torch.randn(V, D, device=DEV)).bfloat16()
    lab = torch.randint(0, V, (M,), device=DEV); lab[::5] = -100
    dw0 = torch.zeros(V, D, device=DEV); dw1 = torch.zeros(V, D, device=DEV, dtype=torch.bfloat16)
    l0, dh0 = TK.linear_ce_fwd_bwd(h.float(), w.float(), lab, dw0)
    l1, dh1 = CK.linear_ce_fwd_bwd(h, w, lab, dw1, chunk_rows=256)
    assert abs(l0.item() - l1.item()) < 2e-3 and rel(dh1, dh0) < 2e-2 and rel(dw1, dw0) < 2e-2


def test_adamw_and_sumsq(K):
    CK, TK = K
    n = 1 << 18
    p = torch.randn(n, device=DEV); g = torch.randn(n, device=DEV).bfloat16()
    m, v = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    lp, lp2 = torch.empty(n, device=DEV, dtype=torch.bfloat16), torch.empty(n, device=DEV, dtype=torch.bfloat16)
    sc = torch.tensor(0.5, device=DEV)
    for step in (1, 2, 3):
        TK.adamw_step(p, g, m, v, lp, 1e-3, 0.9, 0.95, 1e-8, 0.1, step, sc)
        CK.adamw_step(p2, g, m2, v2, lp2, 1e-3, 0.9, 0.95, 1e-8, 0.1, step, sc)
    assert rel(p2, p) < 1e-5 and rel(m2, m) < 1e-5 and rel(v2, v) < 1e-5 and rel(lp2, lp) < 1e-2
    assert abs(CK.sumsq(g).item() / TK.sumsq(g).item() - 1) < 1e-4


@pytest.mark.parametrize("cfg", [(1, 128, 1, 1, 128), (2, 256, 4, 2, 128), (1, 512, 2, 2, 64), (1, 384, 4, 1, 128)])
def test_flash_attention_fwd_bwd(K, cfg):
    CK, TK = K
    B, S, H, KVH, hd = cfg
    torch.manual_seed(1)
    qkv = torch.randn(B * S, (H + 2 * KVH) * hd, device=DEV).bfloat16()
    do = torch.randn(B * S, H * hd, device=DEV).bfloat16()
    sc = hd ** -0.5
    o1, l1 = CK.attn_fwd(qkv, B, S, H, KVH, hd, sc)
    o0, l0 = TK.attn_fwd(qkv, B, S, H, KVH, hd, sc)
    assert rel(o1, o0) < 1e-2 and rel(l1, l0) < 1e-4
    g1 = CK.attn_bwd(do, qkv, o1, l1, B, S, H, KVH, hd, sc)
    g0 = TK.attn_bwd(do, qkv, o0, l0, B, S, H, KVH, hd, sc)
    assert rel(g1, g0) < 1.5e-2


def test_conv1d(K):
    CK, TK = K
    S, C = 200, 512
    x = torch.randn(2 * S, C, device=DEV).bfloat16(); w = (0.5 * torch.randn(C, 4, device=DEV)).bfloat16()
    b = (0.1 * torch.randn(C, device=DEV)).bfloat16(); dy = torch.randn(2 * S, C, device=DEV).bfloat16()
    assert rel(CK.causal_conv1d_fwd(x, w, b, S), TK.causal_conv1d_fwd(x, w, b, S)) < 1e-2
    g0 = TK.causal_conv1d_bwd(dy, x, w, b, S); g1 = CK.causal_conv1d_bwd(dy, x, w, b, S)
    assert rel(g1[0], g0[0]) < 1e-2 and rel(g1[1], g0[1]) < 1e-3 and rel(g1[2], g0[2]) < 1e-3


def test_engine_fused_kernels_match_aten_path():
    """Same model + data: sm_100a kernel path vs ATen path (bf16), loss trajectory and grad norms agree."""
    from fms_fsdp_b200.models.llama import LLaMA, LLaMAConfig
    from fms_fsdp_b200.ops import cuda_kernels as CK
    from fms_fsdp_b200.ops import set_kernel_path
    from fms_fsdp_b200.parallel import ShardedAdamW, ShardedModel
    from fms_fsdp_b200.policies import apply_fsdp_checkpointing, bfSixteen
    from fms_fsdp_b200.models.llama import LLaMABlock

    def run(path):
        set_kernel_path(path)
        torch.manual_seed(0); torch.cuda.manual_seed(0)
        cfg = LLaMAConfig(src_vocab_size=2048, emb_dim=512, nheads=4, kvheads=2, nlayers=3, multiple_of=256, max_expected_seq_len=256)
        with torch.device("meta"):
            m = LLaMA(cfg)
        apply_fsdp_checkpointing(m, LLaMABlock, "1/2")
        eng = ShardedModel(m, mixed_precision=bfSixteen, device=torch.device("cuda", 0))
        opt = ShardedAdamW(eng, lr=1e-3)
        x = torch.randint(0, 2048, (2, 256), generator=torch.Generator().manual_seed(3)).cuda()
        out = []
        for _ in range(4):
            l = eng.forward_backward(x, x); g = eng.clip_grad_norm_(1.0); opt.step(); out.append((l.item(), g.item()))
        return out
    try:
        n0 = CK.launch_count()
        fused = run("fused")
        assert CK.launch_count() - n0 > 100
        aten = run("torch")
    finally:
        set_kernel_path("auto")
    for (lf, gf), (la, ga) in zip(fused, aten):
        assert abs(lf - la) < 3e-2 * abs(la) and abs(gf - ga) < 6e-2 * abs(ga)
    assert fused[-1][0] < fused[0][0]


def test_smoke_entry():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.smoke()


# Real NVLink run (2 ranks).  On one GPU the same kernels are exercised through local pointer tables in
# tests/test_gpu_collectives_1gpu.py.
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_fused_collectives_two_gpus(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541",
                        os.path.join(ROOT, "scripts", "gpu_multi_check.py"), "all", str(tmp_path / "multi_2.json")],
                       env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    import json
    out = json.load(open(tmp_path / "multi_2.json"))
    assert out["allgather_equal"] and out["reduce_scatter_maxdiff"] < 1e-3
    f, t = out["engine_fsdp"]["fused"], out["engine_fsdp"]["torch"]
    assert all(abs(a[1] - b[1]) < 2e-2 * b[1] for a, b in zip(f, t))


@pytest.mark.parametrize("shape", [(2, 256, 8, 64, 1, 128), (1, 384, 8, 64, 2, 64)])
def test_ssd_scan_native_vs_chunked_oracle(K, shape):
    """Mamba2 SSD scan: batched tcgen05 GEMMs + csrc/ssd.cu glue against the fp32 ATen chunked formulation."""
    CK, TK = K
    Bs, S, H, P, G, N = shape
    M = Bs * S
    x = torch.randn(M, H, P, device=DEV).bfloat16().requires_grad_()
    dt = (torch.randn(M, H, device=DEV) * 0.5 - 1.0).bfloat16().requires_grad_()
    A = (-(torch.rand(H, device=DEV) * 4 + 0.5)).requires_grad_()
    Bm = (torch.randn(M, G, N, device=DEV) * 0.3).bfloat16().requires_grad_()
    Cm = (torch.randn(M, G, N, device=DEV) * 0.3).bfloat16().requires_grad_()
    D = torch.randn(H, device=DEV).requires_grad_()
    bias = (torch.randn(H, device=DEV) * 0.2).requires_grad_()
    dy = torch.randn(M, H, P, device=DEV).bfloat16()
    y0 = TK.ssd_scan_chunked(x, dt, A, Bm, Cm, D, bias, S, 128)
    g0 = torch.autograd.grad(y0, [x, dt, A, Bm, Cm, D, bias], dy.float())
    d = lambda t: t.detach()
    y1 = CK.ssd_scan_fwd(d(x), d(dt), d(A), d(Bm), d(Cm), d(D), d(bias), S, 256)
    g1 = CK.ssd_scan_bwd(dy, d(x), d(dt), d(A), d(Bm), d(Cm), d(D), d(bias), S, 256)
    assert g1 is not None, "native SSD path was not taken"
    assert rel(y1, y0) < 2e-2
    for name, a, b in zip(["dx", "ddt", "dA", "dB", "dC", "dD", "dbias"], g1, g0):
        assert rel(a, b) < 3e-2, name


@pytest.mark.parametrize("use_z", [True, False])
def test_selective_scan_native_vs_sequential_oracle(K, use_z):
    """Mamba1 selective scan (csrc/selscan.cu) against the sequential fp32 ATen recurrence."""
    CK, TK = K
    Bs, S, Dm, N = 2, 64, 64, 16
    M = Bs * S
    u = torch.randn(M, Dm, device=DEV).bfloat16().requires_grad_()
    dl = (torch.randn(M, Dm, device=DEV) * 0.5 - 1.0).bfloat16().requires_grad_()
    A = (-(torch.rand(Dm, N, device=DEV) * 4 + 0.5)).requires_grad_()
    Bm = (torch.randn(M, N, device=DEV) * 0.5).bfloat16().requires_grad_()
    Cm = (torch.randn(M, N, device=DEV) * 0.5).bfloat16().requires_grad_()
    D = torch.randn(Dm, device=DEV).requires_grad_()
    bias = (torch.randn(Dm, device=DEV) * 0.2).requires_grad_()
    z = torch.randn(M, Dm, device=DEV).bfloat16().requires_grad_() if use_z else None
    dy = torch.randn(M, Dm, device=DEV).bfloat16()
    y0 = TK.selective_scan_fwd(u, dl, A, Bm, Cm, D, z, bias, S)
    ins = [u, dl, A, Bm, Cm, D] + ([z] if use_z else []) + [bias]
    g0 = list(torch.autograd.grad(y0, ins, dy.float()))
    dd = lambda t: None if t is None else t.detach()
    y1 = CK.selective_scan_fwd(dd(u), dd(dl), dd(A), dd(Bm), dd(Cm), dd(D), dd(z), dd(bias), S)
    g1 = CK.selective_scan_bwd(dy, dd(u), dd(dl), dd(A), dd(Bm), dd(Cm), dd(D), dd(z), dd(bias), S)
    assert g1 is not None, "native selective-scan path was not taken"
    assert rel(y1, y0) < 2e-2
    mine = list(g1[:6]) + ([g1[6]] if use_z else []) + [g1[7]]
    names = ["du", "ddelta", "dA", "dB", "dC", "dD"] + (["dz"] if use_z else []) + ["dbias"]
    for name, a, b in zip(names, mine, g0):
        assert rel(a, b) < 3e-2, name


def test_qkv_attention_rope_fused_in_gemm_and_bwd_epilogues(K):
    """RoPE as the epilogue of the CTA-pair QKV GEMM (forward) and of the dq/dk kernels (backward) against the
    unfused CUDA path (GEMM, in-place RoPE kernel, attention) and its autograd."""
    from fms_fsdp_b200 import ops
    CK, TK = K
    torch.manual_seed(0)
    B, S, D, H, KVH, hd = 2, 256, 512, 4, 2, 128
    tab = TK.rope_table(S, hd, device=DEV)
    h = (torch.randn(B, S, D, device=DEV) * 0.5).bfloat16().requires_grad_()
    w = torch.nn.Parameter((torch.randn((H + 2 * KVH) * hd, D, device=DEV) * 0.05).bfloat16())
    dy = torch.randn(B, S, H * hd, device=DEV).bfloat16()
    y = ops.qkv_attention(h, w, tab, H, KVH, hd)
    y.backward(dy)
    h2 = h.detach().requires_grad_(); w2 = torch.nn.Parameter(w.detach().clone())
    qkv = ops.rope_(ops.linear(h2, w2), tab, S, H, KVH, hd)
    y2 = ops.attention(qkv, H, KVH, hd)
    y2.backward(dy)
    assert rel(y, y2) < 2e-2
    assert rel(h.grad, h2.grad) < 3e-2 and rel(w.grad, w2.grad) < 3e-2


@pytest.mark.parametrize("gate_first", [True, False])
@pytest.mark.parametrize("shape", [(512, 256, 384), (1024, 512, 2816), (8192, 4096, 11008)])
def test_swiglu_fused_into_gemm_epilogues(K, shape, gate_first):
    """SwiGLU as the epilogue of the gate/up GEMM (forward) and of the down-projection dgrad GEMM (backward) against
    the fp32 oracle; the last shape is the Llama2-7B MLP at the benchmark token count."""
    CK, TK = K
    M, D, F = shape
    torch.manual_seed(1)
    x = (torch.randn(M, D, device=DEV) * 0.5).bfloat16()
    w = (torch.randn(2 * F, D, device=DEV) * (D ** -0.5)).bfloat16()
    w2 = (torch.randn(D, F, device=DEV) * (F ** -0.5)).bfloat16()
    dy = (torch.randn(M, D, device=DEV) * 0.5).bfloat16()
    n0 = CK.launch_count()
    gu, act = CK.gated_up_fwd(x, w, gate_first)
    assert CK.launch_count() == n0 + 1, "the fused epilogue was not taken"
    gu0 = x.float() @ w.float().t()
    assert rel(gu, gu0) < 1e-2
    act0 = TK.swiglu_fwd(gu.float(), gate_first)          # activation of the bf16-rounded projection, as the kernel does
    assert rel(act, act0) < 1e-2
    n0 = CK.launch_count()
    dgu = CK.gated_down_bwd(dy, w2, gu, gate_first)
    assert CK.launch_count() == n0 + 1
    dgu0 = TK.swiglu_bwd(dy.float() @ w2.float(), gu.float(), gate_first)
    assert rel(dgu[:, :F], dgu0[:, :F]) < 2e-2 and rel(dgu[:, F:], dgu0[:, F:]) < 2e-2


def test_gated_mlp_node_matches_unfused_ops(K):
    from fms_fsdp_b200 import ops
    torch.manual_seed(2)
    B, S, D, F = 2, 256, 512, 1408                          # F % 128 == 0
    x = (torch.randn(B, S, D, device=DEV) * 0.5).bfloat16().requires_grad_()
    w1 = torch.nn.Parameter((torch.randn(2 * F, D, device=DEV) * 0.04).bfloat16())
    w2 = torch.nn.Parameter((torch.randn(D, F, device=DEV) * 0.03).bfloat16())
    dy = torch.randn(B, S, D, device=DEV).bfloat16()
    y = ops.gated_mlp(x, w1, w2, residual=x)
    y.backward(dy)
    x2 = x.detach().requires_grad_(); a1 = torch.nn.Parameter(w1.detach().clone()); a2 = torch.nn.Parameter(w2.detach().clone())
    y2 = ops.linear(ops.swiglu(ops.linear(x2, a1)), a2, residual=x2)
    y2.backward(dy)
    assert rel(y, y2) < 1e-2
    assert rel(x.grad, x2.grad) < 2e-2 and rel(w1.grad, a1.grad) < 2e-2 and rel(w2.grad, a2.grad) < 2e-2


def test_fp8_rowwise_quant_and_e4m3_gemm(K):
    """Opt-in fp8 forward path: row-wise e4m3 quantisation kernel and the kind::f8f6f4 CTA-pair GEMM against the torch
    float8_e4m3fn oracle (the GEMM is exact on the quantised values up to fp32 summation order and bf16 rounding)."""
    CK, TK = K
    torch.manual_seed(4)
    M, N, Kd = 1024, 768, 512
    x = (torch.randn(M, Kd, device=DEV) * 0.7).bfloat16()
    w = (torch.randn(N, Kd, device=DEV) * 0.05).bfloat16()
    n0 = CK.launch_count()
    xq, sx = CK.quant_rowwise_e4m3(x)
    wq, sw = CK.quant_rowwise_e4m3(w)
    xq0, sx0 = TK.quant_rowwise_e4m3(x)
    assert torch.allclose(sx, sx0, rtol=1e-6)
    dq = xq.view(torch.float8_e4m3fn).float() * sx[:, None]
    assert rel(dq, x) < 0.07                                              # e4m3: 3 mantissa bits
    assert (xq.view(torch.float8_e4m3fn).float() - xq0.view(torch.float8_e4m3fn).float()).abs().max() <= 32  # <= 1 ulp at the top
    y = CK.gemm_fp8(xq, wq, sx, sw)
    assert CK.launch_count() == n0 + 3
    y0 = TK.gemm_fp8(xq, wq, sx, sw)
    assert rel(y, y0) < 1e-2
    assert rel(y, x.float() @ w.float().t()) < 0.08


def test_fp8_linear_trains_like_bf16(K):
    from fms_fsdp_b200 import ops
    from fms_fsdp_b200.ops import functional as Fn
    torch.manual_seed(5)
    x = (torch.randn(2, 256, 512, device=DEV) * 0.5).bfloat16().requires_grad_()
    w = torch.nn.Parameter((torch.randn(1024, 512, device=DEV) * 0.04).bfloat16())
    dy = torch.randn(2, 256, 1024, device=DEV).bfloat16()
    y_ref = ops.linear(x, w)
    Fn.set_gemm_precision("fp8")
    try:
        y = ops.linear(x, w)
        y.backward(dy)
    finally:
        Fn.set_gemm_precision("bf16")
    assert rel(y, y_ref) < 0.08
    x2 = x.detach().requires_grad_(); w2 = torch.nn.Parameter(w.detach().clone())
    ops.linear(x2, w2).backward(dy)
    assert rel(x.grad, x2.grad) < 1e-2 and rel(w.grad, w2.grad) < 1e-2     # the backward is the bf16 backward
