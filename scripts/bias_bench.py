"""Cost of the q/k/v projection bias on one GPU (CUDA events; card name and power limit read in the same run):

* ``bias_grad`` (deterministic column sum of dqkv) at the Qwen2.5-7B training shape: time and achieved HBM bytes/s;
* the QKV + RoPE projection GEMM with and without the bias epilogue at the Qwen2.5-7B and Llama2-7B projection shapes,
  the two variants timed alternately in the same process so that clock and neighbour noise hit both alike.

    python scripts/bias_bench.py [--tokens 8192] [--reps 7] [--iters 50] [--out result.json]

Every timed window launches the same kernel ``--iters`` times back to back: steady-state times.  The GEMM working sets
(170-370 MB) exceed the 126 MB L2; the 75 MB ``dy`` of ``bias_grad`` fits in it, so its bytes/s is partly L2-served.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable ({e!r})"


def time_ms(fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--tokens", type=int, default=8192, help="rows M = batch x seq (bench.py default: 2 x 4096)")
    p.add_argument("--reps", type=int, default=7)
    p.add_argument("--iters", type=int, default=50)
    p.add_argument("--out", default="", help="also write the JSON result to this file")
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bias_bench.py measures GPU kernels; no GPU here")
    from fms_fsdp_b200.ops import cuda_kernels as CK
    from fms_fsdp_b200.ops import torch_kernels as TK
    from fms_fsdp_b200.utils.config_utils import get_model_config
    torch.manual_seed(0)
    M = a.tokens
    res = {"card": card(), "tokens": M, "iters": a.iters, "reps": a.reps}

    # ---- bias gradient at the Qwen2.5-7B QKV width
    q = get_model_config("qwen2.5_7b")
    N = (q.nheads + 2 * q.kv_heads) * q.head_dim
    dy = torch.randn(M, N, device="cuda").bfloat16()
    db = torch.empty(N, device="cuda")
    n0 = CK.launch_count()
    CK.bias_grad(dy, db)
    assert CK.launch_count() == n0 + 2 and CK.fallback_count() == 0
    P = CK._C.bias_grad_partials(M, N)
    t = [time_ms(lambda: CK.bias_grad(dy, db), a.iters) for _ in range(a.reps)]
    ms = statistics.median(t)
    moved = M * N * 2 + 2 * P * N * 4 + N * 4        # dy read, partials written + read, db written
    res["bias_grad"] = {"M": M, "N": N, "partials": P, "ms_median": ms, "ms_all": t, "bytes": moved,
                        "GB_per_s": moved / ms / 1e6}

    # ---- QKV + RoPE projection GEMM, with and without the bias, alternating
    res["qkv_rope_gemm"] = {}
    for name in ("qwen2.5_7b", "llama2_7b"):
        c = get_model_config(name)
        hd, H, KVH, D = c.head_dim, c.nheads, c.kv_heads, c.emb_dim
        N = (H + 2 * KVH) * hd
        S = 4096
        tab = TK.rope_table(S, hd, c.rope_theta, device="cuda")
        x = torch.randn(M, D, device="cuda").bfloat16()
        w = (torch.randn(N, D, device="cuda") * 0.02).bfloat16()
        bias = (torch.randn(N, device="cuda") * 0.1).bfloat16()
        out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
        rope = (tab, S, hd, H, KVH)
        plain = lambda: CK.gemm(x, w, "nt", out=out, rope=rope)              # noqa: E731
        biased = lambda: CK.gemm(x, w, "nt", out=out, rope=rope, bias=bias)  # noqa: E731
        t0, t1 = [], []
        for _ in range(a.reps):
            t0.append(time_ms(plain, a.iters))
            t1.append(time_ms(biased, a.iters))
        assert CK.fallback_count() == 0
        flops = 2.0 * M * N * D
        m0, m1 = statistics.median(t0), statistics.median(t1)
        res["qkv_rope_gemm"][name] = {"M": M, "N": N, "K": D, "ms_no_bias": m0, "ms_bias": m1, "ms_no_bias_all": t0,
                                      "ms_bias_all": t1, "TFLOP_s_no_bias": flops / m0 / 1e9, "TFLOP_s_bias": flops / m1 / 1e9,
                                      "bias_overhead_pct": 100.0 * (m1 - m0) / m0}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
