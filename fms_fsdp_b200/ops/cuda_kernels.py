"""sm_100a primitive set (same signatures as ``torch_kernels``), backed by ``fms_fsdp_b200._C``.

Every function here launches hand-written kernels from ``csrc/`` (tcgen05 GEMM / flash attention,
fused elementwise, peer-memory collectives).  ``launch_count()`` reports how many of OUR kernels
were launched (bench.py's ``gpu_launches``).
"""
from __future__ import annotations

import os

import torch

from fms_fsdp_b200.ops import _ext, torch_kernels

NAME = "cuda"
_C = _ext.require()

_LAYOUT = {"nt": 0, "nn": 1, "tn": 2}
# attention implementation: "tcgen05" (ours) | "sdpa" (library fallback, debugging only)
ATTN_IMPL = os.environ.get("FMS_B200_ATTN_IMPL", "tcgen05")
GEMM_IMPL = os.environ.get("FMS_B200_GEMM_IMPL", "tcgen05")  # "cublas" = library fallback, debugging only
# pairs (of every 4) of softmax exponentials computed on the FMA pipe (packed FFMA2 polynomial) instead of the MUFU
# (measured, profiles/attn_bench_r2.json: the split is performance-neutral -- the row owners are bound by the dependency
# chain S -> exp -> P -> next MMA, not by MUFU throughput -- so the defaults stay at 0 / 1)
_C.set_attn_poly(int(os.environ.get("FMS_B200_ATTN_POLY_FWD", "0")), int(os.environ.get("FMS_B200_ATTN_POLY_BWD", "1")))
_C.set_gemm_2cta(os.environ.get("FMS_B200_GEMM_2CTA", "1") == "1")  # CTA-pair (cta_group::2) GEMM for M >= 256


def launch_count() -> int:
    return int(_C.launch_count())


# Calls that did NOT run one of our kernels but the ATen oracle (unsupported dtype / alignment).  Never silent: the
# first fallback of each op prints one line, every one is counted; bench.py reports the count of its timed region and
# flags a non-zero value.
FALLBACKS: dict = {}


def _fallback(op: str, why: str = ""):
    n = FALLBACKS.get(op, 0)
    FALLBACKS[op] = n + 1
    if n == 0 and os.environ.get("FMS_B200_QUIET_FALLBACK", "0") != "1":
        print(f"[fms_fsdp_b200] '{op}' ran on the ATen fallback{(' (' + why + ')') if why else ''}; "
              "counted in cuda_kernels.FALLBACKS", flush=True)
    return torch_kernels


def fallback_count() -> int:
    return sum(FALLBACKS.values())


def reset_fallback_count():
    FALLBACKS.clear()


def reset_launch_count():
    _C.reset_launch_count()


def _bf16c(t):
    if t.dtype != torch.bfloat16:
        t = t.to(torch.bfloat16)
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------- fused all-gather requests (ag_gemm)
# The sharded runtime queues "gather this unit's parameters" requests; the next eligible GEMM launched on the
# compute stream carries one inside its own kernel (comm warps pulling peer shards over NVLink while the tensor
# core works).  dependent requests (the GEMM's own weight is being gathered) make the TMA producer wait on
# per-chunk ready flags; others are next-unit prefetches.  Anything left over is flushed as a standalone gather.
_AG_QUEUE = []
AG_STATS = {"fused": 0, "flushed": 0, "carrier_gemms": 0}
# A prefetch request is spread over the GEMMs that follow: each carries (its own weight size x AG_SPLIT) bytes of the
# next unit, i.e. bytes proportional to its FLOPs, so a whole unit is in flight for the duration of one block's forward
# instead of stretching a single GEMM (measured on 2 GPUs: 590 -> 924 us when one QKV GEMM carried all 404 MB).
# 0 = old behaviour (one GEMM carries the whole request).
AG_SPLIT = float(os.environ.get("FMS_B200_AG_SPLIT", "1.0"))
_AG_CHUNK = 65536


def push_ag_request(req: dict):
    req["consumed"] = False
    _AG_QUEUE.append(req)


def _standalone_gather(req):
    _C.p2p_gather_range(req["table"], req["full"], req["shard_bytes"], req["begin"], req["end"])
    req["consumed"] = True
    AG_STATS["flushed"] += 1


def flush_ag_request(req=None):
    """Run pending request(s) as plain range gathers (no GEMM came along to carry them)."""
    for r in list(_AG_QUEUE):
        if req is None or r is req:
            _AG_QUEUE.remove(r)
            if not r["consumed"]:
                _standalone_gather(r)


def _try_fused_gather(a, b, layout, out, epi, residual, bias=None) -> bool:
    if not _AG_QUEUE:
        return False
    req = _AG_QUEUE[0]
    M = a.shape[1] if layout == "tn" else a.shape[0]
    ok = (M >= 256 and out.dtype == torch.bfloat16 and _C.get_gemm_2cta()
          and ((layout in ("nt", "nn") and epi in (0, 1)) or (layout == "tn" and epi in (0, 2, 4))
               or (layout == "nt" and epi == 5 and not req["dependent"]) or (layout == "nn" and epi == 6)
               or (layout == "nt" and epi == 3)))
    if ok and req["dependent"]:
        lo = req["full"].data_ptr() + req["begin"]
        ok = lo <= b.data_ptr() < req["full"].data_ptr() + req["end"]
    if not ok:
        if req["dependent"]:          # this GEMM may read the weights right now: they must be there
            _AG_QUEUE.pop(0)
            _standalone_gather(req)
        return False
    begin, end = req["begin"], req["end"]
    hi = end
    split = req.get("split", AG_SPLIT)
    if split > 0 and not req["dependent"]:
        w = out if layout == "tn" else b                       # the weight-shaped operand of this GEMM
        take = int(w.numel() * w.element_size() * split)
        take = max(_AG_CHUNK, (take + _AG_CHUNK - 1) // _AG_CHUNK * _AG_CHUNK)
        hi = min(end, begin + take)
    _C.gemm_ag(a, b, None if epi == 4 else out, _LAYOUT[layout], epi, residual, req["table"], req["full"], req["shard_bytes"], begin,
               hi, req["world"], req["rank"], req["flags"], req["epoch"], bool(req["dependent"]),
               **({} if bias is None else {"bias": bias}))
    AG_STATS["carrier_gemms"] += 1
    if hi >= end:
        _AG_QUEUE.pop(0)
        req["consumed"] = True
        AG_STATS["fused"] += 1
    else:
        req["begin"] = hi                                      # the remainder rides on the following GEMMs
    return True


class PushTarget:
    """"Output" of a wgrad GEMM whose epilogue writes every tile into the staging slots of the rank that owns that
    slice of the unit's flat gradient (fused GEMM -> reduce-scatter, SURVEY.md N8; ``csrc/gemm2_sm100.cu`` P_EPI_PUSH).
    ``table``: int64 device tensor of the ranks' staging-buffer addresses; ``n``: elements per shard; ``off``: element
    offset of this weight inside the flat unit."""
    __slots__ = ("table", "n", "off", "rank", "shape", "dtype", "world")

    def __init__(self, table, n, off, rank, shape, device=None, world=1):
        self.table, self.n, self.off, self.rank, self.shape = table, int(n), int(off), int(rank), tuple(shape)
        self.dtype, self.world = torch.bfloat16, int(world)

    def numel(self):
        return self.shape[0] * self.shape[1]

    def element_size(self):
        return 2


# 1 = rows leave the SM as 128-byte cp.async.bulk stores staged through shared memory; 0 = 16-byte st.global per lane
PUSH_BULK = os.environ.get("FMS_B200_PUSH_BULK", "1") == "1"
# every rank starts its tile sweep rank/world of the way into the raster, so the ranks push to different owners at any time
PUSH_ROTATE = os.environ.get("FMS_B200_PUSH_ROTATE", "1") == "1"
PUSH_STATS = {"gemms": 0, "with_gather": 0}


def push_eligible_shape(shape) -> bool:
    """Weight shapes the push epilogue handles (CTA-pair wgrad GEMM, 16-byte vectors never straddle an owner)."""
    return len(shape) == 2 and shape[0] >= 256 and shape[0] % 8 == 0 and shape[1] % 8 == 0


def _gemm_push(a, b, tgt: PushTarget):
    M, N = a.shape[1], b.shape[1]
    if (a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16 or (M, N) != tgt.shape or not push_eligible_shape((M, N))
            or not _C.get_gemm_2cta() or a.shape[0] % 8):
        raise RuntimeError(f"wgrad {tuple(a.shape)}^T x {tuple(b.shape)} cannot use the push epilogue")
    a = a if a.stride(-1) == 1 else a.contiguous()
    b = b if b.stride(-1) == 1 else b.contiguous()
    _C.set_gemm_push(tgt.table, tgt.n, tgt.off, tgt.rank, PUSH_BULK, tgt.world if PUSH_ROTATE else 1)
    PUSH_STATS["gemms"] += 1
    if _AG_QUEUE and _try_fused_gather(a, b, "tn", tgt, 4, None):
        PUSH_STATS["with_gather"] += 1      # the same kernel pushes its tiles out and pulls the next unit's weights in
        return tgt
    _C.gemm_push(a, b)
    return tgt


# ------------------------------------------------------------------------------------------ GEMM
def _bias_fusable(a, b, layout, out, accumulate, residual, out_dtype, bias):
    """Shapes the bias epilogue takes: CTA-pair nt GEMM with a bf16 output and a contiguous, 16-byte aligned bf16 bias."""
    return (GEMM_IMPL == "tcgen05" and layout == "nt" and a.dtype == b.dtype == bias.dtype == torch.bfloat16
            and residual is None and not accumulate and a.shape[0] >= 256 and _C.get_gemm_2cta()
            and out_dtype in (None, torch.bfloat16) and (out is None or out.dtype == torch.bfloat16)
            and bias.dim() == 1 and bias.numel() == b.shape[0] and bias.is_contiguous() and bias.data_ptr() % 16 == 0)


def gemm(a, b, layout="nt", out=None, accumulate=False, residual=None, out_dtype=None, rope=None, bias=None):
    """``rope=(table [S, hd/2, 2] fp32, S, hd, H, KVH)``: rotary embedding of the q and k heads (the first
    ``(H + KVH) * hd`` output columns) fused into the GEMM epilogue (QKV projection; nt layout).
    ``bias`` [N] bf16 (nt): added in fp32 to the accumulator before the RoPE rotation / store (P_EPI_BIAS)."""
    if isinstance(out, PushTarget):
        if layout != "tn" or accumulate or residual is not None or bias is not None:
            raise RuntimeError("the push epilogue is a plain tn (wgrad) store")
        return _gemm_push(a, b, out)
    if bias is not None and not _bias_fusable(a, b, layout, out, accumulate, residual, out_dtype, bias):
        return _fallback("gemm_bias").gemm(a, b, layout, out=out, accumulate=accumulate, residual=residual,
                                           out_dtype=out_dtype, rope=rope, bias=bias)
    if rope is not None:
        M0 = a.shape[0]
        ok = (GEMM_IMPL == "tcgen05" and layout == "nt" and a.dtype == b.dtype == torch.bfloat16 and residual is None
              and not accumulate and M0 >= 256 and M0 % 8 == 0 and _C.get_gemm_2cta() and rope[2] % 8 == 0
              and a.shape[1] % 8 == 0 and b.shape[0] % 8 == 0 and out_dtype in (None, torch.bfloat16)
              and (out is None or out.dtype == torch.bfloat16))
        if not ok:   # unfused: GEMM, then the in-place RoPE kernel
            y = gemm(a, b, layout, out=out, accumulate=accumulate, residual=residual, out_dtype=out_dtype, bias=bias)
            table, S, hd, H, KVH = rope
            return rope_(y, table, S, H, KVH, hd)
    if GEMM_IMPL != "tcgen05" or a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16:
        return _fallback("gemm").gemm(a, b, layout, out=out, accumulate=accumulate, residual=residual, out_dtype=out_dtype)
    if layout == "nt":
        M, N = a.shape[0], b.shape[0]
    elif layout == "nn":
        M, N = a.shape[0], b.shape[1]
    else:
        M, N = a.shape[1], b.shape[1]
    K = a.shape[1] if layout != "tn" else a.shape[0]
    if (M % 8) or (N % 8) or (K % 8):
        return _fallback("gemm").gemm(a, b, layout, out=out, accumulate=accumulate, residual=residual, out_dtype=out_dtype,
                                      bias=bias)
    if a.stride(-1) != 1:
        a = a.contiguous()
    if b.stride(-1) != 1:
        b = b.contiguous()
    if out is None:
        out = torch.empty(M, N, dtype=out_dtype or a.dtype, device=a.device)
    epi = 0
    if residual is not None:
        if accumulate:
            raise ValueError("residual and accumulate are mutually exclusive")
        epi = 1
    elif accumulate:
        epi = 2
    if rope is not None:
        epi = 3
        _C.set_gemm_rope(rope[0], int(rope[1]), int(rope[2]), int((rope[3] + rope[4]) * rope[2]))   # for the launch below
    if _AG_QUEUE and _try_fused_gather(a, b, layout, out, epi, residual, bias):
        return out
    _C.gemm(a, b, out, _LAYOUT[layout], epi, residual, **({} if bias is None else {"bias": bias}))
    return out


def bias_grad(dy, out, accumulate=False):
    """out[n] (+)= sum_m dy[m, n]: deterministic two-pass column sum (csrc/elementwise.cu bias_grad_*_kernel)."""
    dy2 = dy.reshape(-1, dy.shape[-1])
    if (dy2.dtype != torch.bfloat16 or dy2.shape[1] % 8 or out.dtype not in (torch.bfloat16, torch.float32)
            or not out.is_contiguous() or out.numel() != dy2.shape[1]):
        return _fallback("bias_grad").bias_grad(dy, out, accumulate)
    dy2 = dy2 if dy2.is_contiguous() and dy2.data_ptr() % 16 == 0 else dy2.contiguous()
    _C.bias_grad(dy2, out, bool(accumulate))
    return out


# -------------------------------------------------------- gate/up GEMM + SwiGLU, down-proj dgrad + SwiGLU backward
FUSE_SWIGLU = os.environ.get("FMS_B200_FUSE_SWIGLU", "1") == "1"
# Measured on Llama2-7B, 1 GPU, same box (profiles/step_kernel_table_1gpu_swiglu_{fused,unfused}_r2.txt, ab_1gpu_swiglu_*):
# forward fusion +97 us in the gate/up GEMM, -112 us activation kernel.  The first backward epilogue read gate/up in
# 32-column steps (every 128-byte line fetched twice, loads issued after the TMEM wait): 904 us vs 560 + 155 us unfused;
# with 64-column steps and the loads issued before the TMEM wait the step time equals the unfused one (329.7 vs 329.4 ms)
# while dS [M, F] never reaches memory -- on by default.
FUSE_SWIGLU_BWD = os.environ.get("FMS_B200_FUSE_SWIGLU_BWD", "1") == "1"


def _swiglu_fusable(x, F):
    return (FUSE_SWIGLU and GEMM_IMPL == "tcgen05" and x.dtype == torch.bfloat16 and x.shape[0] >= 256 and x.shape[0] % 8 == 0
            and _C.get_gemm_2cta())


def gated_up_fwd(x, w, gate_first=True):
    """(gu [M, 2F] bf16, silu(gate) * up [M, F]): the activation is the EPILOGUE of the gate/up GEMM -- a CTA pair's
    accumulator holds gate and up of the same 128 features side by side (csrc/gemm2_sm100.cu P_EPI_SWIGLU)."""
    F = w.shape[0] // 2
    if not (_swiglu_fusable(x, F) and w.dtype == torch.bfloat16 and F % 128 == 0 and x.shape[1] % 8 == 0):
        gu = gemm(x, w, "nt")
        return gu, swiglu_fwd(gu, gate_first)
    x = x if x.stride(-1) == 1 else x.contiguous()
    w = w if w.stride(-1) == 1 else w.contiguous()
    gu = torch.empty(x.shape[0], 2 * F, dtype=torch.bfloat16, device=x.device)
    act = torch.empty(x.shape[0], F, dtype=torch.bfloat16, device=x.device)
    _C.set_gemm_swiglu(act, F, bool(gate_first))
    if _AG_QUEUE and _try_fused_gather(x, w, "nt", gu, 5, None):
        return gu, act
    _C.gemm(x, w, gu, 0, 5, None)
    return gu, act


def gated_down_bwd(dy, w2, gu, gate_first=True):
    """d(gu) [M, 2F] = swiglu_bwd(dy @ w2, gu) with the SwiGLU backward as the epilogue of the dgrad GEMM: dS = dy @ w2
    never reaches memory (csrc/gemm2_sm100.cu P_EPI_SWIGLU_BWD)."""
    F = w2.shape[1]
    if not (FUSE_SWIGLU_BWD and _swiglu_fusable(dy, F) and w2.dtype == gu.dtype == torch.bfloat16 and F % 8 == 0 and dy.shape[1] % 8 == 0
            and gu.is_contiguous()):
        return swiglu_bwd(gemm(dy, w2, "nn"), gu, gate_first)
    dy = dy if dy.stride(-1) == 1 else dy.contiguous()
    w2 = w2 if w2.stride(-1) == 1 else w2.contiguous()
    dgu = torch.empty_like(gu)
    _C.set_gemm_swiglu(gu, F, bool(gate_first))
    if _AG_QUEUE and _try_fused_gather(dy, w2, "nn", dgu, 6, None):
        return dgu
    _C.gemm(dy, w2, dgu, 1, 6, None)
    return dgu


# ------------------------------------------------------------------------ optional fp8 (e4m3) forward GEMMs
def quant_rowwise_e4m3(x):
    if x.dtype != torch.bfloat16 or x.dim() != 2 or x.shape[1] % 16 or x.stride(-1) != 1:
        return _fallback("quant_rowwise_e4m3").quant_rowwise_e4m3(x)
    q, sc = _C.quant_rowwise_e4m3(x)
    return q, sc


def gemm_fp8(aq, bq, sa, sb, out=None):
    """e4m3 x e4m3 -> bf16 on the tensor cores (tcgen05.mma kind::f8f6f4, CTA pair), row / column scales in the epilogue."""
    M, K = aq.shape
    N = bq.shape[0]
    if out is None:
        out = torch.empty(M, N, dtype=torch.bfloat16, device=aq.device)
    if K % 16 or N % 8 or not _C.get_gemm_2cta():
        return _fallback("gemm_fp8").gemm_fp8(aq, bq, sa, sb, out)
    _C.gemm_fp8(aq, bq, sa, sb, out)
    return out


# --------------------------------------------------------------------------------------- RMSNorm
def rmsnorm_fwd(x, w, eps):
    if x.dtype != torch.bfloat16 or x.shape[-1] % 8 or x.shape[-1] > 8192:
        return _fallback("rmsnorm_fwd").rmsnorm_fwd(x, w, eps)
    y, rstd = _C.rmsnorm_fwd(x.contiguous(), _bf16c(w), float(eps))
    return y, rstd


def rmsnorm_bwd(dy, x, w, rstd, dres=None):
    """``dres``: optional gradient of the residual branch that forked off ``x``; summed into dx inside the kernel."""
    if dres is not None and (x.dtype != torch.bfloat16 or dres.dtype != torch.bfloat16 or x.shape[-1] % 8 or x.shape[-1] > 8192):
        dx, dw = rmsnorm_bwd(dy, x, w, rstd)
        return dx + dres.reshape(dx.shape).to(dx.dtype), dw
    if x.dtype == torch.float32 and dy.dtype == torch.bfloat16 and x.shape[-1] % 8 == 0 and x.shape[-1] <= 8192:
        dx, dw = _C.rmsnorm_bwd_f32(dy.contiguous(), x.contiguous(), _bf16c(w), rstd)   # fp32 residual stream
        return dx, dw
    if x.dtype != torch.bfloat16 or x.shape[-1] % 8 or x.shape[-1] > 8192:
        return _fallback("rmsnorm_bwd").rmsnorm_bwd(dy, x, w, rstd)
    dx, dw = _C.rmsnorm_bwd(dy.contiguous(), x.contiguous(), _bf16c(w), rstd,
                            None if dres is None else dres.reshape(x.shape).contiguous())
    return dx, dw


def add_rmsnorm_fwd(x, res, w, eps):
    if x.dtype != torch.bfloat16 or res.dtype != torch.float32 or x.shape[-1] % 8 or x.shape[-1] > 8192:
        return _fallback("add_rmsnorm_fwd").add_rmsnorm_fwd(x, res, w, eps)
    y, res_out, rstd = _C.add_rmsnorm_fwd(x.contiguous(), res.contiguous(), _bf16c(w), float(eps))
    return y, res_out, rstd


def rmsnorm_gated_fwd(x, z, w, eps, group_size):
    D = x.shape[-1]
    if x.dtype != torch.bfloat16 or group_size != D or D % 8 or D > 8192:
        return _fallback("rmsnorm_gated_fwd").rmsnorm_gated_fwd(x, z, w, eps, group_size)
    y, rstd = _C.rmsnorm_gated_fwd(x.contiguous(), z.contiguous(), _bf16c(w), float(eps))
    return y, rstd.view(-1, 1)


def rmsnorm_gated_bwd(dy, x, z, w, rstd, group_size):
    D = x.shape[-1]
    if x.dtype != torch.bfloat16 or group_size != D or D % 8 or D > 8192:
        return _fallback("rmsnorm_gated_bwd").rmsnorm_gated_bwd(dy, x, z, w, rstd, group_size)
    dx, dz, dw = _C.rmsnorm_gated_bwd(dy.contiguous(), x.contiguous(), z.contiguous(), _bf16c(w), rstd.reshape(-1))
    return dx, dz, dw

# ------------------------------------------------------------------------------------------ RoPE
rope_table = torch_kernels.rope_table


def rope_(qkv, table, seq_len, nheads, kvheads, head_dim, rot_dim=None, inverse=False, pos_offset=0, interleaved=True):
    rot_dim = head_dim if rot_dim is None else rot_dim
    if qkv.dtype != torch.bfloat16 or rot_dim % 16 or head_dim % 8:
        return _fallback("rope_").rope_(qkv, table, seq_len, nheads, kvheads, head_dim, rot_dim, inverse, pos_offset,
                                   interleaved)
    _C.rope(qkv, table, seq_len, nheads + kvheads, head_dim, rot_dim, bool(inverse), pos_offset, bool(interleaved))
    return qkv


# ------------------------------------------------------------------------------------- attention
def _sdpa_fwd(qkv, B, S, H, KVH, hd, scale):
    q, k, v = torch_kernels._split_qkv(qkv, B, S, H, KVH, hd)
    q, k, v = (t.transpose(1, 2) for t in (q, k, v))
    o = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=True, scale=scale, enable_gqa=(KVH != H))
    return o.transpose(1, 2).reshape(B * S, H * hd).contiguous()


def attn_fwd(qkv, B, S, H, KVH, hd, scale, causal=True):
    if ATTN_IMPL == "tcgen05" and qkv.dtype == torch.bfloat16 and hd in (64, 128) and causal:
        o, lse = _C.attn_fwd(qkv.contiguous(), B, S, H, KVH, hd, float(scale))
        return o, lse
    if ATTN_IMPL == "sdpa":
        return _sdpa_fwd(qkv, B, S, H, KVH, hd, scale), torch.empty(0, device=qkv.device)
    return _fallback("attn_fwd").attn_fwd(qkv, B, S, H, KVH, hd, scale, causal)


def attn_bwd(do, qkv, o, lse, B, S, H, KVH, hd, scale, causal=True, rope_table=None):
    """``rope_table``: the forward applied RoPE (full head_dim, interleaved) to q, k before this attention; return the
    gradient of the UN-rotated projection (inverse rotation fused into the dq / dk epilogues)."""
    if ATTN_IMPL == "tcgen05" and qkv.dtype == torch.bfloat16 and hd in (64, 128) and causal:
        return _C.attn_bwd(do.contiguous(), qkv.contiguous(), o, lse, B, S, H, KVH, hd, float(scale), rope_table)
    if rope_table is not None:
        g = attn_bwd(do, qkv, o, lse, B, S, H, KVH, hd, scale, causal)
        return rope_(g, rope_table, S, H, KVH, hd, inverse=True)
    if ATTN_IMPL == "sdpa":
        with torch.enable_grad():
            leaf = qkv.detach().requires_grad_(True)
            out = _sdpa_fwd(leaf, B, S, H, KVH, hd, scale)
            (g,) = torch.autograd.grad(out, leaf, do)
        return g
    return _fallback("attn_bwd").attn_bwd(do, qkv, o, lse, B, S, H, KVH, hd, scale, causal)


# ---------------------------------------------------------------------------------------- SwiGLU
def swiglu_fwd(gu, gate_first=True):
    if gu.dtype != torch.bfloat16 or (gu.shape[-1] // 2) % 8:
        return _fallback("swiglu_fwd").swiglu_fwd(gu, gate_first)
    return _C.swiglu_fwd(gu.contiguous(), bool(gate_first))


def swiglu_bwd(ds, gu, gate_first=True):
    if gu.dtype != torch.bfloat16 or (gu.shape[-1] // 2) % 8:
        return _fallback("swiglu_bwd").swiglu_bwd(ds, gu, gate_first)
    return _C.swiglu_bwd(ds.contiguous(), gu.contiguous(), bool(gate_first))


# ------------------------------------------------------------------------------------- embedding
def embedding_fwd(tokens, w):
    if w.dtype != torch.bfloat16 or w.shape[1] % 8:
        return _fallback("embedding_fwd").embedding_fwd(tokens, w)
    return _C.embedding_fwd(tokens.contiguous(), w)


def embedding_bwd(dx, tokens, out, accumulate=False):
    if dx.dtype != torch.bfloat16 or dx.shape[-1] % 2 or out.dtype not in (torch.bfloat16, torch.float32):
        return _fallback("embedding_bwd").embedding_bwd(dx, tokens, out, accumulate)
    if not accumulate:
        out.zero_()
    _C.embedding_bwd(dx.contiguous(), tokens.contiguous(), out)
    return out


# ---------------------------------------------------------------------------- fused linear + CE
def linear_ce_fwd_bwd(h, w, labels, dw_out, ignore_index=-100, chunk_rows=4096, accumulate=False):
    M, D = h.shape
    V = w.shape[0]
    if h.dtype != torch.bfloat16 or V % 8 or D % 8 or M % 8:
        return _fallback("linear_ce_fwd_bwd").linear_ce_fwd_bwd(h, w, labels, dw_out, ignore_index, chunk_rows, accumulate)
    labels = labels.reshape(-1)
    if labels.dtype != torch.long:
        labels = labels.long()
    n_valid = torch.zeros((), dtype=torch.float32, device=h.device)
    loss_sum = torch.zeros((), dtype=torch.float32, device=h.device)
    _C.count_valid(labels, ignore_index, n_valid)
    dh = torch.empty_like(h)
    chunk_rows = min(chunk_rows, M)
    logits = torch.empty(chunk_rows, V, dtype=torch.bfloat16, device=h.device)
    first = not accumulate
    for s in range(0, M, chunk_rows):
        e = min(M, s + chunk_rows)
        lg = logits[: e - s]
        gemm(h[s:e], w, "nt", out=lg)
        _C.ce_grad_inplace(lg, labels[s:e], n_valid, loss_sum, ignore_index)   # lg <- (softmax - onehot)/n
        gemm(lg, w, "nn", out=dh[s:e])
        gemm(lg, h[s:e], "tn", out=dw_out, accumulate=not first)
        first = False
    return loss_sum / n_valid.clamp(min=1.0), dh


def cross_entropy_fwd_bwd(logits, labels, ignore_index=-100):
    V = logits.shape[-1]
    if logits.dtype != torch.bfloat16 or V % 8:
        return _fallback("cross_entropy_fwd_bwd").cross_entropy_fwd_bwd(logits, labels, ignore_index)
    labels = labels.reshape(-1).long()
    n_valid = torch.zeros((), dtype=torch.float32, device=logits.device)
    loss_sum = torch.zeros((), dtype=torch.float32, device=logits.device)
    _C.count_valid(labels, ignore_index, n_valid)
    g = logits.clone()
    _C.ce_grad_inplace(g, labels, n_valid, loss_sum, ignore_index)
    return loss_sum / n_valid.clamp(min=1.0), g


# ------------------------------------------------------------------------------------- optimizer
def sumsq(x, out=None):
    if out is None:
        out = torch.zeros((), dtype=torch.float32, device=x.device)
    if x.dtype not in (torch.bfloat16, torch.float32) or x.data_ptr() % 16 or not x.is_contiguous():
        return _fallback("sumsq").sumsq(x, out)
    _C.sumsq(x, out)
    return out


def adamw_step(master, grad, exp_avg, exp_avg_sq, lowp_out, lr, beta1, beta2, eps, weight_decay, step,
               grad_scale=None):
    ok = (master.numel() % 4 == 0 and grad.dtype in (torch.bfloat16, torch.float32)
          and (lowp_out is None or lowp_out.dtype == torch.bfloat16))
    if not ok:
        return _fallback("adamw_step").adamw_step(master, grad, exp_avg, exp_avg_sq, lowp_out, lr, beta1, beta2, eps,
                                        weight_decay, step, grad_scale)
    if grad_scale is not None and grad_scale.dtype != torch.float32:
        grad_scale = grad_scale.float()
    _C.adamw(master, grad, exp_avg, exp_avg_sq, lowp_out, lr, beta1, beta2, eps, weight_decay, step, grad_scale)
    return master


# ----------------------------------------------------------------------------------------- mamba
def causal_conv1d_fwd(x, w, b, seq_len, activation=True):
    if x.dtype != torch.bfloat16 or x.shape[1] % 8 or w.shape[1] > 4:
        return _fallback("causal_conv1d_fwd").causal_conv1d_fwd(x, w, b, seq_len, activation)
    return _C.causal_conv1d_fwd(x.contiguous(), _bf16c(w), None if b is None else _bf16c(b), seq_len, activation)


def causal_conv1d_bwd(dy, x, w, b, seq_len, activation=True):
    if x.dtype != torch.bfloat16 or x.shape[1] % 8 or w.shape[1] > 4:
        return _fallback("causal_conv1d_bwd").causal_conv1d_bwd(dy, x, w, b, seq_len, activation)
    dx, dw, db = _C.causal_conv1d_bwd(dy.contiguous(), x.contiguous(), _bf16c(w), None if b is None else _bf16c(b),
                                      seq_len, activation)
    return dx, dw, (None if b is None else db)


# ------------------------------------------------------------------------------ Mamba2 SSD scan
def _ssd_native_ok(x, dt, Bm, Cm, seq_len):
    return (x.is_cuda and x.dtype == dt.dtype == Bm.dtype == Cm.dtype == torch.bfloat16 and x.dim() == 3
            and seq_len % 128 == 0 and x.shape[2] % 32 == 0 and Bm.shape[2] % 8 == 0 and x.shape[1] % Bm.shape[1] == 0)


def _f32c(t):
    return None if t is None else t.detach().float().contiguous()


def ssd_scan_fwd(x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size, dt_softplus=True):
    """Mamba2 SSD scan (csrc/ssd.cu + batched tcgen05 GEMMs); 128-token internal chunks whatever ``chunk_size``."""
    if not _ssd_native_ok(x, dt, Bm, Cm, seq_len):
        return _fallback("ssd_scan_chunked").ssd_scan_chunked(x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size, dt_softplus)
    return _C.ssd_scan_fwd(x.contiguous(), dt.contiguous(), _f32c(A), Bm.contiguous(), Cm.contiguous(), _f32c(D),
                           _f32c(dt_bias), int(seq_len), bool(dt_softplus))


def ssd_scan_bwd(dy, x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size, dt_softplus=True):
    if not _ssd_native_ok(x, dt, Bm, Cm, seq_len):
        return None                                   # caller differentiates the ATen chunked form instead
    dx, ddt, dA, dB, dC, dD, dbias = _C.ssd_scan_bwd(dy.contiguous(), x.contiguous(), dt.contiguous(), _f32c(A),
                                                     Bm.contiguous(), Cm.contiguous(), _f32c(D), _f32c(dt_bias),
                                                     int(seq_len), bool(dt_softplus))
    return dx, ddt, dA, dB, dC, dD, dbias


# ------------------------------------------------------------------------------ Mamba1 selective scan
def _selscan_native_ok(u, delta, A, Bm, Cm, z, seq_len):
    return (u.is_cuda and u.dtype == delta.dtype == Bm.dtype == Cm.dtype == torch.bfloat16 and u.dim() == 2
            and (z is None or z.dtype == torch.bfloat16) and A.shape[-1] == 16 and seq_len % 32 == 0
            and u.shape[1] % 32 == 0)


def selective_scan_fwd(u, delta, A, Bm, Cm, D, z, delta_bias, seq_len, delta_softplus=True):
    """Mamba1 selective scan (csrc/selscan.cu: warp = channel, lane = timestep, shuffle scans)."""
    if not _selscan_native_ok(u, delta, A, Bm, Cm, z, seq_len):
        return _fallback("selective_scan_fwd").selective_scan_fwd(u, delta, A, Bm, Cm, D, z, delta_bias, seq_len, delta_softplus)
    y, _ = _C.selective_scan_fwd(u.contiguous(), delta.contiguous(), _f32c(A), Bm.contiguous(), Cm.contiguous(), _f32c(D),
                                 None if z is None else z.contiguous(), _f32c(delta_bias), int(seq_len),
                                 bool(delta_softplus), False)
    return y


def selective_scan_bwd(dy, u, delta, A, Bm, Cm, D, z, delta_bias, seq_len, delta_softplus=True):
    if not _selscan_native_ok(u, delta, A, Bm, Cm, z, seq_len):
        return None
    args = (u.contiguous(), delta.contiguous(), _f32c(A), Bm.contiguous(), Cm.contiguous(), _f32c(D),
            None if z is None else z.contiguous(), _f32c(delta_bias))
    _, hc = _C.selective_scan_fwd(*args, int(seq_len), bool(delta_softplus), True)   # block-entry states for the recompute
    du, dd, dA, dB, dC, dD, dz, ddb = _C.selective_scan_bwd(dy.contiguous(), *args, hc, int(seq_len), bool(delta_softplus))
    return du, dd, dA, dB, dC, dD, dz, ddb
