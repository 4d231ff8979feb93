"""ATen implementations of every engine primitive (forward *and* hand-derived backward).

Two jobs: (1) the CPU/gloo plumbing path and numerical oracle for the sm_100a kernels
(tests compare ``cuda_kernels.X`` against ``torch_kernels.X`` and both against autograd of
the naive formula); (2) executable documentation of exactly what each CUDA kernel computes.
Signatures are identical to ``cuda_kernels``.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

NAME = "torch"


# ----------------------------------------------------------------------------------------------
# GEMM family.  layout: "nt": C[M,N] = A[M,K] B[N,K]^T ; "nn": C[M,N] = A[M,K] B[K,N] ;
#                        "tn": C[M,N] = A[K,M]^T B[K,N].  fp32 accumulate, output dtype of `out`/a.
# ----------------------------------------------------------------------------------------------
def gemm(a, b, layout="nt", out=None, accumulate=False, residual=None, out_dtype=None, rope=None, bias=None):
    """``bias`` [N] (nt only): added to the product before the RoPE rotation / residual."""
    if rope is not None:   # (table, S, head_dim, H, KVH): RoPE on the q and k heads of a fused QKV product
        y = gemm(a, b, layout, out=out, accumulate=accumulate, residual=residual, out_dtype=out_dtype, bias=bias)
        table, S, hd, H, KVH = rope
        return rope_(y, table, S, H, KVH, hd)
    if bias is not None:
        if layout != "nt":
            raise ValueError("bias: nt layout only")
        c = torch.addmm(bias.to(a.dtype), a, b.t())
    elif layout == "nt":
        c = a @ b.t()
    elif layout == "nn":
        c = a @ b
    elif layout == "tn":
        c = a.t() @ b
    else:
        raise ValueError(layout)
    if residual is not None:
        c = c + residual
    if out is None:
        return c if out_dtype is None else c.to(out_dtype)
    if accumulate:
        out.add_(c.to(out.dtype))
    else:
        out.copy_(c)
    return out


def bias_grad(dy, out, accumulate=False):
    """out[n] (+)= sum_m dy[m, n] with fp32 accumulation (gradient of a bias added to every row of a GEMM output)."""
    s = dy.reshape(-1, dy.shape[-1]).float().sum(0)
    if accumulate:
        out.add_(s.to(out.dtype))
    else:
        out.copy_(s)
    return out


# ----------------------------------------------------------------------------------------------
# RMSNorm (fp32 math, io in x.dtype).  y = x * rsqrt(mean(x^2)+eps) * w
# ----------------------------------------------------------------------------------------------
def rmsnorm_fwd(x, w, eps):
    xf = x.float()
    rstd = torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)
    y = (xf * rstd * w.float()).to(x.dtype)
    return y, rstd.squeeze(-1)


def rmsnorm_bwd(dy, x, w, rstd, dres=None):
    xf, dyf, wf = x.float(), dy.float(), w.float()
    r = rstd.unsqueeze(-1)
    xhat = xf * r
    g = dyf * wf
    dx = r * (g - xhat * (g * xhat).mean(-1, keepdim=True))
    if dres is not None:
        dx = dx + dres.reshape(dx.shape).float()
    dw = (dyf * xhat).reshape(-1, x.shape[-1]).sum(0)
    return dx.to(x.dtype), dw


def add_rmsnorm_fwd(x, res, w, eps):
    """res_out = res + x (kept in res.dtype, fp32 for Mamba); y = rmsnorm(res_out)."""
    res_out = (res.float() + x.float()).to(res.dtype)
    y, rstd = rmsnorm_fwd(res_out.to(torch.float32), w, eps)
    return y.to(x.dtype), res_out, rstd


def rmsnorm_gated_fwd(x, z, w, eps, group_size):
    """Mamba2 RMSNormGated(norm_before_gate=False): y = rmsnorm_grouped(x * silu(z)) * w."""
    xf = x.float() * F.silu(z.float())
    shp = xf.shape
    xg = xf.reshape(*shp[:-1], shp[-1] // group_size, group_size)
    rstd = torch.rsqrt(xg.pow(2).mean(-1, keepdim=True) + eps)
    y = (xg * rstd).reshape(shp) * w.float()
    return y.to(x.dtype), rstd.squeeze(-1)


def rmsnorm_gated_bwd(dy, x, z, w, rstd, group_size):
    xf, zf, dyf, wf = x.float(), z.float(), dy.float(), w.float()
    sig = torch.sigmoid(zf)
    sz = zf * sig
    u = xf * sz
    shp = u.shape
    G = shp[-1] // group_size
    ug = u.reshape(*shp[:-1], G, group_size)
    r = rstd.unsqueeze(-1)
    uhat = ug * r
    g = (dyf * wf).reshape(*shp[:-1], G, group_size)
    du = (r * (g - uhat * (g * uhat).mean(-1, keepdim=True))).reshape(shp)
    dw = (dyf * uhat.reshape(shp)).reshape(-1, shp[-1]).sum(0)
    dx = du * sz
    dz = du * xf * (sig * (1 + zf * (1 - sig)))
    return dx.to(x.dtype), dz.to(z.dtype), dw


# ----------------------------------------------------------------------------------------------
# RoPE, FMS "interleaved pair" convention: (x[2i], x[2i+1]) rotated by pos * theta^(-2i/rot_dim).
# Operates IN PLACE on the q and k sections of a fused [M, (H+2*KVH)*hd] projection.
# ----------------------------------------------------------------------------------------------
def scaled_inv_freq(inv, scaling):
    """Frequency rescaling of long-context checkpoints (HF ``rope_scaling``): ``linear`` divides every frequency by ``factor``;
    ``llama3`` (Llama 3.1 / 3.2) leaves short wavelengths alone, divides wavelengths beyond
    ``original_max_position_embeddings / low_freq_factor`` by ``factor`` and interpolates in between."""
    kind = scaling.get("rope_type") or scaling.get("type")
    factor = float(scaling["factor"])
    if kind == "linear":
        return inv / factor
    if kind != "llama3":
        raise NotImplementedError(f"rope scaling {kind!r}")
    lo, hi = float(scaling.get("low_freq_factor", 1.0)), float(scaling.get("high_freq_factor", 4.0))
    old_len = float(scaling.get("original_max_position_embeddings", 8192))
    wavelen = 2 * math.pi / inv
    out = torch.where(wavelen > old_len / lo, inv / factor, inv)
    smooth = (old_len / wavelen - lo) / (hi - lo)
    medium = ~(wavelen < old_len / hi) & ~(wavelen > old_len / lo)
    return torch.where(medium, (1 - smooth) * out / factor + smooth * out, out)


def rope_table(max_seq_len, rot_dim, theta=10000.0, ntk_alpha=1.0, device=None, scaling=None):
    ratio = theta * (ntk_alpha ** (rot_dim / (rot_dim - 2))) if ntk_alpha != 1.0 else theta
    inv = 1.0 / (ratio ** (torch.arange(0, rot_dim, 2, device=device, dtype=torch.float32) / rot_dim))
    if scaling:
        inv = scaled_inv_freq(inv, scaling)
    ang = torch.outer(torch.arange(max_seq_len, device=device, dtype=torch.float32), inv)
    return torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous()  # [S, rot_dim/2, 2]


def rope_(qkv, table, seq_len, nheads, kvheads, head_dim, rot_dim=None, inverse=False, pos_offset=0, interleaved=True):
    rot_dim = head_dim if rot_dim is None else rot_dim
    M = qkv.shape[0]
    nrot = nheads + kvheads
    v = qkv.view(M, nheads + 2 * kvheads, head_dim)[:, :nrot, :rot_dim]
    pos = (torch.arange(M, device=qkv.device) % seq_len) + pos_offset
    cs = table[pos]  # [M, rot/2, 2]
    cos, sin = cs[..., 0].unsqueeze(1), cs[..., 1].unsqueeze(1)
    if inverse:
        sin = -sin
    if interleaved:   # FMS convention: pairs (2i, 2i+1)
        x = v.float().reshape(M, nrot, rot_dim // 2, 2)
        x0, x1 = x[..., 0], x[..., 1]
        out = torch.stack([x0 * cos - x1 * sin, x0 * sin + x1 * cos], dim=-1).reshape(M, nrot, rot_dim)
    else:             # GPT-NeoX / HF convention: pairs (i, i + rot/2)
        x = v.float()
        x0, x1 = x[..., : rot_dim // 2], x[..., rot_dim // 2:]
        out = torch.cat([x0 * cos - x1 * sin, x0 * sin + x1 * cos], dim=-1)
    v.copy_(out.to(qkv.dtype))
    return qkv


# ----------------------------------------------------------------------------------------------
# Causal flash attention on the fused projection.  qkv: [B*S, (H+2KVH)*hd]; o: [B*S, H*hd];
# lse: [B, H, S] fp32 (natural log).
# ----------------------------------------------------------------------------------------------
def _split_qkv(qkv, B, S, H, KVH, hd):
    t = qkv.view(B, S, H + 2 * KVH, hd)
    return t[:, :, :H], t[:, :, H:H + KVH], t[:, :, H + KVH:]


def attn_fwd(qkv, B, S, H, KVH, hd, scale, causal=True):
    q, k, v = _split_qkv(qkv, B, S, H, KVH, hd)
    qf, kf, vf = (t.permute(0, 2, 1, 3).float() for t in (q, k, v))
    rep = H // KVH
    if rep > 1:
        kf = kf.repeat_interleave(rep, dim=1)
        vf = vf.repeat_interleave(rep, dim=1)
    s = (qf @ kf.transpose(-1, -2)) * scale
    if causal:
        mask = torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril()
        s = s.masked_fill(~mask, float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    p = torch.exp(s - lse.unsqueeze(-1))
    o = (p @ vf).permute(0, 2, 1, 3).reshape(B * S, H * hd).to(qkv.dtype)
    return o, lse


def attn_bwd(do, qkv, o, lse, B, S, H, KVH, hd, scale, causal=True, rope_table=None):
    if rope_table is not None:   # gradient of the un-rotated projection
        g = attn_bwd(do, qkv, o, lse, B, S, H, KVH, hd, scale, causal)
        return rope_(g, rope_table, S, H, KVH, hd, inverse=True)
    q, k, v = _split_qkv(qkv, B, S, H, KVH, hd)
    qf, kf, vf = (t.permute(0, 2, 1, 3).float() for t in (q, k, v))
    rep = H // KVH
    kx = kf.repeat_interleave(rep, dim=1) if rep > 1 else kf
    vx = vf.repeat_interleave(rep, dim=1) if rep > 1 else vf
    dof = do.view(B, S, H, hd).permute(0, 2, 1, 3).float()
    of = o.view(B, S, H, hd).permute(0, 2, 1, 3).float()
    s = (qf @ kx.transpose(-1, -2)) * scale
    if causal:
        mask = torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril()
        s = s.masked_fill(~mask, float("-inf"))
    p = torch.exp(s - lse.unsqueeze(-1))
    dv = p.transpose(-1, -2) @ dof
    dp = dof @ vx.transpose(-1, -2)
    delta = (dof * of).sum(-1, keepdim=True)
    ds = p * (dp - delta) * scale
    dq = ds @ kx
    dk = ds.transpose(-1, -2) @ qf
    if rep > 1:
        dk = dk.view(B, KVH, rep, S, hd).sum(2)
        dv = dv.view(B, KVH, rep, S, hd).sum(2)
    dqkv = torch.empty_like(qkv)
    t = dqkv.view(B, S, H + 2 * KVH, hd)
    t[:, :, :H] = dq.permute(0, 2, 1, 3).to(qkv.dtype)
    t[:, :, H:H + KVH] = dk.permute(0, 2, 1, 3).to(qkv.dtype)
    t[:, :, H + KVH:] = dv.permute(0, 2, 1, 3).to(qkv.dtype)
    return dqkv


# ----------------------------------------------------------------------------------------------
# Optional fp8 forward path (default off): row-wise scaled e4m3 operands, fp32 accumulation.
# ----------------------------------------------------------------------------------------------
E4M3_MAX = 448.0


def quant_rowwise_e4m3(x):
    """(q uint8 view of float8_e4m3fn [R, K], scale fp32 [R]) with scale = amax(row) / 448."""
    xf = x.float()
    amax = xf.abs().amax(dim=1)
    sc = torch.where(amax > 0, amax / E4M3_MAX, torch.ones_like(amax))
    q = (xf / sc[:, None]).clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)
    return q.view(torch.uint8), sc


def gemm_fp8(aq, bq, sa, sb, out=None):
    """C = (A_q B_q^T) * sa[:, None] * sb[None, :] in bf16 (oracle of csrc/gemm2_sm100.cu b200_gemm2_fp8)."""
    a = aq.view(torch.float8_e4m3fn).float()
    b = bq.view(torch.float8_e4m3fn).float()
    y = ((a @ b.t()) * sa[:, None] * sb[None, :]).to(torch.bfloat16)
    if out is not None:
        out.copy_(y)
        return out
    return y


# ----------------------------------------------------------------------------------------------
# SwiGLU on the fused gate/up projection gu = [gate | up] (FMS wg1_fused row order).
# ----------------------------------------------------------------------------------------------
def swiglu_fwd(gu, gate_first=True):
    F_ = gu.shape[-1] // 2
    a, b = gu[..., :F_].float(), gu[..., F_:].float()
    g, u = (a, b) if gate_first else (b, a)
    return (F.silu(g) * u).to(gu.dtype)


def gated_up_fwd(x, w, gate_first=True):
    """Gate/up projection with the SwiGLU activation: returns (gu [M, 2F], silu(gate) * up [M, F])  (SURVEY.md K6/K7)."""
    gu = gemm(x, w, "nt")
    return gu, swiglu_fwd(gu, gate_first)


def gated_down_bwd(dy, w2, gu, gate_first=True):
    """d(gu) of  y = (silu(gate) * up) @ w2^T :  swiglu_bwd(dy @ w2, gu)  (the CUDA path fuses the two)."""
    return swiglu_bwd(gemm(dy, w2, "nn"), gu, gate_first)


def swiglu_bwd(ds, gu, gate_first=True):
    F_ = gu.shape[-1] // 2
    a, b, d = gu[..., :F_].float(), gu[..., F_:].float(), ds.float()
    g, u = (a, b) if gate_first else (b, a)
    sig = torch.sigmoid(g)
    dg = d * u * sig * (1 + g * (1 - sig))
    du = d * g * sig
    return torch.cat([dg, du] if gate_first else [du, dg], dim=-1).to(gu.dtype)


# ----------------------------------------------------------------------------------------------
# Embedding
# ----------------------------------------------------------------------------------------------
def embedding_fwd(tokens, w):
    return w[tokens.reshape(-1).long()]


def embedding_bwd(dx, tokens, out, accumulate=False):
    if not accumulate:
        out.zero_()
    out.index_add_(0, tokens.reshape(-1).long(), dx.to(out.dtype))
    return out


# ----------------------------------------------------------------------------------------------
# Fused linear + cross-entropy (mean over non-ignored rows).  Never materialises [M,V] logits:
# processes row chunks, computes loss and (already 1/n scaled) gradients in the same pass.
# Returns loss (fp32 scalar), dh [M,D]; dW is written/accumulated into `dw_out` [V,D].
# ----------------------------------------------------------------------------------------------
def linear_ce_fwd_bwd(h, w, labels, dw_out, ignore_index=-100, chunk_rows=4096, accumulate=False):
    M, D = h.shape
    labels = labels.reshape(-1).long()
    valid = labels != ignore_index
    n_valid = valid.sum().clamp(min=1).float()
    dh = torch.empty_like(h)
    loss = torch.zeros((), dtype=torch.float32, device=h.device)
    first = not accumulate
    for s in range(0, M, chunk_rows):
        e = min(M, s + chunk_rows)
        logits = (h[s:e] @ w.t()).float()
        lab = labels[s:e]
        ok = valid[s:e]
        lse = torch.logsumexp(logits, dim=-1)
        safe = lab.clamp(min=0)
        tgt = logits.gather(1, safe.unsqueeze(1)).squeeze(1)
        loss = loss + ((lse - tgt) * ok).sum()
        p = torch.exp(logits - lse.unsqueeze(1))
        p.scatter_add_(1, safe.unsqueeze(1), -torch.ones_like(tgt).unsqueeze(1))
        p = (p * (ok.unsqueeze(1) / n_valid)).to(h.dtype)
        dh[s:e] = p @ w
        gemm(p, h[s:e], "tn", out=dw_out, accumulate=not first)
        first = False
    return loss / n_valid, dh


def cross_entropy_fwd_bwd(logits, labels, ignore_index=-100):
    """Unfused variant for an explicit logits tensor: returns loss and dlogits (1/n scaled)."""
    labels = labels.reshape(-1).long()
    valid = labels != ignore_index
    n_valid = valid.sum().clamp(min=1).float()
    lf = logits.float()
    lse = torch.logsumexp(lf, dim=-1)
    safe = labels.clamp(min=0)
    tgt = lf.gather(1, safe.unsqueeze(1)).squeeze(1)
    loss = ((lse - tgt) * valid).sum() / n_valid
    p = torch.exp(lf - lse.unsqueeze(1))
    p.scatter_add_(1, safe.unsqueeze(1), -torch.ones_like(tgt).unsqueeze(1))
    return loss, (p * (valid.unsqueeze(1) / n_valid)).to(logits.dtype)


# ----------------------------------------------------------------------------------------------
# Optimizer / gradient utilities on flat shards
# ----------------------------------------------------------------------------------------------
def sumsq(x, out=None):
    s = x.float().pow(2).sum()
    if out is None:
        return s
    out.add_(s)
    return out


def adamw_step(master, grad, exp_avg, exp_avg_sq, lowp_out, lr, beta1, beta2, eps, weight_decay, step,
               grad_scale=None):
    """Decoupled-weight-decay Adam on a flat fp32 shard (torch.optim.AdamW semantics).
    grad may be bf16/fp32; grad_scale is an optional 0-dim fp32 tensor (clip coefficient).
    Writes the refreshed low-precision shard into lowp_out (may be None)."""
    g = grad.float()
    if grad_scale is not None:
        g = g * grad_scale
    master.mul_(1.0 - lr * weight_decay)
    exp_avg.mul_(beta1).add_(g, alpha=1.0 - beta1)
    exp_avg_sq.mul_(beta2).addcmul_(g, g, value=1.0 - beta2)
    bc1 = 1.0 - beta1 ** step
    bc2 = 1.0 - beta2 ** step
    denom = (exp_avg_sq.sqrt() / math.sqrt(bc2)).add_(eps)
    master.addcdiv_(exp_avg, denom, value=-lr / bc1)
    if lowp_out is not None:
        lowp_out.copy_(master)
    return master


# ----------------------------------------------------------------------------------------------
# Mamba primitives
# ----------------------------------------------------------------------------------------------
def causal_conv1d_fwd(x, w, b, seq_len, activation=True):
    """x: [B*S, C] channels-last; w: [C, K]; depthwise causal FIR + optional SiLU."""
    M, C = x.shape
    B = M // seq_len
    K = w.shape[1]
    xt = x.view(B, seq_len, C).transpose(1, 2).float()
    y = F.conv1d(F.pad(xt, (K - 1, 0)), w.float().unsqueeze(1), None if b is None else b.float(), groups=C)
    if activation:
        y = F.silu(y)
    return y.transpose(1, 2).reshape(M, C).to(x.dtype)


def causal_conv1d_bwd(dy, x, w, b, seq_len, activation=True):
    M, C = x.shape
    B = M // seq_len
    K = w.shape[1]
    xt = x.view(B, seq_len, C).transpose(1, 2).float()
    xp = F.pad(xt, (K - 1, 0))
    pre = F.conv1d(xp, w.float().unsqueeze(1), None if b is None else b.float(), groups=C)
    d = dy.view(B, seq_len, C).transpose(1, 2).float()
    if activation:
        sig = torch.sigmoid(pre)
        d = d * sig * (1 + pre * (1 - sig))
    # dx[t] = sum_k w[k] * d[t + (K-1-k)]
    dpad = F.pad(d, (0, K - 1))
    dx = F.conv1d(dpad, w.float().flip(1).unsqueeze(1), None, groups=C)
    dw = torch.stack([(xp[:, :, k:k + seq_len] * d).sum((0, 2)) for k in range(K)], dim=1)
    db = None if b is None else d.sum((0, 2))
    return dx.transpose(1, 2).reshape(M, C).to(x.dtype), dw, db


def ssd_scan_fwd(x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size, dt_softplus=True):
    """Mamba2 state-space-dual scan (sequential fp32 oracle; the CUDA kernel is chunked).
    x: [M, H, P]; dt: [M, H]; A: [H] (negative); Bm, Cm: [M, G, N]; D: [H]; returns y [M, H, P]."""
    M, H, P = x.shape
    Bsz = M // seq_len
    G, N = Bm.shape[1], Bm.shape[2]
    xf = x.float().view(Bsz, seq_len, H, P)
    dtf = dt.float().view(Bsz, seq_len, H)
    if dt_bias is not None:
        dtf = dtf + dt_bias.float()
    if dt_softplus:
        dtf = F.softplus(dtf)
    Bf = Bm.float().view(Bsz, seq_len, G, N).repeat_interleave(H // G, dim=2)
    Cf = Cm.float().view(Bsz, seq_len, G, N).repeat_interleave(H // G, dim=2)
    dA = torch.exp(dtf * A.float())  # [B,S,H]
    state = torch.zeros(Bsz, H, P, N, dtype=torch.float32, device=x.device)
    ys = []
    for t in range(seq_len):
        state = state * dA[:, t, :, None, None] + (dtf[:, t, :, None] * xf[:, t])[..., None] * Bf[:, t, :, None, :]
        ys.append((state * Cf[:, t, :, None, :]).sum(-1))
    y = torch.stack(ys, dim=1)
    if D is not None:
        y = y + xf * D.float()[None, None, :, None]
    return y.reshape(M, H, P).to(x.dtype)


def _segsum(x):
    """out[..., i, j] = sum_{j < k <= i} x[..., k]  (lower triangle; -inf above the diagonal)."""
    T = x.size(-1)
    cs = torch.cumsum(x, dim=-1)
    d = cs[..., :, None] - cs[..., None, :]
    mask = torch.tril(torch.ones(T, T, device=x.device, dtype=torch.bool), diagonal=0)
    return d.masked_fill(~mask, float("-inf"))


def ssd_scan_chunked(x, dt, A, Bm, Cm, D, dt_bias, seq_len, chunk_size, dt_softplus=True):
    """Mamba2 SSD in its chunked (state-space dual) matmul form -- differentiable ATen, the formulation the
    tensor-core kernel follows: intra-chunk quadratic term + chunk states + inter-chunk state passing."""
    M, H, P = x.shape
    Bsz = M // seq_len
    G, N = Bm.shape[1], Bm.shape[2]
    L = min(chunk_size, seq_len)
    pad = (-seq_len) % L
    xf = x.float().view(Bsz, seq_len, H, P)
    dtf = dt.float().view(Bsz, seq_len, H)
    if dt_bias is not None:
        dtf = dtf + dt_bias.float()
    if dt_softplus:
        dtf = F.softplus(dtf)
    Bf = Bm.float().view(Bsz, seq_len, G, N).repeat_interleave(H // G, dim=2)
    Cf = Cm.float().view(Bsz, seq_len, G, N).repeat_interleave(H // G, dim=2)
    if pad:
        xf, dtf = F.pad(xf, (0, 0, 0, 0, 0, pad)), F.pad(dtf, (0, 0, 0, pad))
        Bf, Cf = F.pad(Bf, (0, 0, 0, 0, 0, pad)), F.pad(Cf, (0, 0, 0, 0, 0, pad))
    S2 = seq_len + pad
    nc = S2 // L
    X = (xf * dtf.unsqueeze(-1)).view(Bsz, nc, L, H, P)
    Ad = (dtf * A.float()).view(Bsz, nc, L, H).permute(0, 3, 1, 2)        # [b,h,c,L]
    Bc = Bf.view(Bsz, nc, L, H, N)
    Cc = Cf.view(Bsz, nc, L, H, N)
    A_cs = torch.cumsum(Ad, dim=-1)
    Lm = torch.exp(_segsum(Ad))                                              # [b,h,c,L,L]
    Y_diag = torch.einsum("bclhn,bcshn,bhcls,bcshp->bclhp", Cc, Bc, Lm, X)
    decay_states = torch.exp(A_cs[..., -1:] - A_cs)                          # [b,h,c,L]
    states = torch.einsum("bclhn,bhcl,bclhp->bchpn", Bc, decay_states, X)    # [b,c,h,p,n]
    states = torch.cat([torch.zeros_like(states[:, :1]), states], dim=1)
    decay_chunk = torch.exp(_segsum(F.pad(A_cs[..., -1], (1, 0))))           # [b,h,c+1,c+1]
    new_states = torch.einsum("bhzc,bchpn->bzhpn", decay_chunk, states)[:, :-1]
    Y_off = torch.einsum("bclhn,bchpn,bhcl->bclhp", Cc, new_states, torch.exp(A_cs))
    y = (Y_diag + Y_off).reshape(Bsz, S2, H, P)[:, :seq_len]
    if D is not None:
        y = y + xf[:, :seq_len] * D.float()[None, None, :, None]
    return y.reshape(M, H, P).to(x.dtype)


def selective_scan_fwd(u, delta, A, Bm, Cm, D, z, delta_bias, seq_len, delta_softplus=True):
    """Mamba1 selective scan oracle. u, delta, z: [M, Dm]; A: [Dm, N]; Bm, Cm: [M, N]; D: [Dm]."""
    M, Dm = u.shape
    Bsz = M // seq_len
    N = A.shape[1]
    uf = u.float().view(Bsz, seq_len, Dm)
    df = delta.float().view(Bsz, seq_len, Dm)
    if delta_bias is not None:
        df = df + delta_bias.float()
    if delta_softplus:
        df = F.softplus(df)
    Bf = Bm.float().view(Bsz, seq_len, N)
    Cf = Cm.float().view(Bsz, seq_len, N)
    h = torch.zeros(Bsz, Dm, N, dtype=torch.float32, device=u.device)
    ys = []
    for t in range(seq_len):
        h = h * torch.exp(df[:, t, :, None] * A.float()) + (df[:, t] * uf[:, t])[..., None] * Bf[:, t, None, :]
        ys.append((h * Cf[:, t, None, :]).sum(-1))
    y = torch.stack(ys, dim=1)
    if D is not None:
        y = y + uf * D.float()
    if z is not None:
        y = y * F.silu(z.float().view(Bsz, seq_len, Dm))
    return y.reshape(M, Dm).to(u.dtype)
