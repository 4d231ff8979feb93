// Bandwidth-bound kernels of the engine (sm_100a): RMSNorm fwd/bwd, RoPE, SwiGLU fwd/bwd, embedding
// fwd/bwd, softmax-cross-entropy gradient (in place on a logits chunk), fused sharded AdamW, sum of
// squares.  All are single-pass over HBM with 16-byte vector accesses; fp32 math, bf16 I/O.
// SURVEY.md K2/K5/K7/K9/K10(softmax part)/K11/K12.
#include "common.cuh"

namespace b200 {

constexpr int NT = 256;  // threads per CTA for row kernels

B200_DEVINL float block_sum(float v, float* sh) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();  // protect sh from the previous use
  if (l == 0) sh[w] = v;
  __syncthreads();
  float r = (l < (blockDim.x >> 5)) ? sh[l] : 0.f;
  r = warp_sum(r);
  return r;
}
B200_DEVINL float block_max(float v, float* sh) {
  v = warp_max(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  float r = (l < (blockDim.x >> 5)) ? sh[l] : -INFINITY;
  r = warp_max(r);
  return r;
}

B200_DEVINL void load8(const __nv_bfloat16* p, float (&f)[8]) {
  uint4 u = *reinterpret_cast<const uint4*>(p);
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
B200_DEVINL void store8(__nv_bfloat16* p, const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16x2(f[0], f[1]); u.y = pack_bf16x2(f[2], f[3]);
  u.z = pack_bf16x2(f[4], f[5]); u.w = pack_bf16x2(f[6], f[7]);
  *reinterpret_cast<uint4*>(p) = u;
}

// ------------------------------------------------------------------------------------- RMSNorm
// One CTA per row (grid-stride).  Row cached in registers: D <= NT*8*MAXC.
constexpr int MAXC = 4;

B200_DEVINL void unpack8(const uint4& u, float (&f)[8]) {
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

// NC = ceil(D / (NT*8)) 16-byte vectors per thread.  Rows stay in registers as PACKED bf16 (4 regs per vector) so
// 6-8 CTAs are resident per SM and every thread has all of its row's loads in flight before the reduction.
template <int NC>
__global__ void __launch_bounds__(NT, 6) rmsnorm_fwd_kernel(const __nv_bfloat16* __restrict__ x,
                                                            const __nv_bfloat16* __restrict__ w,
                                                            __nv_bfloat16* __restrict__ y, float* __restrict__ rstd,
                                                            int M, int D, float eps) {
  __shared__ float sh[32];
  uint4 wq[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
    wq[c] = (col < D) ? *reinterpret_cast<const uint4*>(w + col) : make_uint4(0, 0, 0, 0);
  }
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    const __nv_bfloat16* xr = x + (size_t)row * D;
    uint4 xq[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      xq[c] = (col < D) ? *reinterpret_cast<const uint4*>(xr + col) : make_uint4(0, 0, 0, 0);
    }
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      float v[8];
      unpack8(xq[c], v);
#pragma unroll
      for (int i = 0; i < 8; ++i) ss += v[i] * v[i];
    }
    ss = block_sum(ss, sh);
    const float r = rsqrtf(ss / (float)D + eps);
    if (threadIdx.x == 0) rstd[row] = r;
    __nv_bfloat16* yr = y + (size_t)row * D;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float v[8], wv[8], o[8];
        unpack8(xq[c], v);
        unpack8(wq[c], wv);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = v[i] * r * wv[i];
        store8(yr + col, o);
      }
    }
  }
}

// dx = r * (g - xhat * mean(g*xhat)),  g = dy*w,  xhat = x*r ;  dw_partial[cta] += dy*xhat
template <int NC>
__global__ void __launch_bounds__(NT, (NC <= 2 ? 4 : 2)) rmsnorm_bwd_kernel(const __nv_bfloat16* __restrict__ dy,
                                                         const __nv_bfloat16* __restrict__ x,
                                                         const __nv_bfloat16* __restrict__ w,
                                                         const float* __restrict__ rstd,
                                                         const __nv_bfloat16* __restrict__ dres,
                                                         __nv_bfloat16* __restrict__ dx, float* __restrict__ dw_part,
                                                         int M, int D) {
  // dres (optional): gradient arriving on the residual branch that forked off x; summed into dx here so autograd
  // never runs a separate accumulate kernel
  __shared__ float sh[32];
  float dwacc[NC][8];
  uint4 wq[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) dwacc[c][i] = 0.f;
    wq[c] = (col < D) ? *reinterpret_cast<const uint4*>(w + col) : make_uint4(0, 0, 0, 0);
  }
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    uint4 dq[NC], xq[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      const bool ok = col < D;
      dq[c] = ok ? *reinterpret_cast<const uint4*>(dy + (size_t)row * D + col) : make_uint4(0, 0, 0, 0);
      xq[c] = ok ? *reinterpret_cast<const uint4*>(x + (size_t)row * D + col) : make_uint4(0, 0, 0, 0);
    }
    const float r = rstd[row];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      float a[8], b[8], wv[8];
      unpack8(dq[c], a);
      unpack8(xq[c], b);
      unpack8(wq[c], wv);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float xh = b[i] * r;
        dot += a[i] * wv[i] * xh;
        dwacc[c][i] += a[i] * xh;
      }
    }
    dot = block_sum(dot, sh) / (float)D;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float a[8], b[8], wv[8], o[8];
        unpack8(dq[c], a);
        unpack8(xq[c], b);
        unpack8(wq[c], wv);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = r * (a[i] * wv[i] - b[i] * r * dot);
        if (dres) {
          float e[8];
          load8(dres + (size_t)row * D + col, e);
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] += e[i];
        }
        store8(dx + (size_t)row * D + col, o);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
    if (col < D) {
      float4* o = reinterpret_cast<float4*>(dw_part + (size_t)blockIdx.x * D + col);
      o[0] = make_float4(dwacc[c][0], dwacc[c][1], dwacc[c][2], dwacc[c][3]);
      o[1] = make_float4(dwacc[c][4], dwacc[c][5], dwacc[c][6], dwacc[c][7]);
    }
  }
}

// out[d] = sum_p part[p, d]   (CTA = 32 columns x 8 row slices)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ part, float* __restrict__ out, int P, int D) {
  __shared__ float sh[8][33];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int d = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (d < D)
    for (int p = slice; p < P; p += 8) s += part[(size_t)p * D + d];
  sh[slice][lane] = s;
  __syncthreads();
  if (slice == 0 && d < D) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sh[k][lane];
    out[d] = t;
  }
}

// ------------------------------------------------------------- fused add + RMSNorm (fp32 residual stream)
// res_out = res + x (fp32) ; y = rmsnorm(res_out) * w (bf16).  Mamba block prologue (SURVEY.md M6).
__global__ void __launch_bounds__(NT) add_rmsnorm_fwd_kernel(const __nv_bfloat16* __restrict__ x,
                                                             const float* __restrict__ res,
                                                             const __nv_bfloat16* __restrict__ w,
                                                             __nv_bfloat16* __restrict__ y, float* __restrict__ res_out,
                                                             float* __restrict__ rstd, int M, int D, float eps) {
  __shared__ float sh[32];
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    float v[MAXC][8];
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float a[8];
        load8(x + (size_t)row * D + col, a);
        const float4* rp = reinterpret_cast<const float4*>(res + (size_t)row * D + col);
        const float4 r0 = rp[0], r1 = rp[1];
        v[c][0] = a[0] + r0.x; v[c][1] = a[1] + r0.y; v[c][2] = a[2] + r0.z; v[c][3] = a[3] + r0.w;
        v[c][4] = a[4] + r1.x; v[c][5] = a[5] + r1.y; v[c][6] = a[6] + r1.z; v[c][7] = a[7] + r1.w;
        float4* op = reinterpret_cast<float4*>(res_out + (size_t)row * D + col);
        op[0] = make_float4(v[c][0], v[c][1], v[c][2], v[c][3]);
        op[1] = make_float4(v[c][4], v[c][5], v[c][6], v[c][7]);
#pragma unroll
        for (int i = 0; i < 8; ++i) ss += v[c][i] * v[c][i];
      }
    }
    ss = block_sum(ss, sh);
    const float r = rsqrtf(ss / (float)D + eps);
    if (threadIdx.x == 0) rstd[row] = r;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float wv[8], o[8];
        load8(w + col, wv);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = v[c][i] * r * wv[i];
        store8(y + (size_t)row * D + col, o);
      }
    }
  }
}

// RMSNorm backward with an fp32 input stream: dx (fp32) = r * (g - xhat * mean(g*xhat)), dw_part += dy * xhat
__global__ void __launch_bounds__(NT) rmsnorm_bwd_f32_kernel(const __nv_bfloat16* __restrict__ dy,
                                                             const float* __restrict__ x,
                                                             const __nv_bfloat16* __restrict__ w,
                                                             const float* __restrict__ rstd, float* __restrict__ dx,
                                                             float* __restrict__ dw_part, int M, int D) {
  __shared__ float sh[32];
  float dwacc[MAXC][8], wv[MAXC][8];
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) dwacc[c][i] = 0.f;
    if (col < D) load8(w + col, wv[c]);
  }
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    const float r = rstd[row];
    float g[MAXC][8], xh[MAXC][8];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float a[8];
        load8(dy + (size_t)row * D + col, a);
        const float4* xp = reinterpret_cast<const float4*>(x + (size_t)row * D + col);
        const float4 x0 = xp[0], x1 = xp[1];
        const float b[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          xh[c][i] = b[i] * r;
          g[c][i] = a[i] * wv[c][i];
          dot += g[c][i] * xh[c][i];
          dwacc[c][i] += a[i] * xh[c][i];
        }
      }
    }
    dot = block_sum(dot, sh) / (float)D;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float4* op = reinterpret_cast<float4*>(dx + (size_t)row * D + col);
        op[0] = make_float4(r * (g[c][0] - xh[c][0] * dot), r * (g[c][1] - xh[c][1] * dot),
                            r * (g[c][2] - xh[c][2] * dot), r * (g[c][3] - xh[c][3] * dot));
        op[1] = make_float4(r * (g[c][4] - xh[c][4] * dot), r * (g[c][5] - xh[c][5] * dot),
                            r * (g[c][6] - xh[c][6] * dot), r * (g[c][7] - xh[c][7] * dot));
      }
    }
  }
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
    if (col < D) {
      float4* o = reinterpret_cast<float4*>(dw_part + (size_t)blockIdx.x * D + col);
      o[0] = make_float4(dwacc[c][0], dwacc[c][1], dwacc[c][2], dwacc[c][3]);
      o[1] = make_float4(dwacc[c][4], dwacc[c][5], dwacc[c][6], dwacc[c][7]);
    }
  }
}

// ----------------------------------------------------- gated RMSNorm (Mamba2 RMSNormGated, norm_before_gate=False)
// y = rmsnorm(x * silu(z)) * w over the whole row (ngroups = 1).  SURVEY.md M5.
__global__ void __launch_bounds__(NT) rmsnorm_gated_fwd_kernel(const __nv_bfloat16* __restrict__ x,
                                                               const __nv_bfloat16* __restrict__ z,
                                                               const __nv_bfloat16* __restrict__ w,
                                                               __nv_bfloat16* __restrict__ y, float* __restrict__ rstd,
                                                               int M, int D, float eps) {
  __shared__ float sh[32];
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    float u[MAXC][8];
    float ss = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float a[8], g[8];
        load8(x + (size_t)row * D + col, a);
        load8(z + (size_t)row * D + col, g);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          u[c][i] = a[i] * g[i] / (1.f + __expf(-g[i]));
          ss += u[c][i] * u[c][i];
        }
      }
    }
    ss = block_sum(ss, sh);
    const float r = rsqrtf(ss / (float)D + eps);
    if (threadIdx.x == 0) rstd[row] = r;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float wv[8], o[8];
        load8(w + col, wv);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = u[c][i] * r * wv[i];
        store8(y + (size_t)row * D + col, o);
      }
    }
  }
}

__global__ void __launch_bounds__(NT) rmsnorm_gated_bwd_kernel(const __nv_bfloat16* __restrict__ dy,
                                                               const __nv_bfloat16* __restrict__ x,
                                                               const __nv_bfloat16* __restrict__ z,
                                                               const __nv_bfloat16* __restrict__ w,
                                                               const float* __restrict__ rstd,
                                                               __nv_bfloat16* __restrict__ dx, __nv_bfloat16* __restrict__ dz,
                                                               float* __restrict__ dw_part, int M, int D) {
  __shared__ float sh[32];
  float dwacc[MAXC][8], wv[MAXC][8];
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) dwacc[c][i] = 0.f;
    if (col < D) load8(w + col, wv[c]);
  }
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    const float r = rstd[row];
    float g[MAXC][8], uh[MAXC][8], xs[MAXC][8], zs[MAXC][8];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float a[8];
        load8(dy + (size_t)row * D + col, a);
        load8(x + (size_t)row * D + col, xs[c]);
        load8(z + (size_t)row * D + col, zs[c]);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float sig = 1.f / (1.f + __expf(-zs[c][i]));
          const float uu = xs[c][i] * zs[c][i] * sig;
          uh[c][i] = uu * r;
          g[c][i] = a[i] * wv[c][i];
          dot += g[c][i] * uh[c][i];
          dwacc[c][i] += a[i] * uh[c][i];
        }
      }
    }
    dot = block_sum(dot, sh) / (float)D;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = (c * NT + threadIdx.x) * 8;
      if (col < D) {
        float ox[8], oz[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float du = r * (g[c][i] - uh[c][i] * dot);
          const float zz = zs[c][i];
          const float sig = 1.f / (1.f + __expf(-zz));
          ox[i] = du * zz * sig;
          oz[i] = du * xs[c][i] * sig * (1.f + zz * (1.f - sig));
        }
        store8(dx + (size_t)row * D + col, ox);
        store8(dz + (size_t)row * D + col, oz);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = (c * NT + threadIdx.x) * 8;
    if (col < D) {
      float4* o = reinterpret_cast<float4*>(dw_part + (size_t)blockIdx.x * D + col);
      o[0] = make_float4(dwacc[c][0], dwacc[c][1], dwacc[c][2], dwacc[c][3]);
      o[1] = make_float4(dwacc[c][4], dwacc[c][5], dwacc[c][6], dwacc[c][7]);
    }
  }
}

// ---------------------------------------------------------------------------------------- RoPE
// In place on heads [0, nrot) of a fused [M, nheads_total*hd] projection; pairs (2i, 2i+1);
// table [S, rot/2, 2] fp32 (cos, sin).  One thread = 8 elements = 4 pairs.
// Half-split (GPT-NeoX / HF / mamba_ssm) convention: pairs (i, i + rot/2).  One thread = 8 pairs.
__global__ void rope_halfsplit_kernel(__nv_bfloat16* __restrict__ qkv, const float* __restrict__ table, int M,
                                      int seq_len, int row_stride, int nrot_heads, int hd, int rot, float sign,
                                      int pos_offset) {
  const int vec_per_head = rot / 16;
  const size_t total = (size_t)M * nrot_heads * vec_per_head;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int vi = (int)(idx % vec_per_head);
    const size_t t = idx / vec_per_head;
    const int head = (int)(t % nrot_heads);
    const size_t row = t / nrot_heads;
    const int pos = (int)(row % seq_len) + pos_offset;
    __nv_bfloat16* p0 = qkv + row * row_stride + head * hd + vi * 8;
    __nv_bfloat16* p1 = p0 + rot / 2;
    float a[8], b[8], oa[8], ob[8];
    load8(p0, a);
    load8(p1, b);
    const float2* cs = reinterpret_cast<const float2*>(table + ((size_t)pos * (rot / 2) + vi * 8) * 2);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float2 c = cs[i];
      const float sn = c.y * sign;
      oa[i] = a[i] * c.x - b[i] * sn;
      ob[i] = a[i] * sn + b[i] * c.x;
    }
    store8(p0, oa);
    store8(p1, ob);
  }
}

__global__ void __launch_bounds__(256) rope_kernel(__nv_bfloat16* __restrict__ qkv, const float* __restrict__ table,
                                                   int M, int seq_len, int row_stride, int nrot_heads, int hd, int rot,
                                                   float sign, int pos_offset) {
  // one CTA per row (grid-stride); 4 independent 16-byte vectors in flight per thread
  const int vph = rot / 8;
  const int per_row = nrot_heads * vph;
  for (int row = blockIdx.x; row < M; row += gridDim.x) {
    const int pos = row % seq_len + pos_offset;
    __nv_bfloat16* base = qkv + (size_t)row * row_stride;
    const float* trow = table + (size_t)pos * rot;          // [rot/2][cos, sin]
    const bool same_vi = (256 % vph) == 0;                    // then v0 + k*256 has the same vi for every k
    for (int v0 = threadIdx.x; v0 < per_row; v0 += 4 * 256) {
      uint4 q[4];
      float4 c0[4], c1[4];
      if (same_vi) {
        const float4* cs = reinterpret_cast<const float4*>(trow + (v0 % vph) * 8);
        c0[0] = cs[0];
        c1[0] = cs[1];
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int v = v0 + k * 256;
        if (v < per_row) {
          const int head = v / vph, vi = v - head * vph;
          q[k] = *reinterpret_cast<const uint4*>(base + head * hd + vi * 8);
          if (!same_vi) {
            const float4* cs = reinterpret_cast<const float4*>(trow + vi * 8);
            c0[k] = cs[0];
            c1[k] = cs[1];
          } else if (k > 0) {
            c0[k] = c0[0];
            c1[k] = c1[0];
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int v = v0 + k * 256;
        if (v < per_row) {
          const int head = v / vph, vi = v - head * vph;
          float f[8], o[8];
          unpack8(q[k], f);
          const float cosv[4] = {c0[k].x, c0[k].z, c1[k].x, c1[k].z};
          const float sinv[4] = {c0[k].y * sign, c0[k].w * sign, c1[k].y * sign, c1[k].w * sign};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            o[2 * i] = f[2 * i] * cosv[i] - f[2 * i + 1] * sinv[i];
            o[2 * i + 1] = f[2 * i] * sinv[i] + f[2 * i + 1] * cosv[i];
          }
          store8(base + head * hd + vi * 8, o);
        }
      }
    }
  }
}

// -------------------------------------------------------------------------------------- SwiGLU
__global__ void swiglu_fwd_kernel(const __nv_bfloat16* __restrict__ gu, __nv_bfloat16* __restrict__ out, size_t M,
                                  int F, int goff, int uoff) {
  const int vec = F / 8;
  const size_t total = M * vec;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / vec;
    const int c = (int)(idx % vec) * 8;
    float g[8], u[8], o[8];
    load8(gu + row * 2 * F + goff + c, g);
    load8(gu + row * 2 * F + uoff + c, u);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = g[i] / (1.f + __expf(-g[i])) * u[i];
    store8(out + row * F + c, o);
  }
}
__global__ void swiglu_bwd_kernel(const __nv_bfloat16* __restrict__ ds, const __nv_bfloat16* __restrict__ gu,
                                  __nv_bfloat16* __restrict__ dgu, size_t M, int F, int goff, int uoff) {
  const int vec = F / 8;
  const size_t total = M * vec;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / vec;
    const int c = (int)(idx % vec) * 8;
    float g[8], u[8], d[8], dg[8], du[8];
    load8(gu + row * 2 * F + goff + c, g);
    load8(gu + row * 2 * F + uoff + c, u);
    load8(ds + row * F + c, d);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float sig = 1.f / (1.f + __expf(-g[i]));
      dg[i] = d[i] * u[i] * sig * (1.f + g[i] * (1.f - sig));
      du[i] = d[i] * g[i] * sig;
    }
    store8(dgu + row * 2 * F + goff + c, dg);
    store8(dgu + row * 2 * F + uoff + c, du);
  }
}

// ----------------------------------------------------------------------------------- embedding
template <typename IdxT>
__global__ void embedding_fwd_kernel(const IdxT* __restrict__ tok, const __nv_bfloat16* __restrict__ w,
                                     __nv_bfloat16* __restrict__ out, size_t M, int D) {
  const int vec = D / 8;
  const size_t total = M * vec;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / vec;
    const int c = (int)(idx % vec) * 8;
    const size_t t = (size_t)tok[row];
    *reinterpret_cast<uint4*>(out + row * D + c) = *reinterpret_cast<const uint4*>(w + t * D + c);
  }
}
template <typename IdxT>
__global__ void embedding_bwd_kernel(const IdxT* __restrict__ tok, const __nv_bfloat16* __restrict__ dx,
                                     __nv_bfloat16* __restrict__ dw, size_t M, int D) {
  const int vec = D / 2;
  const size_t total = M * vec;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / vec;
    const int c = (int)(idx % vec) * 2;
    const size_t t = (size_t)tok[row];
    const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(dx + row * D + c);
    atomicAdd(reinterpret_cast<__nv_bfloat162*>(dw + t * D + c), v);
  }
}
template <typename IdxT>
__global__ void embedding_bwd_f32_kernel(const IdxT* __restrict__ tok, const __nv_bfloat16* __restrict__ dx,
                                         float* __restrict__ dw, size_t M, int D) {
  const size_t total = M * D;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (size_t)gridDim.x * blockDim.x) {
    const size_t row = idx / D;
    const int c = (int)(idx % D);
    atomicAdd(dw + (size_t)tok[row] * D + c, __bfloat162float(dx[idx]));
  }
}

// ------------------------------------------------------------------ softmax cross-entropy gradient
// count of labels != ignore_index  ->  *n_valid (float)
__global__ void count_valid_kernel(const long long* __restrict__ labels, int M, long long ignore, float* n_valid) {
  __shared__ float sh[32];
  float c = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M; i += gridDim.x * blockDim.x)
    c += (labels[i] != ignore) ? 1.f : 0.f;
  c = block_sum(c, sh);
  if (threadIdx.x == 0 && c != 0.f) atomicAdd(n_valid, c);
}
// One CTA per row of a bf16 logits chunk [rows, V] (row stride ld): in place logits -> (softmax - onehot)/n_valid,
// loss_sum += (lse - logit[label]).  Rows with ignored labels get zero gradient.
__global__ void __launch_bounds__(NT) ce_grad_inplace_kernel(__nv_bfloat16* __restrict__ logits,
                                                             const long long* __restrict__ labels,
                                                             const float* __restrict__ n_valid,
                                                             float* __restrict__ loss_sum, int rows, int V, int ld,
                                                             long long ignore) {
  __shared__ float sh[32];
  for (int row = blockIdx.x; row < rows; row += gridDim.x) {
    __nv_bfloat16* lr = logits + (size_t)row * ld;
    const long long lab = labels[row];
    const bool valid = lab != ignore;
    // pass 1: row max
    float mx = -INFINITY;
    for (int c = threadIdx.x * 8; c < V; c += NT * 8) {
      float f[8];
      load8(lr + c, f);
#pragma unroll
      for (int i = 0; i < 8; ++i) mx = fmaxf(mx, f[i]);
    }
    mx = block_max(mx, sh);
    // pass 2: sum exp (row is L2/L1 resident: 2*V bytes)
    float se = 0.f;
    for (int c = threadIdx.x * 8; c < V; c += NT * 8) {
      float f[8];
      load8(lr + c, f);
#pragma unroll
      for (int i = 0; i < 8; ++i) se += __expf(f[i] - mx);
    }
    se = block_sum(se, sh);
    const float lse = mx + __logf(se);
    const float inv_n = valid ? 1.f / fmaxf(*n_valid, 1.f) : 0.f;
    if (threadIdx.x == 0 && valid) atomicAdd(loss_sum, lse - __bfloat162float(lr[lab]));
    __syncthreads();  // the label logit must be read before it is overwritten
    // pass 3: gradient in place
    for (int c = threadIdx.x * 8; c < V; c += NT * 8) {
      float f[8], o[8];
      load8(lr + c, f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float p = __expf(f[i] - lse);
        if (c + i == lab) p -= 1.f;
        o[i] = p * inv_n;
      }
      store8(lr + c, o);
    }
  }
}

// ------------------------------------------------------------------------------ fused AdamW
// Decoupled weight decay Adam on a flat fp32 master shard; applies the clip coefficient; refreshes the
// bf16 compute shard.  (torch.optim.AdamW update order.)
template <typename GradT>
__global__ void adamw_kernel(float* __restrict__ master, const GradT* __restrict__ grad, float* __restrict__ m,
                             float* __restrict__ v, __nv_bfloat16* __restrict__ lowp, size_t n, float lr, float b1,
                             float b2, float eps, float wd, float bc1, float bc2_sqrt,
                             const float* __restrict__ grad_scale) {
  const float gs = grad_scale ? *grad_scale : 1.f;
  const float decay = 1.f - lr * wd;
  const float step_size = lr / bc1;
  for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n;
       i += (size_t)gridDim.x * blockDim.x * 4) {
    float4 p = *reinterpret_cast<const float4*>(master + i);
    float4 mm = *reinterpret_cast<const float4*>(m + i);
    float4 vv = *reinterpret_cast<const float4*>(v + i);
    float g[4];
    if constexpr (sizeof(GradT) == 2) {
      uint2 u = *reinterpret_cast<const uint2*>(grad + i);
      float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
      g[0] = a.x; g[1] = a.y; g[2] = b.x; g[3] = b.y;
    } else {
      float4 gg = *reinterpret_cast<const float4*>(grad + i);
      g[0] = gg.x; g[1] = gg.y; g[2] = gg.z; g[3] = gg.w;
    }
    float pp[4] = {p.x, p.y, p.z, p.w}, ma[4] = {mm.x, mm.y, mm.z, mm.w}, va[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = g[k] * gs;
      pp[k] *= decay;
      ma[k] = b1 * ma[k] + (1.f - b1) * gk;
      va[k] = b2 * va[k] + (1.f - b2) * gk * gk;
      const float denom = sqrtf(va[k]) / bc2_sqrt + eps;
      pp[k] -= step_size * ma[k] / denom;
    }
    *reinterpret_cast<float4*>(master + i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
    *reinterpret_cast<float4*>(m + i) = make_float4(ma[0], ma[1], ma[2], ma[3]);
    *reinterpret_cast<float4*>(v + i) = make_float4(va[0], va[1], va[2], va[3]);
    if (lowp) {
      uint2 o;
      o.x = pack_bf16x2(pp[0], pp[1]);
      o.y = pack_bf16x2(pp[2], pp[3]);
      *reinterpret_cast<uint2*>(lowp + i) = o;
    }
  }
}

template <typename T>
__global__ void sumsq_kernel(const T* __restrict__ x, size_t n, float* __restrict__ out) {
  __shared__ float sh[32];
  constexpr int EPV = 16 / sizeof(T);      // elements per 16-byte vector
  constexpr int UNR = 4;                   // vectors in flight per thread
  const size_t nvec = n / EPV;
  const uint4* xv = reinterpret_cast<const uint4*>(x);
  auto acc = [](const uint4& u) -> float {
    if constexpr (sizeof(T) == 2) {
      float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
      return a.x * a.x + a.y * a.y + b.x * b.x + b.y * b.y + c.x * c.x + c.y * c.y + d.x * d.x + d.y * d.y;
    } else {
      const float f0 = __uint_as_float(u.x), f1 = __uint_as_float(u.y), f2 = __uint_as_float(u.z), f3 = __uint_as_float(u.w);
      return f0 * f0 + f1 * f1 + f2 * f2 + f3 * f3;
    }
  };
  float s = 0.f;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + (UNR - 1) * stride < nvec; i += UNR * stride) {
    uint4 u[UNR];
#pragma unroll
    for (int k = 0; k < UNR; ++k) u[k] = xv[i + k * stride];
#pragma unroll
    for (int k = 0; k < UNR; ++k) s += acc(u[k]);
  }
  for (; i < nvec; i += stride) s += acc(xv[i]);
  // tail (n not a multiple of the vector width)
  if (blockIdx.x == 0 && threadIdx.x < (int)(n - nvec * EPV)) {
    const float t = (float)x[nvec * EPV + threadIdx.x];
    s += t * t;
  }
  s = block_sum(s, sh);
  if (threadIdx.x == 0) atomicAdd(out, s);
}

// ------------------------------------------------------------- bias gradient: db[n] = sum_m dy[m, n]
// Deterministic two-pass column sum.  Pass 1: CTA (column block of 256, row slice p) -- 32 lanes x 8 columns (one
// 16-byte load per row, a warp reads 512 contiguous bytes) x 8 warps striding the slice's rows; the warps' sums are
// combined in a fixed order into part[p, n].  Pass 2: one thread per column adds the P partials in order p = 0..P-1.
// The split depends on (M, N) only, so two runs give bitwise-equal results; no atomics.
constexpr int BG_COLS = 256;
__global__ void __launch_bounds__(256) bias_grad_partial_kernel(const __nv_bfloat16* __restrict__ dy, float* __restrict__ part,
                                                                int M, int N, int rows_per) {
  __shared__ float sh[8][BG_COLS + 4];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * BG_COLS + lane * 8;
  const int r0 = blockIdx.y * rows_per, r1 = min(M, r0 + rows_per);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c < N) {
#pragma unroll 4
    for (int r = r0 + w; r < r1; r += 8) {
      const uint4 v = *reinterpret_cast<const uint4*>(dy + (size_t)r * N + c);
      const float2 a = unpack_bf16x2(v.x), b = unpack_bf16x2(v.y), e = unpack_bf16x2(v.z), f = unpack_bf16x2(v.w);
      s[0] += a.x; s[1] += a.y; s[2] += b.x; s[3] += b.y; s[4] += e.x; s[5] += e.y; s[6] += f.x; s[7] += f.y;
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) sh[w][lane * 8 + i] = s[i];
  __syncthreads();
  const int col = blockIdx.x * BG_COLS + threadIdx.x;
  if (col < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += sh[k][threadIdx.x];
    part[(size_t)blockIdx.y * N + col] = t;
  }
}
template <typename OutT>
__global__ void __launch_bounds__(256) bias_grad_final_kernel(const float* __restrict__ part, OutT* __restrict__ out, int P,
                                                              int N, int accumulate) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= N) return;
  float t = 0.f;
  for (int p = 0; p < P; ++p) t += part[(size_t)p * N + col];
  if (accumulate) t += static_cast<float>(out[col]);
  out[col] = static_cast<OutT>(t);
}

static inline int grid_for(size_t work_items, int threads, int max_blocks = 148 * 8) {
  size_t b = (work_items + threads - 1) / threads;
  if (b < 1) b = 1;
  return (int)(b > (size_t)max_blocks ? max_blocks : b);
}

}  // namespace b200

using namespace b200;
#define CK() return (int)cudaGetLastError()

extern "C" int b200_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd, int M, int D, float eps,
                                cudaStream_t s) {
  if (D % 8 || D > NT * 8 * MAXC) return -1;
  const int grid = M < 148 * 6 ? M : 148 * 6;
  const int nc = (D + NT * 8 - 1) / (NT * 8);
#define B200_RMS_FWD(NCV)                                                                                     \
  rmsnorm_fwd_kernel<NCV><<<grid, NT, 0, s>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)w, (__nv_bfloat16*)y, \
                                              rstd, M, D, eps)
  if (nc == 1) B200_RMS_FWD(1); else if (nc == 2) B200_RMS_FWD(2); else if (nc == 3) B200_RMS_FWD(3); else B200_RMS_FWD(4);
#undef B200_RMS_FWD
  CK();
}
extern "C" int b200_rmsnorm_bwd_grid(int M) { return M < 148 * 4 ? M : 148 * 4; }
extern "C" int b200_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rstd, const void* dres,
                                void* dx, float* dw_part, float* dw, int M, int D, cudaStream_t s) {
  if (D % 8 || D > NT * 8 * MAXC) return -1;
  const int grid = b200_rmsnorm_bwd_grid(M);
  const int nc = (D + NT * 8 - 1) / (NT * 8);
#define B200_RMS_BWD(NCV)                                                                                       \
  rmsnorm_bwd_kernel<NCV><<<grid, NT, 0, s>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x,                 \
                                              (const __nv_bfloat16*)w, rstd, (const __nv_bfloat16*)dres,     \
                                              (__nv_bfloat16*)dx, dw_part, M, D)
  if (nc == 1) B200_RMS_BWD(1); else if (nc == 2) B200_RMS_BWD(2); else if (nc == 3) B200_RMS_BWD(3); else B200_RMS_BWD(4);
#undef B200_RMS_BWD
  colsum_kernel<<<(D + 31) / 32, 256, 0, s>>>(dw_part, dw, grid, D);
  CK();
}
extern "C" int b200_add_rmsnorm_fwd(const void* x, const float* res, const void* w, void* y, float* res_out, float* rstd,
                                    int M, int D, float eps, cudaStream_t s) {
  if (D % 8 || D > NT * 8 * MAXC) return -1;
  add_rmsnorm_fwd_kernel<<<M < 148 * 8 ? M : 148 * 8, NT, 0, s>>>((const __nv_bfloat16*)x, res, (const __nv_bfloat16*)w,
                                                                 (__nv_bfloat16*)y, res_out, rstd, M, D, eps);
  CK();
}
extern "C" int b200_rmsnorm_bwd_f32(const void* dy, const float* x, const void* w, const float* rstd, float* dx,
                                    float* dw_part, float* dw, int M, int D, cudaStream_t s) {
  if (D % 8 || D > NT * 8 * MAXC) return -1;
  const int grid = b200_rmsnorm_bwd_grid(M);
  rmsnorm_bwd_f32_kernel<<<grid, NT, 0, s>>>((const __nv_bfloat16*)dy, x, (const __nv_bfloat16*)w, rstd, dx, dw_part, M, D);
  colsum_kernel<<<(D + 31) / 32, 256, 0, s>>>(dw_part, dw, grid, D);
  CK();
}
extern "C" int b200_rmsnorm_gated_fwd(const void* x, const void* z, const void* w, void* y, float* rstd, int M, int D,
                                      float eps, cudaStream_t s) {
  if (D % 8 || D > NT * 8 * MAXC) return -1;
  rmsnorm_gated_fwd_kernel<<<M < 148 * 8 ? M : 148 * 8, NT, 0, s>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)z,
                                                                   (const __nv_bfloat16*)w, (__nv_bfloat16*)y, rstd, M, D, eps);
  CK();
}
extern "C" int b200_rmsnorm_gated_bwd(const void* dy, const void* x, const void* z, const void* w, const float* rstd,
                                      void* dx, void* dz, float* dw_part, float* dw, int M, int D, cudaStream_t s) {
  if (D % 8 || D > NT * 8 * MAXC) return -1;
  const int grid = b200_rmsnorm_bwd_grid(M);
  rmsnorm_gated_bwd_kernel<<<grid, NT, 0, s>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (const __nv_bfloat16*)z,
                                               (const __nv_bfloat16*)w, rstd, (__nv_bfloat16*)dx, (__nv_bfloat16*)dz, dw_part,
                                               M, D);
  colsum_kernel<<<(D + 31) / 32, 256, 0, s>>>(dw_part, dw, grid, D);
  CK();
}
extern "C" int b200_rope(void* qkv, const float* table, int M, int seq_len, int row_stride, int nrot_heads, int hd,
                         int rot, int inverse, int pos_offset, int interleaved, cudaStream_t s) {
  if (rot % 16 || hd % 8 || row_stride % 8) return -1;
  if (interleaved) {
    rope_kernel<<<(M < 148 * 8 ? M : 148 * 8), 256, 0, s>>>((__nv_bfloat16*)qkv, table, M, seq_len, row_stride, nrot_heads,
                                                     hd, rot, inverse ? -1.f : 1.f, pos_offset);
  } else {
    size_t total = (size_t)M * nrot_heads * (rot / 16);
    rope_halfsplit_kernel<<<grid_for(total, 256), 256, 0, s>>>((__nv_bfloat16*)qkv, table, M, seq_len, row_stride,
                                                               nrot_heads, hd, rot, inverse ? -1.f : 1.f, pos_offset);
  }
  CK();
}
extern "C" int b200_swiglu_fwd(const void* gu, void* out, long long M, int F, int gate_first, cudaStream_t s) {
  if (F % 8) return -1;
  swiglu_fwd_kernel<<<grid_for((size_t)M * (F / 8), 256), 256, 0, s>>>((const __nv_bfloat16*)gu, (__nv_bfloat16*)out,
                                                                       (size_t)M, F, gate_first ? 0 : F,
                                                                       gate_first ? F : 0);
  CK();
}
extern "C" int b200_swiglu_bwd(const void* ds, const void* gu, void* dgu, long long M, int F, int gate_first,
                               cudaStream_t s) {
  if (F % 8) return -1;
  swiglu_bwd_kernel<<<grid_for((size_t)M * (F / 8), 256), 256, 0, s>>>(
      (const __nv_bfloat16*)ds, (const __nv_bfloat16*)gu, (__nv_bfloat16*)dgu, (size_t)M, F, gate_first ? 0 : F,
      gate_first ? F : 0);
  CK();
}
extern "C" int b200_embedding_fwd(const void* tok, int tok_is_i64, const void* w, void* out, long long M, int D,
                                  cudaStream_t s) {
  if (D % 8) return -1;
  int g = grid_for((size_t)M * (D / 8), 256);
  if (tok_is_i64)
    embedding_fwd_kernel<long long><<<g, 256, 0, s>>>((const long long*)tok, (const __nv_bfloat16*)w,
                                                      (__nv_bfloat16*)out, (size_t)M, D);
  else
    embedding_fwd_kernel<int><<<g, 256, 0, s>>>((const int*)tok, (const __nv_bfloat16*)w, (__nv_bfloat16*)out,
                                                (size_t)M, D);
  CK();
}
extern "C" int b200_embedding_bwd(const void* tok, int tok_is_i64, const void* dx, void* dw, int dw_is_f32,
                                  long long M, int D, cudaStream_t s) {
  if (D % 2) return -1;
  if (dw_is_f32) {
    int g = grid_for((size_t)M * D, 256);
    if (tok_is_i64)
      embedding_bwd_f32_kernel<long long><<<g, 256, 0, s>>>((const long long*)tok, (const __nv_bfloat16*)dx,
                                                            (float*)dw, (size_t)M, D);
    else
      embedding_bwd_f32_kernel<int><<<g, 256, 0, s>>>((const int*)tok, (const __nv_bfloat16*)dx, (float*)dw,
                                                      (size_t)M, D);
  } else {
    int g = grid_for((size_t)M * (D / 2), 256);
    if (tok_is_i64)
      embedding_bwd_kernel<long long><<<g, 256, 0, s>>>((const long long*)tok, (const __nv_bfloat16*)dx,
                                                        (__nv_bfloat16*)dw, (size_t)M, D);
    else
      embedding_bwd_kernel<int><<<g, 256, 0, s>>>((const int*)tok, (const __nv_bfloat16*)dx, (__nv_bfloat16*)dw,
                                                  (size_t)M, D);
  }
  CK();
}
extern "C" int b200_count_valid(const long long* labels, int M, long long ignore, float* n_valid, cudaStream_t s) {
  count_valid_kernel<<<grid_for((size_t)M, 256, 64), 256, 0, s>>>(labels, M, ignore, n_valid);
  CK();
}
extern "C" int b200_ce_grad_inplace(void* logits, const long long* labels, const float* n_valid, float* loss_sum,
                                    int rows, int V, int ld, long long ignore, cudaStream_t s) {
  if (V % 8 || ld % 8) return -1;
  ce_grad_inplace_kernel<<<rows < 148 * 8 ? rows : 148 * 8, NT, 0, s>>>((__nv_bfloat16*)logits, labels, n_valid,
                                                                       loss_sum, rows, V, ld, ignore);
  CK();
}
extern "C" int b200_adamw(float* master, const void* grad, int grad_is_bf16, float* m, float* v, void* lowp,
                          long long n, float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt,
                          const float* grad_scale, cudaStream_t s) {
  if (n % 4) return -1;
  int g = grid_for((size_t)n / 4, 256, 148 * 16);
  if (grad_is_bf16)
    adamw_kernel<__nv_bfloat16><<<g, 256, 0, s>>>(master, (const __nv_bfloat16*)grad, m, v, (__nv_bfloat16*)lowp,
                                                  (size_t)n, lr, b1, b2, eps, wd, bc1, bc2_sqrt, grad_scale);
  else
    adamw_kernel<float><<<g, 256, 0, s>>>(master, (const float*)grad, m, v, (__nv_bfloat16*)lowp, (size_t)n, lr, b1,
                                          b2, eps, wd, bc1, bc2_sqrt, grad_scale);
  CK();
}
extern "C" int b200_sumsq(const void* x, int is_bf16, long long n, float* out, cudaStream_t s) {
  if (reinterpret_cast<uintptr_t>(x) & 15) return -1;
  int g = grid_for((size_t)n / 16, 256, 148 * 8);
  if (is_bf16) sumsq_kernel<__nv_bfloat16><<<g, 256, 0, s>>>((const __nv_bfloat16*)x, (size_t)n, out);
  else sumsq_kernel<float><<<g, 256, 0, s>>>((const float*)x, (size_t)n, out);
  CK();
}

// ------------------------------------------------------------------------------------------------------------------
// Row-wise e4m3 quantisation for the optional fp8 forward GEMMs: one warp per row; scale[row] = amax(row) / 448 (the
// largest finite e4m3 value), q = x / scale rounded to nearest, saturating.  The second pass re-reads the row from L1/L2.
namespace b200 {
B200_DEVINL uint32_t cvt_e4m3x4(float a, float b, float c, float d) {
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));   // {second operand -> low byte}
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
  return (uint32_t)lo | ((uint32_t)hi << 16);
}
__global__ void __launch_bounds__(256) quant_rowwise_e4m3_kernel(const __nv_bfloat16* __restrict__ x, uint8_t* __restrict__ q,
                                                                 float* __restrict__ scale, int rows, int K, int ldx, int ldq) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const __nv_bfloat16* xr = x + (size_t)row * ldx;
  float amax = 0.f;
  for (int c = lane * 8; c < K; c += 256) {
    const uint4 v = *reinterpret_cast<const uint4*>(xr + c);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = unpack_bf16x2(w[i]);
      amax = fmaxf(amax, fmaxf(fabsf(f.x), fabsf(f.y)));
    }
  }
  amax = warp_max(amax);
  const float sc = amax > 0.f ? amax * (1.f / 448.f) : 1.f;
  const float inv = 1.f / sc;
  if (lane == 0) scale[row] = sc;
  uint8_t* qr = q + (size_t)row * ldq;
  for (int c = lane * 8; c < K; c += 256) {
    const uint4 v = *reinterpret_cast<const uint4*>(xr + c);
    const float2 a = unpack_bf16x2(v.x), b = unpack_bf16x2(v.y), e = unpack_bf16x2(v.z), f = unpack_bf16x2(v.w);
    uint2 o;
    o.x = cvt_e4m3x4(a.x * inv, a.y * inv, b.x * inv, b.y * inv);
    o.y = cvt_e4m3x4(e.x * inv, e.y * inv, f.x * inv, f.y * inv);
    *reinterpret_cast<uint2*>(qr + c) = o;
  }
}
}  // namespace b200

extern "C" int b200_quant_rowwise_e4m3(const void* x, void* q, float* scale, int rows, int K, int ldx, int ldq, cudaStream_t s) {
  if ((K % 8) || (ldx % 8) || (ldq % 8)) return -1;
  const int warps = 8;
  b200::quant_rowwise_e4m3_kernel<<<(rows + warps - 1) / warps, warps * 32, 0, s>>>((const __nv_bfloat16*)x, (uint8_t*)q, scale,
                                                                                   rows, K, ldx, ldq);
  return (int)cudaGetLastError();
}

// db[N] (bf16 or fp32; written, or added to when accumulate) = column sums of dy [M, N] bf16 (row pitch N).
// part: fp32 workspace of b200_bias_grad_partials(M, N) x N elements.
extern "C" int b200_bias_grad_partials(int M, int N) {
  const int col_blocks = (N + b200::BG_COLS - 1) / b200::BG_COLS;
  int P = (148 * 4 + col_blocks - 1) / col_blocks;     // about four CTAs per SM in pass 1
  const int max_p = (M + 63) / 64;                     // at least 64 rows per slice
  if (P > max_p) P = max_p;
  if (P < 1) P = 1;
  const int rows_per = (M + P - 1) / P;
  return M > 0 ? (M + rows_per - 1) / rows_per : 1;
}
extern "C" int b200_bias_grad(const void* dy, float* part, void* db, int db_is_f32, int M, int N, int accumulate,
                              cudaStream_t s) {
  if ((N % 8) || M < 0 || (reinterpret_cast<uintptr_t>(dy) & 15)) return -1;
  const int P = b200_bias_grad_partials(M, N);
  const int rows_per = M > 0 ? (M + P - 1) / P : 1;
  b200::bias_grad_partial_kernel<<<dim3((N + b200::BG_COLS - 1) / b200::BG_COLS, P), 256, 0, s>>>(
      (const __nv_bfloat16*)dy, part, M, N, rows_per);
  if (db_is_f32)
    b200::bias_grad_final_kernel<float><<<(N + 255) / 256, 256, 0, s>>>(part, (float*)db, P, N, accumulate);
  else
    b200::bias_grad_final_kernel<__nv_bfloat16><<<(N + 255) / 256, 256, 0, s>>>(part, (__nv_bfloat16*)db, P, N, accumulate);
  return (int)cudaGetLastError();
}
