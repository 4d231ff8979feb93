// 2-CTA (cta_group::2) persistent bf16 GEMM for sm_100a: a cluster of two CTAs computes a 256x256 output
// tile with ONE tcgen05.mma stream issued by the leader CTA.  Each CTA stages 128 rows of A and 128 of the
// 256 B rows per k-block (32 KiB/stage instead of 48 KiB) -- the single-CTA kernel in gemm_sm100.cu is
// shared-memory-bandwidth bound (TMA writes + UMMA operand reads = 192 B/clk/SM > 128 B/clk); pairing halves
// the B traffic per SM (128 B/clk) and lets the ring go 6 stages deep.
//
// Same operand layouts / epilogues / warp roles as gemm_sm100.cu.  Differences:
//   * __cluster_dims__(2,1,1); TMEM allocated with cta_group::2; TMA loads use the cta_group::2 form so the
//     bytes of BOTH CTAs complete on the leader's "full" barrier;
//   * only the leader's warp 1 issues MMAs; tcgen05.commit multicasts to the "empty"/"accumulator full"
//     barriers of both CTAs; both CTAs' epilogue warps arrive on the leader's "accumulator empty" barrier.
#include "common.cuh"
#include "tensormap.h"

namespace b200 {

constexpr int P_BM = 256;       // rows per CTA pair
constexpr int C_BM = 128;       // rows per CTA
constexpr int P_BN = 256;       // tile columns
constexpr int C_BN = 128;       // B rows staged per CTA
constexpr int P_BK = 64;
constexpr int P_STAGES = 6;
constexpr int PA_BYTES = C_BM * P_BK * 2;   // 16 KiB
constexpr int PB_BYTES = C_BN * P_BK * 2;   // 16 KiB
constexpr int P_STAGE_BYTES = PA_BYTES + PB_BYTES;
constexpr int P_THREADS = 192;
constexpr int P_SMEM = P_STAGES * P_STAGE_BYTES + 1024 + 256;
// push epilogue: each epilogue warp stages 32 rows x 64 bf16 columns (128 B, row pitch 144 B: 16-byte accesses of a
// quarter-warp hit 32 distinct banks) so that every row leaves the SM as ONE 128-byte bulk store over NVLink
constexpr int PUSH_ROW_PITCH = 144;
constexpr int PUSH_STAGE_BYTES = 4 * 32 * PUSH_ROW_PITCH;   // 18 KiB per CTA

enum { P_EPI_STORE = 0, P_EPI_RESIDUAL = 1, P_EPI_ACCUM = 2, P_EPI_ROPE = 3, P_EPI_PUSH = 4, P_EPI_SWIGLU = 5,
       P_EPI_SWIGLU_BWD = 6, P_EPI_SCALE = 7 };
// flag OR-ed into P_EPI_STORE / P_EPI_ROPE: add the bf16 bias b[col] (16-byte aligned, [N]; passed in Gemm2Params::R)
// to the fp32 accumulator before anything else the epilogue does (qkv = x W^T + b, then RoPE).  A flag bit of the
// same template argument keeps the bias-free instantiations' names, parameter layout and code exactly as they were.
constexpr int P_EPI_BIAS = 16;


// L2-friendly rasterisation: sweep all n-tiles for a band of GROUP_M m-tiles before moving to the next band, so the
// band's A rows (GROUP_M x 256 x K) stay L2-resident while B streams through once per band.
constexpr int P_GROUP_M = 8;
B200_DEVINL void tile_coords2(int t, int m_tiles, int n_tiles, int& mt, int& nt) {
  const int per_band = P_GROUP_M * n_tiles;
  const int band = t / per_band;
  const int first_m = band * P_GROUP_M;
  const int band_m = min(P_GROUP_M, m_tiles - first_m);
  const int r = t - band * per_band;
  mt = first_m + r % band_m;
  nt = r / band_m;
}

// ---- fused all-gather (ag_gemm): extra "comm" warps of the same persistent GEMM pull a unit's parameter shards from
// the 7 peers over NVLink (16-byte ld.relaxed.sys on symmetric-heap addresses) into the local gathered buffer and
// publish per-chunk ready flags.  dependent=1: the B operand of THIS GEMM lives in that buffer, so the TMA producer
// acquires the flags of the chunks under each B tile before issuing its loads -- weights flow peer HBM -> NVLink ->
// local L2 -> TMA -> smem -> tcgen05 tile by tile while the tensor core works on the tiles that already landed.
// dependent=0: the gather is the NEXT unit's prefetch riding inside this GEMM.
constexpr int AG_CHUNK = 65536;       // bytes per ready flag
constexpr int AG_WARPS = 2;           // comm warps per CTA
struct AgParams {
  const void* const* peer_shards;     // device table [world] of shard base addresses (own rank included)
  uint8_t* full;                      // local gathered buffer
  unsigned long long shard_bytes;
  unsigned long long begin, end;      // byte range of `full` to gather
  int world, rank;
  uint32_t* flags;                    // [ceil(total/AG_CHUNK)] epochs, local memory
  uint32_t epoch;
  int dependent;
  unsigned long long b_off;           // byte offset of the B matrix inside `full`
  unsigned long long b_row_bytes;     // bytes per stored B row (ldb * 2)
};

B200_DEVINL uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
B200_DEVINL void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
B200_DEVINL uint4 ld_peer_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.relaxed.sys.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
// block until chunks [lo, hi] of the gathered buffer have been published for this epoch
B200_DEVINL void ag_wait_chunks(const AgParams& ag, unsigned long long byte_lo, unsigned long long byte_hi) {
  if (byte_lo < ag.begin) byte_lo = ag.begin;
  if (byte_hi > ag.end) byte_hi = ag.end;
  if (byte_hi <= byte_lo) return;
  const unsigned c0 = (unsigned)(byte_lo / AG_CHUNK), c1 = (unsigned)((byte_hi - 1) / AG_CHUNK);
  for (unsigned c = c0; c <= c1; ++c) {
    uint64_t t0 = 0;
    uint32_t spins = 0;
    while (ld_acquire_gpu(ag.flags + c) != ag.epoch) {
      if ((++spins & 0x3ff) == 0) {
        uint64_t now = global_timer_ns();
        if (t0 == 0) t0 = now;
        else if (now - t0 > B200_WAIT_TIMEOUT_NS) __trap();
      }
    }
  }
  asm volatile("fence.proxy.async;" ::: "memory");  // generic-proxy writes of the comm warps -> TMA (async proxy) reads
}

struct Gemm2Params {
  int M, N, K;
  int ldc, ldr;
  void* C;
  const void* R;
  int m_tiles, n_tiles;  // in units of 256 x 256
  // P_EPI_ROPE (QKV projection): rotate adjacent column pairs of the first rope_cols columns by the angle of
  // (row % rope_S, (col % rope_hd) / 2) before the bf16 store; table is [S][hd/2][cos, sin] fp32 (SURVEY.md K2)
  const float* rope;
  int rope_S, rope_hd, rope_cols;
  // P_EPI_PUSH (fused wgrad GEMM -> reduce-scatter, SURVEY.md N8): the wgrad tile is not stored to C but pushed over
  // NVLink into the staging buffer of the rank that OWNS that slice of the unit's flat gradient:
  //   e = push_off + row * ldc + col ; owner = e / push_n ; dst = push_bases[owner] + push_rank * push_n + (e - owner * push_n)
  // so that after one cross-rank flag round each owner sums `world` LOCAL slots (no NVLink traffic of its own).
  // push_bulk = 1: rows are staged in shared memory and leave as 128-byte cp.async.bulk stores (one per row and
  // 64-column chunk); 0: 16-byte st.global per lane (kept as the reference path for the numerics test).
  void* const* push_bases;
  long long push_n, push_off;
  int push_rank, push_bulk;
  // every CTA pair starts its sweep `tile_rot` tiles into the raster (wraps around).  The push epilogue sets it to
  // rank * tiles / world: all ranks run the same wgrad GEMM at the same time with the same raster, so without the
  // rotation all W ranks write into the SAME owner's staging buffer at once (W -> 1 incast on that GPU's NVLink ingress,
  // ~7 x 175 GB/s) while the other owners' links idle.
  int tile_rot;
  // P_EPI_SWIGLU (gate/up projection, nt; SURVEY.md K6/K7): B is the fused [2F, K] weight.  The CTA pair's 256-wide
  // accumulator holds rows [n0, n0+128) of the FIRST half of the weight in columns [0,128) and the same features of the
  // SECOND half in columns [128,256) (CTA rank r stages weight rows n0 + r*F), so every epilogue lane has gate and up of
  // the same feature: it stores the bf16 projection to C [M, 2F] (needed by the backward) AND silu(gate) * up to
  // aux [M, F].  N of the launch = F.
  // P_EPI_SWIGLU_BWD (down-projection dgrad, nn): the accumulator is dS [M, F]; the epilogue reads gate / up from
  // aux = the saved projection [M, 2F] and stores d(gate) | d(up) to C [M, 2F] -- dS itself never reaches memory.
  void* aux;
  int ld_aux, swi_F, swi_gate_first;
  // P_EPI_SCALE (fp8 e4m3 operands, FP8 = true): C = acc * scale_a[row] * scale_b[col]  (row-wise scales of both
  // quantised operands; the optional reduced-precision forward path, default off)
  const float* scale_a;
  const float* scale_b;
};

B200_DEVINL float sigmoidf_fast(float x) { return __frcp_rn(1.f + exp2f(-1.4426950408889634f * x)); }

B200_DEVINL void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}

template <bool A_MN, bool B_MN, int EPI_BITS, typename OutT, bool AG, bool FP8 = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(P_THREADS + (AG ? 32 * AG_WARPS : 0), 1)
gemm2_bf16_tcgen05(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, Gemm2Params p,
                   AgParams ag) {
  constexpr int EPI = EPI_BITS & ~P_EPI_BIAS;
  constexpr bool BIAS = (EPI_BITS & P_EPI_BIAS) != 0;
  static_assert(!BIAS || ((EPI == P_EPI_STORE || EPI == P_EPI_ROPE) && sizeof(OutT) == 2), "bias: bf16 store / RoPE only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* bar_base = smem + P_STAGES * P_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(bar_base);   // leader's copy is the one in use
  uint64_t* empty_bar = full_bar + P_STAGES;                    // per CTA
  uint64_t* tfull_bar = empty_bar + P_STAGES;                   // per CTA
  uint64_t* tempty_bar = tfull_bar + 2;                         // leader's copy is the one in use
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  // elements per k-block: one 128-byte swizzle atom per row = 64 bf16 or 128 e4m3
  constexpr int BKE = FP8 ? 2 * P_BK : P_BK;
  static_assert(!FP8 || (!A_MN && !B_MN && !AG), "fp8 operands: K-major (nt) only, no fused gather");
  const int num_kb = (p.K + BKE - 1) / BKE;
  const int num_tiles = p.m_tiles * p.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < P_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 8);  // 4 epilogue warps x 2 CTAs
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2cta(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // both CTAs' barriers are initialised before anyone signals across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (one per CTA: its own A rows and its half of B) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = pair; t < num_tiles; t += n_pairs) {
        int mt, nt;
        tile_coords2((t + p.tile_rot) % num_tiles, p.m_tiles, p.n_tiles, mt, nt);
        const int m0 = mt * P_BM + (int)rank * C_BM;
        const int n0 = (EPI == P_EPI_SWIGLU) ? nt * C_BN + (int)rank * p.swi_F : nt * P_BN + (int)rank * C_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * P_STAGE_BYTES;
          uint8_t* sb = sa + PA_BYTES;
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * P_STAGE_BYTES);
          const int k0 = kb * BKE;
          if constexpr (AG) {
            if (ag.dependent) {
              // stored rows of B under this CTA's loads: K-major -> rows [n0, n0+128) (once per tile);
              // MN-major -> rows [k0, k0+64) (every k-block)
              if constexpr (!B_MN) {
                if (kb == 0) ag_wait_chunks(ag, ag.b_off + (unsigned long long)n0 * ag.b_row_bytes,
                                            ag.b_off + (unsigned long long)min(n0 + C_BN, p.N) * ag.b_row_bytes);
              } else {
                ag_wait_chunks(ag, ag.b_off + (unsigned long long)k0 * ag.b_row_bytes,
                               ag.b_off + (unsigned long long)min(k0 + P_BK, p.K) * ag.b_row_bytes);
              }
            }
          }
          if constexpr (!A_MN) {
            tma_load_2d_2cta(sa, &tmA, &full_bar[stage], k0, m0);
          } else {
#pragma unroll
            for (int j = 0; j < C_BM / 64; ++j)
              tma_load_2d_2cta(sa + j * (64 * P_BK * 2), &tmA, &full_bar[stage], m0 + 64 * j, k0);
          }
          if constexpr (!B_MN) {
            tma_load_2d_2cta(sb, &tmB, &full_bar[stage], k0, n0);
          } else {
#pragma unroll
            for (int j = 0; j < C_BN / 64; ++j)
              tma_load_2d_2cta(sb + j * (64 * P_BK * 2), &tmB, &full_bar[stage], n0 + 64 * j, k0);
          }
          if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      constexpr uint32_t idesc = FP8 ? make_idesc_e4m3(P_BM, P_BN) : make_idesc_bf16(P_BM, P_BN, A_MN, B_MN);
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int t = pair; t < num_tiles; t += n_pairs) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * P_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (elect_one()) {   // single elected lane: back-to-back UTCHMMA, descriptors = per-stage base + constant
            const uint32_t sa = smem_u32(smem + stage * P_STAGE_BYTES);
            const uint32_t sb = sa + PA_BYTES;
            const uint64_t a0 = make_smem_desc(sa, A_MN ? 64 * P_BK * 2 : 0, 1024);
            const uint64_t b0 = make_smem_desc(sb, B_MN ? 64 * P_BK * 2 : 0, 1024);
#pragma unroll
            for (int k = 0; k < P_BK / 16; ++k) {
              const uint64_t adesc = a0 + ((A_MN ? k * 2048 : k * 32) >> 4);
              const uint64_t bdesc = b0 + ((B_MN ? k * 2048 : k * 32) >> 4);
              if constexpr (FP8) umma_e4m3_ss_2cta(tmem_d, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
              else umma_bf16_ss_2cta(tmem_d, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit_2cta_mcast(&empty_bar[stage], 0x3);
            if (kb == num_kb - 1) umma_commit_2cta_mcast(&tfull_bar[acc], 0x3);
          }
          __syncwarp();
          if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (AG && warp >= 6) {
    // ===================== comm warps: pull peer shards into the local gathered buffer =====================
    if constexpr (AG) {
      const int ct = (warp - 6) * 32 + lane;              // 0 .. 63
      const unsigned long long total = ag.end - ag.begin;
      const unsigned n_chunks = (unsigned)((total + AG_CHUNK - 1) / AG_CHUNK);
      const unsigned first = (unsigned)(ag.begin / AG_CHUNK);
      // rotate the start so the 8 ranks do not all hit the same peer first
      const unsigned rot = (unsigned)(((unsigned long long)ag.rank * n_chunks) / (unsigned)ag.world);
      for (unsigned i = blockIdx.x; i < n_chunks; i += gridDim.x) {
        const unsigned ci = ag.dependent ? i : (i + rot) % n_chunks;   // dependent mode keeps B-first order
        const unsigned long long lo = ag.begin + (unsigned long long)ci * AG_CHUNK;
        const unsigned long long hi = (lo + AG_CHUNK < ag.end) ? lo + AG_CHUNK : ag.end;
        const unsigned nvec = (unsigned)((hi - lo) / 16);
        const unsigned src_lo = (unsigned)(lo / ag.shard_bytes), src_hi = (unsigned)((hi - 1) / ag.shard_bytes);
        const uint8_t* base_lo = reinterpret_cast<const uint8_t*>(ag.peer_shards[src_lo]) - (unsigned long long)src_lo * ag.shard_bytes;
        const uint8_t* base_hi = reinterpret_cast<const uint8_t*>(ag.peer_shards[src_hi]) - (unsigned long long)src_hi * ag.shard_bytes;
        const unsigned long long split = (unsigned long long)src_hi * ag.shard_bytes;  // a chunk spans <= 2 shards
        for (unsigned v0 = ct; v0 < nvec; v0 += 64 * 8) {
          uint4 buf[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const unsigned v = v0 + u * 64;
            if (v < nvec) {
              const unsigned long long off = lo + (unsigned long long)v * 16;
              buf[u] = ld_peer_v4(((src_lo != src_hi && off >= split) ? base_hi : base_lo) + off);
            }
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const unsigned v = v0 + u * 64;
            if (v < nvec) *reinterpret_cast<uint4*>(ag.full + lo + (unsigned long long)v * 16) = buf[u];
          }
        }
        __threadfence();
        asm volatile("bar.sync 2, 64;" ::: "memory");      // both comm warps finished this chunk
        if (ct == 0) {
          asm volatile("fence.proxy.async;" ::: "memory");
          st_release_gpu(ag.flags + first + ci, ag.epoch);
        }
      }
    }
  } else {
    // ===================== epilogue (both CTAs: own 128 accumulator lanes) =====================
    const int q = warp & 3;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = pair; t < num_tiles; t += n_pairs) {
      int mt, nt;
      tile_coords2((t + p.tile_rot) % num_tiles, p.m_tiles, p.n_tiles, mt, nt);
      const int m0 = mt * P_BM + (int)rank * C_BM;
      const int n0 = nt * P_BN;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const int row = m0 + q * 32 + lane;
      const bool row_ok = row < p.M;
      OutT* crow = reinterpret_cast<OutT*>(p.C) + static_cast<size_t>(row) * p.ldc;
      const __nv_bfloat16* rrow = reinterpret_cast<const __nv_bfloat16*>(p.R) + static_cast<size_t>(row) * p.ldr;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * P_BN;
      if constexpr (EPI == P_EPI_SWIGLU) {
        // columns [0,128) = first half of the fused projection, [128,256) = second half, same 128 features
        const int f0 = nt * C_BN;
        __nv_bfloat16* arow = reinterpret_cast<__nv_bfloat16*>(p.aux) + static_cast<size_t>(row) * p.ld_aux;
#pragma unroll 1
        for (int c = 0; c < C_BN; c += 32) {
          uint32_t a[32], b[32];
          tmem_ld_32x32b_x32(taddr + c, a);
          tmem_ld_32x32b_x32(taddr + C_BN + c, b);
          tmem_ld_wait();
          if (row_ok && f0 + c < p.swi_F) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              uint4 o1, o2, oa;
              uint32_t* w1 = reinterpret_cast<uint32_t*>(&o1);
              uint32_t* w2 = reinterpret_cast<uint32_t*>(&o2);
              uint32_t* wa = reinterpret_cast<uint32_t*>(&oa);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                w1[i] = pack_bf16x2(__uint_as_float(a[g * 8 + 2 * i]), __uint_as_float(a[g * 8 + 2 * i + 1]));
                w2[i] = pack_bf16x2(__uint_as_float(b[g * 8 + 2 * i]), __uint_as_float(b[g * 8 + 2 * i + 1]));
                // activation from the ROUNDED projection: forward and backward see the same gate / up values
                const float2 x1 = unpack_bf16x2(w1[i]), x2 = unpack_bf16x2(w2[i]);
                const float2 gt = p.swi_gate_first ? x1 : x2, up = p.swi_gate_first ? x2 : x1;
                wa[i] = pack_bf16x2(gt.x * sigmoidf_fast(gt.x) * up.x, gt.y * sigmoidf_fast(gt.y) * up.y);
              }
              const int col = f0 + c + g * 8;
              *reinterpret_cast<uint4*>(crow + col) = o1;
              *reinterpret_cast<uint4*>(crow + p.swi_F + col) = o2;
              *reinterpret_cast<uint4*>(arow + col) = oa;
            }
          }
        }
      } else if constexpr (EPI == P_EPI_SWIGLU_BWD) {
        const __nv_bfloat16* grow = reinterpret_cast<const __nv_bfloat16*>(p.aux) + static_cast<size_t>(row) * p.ld_aux;
        // 64 columns per step: every lane reads whole 128-byte lines of its row's gate and up values (all 16 loads are
        // issued before the TMEM wait, so their latency overlaps it) -- 32-column steps fetched every line twice
#pragma unroll 1
        for (int c = 0; c < P_BN; c += 64) {
          const int col = n0 + c;
          const bool live = row_ok && col < p.N;
          uint4 r1[8], r2[8];
          if (live) {
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              if (col + g * 8 < p.N) {
                r1[g] = *reinterpret_cast<const uint4*>(grow + col + g * 8);
                r2[g] = *reinterpret_cast<const uint4*>(grow + p.swi_F + col + g * 8);
              }
            }
          }
          uint32_t d[64];
          tmem_ld_32x32b_x32(taddr + c, *reinterpret_cast<uint32_t(*)[32]>(&d[0]));
          tmem_ld_32x32b_x32(taddr + c + 32, *reinterpret_cast<uint32_t(*)[32]>(&d[32]));
          tmem_ld_wait();
          if (live) {
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              if (col + g * 8 >= p.N) break;
              const uint32_t* q1 = reinterpret_cast<const uint32_t*>(&r1[g]);
              const uint32_t* q2 = reinterpret_cast<const uint32_t*>(&r2[g]);
              uint4 o1, o2;
              uint32_t* w1 = reinterpret_cast<uint32_t*>(&o1);
              uint32_t* w2 = reinterpret_cast<uint32_t*>(&o2);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float2 x1 = unpack_bf16x2(q1[i]), x2 = unpack_bf16x2(q2[i]);
                const float2 gt = p.swi_gate_first ? x1 : x2, up = p.swi_gate_first ? x2 : x1;
                const float ds0 = __uint_as_float(d[g * 8 + 2 * i]), ds1 = __uint_as_float(d[g * 8 + 2 * i + 1]);
                const float s0 = sigmoidf_fast(gt.x), s1 = sigmoidf_fast(gt.y);
                const float dg0 = ds0 * up.x * s0 * (1.f + gt.x * (1.f - s0)), dg1 = ds1 * up.y * s1 * (1.f + gt.y * (1.f - s1));
                const float du0 = ds0 * gt.x * s0, du1 = ds1 * gt.y * s1;
                const uint32_t pg = pack_bf16x2(dg0, dg1), pu = pack_bf16x2(du0, du1);
                w1[i] = p.swi_gate_first ? pg : pu;
                w2[i] = p.swi_gate_first ? pu : pg;
              }
              *reinterpret_cast<uint4*>(crow + col + g * 8) = o1;
              *reinterpret_cast<uint4*>(crow + p.swi_F + col + g * 8) = o2;
            }
          }
        }
      } else {
#pragma unroll 1
      for (int c = 0; c < P_BN; c += 64) {
        uint4 bias8[BIAS ? 8 : 1];
        if constexpr (BIAS) {   // the chunk's 64 bias values, loaded before the TMEM wait so that their latency overlaps it;
                                // every lane of the warp reads the same bytes (broadcast)
#pragma unroll
          for (int g = 0; g < 8; ++g)
            if (n0 + c + g * 8 < p.N)
              bias8[g] = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.R) + n0 + c + g * 8);
        }
        uint32_t v0[32], v1[32];
        tmem_ld_32x32b_x32(taddr + c, v0);
        tmem_ld_32x32b_x32(taddr + c + 32, v1);
        tmem_ld_wait();
        const int col = n0 + c;
        if constexpr (EPI == P_EPI_PUSH) {
          if (p.push_bulk) {
            uint8_t* stg = bar_base + 256 + (q * 32 + lane) * PUSH_ROW_PITCH;
            // the bulk store issued from this staging row two chunks ago has finished READING it
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            if (row_ok && col < p.N) {
              const int ncols = min(64, p.N - col);            // multiple of 8
#pragma unroll
              for (int g = 0; g < 8; ++g) {
                const uint32_t* v = (g < 4) ? (v0 + g * 8) : (v1 + (g - 4) * 8);
                uint4 o;
                o.x = pack_bf16x2(__uint_as_float(v[0]), __uint_as_float(v[1]));
                o.y = pack_bf16x2(__uint_as_float(v[2]), __uint_as_float(v[3]));
                o.z = pack_bf16x2(__uint_as_float(v[4]), __uint_as_float(v[5]));
                o.w = pack_bf16x2(__uint_as_float(v[6]), __uint_as_float(v[7]));
                *reinterpret_cast<uint4*>(stg + g * 16) = o;
              }
              asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic smem writes -> async-proxy reads
              const long long e = p.push_off + (long long)row * p.ldc + col;
              if (ncols == 64 && (e & 63) == 0 && (p.push_n & 63) == 0) {
                const long long owner = e / p.push_n;
                bulk_store_s2g(reinterpret_cast<__nv_bfloat16*>(p.push_bases[owner]) +
                                   ((long long)p.push_rank * p.push_n + (e - owner * p.push_n)), stg, 128);
              } else {   // a chunk that may straddle two owners / a ragged right edge: one 16-byte store per vector
                for (int g = 0; g * 8 < ncols; ++g) {
                  const long long e8 = e + g * 8;
                  const long long owner = e8 / p.push_n;
                  bulk_store_s2g(reinterpret_cast<__nv_bfloat16*>(p.push_bases[owner]) +
                                     ((long long)p.push_rank * p.push_n + (e8 - owner * p.push_n)), stg + g * 16, 16);
                }
              }
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            continue;
          }
        }
        if (row_ok && col < p.N) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t* v = h ? v1 : v0;
            const int cb = col + 32 * h;
            if (cb >= p.N) break;
            if constexpr (sizeof(OutT) == 2) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                if (cb + g * 8 >= p.N) break;
                float f[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(v[g * 8 + i]);
                if constexpr (BIAS) {
                  const uint4 bv = bias8[h * 4 + g];
                  const float2 b0 = unpack_bf16x2(bv.x), b1 = unpack_bf16x2(bv.y), b2 = unpack_bf16x2(bv.z),
                               b3 = unpack_bf16x2(bv.w);
                  f[0] += b0.x; f[1] += b0.y; f[2] += b1.x; f[3] += b1.y; f[4] += b2.x; f[5] += b2.y; f[6] += b3.x; f[7] += b3.y;
                }
                if constexpr (EPI == P_EPI_PUSH) {
                  const long long e = p.push_off + (long long)row * p.ldc + (cb + g * 8);
                  const long long owner = e / p.push_n;
                  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.push_bases[owner]) +
                                       ((long long)p.push_rank * p.push_n + (e - owner * p.push_n));
                  uint4 o;
                  o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
                  o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
                  *reinterpret_cast<uint4*>(dst) = o;     // peer (or local) store; made visible by the flag round that follows
                  continue;
                }
                if constexpr (EPI == P_EPI_SCALE) {
                  const float sa = p.scale_a[row];
                  const float4 b0 = *reinterpret_cast<const float4*>(p.scale_b + cb + g * 8);
                  const float4 b1 = *reinterpret_cast<const float4*>(p.scale_b + cb + g * 8 + 4);
                  f[0] *= sa * b0.x; f[1] *= sa * b0.y; f[2] *= sa * b0.z; f[3] *= sa * b0.w;
                  f[4] *= sa * b1.x; f[5] *= sa * b1.y; f[6] *= sa * b1.z; f[7] *= sa * b1.w;
                } else if constexpr (EPI == P_EPI_ROPE) {
                  const int c8 = cb + g * 8;
                  if (c8 < p.rope_cols) {
                    const float4* tp = reinterpret_cast<const float4*>(
                        p.rope + ((size_t)(row % p.rope_S) * (p.rope_hd >> 1) + ((c8 % p.rope_hd) >> 1)) * 2);
                    const float4 t0 = tp[0], t1 = tp[1];
                    const float cs[4] = {t0.x, t0.z, t1.x, t1.z}, sn[4] = {t0.y, t0.w, t1.y, t1.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                      const float a0 = f[2 * i], a1 = f[2 * i + 1];
                      f[2 * i] = a0 * cs[i] - a1 * sn[i];
                      f[2 * i + 1] = a0 * sn[i] + a1 * cs[i];
                    }
                  }
                } else if constexpr (EPI != P_EPI_STORE && EPI != P_EPI_SCALE) {
                  const __nv_bfloat16* src = (EPI == P_EPI_RESIDUAL) ? (rrow + cb + g * 8)
                                                                     : (reinterpret_cast<const __nv_bfloat16*>(crow) + cb + g * 8);
                  uint4 r = *reinterpret_cast<const uint4*>(src);
                  float2 a = unpack_bf16x2(r.x), b = unpack_bf16x2(r.y), c2 = unpack_bf16x2(r.z), d = unpack_bf16x2(r.w);
                  f[0] += a.x; f[1] += a.y; f[2] += b.x; f[3] += b.y; f[4] += c2.x; f[5] += c2.y; f[6] += d.x; f[7] += d.y;
                }
                uint4 o;
                o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
                o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
                *reinterpret_cast<uint4*>(crow + cb + g * 8) = o;
              }
            } else {
#pragma unroll
              for (int g = 0; g < 8; ++g) {
                if (cb + g * 4 >= p.N) break;
                float4 o;
                o.x = __uint_as_float(v[g * 4 + 0]); o.y = __uint_as_float(v[g * 4 + 1]);
                o.z = __uint_as_float(v[g * 4 + 2]); o.w = __uint_as_float(v[g * 4 + 3]);
                if constexpr (EPI == P_EPI_RESIDUAL) {
                  uint2 r = *reinterpret_cast<const uint2*>(rrow + cb + g * 4);
                  float2 a = unpack_bf16x2(r.x), b = unpack_bf16x2(r.y);
                  o.x += a.x; o.y += a.y; o.z += b.x; o.w += b.y;
                } else if constexpr (EPI == P_EPI_ACCUM) {
                  float4 r = *reinterpret_cast<const float4*>(crow + cb + g * 4);
                  o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
                }
                *reinterpret_cast<float4*>(crow + cb + g * 4) = o;
              }
            }
          }
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tempty_bar[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if constexpr (EPI == P_EPI_PUSH) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all pushed rows are out
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer may still be reading our smem / signalling our barriers
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

template <bool A_MN, bool B_MN, int EPI, typename OutT>
static int launch2_ag(const CUtensorMap& tmA, const CUtensorMap& tmB, const Gemm2Params& p, const AgParams& ag,
                      cudaStream_t stream) {
  auto kern = gemm2_bf16_tcgen05<A_MN, B_MN, EPI, OutT, true>;
  constexpr int smem = P_SMEM + (EPI == P_EPI_PUSH ? PUSH_STAGE_BYTES : 0);
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  // the comm warps of ALL SMs carry the gather, so always launch the full machine even for few tiles
  int pairs = sm_count() / 2;
  kern<<<pairs * 2, P_THREADS + 32 * AG_WARPS, smem, stream>>>(tmA, tmB, p, ag);
  return (int)cudaGetLastError();
}

template <bool A_MN, bool B_MN, int EPI, typename OutT>
static int launch2(const CUtensorMap& tmA, const CUtensorMap& tmB, const Gemm2Params& p, cudaStream_t stream) {
  auto kern = gemm2_bf16_tcgen05<A_MN, B_MN, EPI, OutT, false>;
  constexpr int smem = P_SMEM + (EPI == P_EPI_PUSH ? PUSH_STAGE_BYTES : 0);
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  int tiles = p.m_tiles * p.n_tiles;
  int pairs = sm_count() / 2;
  if (tiles < pairs) pairs = tiles;
  kern<<<pairs * 2, P_THREADS, smem, stream>>>(tmA, tmB, p, AgParams{});
  return (int)cudaGetLastError();
}

static int launch2_fp8(const CUtensorMap& tmA, const CUtensorMap& tmB, const Gemm2Params& p, cudaStream_t stream) {
  auto kern = gemm2_bf16_tcgen05<false, false, P_EPI_SCALE, __nv_bfloat16, false, true>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM);
    if (e != cudaSuccess) return (int)e;
    configured = true;
  }
  int tiles = p.m_tiles * p.n_tiles;
  int pairs = sm_count() / 2;
  if (tiles < pairs) pairs = tiles;
  kern<<<pairs * 2, P_THREADS, P_SMEM, stream>>>(tmA, tmB, p, AgParams{});
  return (int)cudaGetLastError();
}

template <bool A_MN, bool B_MN>
static int dispatch2(const CUtensorMap& a, const CUtensorMap& b, const Gemm2Params& p, int epi, int out_fp32,
                     cudaStream_t s) {
  if (out_fp32) {
    if (epi == P_EPI_STORE) return launch2<A_MN, B_MN, P_EPI_STORE, float>(a, b, p, s);
    if (epi == P_EPI_RESIDUAL) return launch2<A_MN, B_MN, P_EPI_RESIDUAL, float>(a, b, p, s);
    return launch2<A_MN, B_MN, P_EPI_ACCUM, float>(a, b, p, s);
  }
  if (epi == P_EPI_STORE) return launch2<A_MN, B_MN, P_EPI_STORE, __nv_bfloat16>(a, b, p, s);
  if (epi == P_EPI_RESIDUAL) return launch2<A_MN, B_MN, P_EPI_RESIDUAL, __nv_bfloat16>(a, b, p, s);
  return launch2<A_MN, B_MN, P_EPI_ACCUM, __nv_bfloat16>(a, b, p, s);
}

// RoPE epilogue parameters of the NEXT epi == P_EPI_ROPE launch (set immediately before it by the single host thread
// that owns the stream; keeps the two launcher signatures unchanged)
static const float* g_rope_table = nullptr;
static int g_rope_S = 1, g_rope_hd = 2, g_rope_cols = 0;
// same convention for the push epilogue
static void* const* g_push_bases = nullptr;
static long long g_push_n = 1, g_push_off = 0;
static int g_push_rank = 0, g_push_bulk = 1, g_push_world = 1;
// same convention for the SwiGLU epilogues: aux = activation output (forward) / saved projection (backward)
static void* g_swi_aux = nullptr;
static int g_swi_ld = 0, g_swi_F = 0, g_swi_gate_first = 1;

}  // namespace b200

extern "C" void b200_gemm2_set_rope(const float* table, int S, int hd, int cols) {
  b200::g_rope_table = table; b200::g_rope_S = S; b200::g_rope_hd = hd; b200::g_rope_cols = cols;
}

// world > 1: rotate the tile raster by rank * tiles / world (0 / 1 = no rotation)
extern "C" void b200_gemm2_set_push(void* const* bases, long long n, long long off, int rank, int bulk, int world) {
  b200::g_push_bases = bases; b200::g_push_n = n; b200::g_push_off = off; b200::g_push_rank = rank; b200::g_push_bulk = bulk;
  b200::g_push_world = world < 1 ? 1 : world;
}

extern "C" void b200_gemm2_set_swiglu(void* aux, int ld_aux, int F, int gate_first) {
  b200::g_swi_aux = aux; b200::g_swi_ld = ld_aux; b200::g_swi_F = F; b200::g_swi_gate_first = gate_first;
}

extern "C" int b200_gemm2_bf16(const void* A, const void* B, void* C, const void* R, int M, int N, int K, int lda,
                               int ldb, int ldc, int ldr, int a_mn, int b_mn, int epi, int out_fp32,
                               cudaStream_t stream) {
  using namespace b200;
  CUtensorMap tmA, tmB;
  int rc;
  if (!a_mn) rc = make_tmap_2d_bf16(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, P_BK, C_BM);
  else       rc = make_tmap_2d_bf16(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, 64, P_BK);
  if (rc) return 1000 - rc;
  if (!b_mn) rc = make_tmap_2d_bf16(&tmB, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, P_BK, C_BN);
  else       rc = make_tmap_2d_bf16(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, 64, P_BK);
  if (rc) return 2000 - rc;
  Gemm2Params p;
  p.M = M; p.N = N; p.K = K; p.ldc = ldc; p.ldr = ldr; p.C = C; p.R = R;
  p.m_tiles = (M + P_BM - 1) / P_BM;
  p.n_tiles = (N + P_BN - 1) / P_BN;
  p.rope = g_rope_table; p.rope_S = g_rope_S; p.rope_hd = g_rope_hd; p.rope_cols = g_rope_cols;
  p.push_bases = g_push_bases; p.push_n = g_push_n; p.push_off = g_push_off; p.push_rank = g_push_rank;
  p.push_bulk = g_push_bulk;
  p.tile_rot = 0;
  p.aux = g_swi_aux; p.ld_aux = g_swi_ld; p.swi_F = g_swi_F; p.swi_gate_first = g_swi_gate_first;
  if (epi == P_EPI_PUSH && g_push_world > 1) {
    const int per_band = P_GROUP_M * p.n_tiles, tiles = p.m_tiles * p.n_tiles;
    const int bands = (tiles + per_band - 1) / per_band;
    p.tile_rot = (int)(((long long)(g_push_rank % g_push_world) * bands / g_push_world) * per_band) % tiles;
  }
  if (epi == P_EPI_SWIGLU) {   // nt; N = 2F rows of the fused weight, tiles of 128 features
    if (a_mn || b_mn || out_fp32 || !p.aux || p.swi_F <= 0 || N != 2 * p.swi_F || (p.swi_F % C_BN) || (p.ld_aux % 8)) return -11;
    p.N = p.swi_F;
    p.n_tiles = p.swi_F / C_BN;
    return launch2<false, false, P_EPI_SWIGLU, __nv_bfloat16>(tmA, tmB, p, stream);
  }
  if (epi == P_EPI_SWIGLU_BWD) {   // nn; N = F columns of dS, output [M, 2F]
    if (a_mn || !b_mn || out_fp32 || !p.aux || p.swi_F != N || (N % 8) || (p.ld_aux % 8)) return -12;
    return launch2<false, true, P_EPI_SWIGLU_BWD, __nv_bfloat16>(tmA, tmB, p, stream);
  }
  if (epi == P_EPI_ROPE) {
    if (a_mn || b_mn || out_fp32 || !p.rope || (p.rope_hd % 8) || (p.rope_cols % 8)) return -8;
    return launch2<false, false, P_EPI_ROPE, __nv_bfloat16>(tmA, tmB, p, stream);
  }
  if (epi & P_EPI_BIAS) {   // R = bias [N] bf16; nt, bf16 output
    if (a_mn || b_mn || out_fp32 || !R || (reinterpret_cast<uintptr_t>(R) & 15) || (N % 8)) return -14;
    if (epi == (P_EPI_ROPE | P_EPI_BIAS)) {
      if (!p.rope || (p.rope_hd % 8) || (p.rope_cols % 8)) return -8;
      return launch2<false, false, P_EPI_ROPE | P_EPI_BIAS, __nv_bfloat16>(tmA, tmB, p, stream);
    }
    if (epi == (P_EPI_STORE | P_EPI_BIAS)) return launch2<false, false, P_EPI_STORE | P_EPI_BIAS, __nv_bfloat16>(tmA, tmB, p, stream);
    return -14;
  }
  if (epi == P_EPI_PUSH) {   // wgrad (tn) only; every 8-element vector must stay inside one owner's slice
    if (!a_mn || !b_mn || out_fp32 || !p.push_bases || p.push_n <= 0 || (p.push_n % 8) || (p.push_off % 8) || (ldc % 8))
      return -9;
    return launch2<true, true, P_EPI_PUSH, __nv_bfloat16>(tmA, tmB, p, stream);
  }
  if (a_mn) {
    if (b_mn) return dispatch2<true, true>(tmA, tmB, p, epi, out_fp32, stream);
    return dispatch2<true, false>(tmA, tmB, p, epi, out_fp32, stream);
  }
  if (b_mn) return dispatch2<false, true>(tmA, tmB, p, epi, out_fp32, stream);
  return dispatch2<false, false>(tmA, tmB, p, epi, out_fp32, stream);
}

// GEMM + fused all-gather.  Supported: bf16 output, EPI store|residual, layouts nt (forward first GEMM) and
// nn / tn (backward first GEMMs).
extern "C" int b200_gemm2_ag_bf16(const void* A, const void* B, void* C, const void* R, int M, int N, int K, int lda,
                                  int ldb, int ldc, int ldr, int a_mn, int b_mn, int epi,
                                  const void* const* peer_shards, void* full, unsigned long long shard_bytes,
                                  unsigned long long begin, unsigned long long end, int world, int rank,
                                  uint32_t* flags, uint32_t epoch, int dependent, cudaStream_t stream) {
  using namespace b200;
  if ((begin % 16) || (end % 16) || (begin % AG_CHUNK)) return -5;
  CUtensorMap tmA, tmB;
  int rc;
  if (!a_mn) rc = make_tmap_2d_bf16(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, P_BK, C_BM);
  else       rc = make_tmap_2d_bf16(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, 64, P_BK);
  if (rc) return 1000 - rc;
  if (!b_mn) rc = make_tmap_2d_bf16(&tmB, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, P_BK, C_BN);
  else       rc = make_tmap_2d_bf16(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, 64, P_BK);
  if (rc) return 2000 - rc;
  Gemm2Params p;
  p.M = M; p.N = N; p.K = K; p.ldc = ldc; p.ldr = ldr; p.C = C; p.R = R;
  p.m_tiles = (M + P_BM - 1) / P_BM;
  p.n_tiles = (N + P_BN - 1) / P_BN;
  p.rope = g_rope_table; p.rope_S = g_rope_S; p.rope_hd = g_rope_hd; p.rope_cols = g_rope_cols;
  p.push_bases = g_push_bases; p.push_n = g_push_n; p.push_off = g_push_off; p.push_rank = g_push_rank;
  p.push_bulk = g_push_bulk;
  p.tile_rot = 0;
  p.aux = g_swi_aux; p.ld_aux = g_swi_ld; p.swi_F = g_swi_F; p.swi_gate_first = g_swi_gate_first;
  if (epi == P_EPI_PUSH && g_push_world > 1) {
    const int per_band = P_GROUP_M * p.n_tiles, tiles = p.m_tiles * p.n_tiles;
    const int bands = (tiles + per_band - 1) / per_band;
    p.tile_rot = (int)(((long long)(g_push_rank % g_push_world) * bands / g_push_world) * per_band) % tiles;
  }
  if (epi == P_EPI_SWIGLU) {
    if (a_mn || b_mn || !p.aux || p.swi_F <= 0 || N != 2 * p.swi_F || (p.swi_F % C_BN) || (p.ld_aux % 8) || dependent) return -11;
    p.N = p.swi_F;
    p.n_tiles = p.swi_F / C_BN;
  }
  if (epi == P_EPI_SWIGLU_BWD && (a_mn || !b_mn || !p.aux || p.swi_F != N || (N % 8) || (p.ld_aux % 8))) return -12;
  AgParams ag;
  ag.peer_shards = peer_shards; ag.full = (uint8_t*)full; ag.shard_bytes = shard_bytes; ag.begin = begin; ag.end = end;
  ag.world = world; ag.rank = rank; ag.flags = flags; ag.epoch = epoch; ag.dependent = dependent;
  ag.b_off = (unsigned long long)((const uint8_t*)B - (const uint8_t*)full);
  ag.b_row_bytes = (unsigned long long)ldb * 2;
  if (dependent && ((const uint8_t*)B < (const uint8_t*)full)) return -6;
#define AGL(AM, BM_, E) return launch2_ag<AM, BM_, E, __nv_bfloat16>(tmA, tmB, p, ag, stream)
  if (epi == P_EPI_ROPE) {
    if (a_mn || b_mn || !p.rope || (p.rope_hd % 8) || (p.rope_cols % 8)) return -8;
    AGL(false, false, P_EPI_ROPE);
  }
  if (epi & P_EPI_BIAS) {   // R = bias [N] bf16; nt
    if (a_mn || b_mn || !R || (reinterpret_cast<uintptr_t>(R) & 15) || (N % 8)) return -14;
    if (epi == (P_EPI_ROPE | P_EPI_BIAS)) {
      if (!p.rope || (p.rope_hd % 8) || (p.rope_cols % 8)) return -8;
      AGL(false, false, P_EPI_ROPE | P_EPI_BIAS);
    }
    if (epi == (P_EPI_STORE | P_EPI_BIAS)) AGL(false, false, P_EPI_STORE | P_EPI_BIAS);
    return -14;
  }
  if (!a_mn && !b_mn) {
    if (epi == P_EPI_SWIGLU) AGL(false, false, P_EPI_SWIGLU);
    if (epi == P_EPI_RESIDUAL) AGL(false, false, P_EPI_RESIDUAL);
    AGL(false, false, P_EPI_STORE);
  }
  if (!a_mn && b_mn) {
    if (epi == P_EPI_SWIGLU_BWD) AGL(false, true, P_EPI_SWIGLU_BWD);
    if (epi == P_EPI_RESIDUAL) AGL(false, true, P_EPI_RESIDUAL);
    AGL(false, true, P_EPI_STORE);
  }
  if (a_mn && b_mn) {
    if (epi == P_EPI_PUSH) {   // wgrad that pushes its tiles to the owners AND carries the next unit's all-gather
      if (!p.push_bases || p.push_n <= 0 || (p.push_n % 8) || (p.push_off % 8) || (ldc % 8)) return -9;
      AGL(true, true, P_EPI_PUSH);
    }
    if (epi == P_EPI_ACCUM) AGL(true, true, P_EPI_ACCUM);
    AGL(true, true, P_EPI_STORE);
  }
#undef AGL
  return -7;
}

// C[M, N] (bf16) = (A_q[M, K] x B_q[N, K]^T) * scale_a[M] * scale_b[N]  with e4m3 operands on the tensor cores
// (tcgen05.mma kind::f8f6f4, fp32 accumulate).  K (bytes = elements) must be a multiple of 16; rows 16-byte aligned.
extern "C" int b200_gemm2_fp8(const void* A, const void* B, void* C, const float* scale_a, const float* scale_b, int M, int N,
                              int K, int lda, int ldb, int ldc, cudaStream_t stream) {
  using namespace b200;
  if ((K % 16) || (lda % 16) || (ldb % 16) || (N % 8) || (ldc % 8) || M < 1) return -13;
  CUtensorMap tmA, tmB;
  if (make_tmap_2d_u8(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, 2 * P_BK, C_BM)) return 1001;
  if (make_tmap_2d_u8(&tmB, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, 2 * P_BK, C_BN)) return 2001;
  Gemm2Params p{};
  p.M = M; p.N = N; p.K = K; p.ldc = ldc; p.ldr = 0; p.C = C; p.R = nullptr;
  p.m_tiles = (M + P_BM - 1) / P_BM;
  p.n_tiles = (N + P_BN - 1) / P_BN;
  p.tile_rot = 0;
  p.scale_a = scale_a; p.scale_b = scale_b;
  return launch2_fp8(tmA, tmB, p, stream);
}
