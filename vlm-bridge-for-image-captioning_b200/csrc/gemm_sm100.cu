// Persistent, warp-specialised bf16 GEMM for sm_100a: TMA -> 128B-swizzled shared memory ->
// tcgen05.mma (cta_group::1, 128 x BLOCK_N x 16) -> double-buffered TMEM accumulators ->
// tcgen05.ld epilogue with fused bias / GELU / dropout / residual.
//
// Replaces every nn.Linear of the reference bridge (bridge_module.py:98-100,118,196-198,216,
// 292,295) and the dgrad / wgrad matmuls autograd derives from them.
//
// Roles (320 threads, one CTA per SM):
//   warp 8      TMA producer   : waits empty[s], arms full[s] with the stage byte count, issues
//                                the A and B tile loads
//   warp 9      MMA issuer     : owns TMEM (alloc/dealloc); waits full[s]; lane 0 issues 4
//                                tcgen05.mma per 64-wide k block and commits to empty[s]; after the
//                                last k block commits to tmem_full[acc]
//   warps 0..7  epilogue       : wait tmem_full[acc]; two warps share each 32-lane TMEM quadrant
//                                (alternating 32-column chunks); tcgen05.ld (thread = one output
//                                row, 32 columns), transpose through shared memory, fused epilogue
//                                with the residual / aux / bias operands of the NEXT chunk already
//                                in flight; then arrive on tmem_empty[acc]
// The accumulator is double buffered (2 x BLOCK_N TMEM columns) so the epilogue of tile i
// overlaps the main loop of tile i+1. The two single-thread roles sit on the HIGHEST warp ids: the
// SM sub-partition arbiter prefers higher warp ids, so the arithmetic-heavy epilogue warps that
// share their schedulers can never delay a TMA issue or an MMA issue.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include <mutex>

#include "../../include/b200_bridge.h"
#include "common.cuh"
#include "launch.h"

namespace b200b {

struct GemmKernelParams {
  int m, n, k;
  int num_m_blocks, num_n_blocks, num_k_blocks;
  void* out;
  long long ldo;
  void* aux;
  long long ldaux;
  const float* bias;
  const float* resid;
  long long ldr;
  float beta;
  DropoutCfg drop;
  uint32_t drop_stream;
};

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kUmmaK = 16;
constexpr int kEpiWarps = 8;
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;
constexpr int kProducerWarp = kEpiWarps;      // warp 8
constexpr int kMmaWarp = kEpiWarps + 1;       // warp 9

template <int BLOCK_N>
struct GemmCfg {
  static constexpr int kStages = (BLOCK_N == 256) ? 4 : 6;
  static constexpr uint32_t kABytes = kBlockM * kBlockK * 2;
  static constexpr uint32_t kBBytes = BLOCK_N * kBlockK * 2;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kTmemCols = 2 * BLOCK_N;
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + 1024 + kEpiWarps * 32 * 33 * 4;
};

// ---- fused epilogue -----------------------------------------------------------------------------
// Work unit: a GROUP = 4 passes of (4 rows x 8 lanes x 4 columns) = 16 rows x 32 columns of one
// warp's 32 x 32 chunk. The loop over (chunk, group) is deliberately NOT unrolled: the first version
// unrolled all 8 passes of all chunks and its ~10k SASS instructions thrashed the instruction cache
// (ncu: stall_no_inst 41% of samples, profiles/r01_ncu_gemm_gelu_v3_*). One group body is ~0.5k
// instructions. Global operands of the NEXT group (residual rows, saved pre-activations, bias) are
// fetched before the arithmetic of the current one, and those of a tile's first group before the
// accumulator is even ready, so no load latency sits between a load and the store that needs it.
constexpr int kGroupPasses = 4;

template <int EPI>
struct EpiOperands {
  float4 bias;                 // BF16_BIAS, BF16_BIAS_GELU, F32_BIAS_RESID
  float4 resid[kGroupPasses];  // F32_BIAS_RESID
  uint2 aux[kGroupPasses];     // BF16_DGELU (the saved pre-activation u)
};                             // members an epilogue does not use are never touched: no registers

template <int EPI>
constexpr bool kEpiHasDropout =
    (EPI == B200B_EPI_BF16_BIAS_GELU || EPI == B200B_EPI_F32_BIAS_RESID || EPI == B200B_EPI_BF16_DGELU);

// rows row0 + 4*pass + r_sub (pass < 4), columns [col, col+4)
template <int EPI>
__device__ __forceinline__ void epi_fetch(const GemmKernelParams& p, int row0, int col, int r_sub,
                                          EpiOperands<EPI>& o) {
  const bool col_ok = col < p.n;
  if constexpr (EPI == B200B_EPI_BF16_BIAS || EPI == B200B_EPI_BF16_BIAS_GELU || EPI == B200B_EPI_F32_BIAS_RESID) {
    o.bias = (p.bias != nullptr && col_ok) ? __ldg(reinterpret_cast<const float4*>(p.bias + col))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if constexpr (EPI == B200B_EPI_F32_BIAS_RESID) {
#pragma unroll
    for (int pass = 0; pass < kGroupPasses; ++pass) {
      const int r = row0 + 4 * pass + r_sub;
      o.resid[pass] = (col_ok && r < p.m) ? *reinterpret_cast<const float4*>(p.resid + (long long)r * p.ldr + col)
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  if constexpr (EPI == B200B_EPI_BF16_DGELU) {
#pragma unroll
    for (int pass = 0; pass < kGroupPasses; ++pass) {
      const int r = row0 + 4 * pass + r_sub;
      o.aux[pass] = (col_ok && r < p.m)
                        ? *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p.aux) +
                                                          (long long)r * p.ldaux + col)
                        : make_uint2(0u, 0u);
    }
  }
}

// One copy of the 10 Philox rounds per kernel instead of one per call site.
static __device__ __noinline__ uint4 dropout_bits8_call(uint32_t seed_lo, uint32_t seed_hi, uint32_t stream,
                                                        uint32_t group_lo, uint32_t group_hi) {
  return philox4x32_10(make_uint4(group_lo, group_hi, stream, 0x0b200b00u), make_uint2(seed_lo, seed_hi));
}

// Dropout decisions of one group: the two lanes that share an 8-element dropout group (lane ^ 1)
// each run Philox for one of two consecutive passes and swap the halves they do not need.
// Executed by all 32 lanes (shuffles); dropout disabled -> thr == 0 keeps everything.
__device__ __forceinline__ void epi_dropout_bits(const GemmKernelParams& p, uint2 seed, int row0, int col, int r_sub,
                                                 int cg, uint2 (&w)[kGroupPasses]) {
#pragma unroll
  for (int i = 0; i < kGroupPasses; ++i) w[i] = make_uint2(0u, 0u);
  if (p.drop.thr == 0) return;  // warp-uniform
  const bool odd = (cg & 1) != 0;
#pragma unroll
  for (int pp = 0; pp < kGroupPasses; pp += 2) {
    const int row = row0 + 4 * (pp + (odd ? 1 : 0)) + r_sub;
    const uint64_t group = ((uint64_t)row * (uint64_t)p.n + (uint64_t)col) >> 3;
    const uint4 b = dropout_bits8_call(seed.x, seed.y, p.drop_stream, (uint32_t)group,
                                       (uint32_t)(group >> 32));
    const uint32_t r0 = __shfl_xor_sync(0xffffffffu, odd ? b.x : b.z, 1);
    const uint32_t r1 = __shfl_xor_sync(0xffffffffu, odd ? b.y : b.w, 1);
    w[pp] = odd ? make_uint2(r0, r1) : make_uint2(b.x, b.y);
    w[pp + 1] = odd ? make_uint2(b.z, b.w) : make_uint2(r0, r1);
  }
}
__device__ __forceinline__ bool keep4(const uint2& w, int i, uint32_t thr) {
  const uint32_t v = (i < 2) ? w.x : w.y;
  return ((i & 1) ? (v >> 16) : (v & 0xffffu)) >= thr;
}

// epilogue of 4 consecutive columns of one row; `w` = the 4 x 16 dropout bits of these elements
template <int EPI>
__device__ __forceinline__ void epilogue4(const GemmKernelParams& p, int row, int col, float4 acc, const float4& bias,
                                          const float4& resid, const uint2& aux, const uint2& w, bool store) {
  float f[4] = {acc.x, acc.y, acc.z, acc.w};
  const uint32_t thr = p.drop.thr;
  const float scale = p.drop.scale;  // 1.0f when dropout is off

  if constexpr (EPI == B200B_EPI_BF16_BIAS || EPI == B200B_EPI_BF16_BIAS_GELU ||
                EPI == B200B_EPI_F32_BIAS_RESID) {
    f[0] += bias.x; f[1] += bias.y; f[2] += bias.z; f[3] += bias.w;
  }

  if constexpr (EPI == B200B_EPI_BF16_BIAS) {
    uint2 o;
    o.x = pack_bf16(f[0], f[1]); o.y = pack_bf16(f[2], f[3]);
    if (store) *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)row * p.ldo + col) = o;
  } else if constexpr (EPI == B200B_EPI_BF16_BIAS_GELU) {
    float h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      f[i] = bf16_round(f[i]);          // the reference Linear output is bf16 under autocast
      h[i] = bf16_round(gelu_erf(f[i]));
      h[i] = keep4(w, i, thr) ? h[i] * scale : 0.0f;
    }
    uint2 u, o;
    u.x = pack_bf16(f[0], f[1]); u.y = pack_bf16(f[2], f[3]);
    o.x = pack_bf16(h[0], h[1]); o.y = pack_bf16(h[2], h[3]);
    if (store) {
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.aux) + (long long)row * p.ldaux + col) = u;
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)row * p.ldo + col) = o;
    }
  } else if constexpr (EPI == B200B_EPI_F32_BIAS_RESID) {
    const float r[4] = {resid.x, resid.y, resid.z, resid.w};
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float y = bf16_round(f[i]);
      if (thr != 0) y = keep4(w, i, thr) ? bf16_round(y * scale) : 0.0f;
      o[i] = r[i] + y;
    }
    if (store)
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (long long)row * p.ldo + col) =
          make_float4(o[0], o[1], o[2], o[3]);
  } else if constexpr (EPI == B200B_EPI_BF16_DGELU) {
    const float u[4] = {bf16_lo(aux.x), bf16_hi(aux.x), bf16_lo(aux.y), bf16_hi(aux.y)};
    float g[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float d = bf16_round(f[i]);
      if (thr != 0) d = keep4(w, i, thr) ? bf16_round(d * scale) : 0.0f;
      g[i] = d * gelu_erf_grad(u[i]);
    }
    uint2 o;
    o.x = pack_bf16(g[0], g[1]); o.y = pack_bf16(g[2], g[3]);
    if (store) *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)row * p.ldo + col) = o;
  } else {  // B200B_EPI_F32
    float* op = reinterpret_cast<float*>(p.out) + (long long)row * p.ldo + col;
    if (store) {
      if (p.beta != 0.0f) {
        const float4 o0 = *reinterpret_cast<const float4*>(op);
        f[0] += p.beta * o0.x; f[1] += p.beta * o0.y; f[2] += p.beta * o0.z; f[3] += p.beta * o0.w;
      }
      *reinterpret_cast<float4*>(op) = make_float4(f[0], f[1], f[2], f[3]);
    }
  }
}

// Shared pieces of the two kernels ---------------------------------------------------------------

// Drain this CTA's 128 x BLOCK_N accumulator stage through the fused epilogue.
// tcgen05.ld hands each thread one accumulator ROW (32 columns at a time); storing from that
// layout would touch 32 different cache lines per instruction. Each warp therefore transposes its
// 32 x 32 chunk through a private padded shared-memory tile so that 8 consecutive lanes own one
// row's 32 columns (4 each): every global load/store instruction then covers 4 full 128-byte
// (fp32) or 64-byte (bf16) row segments.
// Two warps serve each TMEM lane quadrant: warp `half` (0/1) takes the 32-column chunks
// half, half+2, ... of the tile.
constexpr int kEpiLd = 33;                                  // padded row, words (conflict free both ways)
constexpr uint32_t kEpiBytesPerWarp = 32 * kEpiLd * 4;      // 4224 B
constexpr uint32_t kEpiBytes = kEpiWarps * kEpiBytesPerWarp;

// The tile's first group of epilogue operands: issued BEFORE waiting for the accumulator.
template <int BLOCK_N, int EPI>
__device__ __forceinline__ void drain_prefetch(const GemmKernelParams& p, int row0, int n_idx, int half, int lane,
                                               EpiOperands<EPI>& ops) {
  epi_fetch<EPI>(p, row0, n_idx + 32 * half + 4 * (lane & 7), lane >> 3, ops);
}

template <int BLOCK_N, int EPI>
__device__ __forceinline__ void drain_accumulator(const GemmKernelParams& p, uint32_t t_row, int row0 /*of this warp*/,
                                                  int n_idx, float* stage /*this warp's tile*/, int lane, int half,
                                                  EpiOperands<EPI>& ops /*prefetched for the first group*/,
                                                  uint2 seed /*resolved dropout seed*/) {
  const int r_sub = lane >> 3, cg = lane & 7;
  constexpr int kChunks = BLOCK_N / 64;  // chunks per warp
#pragma unroll 1
  for (int i = 0; i < kChunks; ++i) {
    const int c0 = 32 * (2 * i + half);
    if (n_idx + c0 >= p.n) break;  // warp-uniform
    {
      uint32_t v[32];
      tmem_ld_32x32(t_row + (uint32_t)c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) stage[lane * kEpiLd + j] = __uint_as_float(v[j]);
    }
    __syncwarp();
    const int col = n_idx + c0 + 4 * cg;
#pragma unroll 1
    for (int grp = 0; grp < 8 / kGroupPasses; ++grp) {
      const int grow0 = row0 + 4 * kGroupPasses * grp;
      // operands of the next group: same chunk, next 16 rows -- or the first 16 rows of this warp's next chunk
      EpiOperands<EPI> nxt;
      {
        const bool last_grp = grp == 8 / kGroupPasses - 1;
        const int nrow0 = last_grp ? row0 : grow0 + 4 * kGroupPasses;
        const int ncol = last_grp ? col + 64 : col;
        if (!(last_grp && i + 1 == kChunks)) epi_fetch<EPI>(p, nrow0, ncol, r_sub, nxt);
      }
      uint2 w[kGroupPasses];
      if constexpr (kEpiHasDropout<EPI>) epi_dropout_bits(p, seed, grow0, col, r_sub, cg, w);
#pragma unroll
      for (int pass = 0; pass < kGroupPasses; ++pass) {
        const int r = 4 * (kGroupPasses * grp + pass) + r_sub;
        const float* sp = stage + r * kEpiLd + 4 * cg;
        const float4 acc = make_float4(sp[0], sp[1], sp[2], sp[3]);
        epilogue4<EPI>(p, row0 + r, col, acc, ops.bias, ops.resid[pass], ops.aux[pass], w[pass],
                       col < p.n && row0 + r < p.m);
      }
      ops = nxt;
    }
    __syncwarp();
  }
}

// The 64-bit shared-memory descriptors differ between k steps / stages only in the 14-bit start
// address field, so the issuing thread keeps the constant high words and adds to the low word.
template <bool MN>
struct DescConsts {
  static constexpr uint32_t kLbo = MN ? 8192u : 16u;
  static constexpr uint32_t kKStep16 = (MN ? 2048u : 32u) >> 4;  // start-address units per 16-wide k step
};
__device__ __forceinline__ uint64_t desc_with_lo(uint64_t base, uint32_t add16) {
  return base + (uint64_t)add16;  // never carries out of the 14-bit field: smem addresses < 256 KiB
}

template <int BLOCK_N, bool A_MN, bool B_MN, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                    const GemmKernelParams p) {
  using Cfg = GemmCfg<BLOCK_N>;
  constexpr int kStages = Cfg::kStages;

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kStages];
  __shared__ __align__(8) uint64_t empty_bar[kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // 32-bit shared addresses, computed once
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem0 - smem_u32(smem_raw));
  const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
  const uint32_t tfull0 = smem_u32(tmem_full_bar), tempty0 = smem_u32(tmem_empty_bar);

  if (warp == kProducerWarp && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tmem_full_bar[0], 1);
    mbar_init(&tmem_full_bar[1], 1);
    mbar_init(&tmem_empty_bar[0], 32 * kEpiWarps);
    mbar_init(&tmem_empty_bar[1], 32 * kEpiWarps);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc(&tmem_base_smem, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t tmem_base = tmem_base_smem;
  const int num_tiles = p.num_m_blocks * p.num_n_blocks;

  if (warp == kProducerWarp) {
    // ------------------------------- TMA producer -------------------------------------------
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m_idx = (tile % p.num_m_blocks) * kBlockM;
      const int n_idx = (tile / p.num_m_blocks) * BLOCK_N;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait_a(empty0 + 8u * stage, phase ^ 1);
        if (elect_one()) {
          const uint32_t sa = smem0 + (uint32_t)stage * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          const uint32_t fb = full0 + 8u * stage;
          mbar_arrive_expect_tx_a(fb, Cfg::kStageBytes);
          const int k_idx = kb * kBlockK;
          if constexpr (!A_MN) {
            tma_load_2d_a(sa, &tm_a, fb, k_idx, m_idx);  // box {64 k, 128 rows}
          } else {
#pragma unroll
            for (int j = 0; j < kBlockM / 64; ++j)       // box {64 m, 64 k} per atom
              tma_load_2d_a(sa + j * 8192, &tm_a, fb, m_idx + 64 * j, k_idx);
          }
          if constexpr (!B_MN) {
            tma_load_2d_a(sb, &tm_b, fb, k_idx, n_idx);  // box {64 k, BLOCK_N rows}
          } else {
#pragma unroll
            for (int j = 0; j < BLOCK_N / 64; ++j)
              tma_load_2d_a(sb + j * 8192, &tm_b, fb, n_idx + 64 * j, k_idx);
          }
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------- MMA issuer ---------------------------------------------
    constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, BLOCK_N, A_MN, B_MN);
    // K-major: 8-row groups 1024 B apart; advancing 16 k elements = +32 B inside the swizzle row.
    // MN-major: 64-wide MN atoms 8192 B apart (LBO), 8-k-row groups 1024 B apart (SBO);
    //           advancing 16 k rows = +2048 B.
    const uint64_t adesc0 = umma_smem_desc(smem0, DescConsts<A_MN>::kLbo, 1024u);
    const uint64_t bdesc0 = umma_smem_desc(smem0 + Cfg::kABytes, DescConsts<B_MN>::kLbo, 1024u);
    int stage = 0;
    uint32_t phase = 0;
    int iter = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
      const int acc = iter & 1;
      const uint32_t acc_phase = (iter >> 1) & 1;
      mbar_wait_a(tempty0 + 8u * acc, acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait_a(full0 + 8u * stage, phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t soff16 = ((uint32_t)stage * Cfg::kStageBytes) >> 4;
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) {
            umma_bf16(d_tmem, desc_with_lo(adesc0, soff16 + k * DescConsts<A_MN>::kKStep16),
                      desc_with_lo(bdesc0, soff16 + k * DescConsts<B_MN>::kKStep16), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit_a(empty0 + 8u * stage);                              // frees the smem stage
          if (kb == p.num_k_blocks - 1) umma_commit_a(tfull0 + 8u * acc);  // accumulator ready
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ------------------------------- epilogue -----------------------------------------------
    const int quad = warp & 3;  // TMEM lanes [32*quad, 32*quad+32) are visible to this warp
    const int half = warp >> 2;
    float* epi_stage =
        reinterpret_cast<float*>(smem_gen + (size_t)kStages * Cfg::kStageBytes) + warp * 32 * kEpiLd;
    const DropoutCfg drop = dropout_resolve(p.drop);
    const uint2 seed = make_uint2(drop.seed_lo, drop.seed_hi);
    int iter = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
      const int acc = iter & 1;
      const uint32_t acc_phase = (iter >> 1) & 1;
      const int m_idx = (tile % p.num_m_blocks) * kBlockM;
      const int n_idx = (tile / p.num_m_blocks) * BLOCK_N;
      EpiOperands<EPI> ops;
      drain_prefetch<BLOCK_N, EPI>(p, m_idx + quad * 32, n_idx, half, lane, ops);
      mbar_wait_a(tfull0 + 8u * acc, acc_phase);
      tc_fence_after();
      drain_accumulator<BLOCK_N, EPI>(p, tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BLOCK_N),
                                      m_idx + quad * 32, n_idx, epi_stage, lane, half, ops, seed);
      tc_fence_before();
      mbar_arrive_a(tempty0 + 8u * acc);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// ================================================================================================
// CTA-pair variant (cta_group::2): a cluster of two CTAs on one TPC computes a 256 x BLOCK_N tile.
// Each CTA stages its own 128 rows of A and HALF of the B tile (BLOCK_N/2 rows) per k block; the
// even CTA's MMA thread issues one 256 x BLOCK_N x 16 tcgen05.mma per k step that reads both CTAs'
// shared memory, so every B element is fetched from L2 once per 256 output rows instead of once
// per 128. Each CTA's TMEM holds its own 128 accumulator rows (all BLOCK_N columns) and is drained
// by its own epilogue warps.
//   full[s]        lives in the even CTA; both CTAs' TMA loads credit it (2 x stage bytes)
//   empty[s]       one per CTA, released by a multicast tcgen05.commit
//   tmem_full[a]   one per CTA, multicast commit after the last k block
//   tmem_empty[a]  even CTA only, 256 arrivals (128 local + 128 remote epilogue threads)
// ================================================================================================
template <int BLOCK_N>
struct GemmPairCfg {
  static constexpr int kStages = (BLOCK_N == 256) ? 5 : 7;  // leaves ~25 KB of the SM for a co-resident exchange CTA
  static constexpr uint32_t kABytes = kBlockM * kBlockK * 2;          // this CTA's 128 rows
  static constexpr uint32_t kBBytes = (BLOCK_N / 2) * kBlockK * 2;    // this CTA's half of B
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kTmemCols = 2 * BLOCK_N;
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + 1024 + kEpiBytes;
};

template <int BLOCK_N, bool A_MN, bool B_MN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_pair_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                         const GemmKernelParams p) {
  using Cfg = GemmPairCfg<BLOCK_N>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kHalfN = BLOCK_N / 2;

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kStages];
  __shared__ __align__(8) uint64_t empty_bar[kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int pair_id = (int)cluster_id_x();
  const int num_pairs = (int)cluster_nctaid_x();
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem0 - smem_u32(smem_raw));
  const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
  const uint32_t tfull0 = smem_u32(tmem_full_bar), tempty0 = smem_u32(tmem_empty_bar);
  const uint32_t full0_even = full0 & 0xFEFFFFFFu;          // same offset in the pair's even CTA
  const uint32_t tempty0_even = mapa_u32(tempty0, 0);

  if (warp == kProducerWarp && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tmem_full_bar[0], 1);
    mbar_init(&tmem_full_bar[1], 1);
    mbar_init(&tmem_empty_bar[0], 2 * 32 * kEpiWarps);   // local + remote epilogue threads
    mbar_init(&tmem_empty_bar[1], 2 * 32 * kEpiWarps);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc_pair(&tmem_base_smem, Cfg::kTmemCols);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();  // barriers of both CTAs are initialised before any remote arrive / TMA credit
  tc_fence_after();
  // everything above is CTA-local set-up; it may overlap the tail of the previous kernel on the stream
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t tmem_base = tmem_base_smem;
  const int num_tiles = p.num_m_blocks * p.num_n_blocks;  // num_m_blocks counts 256-row pair tiles

  if (warp == kProducerWarp) {
    // ------------------------------- TMA producer (both CTAs) --------------------------------
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
      const int m_idx = (tile % p.num_m_blocks) * (2 * kBlockM) + (int)cta_rank * kBlockM;
      const int n_idx = (tile / p.num_m_blocks) * BLOCK_N + (int)cta_rank * kHalfN;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait_a(empty0 + 8u * stage, phase ^ 1);
        if (elect_one()) {
          const uint32_t sa = smem0 + (uint32_t)stage * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          const uint32_t fb = full0_even + 8u * stage;
          if (leader) mbar_arrive_expect_tx_a(full0 + 8u * stage, 2 * Cfg::kStageBytes);
          const int k_idx = kb * kBlockK;
          if constexpr (!A_MN) {
            tma_load_2d_pair_a(sa, &tm_a, fb, k_idx, m_idx);
          } else {
#pragma unroll
            for (int j = 0; j < kBlockM / 64; ++j) tma_load_2d_pair_a(sa + j * 8192, &tm_a, fb, m_idx + 64 * j, k_idx);
          }
          if constexpr (!B_MN) {
            tma_load_2d_pair_a(sb, &tm_b, fb, k_idx, n_idx);
          } else {
#pragma unroll
            for (int j = 0; j < kHalfN / 64; ++j) tma_load_2d_pair_a(sb + j * 8192, &tm_b, fb, n_idx + 64 * j, k_idx);
          }
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------- MMA issuer (even CTA only) ------------------------------
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * kBlockM, BLOCK_N, A_MN, B_MN);
      const uint64_t adesc0 = umma_smem_desc(smem0, DescConsts<A_MN>::kLbo, 1024u);
      const uint64_t bdesc0 = umma_smem_desc(smem0 + Cfg::kABytes, DescConsts<B_MN>::kLbo, 1024u);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++iter) {
        const int acc = iter & 1;
        const uint32_t acc_phase = (iter >> 1) & 1;
        mbar_wait_a(tempty0 + 8u * acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          mbar_wait_a(full0 + 8u * stage, phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t soff16 = ((uint32_t)stage * Cfg::kStageBytes) >> 4;
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              umma_bf16_pair(d_tmem, desc_with_lo(adesc0, soff16 + k * DescConsts<A_MN>::kKStep16),
                             desc_with_lo(bdesc0, soff16 + k * DescConsts<B_MN>::kKStep16), idesc,
                             (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit_pair_a(empty0 + 8u * stage, 0b11);
            if (kb == p.num_k_blocks - 1) umma_commit_pair_a(tfull0 + 8u * acc, 0b11);
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------- epilogue (both CTAs, own 128 rows) ----------------------
    const int quad = warp & 3;
    const int half = warp >> 2;
    float* epi_stage =
        reinterpret_cast<float*>(smem_gen + (size_t)kStages * Cfg::kStageBytes) + warp * 32 * kEpiLd;
    const DropoutCfg drop = dropout_resolve(p.drop);
    const uint2 seed = make_uint2(drop.seed_lo, drop.seed_hi);
    int iter = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++iter) {
      const int acc = iter & 1;
      const uint32_t acc_phase = (iter >> 1) & 1;
      const int m_idx = (tile % p.num_m_blocks) * (2 * kBlockM) + (int)cta_rank * kBlockM;
      const int n_idx = (tile / p.num_m_blocks) * BLOCK_N;
      EpiOperands<EPI> ops;
      drain_prefetch<BLOCK_N, EPI>(p, m_idx + quad * 32, n_idx, half, lane, ops);
      mbar_wait_a(tfull0 + 8u * acc, acc_phase);
      tc_fence_after();
      drain_accumulator<BLOCK_N, EPI>(p, tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BLOCK_N),
                                      m_idx + quad * 32, n_idx, epi_stage, lane, half, ops, seed);
      tc_fence_before();
      mbar_arrive_cluster_a(tempty0_even + 8u * acc);  // the even CTA's MMA thread owns the accumulator handshake
    }
  }

  tc_fence_before();
  cluster_sync_all();  // no CTA may exit (or free TMEM) while its peer can still touch its smem / barriers
  if (warp == kMmaWarp) tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// Two independent GEMMs in ONE persistent launch: the data gradient and the weight gradient of a Linear
// (dX = dY W and dW = dY^T X, autograd of bridge_module.py:98,118,196-198,216) share nothing but dY and do not
// depend on each other. For the 2304-wide projections at T = 1024 rows each of them alone is a bad fit for 74
// CTA pairs -- the dgrad is 72 pair tiles (one tile per pair: launch ramp, pipeline fill and the whole epilogue
// exposed, ~5 us of MMA inside ~14 us), the wgrad 162 tiles (2.2 waves, 18 us) -- while together they are 234
// tiles of 36 / 16 k-blocks = 70 k-block units per pair with one ramp and every epilogue but the last overlapped
// by the next tile's main loop.
//   problem 0: A K-major, B MN-major (dgrad form),  epilogue EPI0
//   problem 1: A MN-major, B MN-major (wgrad form), epilogue EPI1
// Both use 256 x 128 pair tiles. Tiles are numbered problem 0 first (its tiles are the long ones), then problem 1;
// pair p takes tiles p, p + P, ... Per tile the three roles pick the problem's tensor maps, instruction
// descriptor, A-operand descriptor form and epilogue; everything else is the single-problem kernel above, and a
// tile's arithmetic is identical to it (same k order), so results are bit-equal to two separate launches.
// ------------------------------------------------------------------------------------------------
template <int EPI0, int EPI1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_pair_dual_kernel(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_b0,
                              const __grid_constant__ CUtensorMap tm_a1, const __grid_constant__ CUtensorMap tm_b1,
                              const GemmKernelParams p0, const GemmKernelParams p1) {
  constexpr int BLOCK_N = 128;
  using Cfg = GemmPairCfg<BLOCK_N>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kHalfN = BLOCK_N / 2;

  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kStages];
  __shared__ __align__(8) uint64_t empty_bar[kStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int pair_id = (int)cluster_id_x();
  const int num_pairs = (int)cluster_nctaid_x();
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem0 - smem_u32(smem_raw));
  const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
  const uint32_t tfull0 = smem_u32(tmem_full_bar), tempty0 = smem_u32(tmem_empty_bar);
  const uint32_t full0_even = full0 & 0xFEFFFFFFu;
  const uint32_t tempty0_even = mapa_u32(tempty0, 0);

  if (warp == kProducerWarp && lane == 0) {
    tma_prefetch_desc(&tm_a0);
    tma_prefetch_desc(&tm_b0);
    tma_prefetch_desc(&tm_a1);
    tma_prefetch_desc(&tm_b1);
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tmem_full_bar[0], 1);
    mbar_init(&tmem_full_bar[1], 1);
    mbar_init(&tmem_empty_bar[0], 2 * 32 * kEpiWarps);
    mbar_init(&tmem_empty_bar[1], 2 * 32 * kEpiWarps);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    tmem_alloc_pair(&tmem_base_smem, Cfg::kTmemCols);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t tmem_base = tmem_base_smem;
  const int tiles0 = p0.num_m_blocks * p0.num_n_blocks;
  const int num_tiles = tiles0 + p1.num_m_blocks * p1.num_n_blocks;

  if (warp == kProducerWarp) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs) {
      const bool second = tile >= tiles0;
      const int lt = second ? tile - tiles0 : tile;
      const int mb = second ? p1.num_m_blocks : p0.num_m_blocks;
      const int nkb = second ? p1.num_k_blocks : p0.num_k_blocks;
      const CUtensorMap* ta = second ? &tm_a1 : &tm_a0;
      const CUtensorMap* tb = second ? &tm_b1 : &tm_b0;
      const int m_idx = (lt % mb) * (2 * kBlockM) + (int)cta_rank * kBlockM;
      const int n_idx = (lt / mb) * BLOCK_N + (int)cta_rank * kHalfN;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait_a(empty0 + 8u * stage, phase ^ 1);
        if (elect_one()) {
          const uint32_t sa = smem0 + (uint32_t)stage * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          const uint32_t fb = full0_even + 8u * stage;
          if (leader) mbar_arrive_expect_tx_a(full0 + 8u * stage, 2 * Cfg::kStageBytes);
          const int k_idx = kb * kBlockK;
          if (!second) {
            tma_load_2d_pair_a(sa, ta, fb, k_idx, m_idx);                       // A K-major: box {64 k, 128 rows}
          } else {
#pragma unroll
            for (int j = 0; j < kBlockM / 64; ++j) tma_load_2d_pair_a(sa + j * 8192, ta, fb, m_idx + 64 * j, k_idx);
          }
#pragma unroll
          for (int j = 0; j < kHalfN / 64; ++j) tma_load_2d_pair_a(sb + j * 8192, tb, fb, n_idx + 64 * j, k_idx);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == kMmaWarp) {
    if (leader) {
      constexpr uint32_t idesc0 = umma_idesc_bf16(2 * kBlockM, BLOCK_N, false, true);
      constexpr uint32_t idesc1 = umma_idesc_bf16(2 * kBlockM, BLOCK_N, true, true);
      const uint64_t adesc_k = umma_smem_desc(smem0, DescConsts<false>::kLbo, 1024u);
      const uint64_t adesc_mn = umma_smem_desc(smem0, DescConsts<true>::kLbo, 1024u);
      const uint64_t bdesc0 = umma_smem_desc(smem0 + Cfg::kABytes, DescConsts<true>::kLbo, 1024u);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++iter) {
        const bool second = tile >= tiles0;
        const int nkb = second ? p1.num_k_blocks : p0.num_k_blocks;
        const uint32_t idesc = second ? idesc1 : idesc0;
        const uint64_t adesc0 = second ? adesc_mn : adesc_k;
        const uint32_t a_kstep = second ? DescConsts<true>::kKStep16 : DescConsts<false>::kKStep16;
        const int acc = iter & 1;
        const uint32_t acc_phase = (iter >> 1) & 1;
        mbar_wait_a(tempty0 + 8u * acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait_a(full0 + 8u * stage, phase);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t soff16 = ((uint32_t)stage * Cfg::kStageBytes) >> 4;
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              umma_bf16_pair(d_tmem, desc_with_lo(adesc0, soff16 + k * a_kstep),
                             desc_with_lo(bdesc0, soff16 + k * DescConsts<true>::kKStep16), idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit_pair_a(empty0 + 8u * stage, 0b11);
            if (kb == nkb - 1) umma_commit_pair_a(tfull0 + 8u * acc, 0b11);
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    const int quad = warp & 3;
    const int half = warp >> 2;
    float* epi_stage =
        reinterpret_cast<float*>(smem_gen + (size_t)kStages * Cfg::kStageBytes) + warp * 32 * kEpiLd;
    const uint2 seed = make_uint2(0u, 0u);   // neither epilogue of a gradient pair draws dropout bits
    int iter = 0;
    for (int tile = pair_id; tile < num_tiles; tile += num_pairs, ++iter) {
      const bool second = tile >= tiles0;
      const int lt = second ? tile - tiles0 : tile;
      const int mb = second ? p1.num_m_blocks : p0.num_m_blocks;
      const int acc = iter & 1;
      const uint32_t acc_phase = (iter >> 1) & 1;
      const int m_idx = (lt % mb) * (2 * kBlockM) + (int)cta_rank * kBlockM;
      const int n_idx = (lt / mb) * BLOCK_N;
      const uint32_t t_row = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BLOCK_N);
      if (!second) {
        EpiOperands<EPI0> ops;
        drain_prefetch<BLOCK_N, EPI0>(p0, m_idx + quad * 32, n_idx, half, lane, ops);
        mbar_wait_a(tfull0 + 8u * acc, acc_phase);
        tc_fence_after();
        drain_accumulator<BLOCK_N, EPI0>(p0, t_row, m_idx + quad * 32, n_idx, epi_stage, lane, half, ops, seed);
      } else {
        EpiOperands<EPI1> ops;
        drain_prefetch<BLOCK_N, EPI1>(p1, m_idx + quad * 32, n_idx, half, lane, ops);
        mbar_wait_a(tfull0 + 8u * acc, acc_phase);
        tc_fence_after();
        drain_accumulator<BLOCK_N, EPI1>(p1, t_row, m_idx + quad * 32, n_idx, epi_stage, lane, half, ops, seed);
      }
      tc_fence_before();
      mbar_arrive_cluster_a(tempty0_even + 8u * acc);
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == kMmaWarp) tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

// bf16 row-major 2-D tensor [outer, inner] (inner contiguous), 128B swizzle, box {64, box_outer}
static int make_tmap_bf16(CUtensorMap* tm, const void* base, uint64_t inner, uint64_t outer,
                          uint64_t ld_elems, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) {
    set_last_error("cuTensorMapEncodeTiled not available from the driver");
    return B200B_ERR_DRIVER;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {64, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed (%d): inner=%llu outer=%llu ld=%llu box_outer=%u base=%p", (int)r,
                   (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld_elems, box_outer, base);
    return B200B_ERR_TENSORMAP;
  }
  return B200B_OK;
}

template <bool PAIR, int BLOCK_N, bool A_MN, bool B_MN, int EPI>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const GemmKernelParams& p, int grid,
                       cudaStream_t stream) {
  static bool configured = false;  // benign race: attribute set is idempotent
  if constexpr (PAIR) {
    auto kern = gemm_tcgen05_pair_kernel<BLOCK_N, A_MN, B_MN, EPI>;
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)GemmPairCfg<BLOCK_N>::kSmemBytes);
      if (e != cudaSuccess) {
        set_last_error("cudaFuncSetAttribute(gemm pair) failed: %s", cudaGetErrorString(e));
        return (int)e;
      }
      configured = true;
    }
    launch_pdl(kPdlGemm, kern, dim3(grid), dim3(kGemmThreads), GemmPairCfg<BLOCK_N>::kSmemBytes, stream, ta, tb, p);
    return check_launch("gemm_tcgen05_pair_kernel", stream);
  } else {
    auto kern = gemm_tcgen05_kernel<BLOCK_N, A_MN, B_MN, EPI>;
    if (!configured) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)GemmCfg<BLOCK_N>::kSmemBytes);
      if (e != cudaSuccess) {
        set_last_error("cudaFuncSetAttribute(gemm) failed: %s", cudaGetErrorString(e));
        return (int)e;
      }
      configured = true;
    }
    launch_pdl(kPdlGemm, kern, dim3(grid), dim3(kGemmThreads), GemmCfg<BLOCK_N>::kSmemBytes, stream, ta, tb, p);
    return check_launch("gemm_tcgen05_kernel", stream);
  }
}

template <bool PAIR, int BLOCK_N, bool A_MN, bool B_MN>
static int dispatch_epi(int epi, const CUtensorMap& ta, const CUtensorMap& tb, const GemmKernelParams& p, int grid,
                        cudaStream_t stream) {
  switch (epi) {
    case B200B_EPI_BF16_BIAS:
      return launch_gemm<PAIR, BLOCK_N, A_MN, B_MN, B200B_EPI_BF16_BIAS>(ta, tb, p, grid, stream);
    case B200B_EPI_BF16_DGELU:
      return launch_gemm<PAIR, BLOCK_N, A_MN, B_MN, B200B_EPI_BF16_DGELU>(ta, tb, p, grid, stream);
    case B200B_EPI_F32:
      return launch_gemm<PAIR, BLOCK_N, A_MN, B_MN, B200B_EPI_F32>(ta, tb, p, grid, stream);
    default:
      break;
  }
  if constexpr (!A_MN && !B_MN) {
    switch (epi) {
      case B200B_EPI_BF16_BIAS_GELU:
        return launch_gemm<PAIR, BLOCK_N, false, false, B200B_EPI_BF16_BIAS_GELU>(ta, tb, p, grid, stream);
      case B200B_EPI_F32_BIAS_RESID:
        return launch_gemm<PAIR, BLOCK_N, false, false, B200B_EPI_F32_BIAS_RESID>(ta, tb, p, grid, stream);
      default:
        break;
    }
  }
  set_last_error("gemm: epilogue %d not built for a_major=%d b_major=%d", epi, (int)A_MN, (int)B_MN);
  return B200B_ERR_ARG;
}

template <bool PAIR, int BLOCK_N>
static int dispatch_major(int a_mn, int b_mn, int epi, const CUtensorMap& ta, const CUtensorMap& tb,
                          const GemmKernelParams& p, int grid, cudaStream_t stream) {
  if (!a_mn && !b_mn) return dispatch_epi<PAIR, BLOCK_N, false, false>(epi, ta, tb, p, grid, stream);
  if (!a_mn && b_mn) return dispatch_epi<PAIR, BLOCK_N, false, true>(epi, ta, tb, p, grid, stream);
  if (a_mn && b_mn) return dispatch_epi<PAIR, BLOCK_N, true, true>(epi, ta, tb, p, grid, stream);
  set_last_error("gemm: a_major=1,b_major=0 is not built");
  return B200B_ERR_ARG;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Tile configuration: CTAs per tile (1 or 2) and tile width. The cost model counts waves of
// tiles over the SMs times a per-tile cost proportional to the tile's k-loop length, with a
// penalty for configurations that fetch more operand bytes from L2 per flop (measured: the main
// loop is paced by operand delivery, not by the tensor pipe, for 128-row tiles).
struct TileChoice {
  int cta_group, block_n;
};

TileChoice choose_tile(int m, int n, int num_sms) {
  // CTA pairs beat single CTAs on every bridge shape measured (profiles/r01_gemm_tile_sweep.jsonl);
  // the width is chosen by counting waves of pair tiles over the num_sms/2 pairs. 128-wide tiles
  // sustain ~88% of the 256-wide main-loop rate.
  const long long units = num_sms >= 2 ? num_sms / 2 : 1;
  double best = 1e300;
  TileChoice out{2, 256};
  const int widths[2] = {256, 128};
  for (int bn : widths) {
    const long long tiles = ((m + 255) / 256) * (long long)((n + bn - 1) / bn);
    const long long waves = (tiles + units - 1) / units;
    const double cost = (double)waves * bn / (bn == 256 ? 1.0 : 0.88);
    if (cost < best) { best = cost; out = {2, bn}; }
  }
  return out;
}

}  // namespace b200b

using namespace b200b;

extern "C" int b200b_gemm(const b200b_gemm_args* a, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (a == nullptr || a->a == nullptr || a->b == nullptr || a->out == nullptr) {
    set_last_error("gemm: null argument");
    return B200B_ERR_ARG;
  }
  // m and k may be ragged (TMA zero-fills out-of-bounds box elements; the epilogue masks rows);
  // n must be a multiple of 8 because the epilogue stores 8 columns at a time.
  if (a->m <= 0 || a->n <= 0 || a->k <= 0 || (a->n % 8) != 0) {
    set_last_error("gemm: need m,n,k > 0 and n a multiple of 8 (got m=%d n=%d k=%d)", a->m, a->n, a->k);
    return B200B_ERR_SHAPE;
  }
  const int epi = a->epilogue;
  if (epi < 0 || epi > B200B_EPI_F32) {
    set_last_error("gemm: bad epilogue %d", epi);
    return B200B_ERR_ARG;
  }
  const bool out_f32 = (epi == B200B_EPI_F32_BIAS_RESID || epi == B200B_EPI_F32);
  if (!aligned16(a->a) || !aligned16(a->b) || !aligned16(a->out) || (a->lda % 8) || (a->ldb % 8) ||
      (a->ldo % (out_f32 ? 4 : 8))) {
    set_last_error("gemm: operands must be 16-byte aligned with 16-byte aligned row pitch");
    return B200B_ERR_ALIGN;
  }
  if (a->bias != nullptr && !aligned16(a->bias)) {
    set_last_error("gemm: bias must be 16-byte aligned");
    return B200B_ERR_ALIGN;
  }
  if (epi == B200B_EPI_BF16_BIAS_GELU || epi == B200B_EPI_BF16_DGELU) {
    if (a->aux == nullptr || !aligned16(a->aux) || (a->ldaux % 8)) {
      set_last_error("gemm: epilogue %d needs a 16-byte aligned aux tensor", epi);
      return B200B_ERR_ARG;
    }
  }
  if (epi == B200B_EPI_F32_BIAS_RESID) {
    if (a->resid == nullptr || !aligned16(a->resid) || (a->ldr % 4)) {
      set_last_error("gemm: residual epilogue needs a 16-byte aligned resid tensor");
      return B200B_ERR_ARG;
    }
  }
  if (!(a->dropout_p >= 0.0f && a->dropout_p < 1.0f)) {
    set_last_error("gemm: dropout_p must be in [0,1)");
    return B200B_ERR_ARG;
  }
  int num_sms = 0;
  int rc = device_sm_count(&num_sms);
  if (rc != B200B_OK) return rc;

  int block_n = a->block_n;
  int cta_group = (int)a->cta_group;
  if (block_n == 0 || cta_group == 0) {
    const TileChoice c = choose_tile(a->m, a->n, num_sms);
    if (block_n == 0 && cta_group == 0) { block_n = c.block_n; cta_group = c.cta_group; }
    else if (block_n == 0) block_n = 256;
    else cta_group = 1;
  }
  if ((block_n != 128 && block_n != 256) || (cta_group != 1 && cta_group != 2)) {
    set_last_error("gemm: block_n must be 0, 128 or 256 and cta_group 0, 1 or 2");
    return B200B_ERR_ARG;
  }
  // A CTA pair occupies two SMs. Under an SM limit of 1 the tiles run on single CTAs instead: the
  // per-element k order is the same, so the result is too.
  if (num_sms < 2) cta_group = 1;
  const bool pair = cta_group == 2;
  // rows of the B tile one CTA stages: the whole tile, or half of it in a CTA pair
  const int b_rows = pair ? block_n / 2 : block_n;

  CUtensorMap ta, tb;
  if (!a->a_major) rc = make_tmap_bf16(&ta, a->a, (uint64_t)a->k, (uint64_t)a->m, (uint64_t)a->lda, kBlockM);
  else             rc = make_tmap_bf16(&ta, a->a, (uint64_t)a->m, (uint64_t)a->k, (uint64_t)a->lda, kBlockK);
  if (rc != B200B_OK) return rc;
  if (!a->b_major) rc = make_tmap_bf16(&tb, a->b, (uint64_t)a->k, (uint64_t)a->n, (uint64_t)a->ldb, (uint32_t)b_rows);
  else             rc = make_tmap_bf16(&tb, a->b, (uint64_t)a->n, (uint64_t)a->k, (uint64_t)a->ldb, kBlockK);
  if (rc != B200B_OK) return rc;

  GemmKernelParams p;
  p.m = a->m; p.n = a->n; p.k = a->k;
  const int tile_m = pair ? 2 * kBlockM : kBlockM;
  p.num_m_blocks = (a->m + tile_m - 1) / tile_m;
  p.num_n_blocks = (a->n + block_n - 1) / block_n;
  p.num_k_blocks = (a->k + kBlockK - 1) / kBlockK;
  p.out = a->out; p.ldo = a->ldo;
  p.aux = a->aux; p.ldaux = a->ldaux;
  p.bias = a->bias;
  p.resid = a->resid; p.ldr = a->ldr;
  p.beta = a->beta;
  p.drop_stream = a->dropout_stream;
  p.drop = make_dropout_cfg(a->dropout_p, a->seed, &p.drop_stream);

  const long long tiles = (long long)p.num_m_blocks * p.num_n_blocks;
  if (pair) {
    const long long pairs = num_sms / 2;
    const int grid = 2 * (int)(tiles < pairs ? tiles : pairs);
    if (block_n == 256) return dispatch_major<true, 256>(a->a_major, a->b_major, epi, ta, tb, p, grid, stream);
    return dispatch_major<true, 128>(a->a_major, a->b_major, epi, ta, tb, p, grid, stream);
  }
  const int grid = (int)(tiles < num_sms ? tiles : num_sms);
  if (block_n == 256) return dispatch_major<false, 256>(a->a_major, a->b_major, epi, ta, tb, p, grid, stream);
  return dispatch_major<false, 128>(a->a_major, a->b_major, epi, ta, tb, p, grid, stream);
}

// ---- the grouped dgrad + wgrad launch ------------------------------------------------------------
namespace b200b {

static void fill_params(const b200b_gemm_args* a, GemmKernelParams* p) {
  p->m = a->m; p->n = a->n; p->k = a->k;
  p->num_m_blocks = (a->m + 2 * kBlockM - 1) / (2 * kBlockM);
  p->num_n_blocks = (a->n + 127) / 128;
  p->num_k_blocks = (a->k + kBlockK - 1) / kBlockK;
  p->out = a->out; p->ldo = a->ldo;
  p->aux = nullptr; p->ldaux = 0;
  p->bias = a->bias;
  p->resid = nullptr; p->ldr = 0;
  p->beta = a->beta;
  p->drop_stream = 0;
  p->drop = make_dropout_cfg(0.f, 0, nullptr);
}

template <int EPI1>
static int launch_dual(const CUtensorMap& ta0, const CUtensorMap& tb0, const CUtensorMap& ta1, const CUtensorMap& tb1,
                       const GemmKernelParams& p0, const GemmKernelParams& p1, int grid, cudaStream_t stream) {
  static bool configured = false;  // benign race: attribute set is idempotent
  auto kern = gemm_tcgen05_pair_dual_kernel<B200B_EPI_BF16_BIAS, EPI1>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GemmPairCfg<128>::kSmemBytes);
    if (e != cudaSuccess) {
      set_last_error("cudaFuncSetAttribute(gemm dual) failed: %s", cudaGetErrorString(e));
      return (int)e;
    }
    configured = true;
  }
  launch_pdl(kPdlGemm, kern, dim3(grid), dim3(kGemmThreads), GemmPairCfg<128>::kSmemBytes, stream, ta0, tb0, ta1, tb1, p0, p1);
  return check_launch("gemm_tcgen05_pair_dual_kernel", stream);
}

static int g_gemm_dual = -1;   // 1 = grouped launch where it applies (default); B200B_GEMM_DUAL=0 / b200b_gemm_set_dual(0): two launches

}  // namespace b200b

extern "C" int b200b_gemm_set_dual(int on) {
  if (g_gemm_dual < 0) {
    const char* e = getenv("B200B_GEMM_DUAL");
    g_gemm_dual = e ? atoi(e) : 1;
  }
  const int prev = g_gemm_dual;
  if (on >= 0) g_gemm_dual = on;
  return prev;
}

extern "C" int b200b_gemm_dual(const b200b_gemm_args* dgrad, const b200b_gemm_args* wgrad, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (dgrad == nullptr || wgrad == nullptr) {
    set_last_error("gemm_dual: null argument");
    return B200B_ERR_ARG;
  }
  int num_sms = 0;
  int rc = device_sm_count(&num_sms);
  if (rc != B200B_OK) return rc;
  // The grouped kernel covers exactly the pair it was written for: dgrad form (A K-major, B MN-major, bf16 out, no
  // bias) + wgrad form (A and B MN-major, fp32 or bf16 out, no bias, beta = 0), both on 256 x 128 pair tiles, no
  // dropout, at least one CTA pair under the SM limit. Anything else runs as the two launches it stands for.
  const bool eligible =
      b200b_gemm_set_dual(-1) != 0 && num_sms >= 2 && dgrad->a_major == 0 && dgrad->b_major == 1 && dgrad->epilogue == B200B_EPI_BF16_BIAS &&
      dgrad->bias == nullptr && wgrad->a_major == 1 && wgrad->b_major == 1 &&
      (wgrad->epilogue == B200B_EPI_F32 || wgrad->epilogue == B200B_EPI_BF16_BIAS) && wgrad->bias == nullptr &&
      wgrad->beta == 0.f && dgrad->dropout_p == 0.f && wgrad->dropout_p == 0.f && dgrad->block_n == 0 && wgrad->block_n == 0 &&
      dgrad->cta_group == 0 && wgrad->cta_group == 0 && dgrad->m > 0 && dgrad->n > 0 && dgrad->k > 0 && wgrad->m > 0 &&
      wgrad->n > 0 && wgrad->k > 0 && (dgrad->n % 8) == 0 && (wgrad->n % 8) == 0 &&
      choose_tile(dgrad->m, dgrad->n, num_sms).block_n == 128 && choose_tile(wgrad->m, wgrad->n, num_sms).block_n == 128 &&
      aligned16(dgrad->a) && aligned16(dgrad->b) && aligned16(dgrad->out) && aligned16(wgrad->a) && aligned16(wgrad->b) &&
      aligned16(wgrad->out) && (dgrad->lda % 8) == 0 && (dgrad->ldb % 8) == 0 && (dgrad->ldo % 8) == 0 &&
      (wgrad->lda % 8) == 0 && (wgrad->ldb % 8) == 0 && (wgrad->ldo % (wgrad->epilogue == B200B_EPI_F32 ? 4 : 8)) == 0;
  if (!eligible) {
    rc = b200b_gemm(wgrad, stream_);
    if (rc != B200B_OK) return rc;
    return b200b_gemm(dgrad, stream_);
  }
  CUtensorMap ta0, tb0, ta1, tb1;
  if ((rc = make_tmap_bf16(&ta0, dgrad->a, (uint64_t)dgrad->k, (uint64_t)dgrad->m, (uint64_t)dgrad->lda, kBlockM)) != B200B_OK) return rc;
  if ((rc = make_tmap_bf16(&tb0, dgrad->b, (uint64_t)dgrad->n, (uint64_t)dgrad->k, (uint64_t)dgrad->ldb, kBlockK)) != B200B_OK) return rc;
  if ((rc = make_tmap_bf16(&ta1, wgrad->a, (uint64_t)wgrad->m, (uint64_t)wgrad->k, (uint64_t)wgrad->lda, kBlockK)) != B200B_OK) return rc;
  if ((rc = make_tmap_bf16(&tb1, wgrad->b, (uint64_t)wgrad->n, (uint64_t)wgrad->k, (uint64_t)wgrad->ldb, kBlockK)) != B200B_OK) return rc;
  GemmKernelParams p0, p1;
  fill_params(dgrad, &p0);
  fill_params(wgrad, &p1);
  const long long tiles = (long long)p0.num_m_blocks * p0.num_n_blocks + (long long)p1.num_m_blocks * p1.num_n_blocks;
  const long long pairs = num_sms / 2;
  const int grid = 2 * (int)(tiles < pairs ? tiles : pairs);
  if (wgrad->epilogue == B200B_EPI_F32) return launch_dual<B200B_EPI_F32>(ta0, tb0, ta1, tb1, p0, p1, grid, stream);
  return launch_dual<B200B_EPI_BF16_BIAS>(ta0, tb0, ta1, tb1, p0, p1, grid, stream);
}
