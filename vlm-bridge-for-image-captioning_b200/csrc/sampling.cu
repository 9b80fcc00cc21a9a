// Temperature / top-p sampling of one token per row of the vocabulary logits (decode, SURVEY.md 8a row a12).
// Replaces, per decode step of FullModel.generate_caption(do_sample=True) (full_model.py:264-350):
//   NaN / Inf guards -> logits / temperature -> top-p filter (sort, softmax, cumsum, scatter) -> multinomial
// which in PyTorch is a full-row sort plus four more passes and launches over [rows, V] floats.
//
// Here one row is split over a cluster of CS CTAs (csrc/sampling.cu, sample_cluster_size): each CTA copies its
// slice of the row from HBM into shared memory once, and every later pass runs on chip; the per-CTA partials
// (row max and guard flags, count and mass histograms, the final argmax) are combined through distributed shared memory.
// The rule (b200_bridge.h, b200b_sample_tokens_top_k):
//   1. guards: a row with a NaN becomes all zeros; else a row with an Inf is clamped to [-100, 100];
//   2. z = x / T in fp32;
//   3a. 0 < top_k < V: token i passes iff z_i >= the k-th largest z (duplicates counted, ties pass together); the
//      threshold is a radix select BY COUNT over an order-preserving 32-bit image of z: three histogram passes
//      (11 + 11 + 10 bits) of token counts, combined over the cluster in rank order (integers: every CTA picks the
//      same threshold); skipped when top_k == 0 or top_k >= V;
//   3b. of the tokens that passed 3a, token i is kept iff the softmax mass of the passing tokens with strictly
//      larger z is < top_p times the mass of all passing tokens; the threshold is the same radix select BY MASS:
//      three histogram passes of exp(z - zmax) in 2^-40 fixed point over the passing keys (integer adds: the same
//      sums in any order, so the choice is deterministic and identical in every CTA of the cluster); skipped when
//      top_p == 1;
//   4. argmax over kept tokens of z + g, g = -ln(-ln u) (Gumbel-max: an exact draw from the renormalised nucleus),
//      ties to the smallest index; u from Philox4x32-10 as documented in the header.
#include <math.h>

#include <cooperative_groups.h>

#include "common.cuh"
#include "launch.h"

namespace cg = cooperative_groups;

namespace b200b {

constexpr int kSampThreads = 512;
constexpr int kSampBins = 2048;                       // 11-bit radix digit
constexpr int kSampBinsPerThread = kSampBins / kSampThreads;
constexpr int kSampMaxCluster = 8;                    // portable cluster size limit
constexpr long long kSampSliceBytes = 176 * 1024;     // logits slice per CTA (+ 24.6 KB of histograms)
constexpr uint32_t kSampleTag = 0x5a3b1e00u;          // 4th Philox counter word; dropout uses 0x0b200b00
constexpr float kSampLog2e = 1.4426950408889634f;
constexpr float kSampMassOne = 1099511627776.0f;      // 2^40: fixed-point unit of exp(z - zmax) <= 1

struct SampStats {
  float max;            // largest logit of the slice, NaN ignored
  uint32_t flags;       // 1: a NaN was seen, 2: an Inf was seen
  float best_key;       // largest z + g over the kept tokens of the slice
  uint32_t pad;
  long long best_idx;   // its vocabulary index (smallest on ties)
};

// order-preserving image of a float (larger z -> larger key); -0 and +0 map to the same key
__device__ __forceinline__ uint32_t samp_key(float z) {
  const uint32_t b = __float_as_uint(z == 0.0f ? 0.0f : z);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ bool samp_better(float k1, long long i1, float k2, long long i2) {
  return k1 > k2 || (k1 == k2 && i1 < i2);
}

// -ln(-ln u) for u = ((w >> 8) + 0.5) 2^-24. u takes 25 significant bits, one more than fp32 holds, so it is
// carried exactly as u (u < 1/2) or as 1 - u (u > 1/2; both < 2^24 units of 2^-25): rounding u itself would turn
// the largest u into 1.0 and g into +inf.
__device__ __forceinline__ float samp_gumbel(uint32_t w) {
  const uint32_t m = w >> 8;
  float nlu;   // -ln u > 0
  if (m < (1u << 23)) {
    nlu = -logf((float)(2u * m + 1u) * 2.98023223876953125e-8f);                  // 2^-25
  } else {
    nlu = -log1pf(-(float)((1u << 25) - 2u * m - 1u) * 2.98023223876953125e-8f);
  }
  return -logf(nlu);
}

template <typename T>
__device__ __forceinline__ float samp_f(T v) {
  if constexpr (sizeof(T) == 2) return __bfloat162float(v);
  else return v;
}

template <bool BF16, int CS>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(kSampThreads, 1)
    sample_kernel(const void* __restrict__ logits, long long ld, long long vocab, long long slice, float temperature,
                  uint32_t top_k, float top_p, const unsigned long long* __restrict__ seed_ptr, uint32_t step,
                  long long* __restrict__ ids_out, long long ids_stride) {
  using T = typename std::conditional<BF16, __nv_bfloat16, float>::type;
  constexpr int kVec = 16 / (int)sizeof(T);
  extern __shared__ __align__(16) unsigned char samp_smem[];
  T* xs = reinterpret_cast<T*>(samp_smem);
  __shared__ uint32_t hmass_lo[kSampBins], hmass_hi[kSampBins];   // fixed-point mass, low / high word
  __shared__ uint32_t hcnt[kSampBins];
  __shared__ SampStats st;
  __shared__ float red_f[kSampThreads / 32];
  __shared__ uint32_t red_u[kSampThreads / 32];
  __shared__ long long red_i[kSampThreads / 32];
  __shared__ unsigned long long red_m[kSampThreads / 32];
  __shared__ unsigned long long sel_above;

  cg::cluster_group cluster = cg::this_cluster();
  const uint32_t rank = cluster.block_rank();
  const uint32_t row = blockIdx.x / CS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long lo = (long long)rank * slice;
  const int n = (int)max(0LL, min(slice, vocab - lo));

  pdl_prologue_late_trigger();
  const unsigned long long seed = __ldg(seed_ptr);

  // ---- pass 0: the slice HBM -> shared memory; max (NaN ignored), NaN / Inf flags ----
  const T* src = reinterpret_cast<const T*>(logits) + (long long)row * ld + lo;
  float mx = -INFINITY;
  uint32_t flags = 0;
  auto note = [&](float f) {
    mx = fmaxf(mx, f);
    flags |= (f != f) ? 1u : 0u;
    flags |= (fabsf(f) == INFINITY) ? 2u : 0u;
  };
  const int nv = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) ? n / kVec : 0;
  const uint4* src4 = reinterpret_cast<const uint4*>(src);
  uint4* xs4 = reinterpret_cast<uint4*>(xs);
  for (int v0 = tid; v0 < nv; v0 += 4 * kSampThreads) {
    uint4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int v = v0 + u * kSampThreads;
      if (v < nv) q[u] = __ldcs(src4 + v);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int v = v0 + u * kSampThreads;
      if (v < nv) {
        xs4[v] = q[u];
        const T* e = reinterpret_cast<const T*>(&q[u]);
#pragma unroll
        for (int j = 0; j < kVec; ++j) note(samp_f(e[j]));
      }
    }
  }
  for (int i = nv * kVec + tid; i < n; i += kSampThreads) {
    const T v = src[i];
    xs[i] = v;
    note(samp_f(v));
  }
  mx = warp_max(mx);
  flags = __reduce_or_sync(0xffffffffu, flags);
  if (lane == 0) {
    red_f[warp] = mx;
    red_u[warp] = flags;
  }
  __syncthreads();
  if (tid == 0) {
    float m = -INFINITY;
    uint32_t f = 0;
    for (int w = 0; w < kSampThreads / 32; ++w) {
      m = fmaxf(m, red_f[w]);
      f |= red_u[w];
    }
    st.max = m;
    st.flags = f;
  }
  cluster.sync();
  float gmax = -INFINITY;
  uint32_t gflags = 0;
  for (int r = 0; r < CS; ++r) {
    const SampStats* p = cluster.map_shared_rank(&st, r);
    gmax = fmaxf(gmax, p->max);
    gflags |= p->flags;
  }
  const bool nan_row = gflags & 1u, inf_row = gflags & 2u;
  auto zof = [&](T v) {
    float x = samp_f(v);
    x = nan_row ? 0.0f : (inf_row ? fminf(fmaxf(x, -100.0f), 100.0f) : x);
    return x / temperature;
  };
  const float zmax = (nan_row ? 0.0f : (inf_row ? fminf(fmaxf(gmax, -100.0f), 100.0f) : gmax)) / temperature;

  // ---- thresholds. kth: tokens with samp_key(z) >= kth are kept (0 keeps every token: keys are >= 0x007FFFFF).
  // kth_k: the top-k threshold (0: no top-k filter). The nucleus: the smallest present key k with
  // mass(key > k) < top_p * S, where its histograms count only keys >= kth_k (S: their mass), so every picked bin
  // holds such a key and the nucleus threshold ends >= kth_k. TopkFilter::value adds the `key >= kth_k` test to the
  // mass pass (a separate instantiation: the top_k == 0 path runs the loop without it).
  uint32_t kth = 0, kth_k = 0;
  auto nucleus = [&](auto topk_filter) {
    using TopkFilter = decltype(topk_filter);
    uint32_t prefix = 0;
    unsigned long long above = 0;   // mass of the tokens whose key lies above the current prefix range
    double limit = 0.0;
    for (int level = 0; level < 3; ++level) {
      const int shift = level == 0 ? 21 : (level == 1 ? 10 : 0);
      const uint32_t pmask = level == 0 ? 0u : (level == 1 ? 0xFFE00000u : 0xFFFFFC00u);
      const uint32_t dmask = level == 2 ? 0x3FFu : 0x7FFu;
      for (int b = tid; b < kSampBins; b += kSampThreads) {
        hmass_lo[b] = 0;
        hmass_hi[b] = 0;
        hcnt[b] = 0;
      }
      __syncthreads();
      for (int i = tid; i < n; i += kSampThreads) {
        const float z = zof(xs[i]);
        const uint32_t k = samp_key(z);
        if ((k & pmask) == prefix && (!TopkFilter::value || k >= kth_k)) {
          const uint32_t d = (k >> shift) & dmask;
          const unsigned long long m = __float2ull_rz(ex2_approx((z - zmax) * kSampLog2e) * kSampMassOne);
          // a 64-bit shared atomic add is a compare-and-swap loop, and logits crowd into a few exponent bins:
          // add the low word with the native 32-bit atomic and carry into the high word when it wraps (the
          // two words end as the exact 64-bit sum whatever the order)
          const uint32_t mlo = (uint32_t)m, old = atomicAdd(&hmass_lo[d], mlo);
          const uint32_t mhi = (uint32_t)(m >> 32) + (old + mlo < old ? 1u : 0u);
          if (mhi) atomicAdd(&hmass_hi[d], mhi);
          atomicAdd(&hcnt[d], 1u);
        }
      }
      cluster.sync();
      // the cluster's histogram, this thread's kSampBinsPerThread consecutive bins, summed in rank order
      unsigned long long mm[kSampBinsPerThread];
      uint32_t cc[kSampBinsPerThread];
#pragma unroll
      for (int j = 0; j < kSampBinsPerThread; ++j) {
        mm[j] = 0;
        cc[j] = 0;
      }
      for (int r = 0; r < CS; ++r) {
        const uint32_t* pl = cluster.map_shared_rank(hmass_lo, r);
        const uint32_t* ph = cluster.map_shared_rank(hmass_hi, r);
        const uint32_t* pc = cluster.map_shared_rank(hcnt, r);
#pragma unroll
        for (int j = 0; j < kSampBinsPerThread; ++j) {
          const int b = tid * kSampBinsPerThread + j;
          mm[j] += ((unsigned long long)ph[b] << 32) | pl[b];
          cc[j] += pc[b];
        }
      }
      cluster.sync();   // every CTA has read this CTA's histogram before the next level clears it
      // mass above each bin: suffix sums over the bins of higher threads, then within the thread
      unsigned long long tot = 0;
#pragma unroll
      for (int j = 0; j < kSampBinsPerThread; ++j) tot += mm[j];
      unsigned long long suf = tot;   // inclusive suffix over the lanes >= this one
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += t;
      }
      if (lane == 0) red_m[warp] = suf;
      __syncthreads();
      unsigned long long higher = suf - tot, total = 0;
      for (int w = 0; w < kSampThreads / 32; ++w) {
        if (w > warp) higher += red_m[w];
        total += red_m[w];
      }
      if (level == 0) limit = (double)top_p * (double)total;
      uint32_t pick = 0xFFFFFFFFu;
      unsigned long long pick_above = 0;
      unsigned long long a = above + higher;   // mass above bin j after the loop step
#pragma unroll
      for (int j = kSampBinsPerThread - 1; j >= 0; --j) {
        if (cc[j] > 0 && (double)a < limit) {
          pick = (uint32_t)(tid * kSampBinsPerThread + j);
          pick_above = a;
        }
        a += mm[j];
      }
      const uint32_t wpick = __reduce_min_sync(0xffffffffu, pick);
      if (lane == 0) red_u[warp] = wpick;
      __syncthreads();
      uint32_t bpick = 0xFFFFFFFFu;
      for (int w = 0; w < kSampThreads / 32; ++w) bpick = min(bpick, red_u[w]);
      if (pick == bpick && pick != 0xFFFFFFFFu) sel_above = pick_above;
      __syncthreads();
      // a bin always qualifies (the top non-empty one has mass above == `above` < limit); guard regardless
      if (bpick == 0xFFFFFFFFu) break;
      prefix |= bpick << shift;
      above = sel_above;
      if (level == 2) kth = prefix;
      __syncthreads();   // sel_above / red_u are rewritten by the next level
    }
  };

  // ---- top-k threshold kth_k: the key of the top_k-th largest z, counting duplicates ----
  if (top_k != 0) {
    uint32_t prefix = 0, above = 0;   // tokens whose key lies above the current prefix range
    for (int level = 0; level < 3; ++level) {
      const int shift = level == 0 ? 21 : (level == 1 ? 10 : 0);
      const uint32_t pmask = level == 0 ? 0u : (level == 1 ? 0xFFE00000u : 0xFFFFFC00u);
      const uint32_t dmask = level == 2 ? 0x3FFu : 0x7FFu;
      for (int b = tid; b < kSampBins; b += kSampThreads) hcnt[b] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += kSampThreads) {
        const uint32_t k = samp_key(zof(xs[i]));
        if ((k & pmask) == prefix) atomicAdd(&hcnt[(k >> shift) & dmask], 1u);
      }
      cluster.sync();
      uint32_t cc[kSampBinsPerThread];
#pragma unroll
      for (int j = 0; j < kSampBinsPerThread; ++j) cc[j] = 0;
      for (int r = 0; r < CS; ++r) {
        const uint32_t* pc = cluster.map_shared_rank(hcnt, r);
#pragma unroll
        for (int j = 0; j < kSampBinsPerThread; ++j) cc[j] += pc[tid * kSampBinsPerThread + j];
      }
      cluster.sync();   // every CTA has read this CTA's histogram before the next level clears it
      uint32_t tot = 0;
#pragma unroll
      for (int j = 0; j < kSampBinsPerThread; ++j) tot += cc[j];
      uint32_t suf = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += t;
      }
      if (lane == 0) red_m[warp] = suf;
      __syncthreads();
      uint32_t higher = suf - tot;
      for (int w = warp + 1; w < kSampThreads / 32; ++w) higher += (uint32_t)red_m[w];
      // the one bin with count(key above it) < top_k <= count(key above it) + its count
      uint32_t pick = 0xFFFFFFFFu, pick_above = 0;
      uint32_t a = above + higher;
#pragma unroll
      for (int j = kSampBinsPerThread - 1; j >= 0; --j) {
        if (a < top_k && a + cc[j] >= top_k) {
          pick = (uint32_t)(tid * kSampBinsPerThread + j);
          pick_above = a;
        }
        a += cc[j];
      }
      const uint32_t wpick = __reduce_min_sync(0xffffffffu, pick);
      if (lane == 0) red_u[warp] = wpick;
      __syncthreads();
      uint32_t bpick = 0xFFFFFFFFu;
      for (int w = 0; w < kSampThreads / 32; ++w) bpick = min(bpick, red_u[w]);
      if (pick == bpick && pick != 0xFFFFFFFFu) sel_above = pick_above;
      __syncthreads();
      // a bin always qualifies (top_k < V tokens in all); guard regardless
      if (bpick == 0xFFFFFFFFu) break;
      prefix |= bpick << shift;
      above = (uint32_t)sel_above;
      if (level == 2) kth_k = prefix;
      __syncthreads();   // sel_above / red_u / red_m are rewritten by the next level
    }
    kth = kth_k;
    if (top_p < 1.0f) nucleus(std::true_type{});
  } else if (top_p < 1.0f) {
    nucleus(std::false_type{});
  }

  // ---- draw: argmax over the kept tokens of z + Gumbel noise ----
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  float best = -INFINITY;
  long long best_i = 0x7fffffffffffffffLL;
  const int ngroups = (n + 3) >> 2;
  for (int g = tid; g < ngroups; g += kSampThreads) {
    float z[4];
    bool keep[4];
    bool any = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int i = g * 4 + e;
      z[e] = i < n ? zof(xs[i]) : 0.0f;
      keep[e] = i < n && samp_key(z[e]) >= kth;
      any |= keep[e];
    }
    if (!any) continue;
    const long long gi = (lo >> 2) + g;   // lo is a multiple of 8: groups of 4 are aligned to the vocabulary
    const uint4 w4 = philox4x32_10(make_uint4((uint32_t)gi, row, step, kSampleTag), key);
    const uint32_t ws[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (!keep[e]) continue;
      const float k = z[e] + samp_gumbel(ws[e]);
      const long long idx = lo + g * 4 + e;
      if (samp_better(k, idx, best, best_i)) {
        best = k;
        best_i = idx;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float k2 = __shfl_xor_sync(0xffffffffu, best, o);
    const long long i2 = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (samp_better(k2, i2, best, best_i)) {
      best = k2;
      best_i = i2;
    }
  }
  if (lane == 0) {
    red_f[warp] = best;
    red_i[warp] = best_i;
  }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kSampThreads / 32; ++w)
      if (samp_better(red_f[w], red_i[w], best, best_i)) {
        best = red_f[w];
        best_i = red_i[w];
      }
    st.best_key = best;
    st.best_idx = best_i;
  }
  cluster.sync();
  if (rank == 0 && tid == 0) {
    for (int r = 1; r < CS; ++r) {
      const SampStats* p = cluster.map_shared_rank(&st, r);
      if (samp_better(p->best_key, p->best_idx, best, best_i)) {
        best = p->best_key;
        best_i = p->best_idx;
      }
    }
    ids_out[(long long)row * ids_stride] = best_i;
  }
  cluster.sync();   // no CTA leaves while rank 0 still reads its shared memory
}

// Cluster size: the fewest CTAs whose slices fit kSampSliceBytes, doubled (up to kSampMaxCluster) while the
// rows * CTAs do not cover the SMs and every CTA keeps at least 4096 tokens. 0 if the row does not fit.
// The beam-step kernel (csrc/beam.cu) splits its rows by the same rule.
int sample_cluster_size(long long rows, long long vocab, int esz, int sms, long long* slice) {
  auto slice_of = [&](int c) { return ((vocab + c - 1) / c + 7) / 8 * 8; };
  int c = 1;
  while (c <= kSampMaxCluster && slice_of(c) * esz > kSampSliceBytes) c *= 2;
  if (c > kSampMaxCluster) return 0;
  while (c < kSampMaxCluster && rows * c < sms && vocab >= 2LL * c * 4096) c *= 2;
  *slice = slice_of(c);
  return c;
}

template <bool BF16, int CS>
static int sample_launch(const void* logits, long long ld, long long rows, long long vocab, long long slice,
                         float temperature, uint32_t top_k, float top_p, const unsigned long long* seed,
                         uint32_t step, long long* ids_out, long long ids_stride, cudaStream_t stream) {
  auto kern = sample_kernel<BF16, CS>;
  const size_t smem = (size_t)slice * (BF16 ? 2 : 4);
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_last_error("sample_tokens: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  e = launch_pdl(kPdlRows, kern, dim3((unsigned)(rows * CS)), dim3(kSampThreads), smem, stream, logits, ld, vocab,
                 slice, temperature, top_k, top_p, seed, step, ids_out, ids_stride);
  if (e != cudaSuccess) {
    set_last_error("sample_tokens: launch failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  return check_launch("sample_tokens", stream);
}

}  // namespace b200b

using namespace b200b;

extern "C" int b200b_sample_tokens_top_k(const void* logits, int dtype, int64_t ld, int64_t rows, int64_t vocab,
                                         float temperature, int64_t top_k, float top_p,
                                         const unsigned long long* seed, int64_t step, int64_t* ids_out,
                                         int64_t ids_stride, void* stream_) {
  if (!logits || !seed || !ids_out) {
    set_last_error("sample_tokens: null pointer");
    return B200B_ERR_ARG;
  }
  if (dtype != 0 && dtype != 1) {
    set_last_error("sample_tokens: dtype must be 0 (f32) or 1 (bf16)");
    return B200B_ERR_ARG;
  }
  if (rows < 1 || vocab < 1) {
    set_last_error("sample_tokens: rows and vocab must be >= 1");
    return B200B_ERR_SHAPE;
  }
  if (ld < vocab) {
    set_last_error("sample_tokens: ld < vocab");
    return B200B_ERR_ARG;
  }
  if (!(temperature > 0.0f) || !isfinite(temperature)) {
    set_last_error("sample_tokens: temperature must be finite and > 0");
    return B200B_ERR_ARG;
  }
  if (!(top_p > 0.0f && top_p <= 1.0f)) {
    set_last_error("sample_tokens: top_p must be in (0, 1]");
    return B200B_ERR_ARG;
  }
  if (top_k < 0) {
    set_last_error("sample_tokens: top_k must be >= 0");
    return B200B_ERR_ARG;
  }
  if (rows > 0x7fffffffLL / kSampMaxCluster) {
    set_last_error("sample_tokens: too many rows");
    return B200B_ERR_SHAPE;
  }
  const int esz = dtype == 1 ? 2 : 4;
  long long slice = 0;
  if (sample_cluster_size(rows, vocab, esz, 1, &slice) == 0) {
    set_last_error("sample_tokens: vocab %lld exceeds the limit of %lld tokens for this dtype", (long long)vocab,
                   (long long)(kSampMaxCluster * (kSampSliceBytes / esz)));
    return B200B_ERR_SHAPE;
  }
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc != B200B_OK) return rc;
  const int cs = sample_cluster_size(rows, vocab, esz, sms, &slice);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  long long* out = reinterpret_cast<long long*>(ids_out);
  const uint32_t t = (uint32_t)step;
  const uint32_t k = top_k < vocab ? (uint32_t)top_k : 0u;   // top_k >= vocab keeps every token, as top_k == 0
#define SAMPLE_CASE(BF, C)                                                                                         \
  if (cs == C)                                                                                                     \
    return sample_launch<BF, C>(logits, ld, rows, vocab, slice, temperature, k, top_p, seed, t, out, ids_stride, \
                                stream);
  if (dtype == 1) {
    SAMPLE_CASE(true, 1) SAMPLE_CASE(true, 2) SAMPLE_CASE(true, 4) SAMPLE_CASE(true, 8)
  } else {
    SAMPLE_CASE(false, 1) SAMPLE_CASE(false, 2) SAMPLE_CASE(false, 4) SAMPLE_CASE(false, 8)
  }
#undef SAMPLE_CASE
  set_last_error("sample_tokens: no kernel for cluster size %d", cs);
  return B200B_ERR_SHAPE;
}

extern "C" int b200b_sample_tokens(const void* logits, int dtype, int64_t ld, int64_t rows, int64_t vocab,
                                   float temperature, float top_p, const unsigned long long* seed, int64_t step,
                                   int64_t* ids_out, int64_t ids_stride, void* stream) {
  return b200b_sample_tokens_top_k(logits, dtype, ld, rows, vocab, temperature, 0, top_p, seed, step, ids_out,
                                   ids_stride, stream);
}
