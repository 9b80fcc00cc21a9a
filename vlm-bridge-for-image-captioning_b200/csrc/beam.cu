// Beam search step over the vocabulary logits of batch * K beam rows (decode, SURVEY.md 8a row a12).
// Replaces, per step of generate(num_beams=K): log_softmax over [B*K, V], add the beam scores, topk(2K) over the
// K*V candidates of each image, and the Python bookkeeping of BeamHypotheses -- four passes over the logits and a
// handful of small launches and host loops.
//
// Two launches (the rule is stated in b200_bridge.h, b200b_beam_step):
//  * beam_topk_kernel: one row split over a cluster of CS CTAs (sample_cluster_size, the sampler's rule). Each
//    thread streams its share of the slice from HBM once, keeping the running max / sum of exp (rescaled once per
//    16 or 32 loaded values), the NaN / Inf flags and its 2K best (z desc, v asc) in registers. The lists are
//    merged per warp with shuffles, per CTA through shared memory, and per cluster by rank 0 through distributed
//    shared memory. A row whose flags show a NaN or an Inf is scanned a second time with the guard applied; other
//    rows pay nothing for it. Out: the row's 2K best z and v, and lse, in the workspace.
//  * beam_select_kernel: one CTA per image. Ranks the K * 2K candidates by (c desc, z desc, flat asc), walks the
//    first 2K (EOS offers, new beams), updates the finished set and the done flag, and copies the ids rows.
#include <float.h>
#include <math.h>

#include <cooperative_groups.h>

#include "common.cuh"
#include "launch.h"

namespace cg = cooperative_groups;

namespace b200b {

constexpr int kBeamThreads = 256;
constexpr int kBeamMaxK = 8;
constexpr int kBeamList = 2 * kBeamMaxK;             // per-thread list capacity (2K <= 16)
constexpr int kBeamWarps = kBeamThreads / 32;
constexpr int kSelThreads = kBeamMaxK * kBeamList;   // one select thread per candidate (K * 2K <= 128)
constexpr uint32_t kBeamEmpty = 0xFFFFFFFFu;         // list slot holding no token (value -inf)
constexpr float kBeamLog2e = 1.4426950408889634f;

// (z1, v1) comes before (z2, v2): larger z, ties to the smaller index; an empty slot (-inf, kBeamEmpty) comes
// after every token, and a NaN never comes before anything
__device__ __forceinline__ bool beam_before(float z1, uint32_t v1, float z2, uint32_t v2) {
  return z1 > z2 || (z1 == z2 && v1 < v2);
}

// insert (z, v) into the sorted list (lz, lv); the last entry falls off. Constant indices only: registers.
__device__ __forceinline__ void beam_insert(float (&lz)[kBeamList], uint32_t (&lv)[kBeamList], float z, uint32_t v) {
#pragma unroll
  for (int j = kBeamList - 1; j >= 0; --j) {
    const int p = j > 0 ? j - 1 : 0;
    const bool here = beam_before(z, v, lz[j], lv[j]);
    const bool above = j > 0 && beam_before(z, v, lz[p], lv[p]);
    if (here) {
      lz[j] = above ? lz[p] : z;
      lv[j] = above ? lv[p] : v;
    }
  }
}

// (z, v) into the list if it comes before its last entry
__device__ __forceinline__ void beam_take(float (&lz)[kBeamList], uint32_t (&lv)[kBeamList], float z, uint32_t v) {
  if (beam_before(z, v, lz[kBeamList - 1], lv[kBeamList - 1])) beam_insert(lz, lv, z, v);
}

// s * exp(m - M), 0 for an empty partial (m = -inf)
__device__ __forceinline__ float beam_rescale(float s, float m, float M) {
  return m == -INFINITY ? 0.0f : s * ex2_approx((m - M) * kBeamLog2e);
}

template <typename T>
__device__ __forceinline__ float beam_f(T v) {
  if constexpr (sizeof(T) == 2) return __bfloat162float(v);
  else return v;
}

// mode 0: the raw value; 1: a row with a NaN (all zeros); 2: a row with an Inf (clamped to [-100, 100])
__device__ __forceinline__ float beam_guard(float f, int mode) {
  return mode == 1 ? 0.0f : (mode == 2 ? fminf(fmaxf(f, -100.0f), 100.0f) : f);
}

struct BeamPartial {
  float z[kBeamList];
  uint32_t v[kBeamList];
  float m, s;
  uint32_t flags;   // 1: a NaN was seen, 2: an Inf was seen (raw values)
};

// One pass over this thread's share of the slice [lo, lo + n) (vocabulary indices): 2K best (z, v), running max m
// and sum s of exp(z - m), flags. The live list is the last n2k slots; the slots before it hold (+inf, 0), which
// no value displaces, so the bar is always the last slot and every register index is a constant (a runtime index
// into the list would move it to local memory).
template <typename T>
__device__ __forceinline__ void beam_scan(const T* __restrict__ src, int n, uint32_t lo, int mode, int n2k,
                                          float (&lz)[kBeamList], uint32_t (&lv)[kBeamList], float& m, float& s,
                                          uint32_t& flags) {
  constexpr int kVec = 16 / (int)sizeof(T);
  constexpr int kUnroll = 4;
  const int tid = threadIdx.x;
#pragma unroll
  for (int j = 0; j < kBeamList; ++j) {
    const bool dead = j < kBeamList - n2k;
    lz[j] = dead ? INFINITY : -INFINITY;
    lv[j] = dead ? 0u : kBeamEmpty;
  }
  m = -INFINITY;
  s = 0.0f;
  flags = 0;
  const int nv = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) ? n / kVec : 0;
  const uint4* src4 = reinterpret_cast<const uint4*>(src);
  for (int v0 = tid; v0 < nv; v0 += kUnroll * kBeamThreads) {
    uint4 q[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int v = v0 + u * kBeamThreads;
      if (v < nv) q[u] = mode == 0 ? __ldcs(src4 + v) : __ldg(src4 + v);
    }
    float cm = -INFINITY;
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      if (v0 + u * kBeamThreads < nv) {
        const T* e = reinterpret_cast<const T*>(&q[u]);
#pragma unroll
        for (int j = 0; j < kVec; ++j) {
          const float x = beam_f(e[j]);
          flags |= (x != x) ? 1u : 0u;
          flags |= (fabsf(x) == INFINITY) ? 2u : 0u;
          cm = fmaxf(cm, beam_guard(x, mode));
        }
      }
    }
    if (cm > m) {
      s = beam_rescale(s, m, cm);
      m = cm;
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int v = v0 + u * kBeamThreads;
      if (v < nv) {
        const T* e = reinterpret_cast<const T*>(&q[u]);
#pragma unroll
        for (int j = 0; j < kVec; ++j) {
          const float f = beam_guard(beam_f(e[j]), mode);
          s += ex2_approx((f - m) * kBeamLog2e);
          beam_take(lz, lv, f, lo + (uint32_t)(v * kVec + j));
        }
      }
    }
  }
  for (int i = nv * kVec + tid; i < n; i += kBeamThreads) {
    const float x = beam_f(src[i]);
    flags |= (x != x) ? 1u : 0u;
    flags |= (fabsf(x) == INFINITY) ? 2u : 0u;
    const float f = beam_guard(x, mode);
    if (f > m) {
      s = beam_rescale(s, m, f);
      m = f;
    }
    s += ex2_approx((f - m) * kBeamLog2e);
    beam_take(lz, lv, f, lo + (uint32_t)i);
  }
}

// warp-wide first of (z, v) (every lane gets it)
__device__ __forceinline__ void beam_warp_first(float& z, uint32_t& v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float z2 = __shfl_xor_sync(0xffffffffu, z, o);
    const uint32_t v2 = __shfl_xor_sync(0xffffffffu, v, o);
    if (beam_before(z2, v2, z, v)) {
      z = z2;
      v = v2;
    }
  }
}

// this CTA's partial (2K best, m, s, flags) from the threads' registers into `out`. Every thread's live list goes
// to shared memory first, so that the merge can walk it with a runtime index.
__device__ __forceinline__ void beam_cta_reduce(const float (&lz)[kBeamList], const uint32_t (&lv)[kBeamList], float m,
                                                float s, uint32_t flags, int n2k, float (*lists_z)[kBeamList],
                                                uint32_t (*lists_v)[kBeamList], BeamPartial* warp_parts,
                                                BeamPartial* out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
  for (int j = 0; j < kBeamList; ++j)
    if (j >= kBeamList - n2k) {
      lists_z[tid][j - (kBeamList - n2k)] = lz[j];
      lists_v[tid][j - (kBeamList - n2k)] = lv[j];
    }
  __syncwarp();
  // per warp: n2k rounds of "first head among the lanes; its owner moves on"
  int p = 0;
  for (int r = 0; r < n2k; ++r) {
    float z = p < n2k ? lists_z[tid][p] : -INFINITY;
    uint32_t v = p < n2k ? lists_v[tid][p] : kBeamEmpty;
    const uint32_t mv = v;
    beam_warp_first(z, v);
    if (lane == 0) {
      warp_parts[warp].z[r] = z;
      warp_parts[warp].v[r] = v;
    }
    if (v != kBeamEmpty && mv == v) ++p;   // indices are distinct across threads: one owner
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
    const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
    const float M = fmaxf(m, m2);
    s = beam_rescale(s, m, M) + beam_rescale(s2, m2, M);
    m = M;
  }
  flags = __reduce_or_sync(0xffffffffu, flags);
  if (lane == 0) {
    warp_parts[warp].m = m;
    warp_parts[warp].s = s;
    warp_parts[warp].flags = flags;
  }
  __syncthreads();
  if (warp == 0) {
    int q = 0;   // lane w < kBeamWarps walks warp w's list
    for (int r = 0; r < n2k; ++r) {
      float z = -INFINITY;
      uint32_t v = kBeamEmpty;
      if (lane < kBeamWarps && q < n2k) {
        z = warp_parts[lane].z[q];
        v = warp_parts[lane].v[q];
      }
      const uint32_t mv = v;
      beam_warp_first(z, v);
      if (lane == 0) {
        out->z[r] = z;
        out->v[r] = v;
      }
      if (v != kBeamEmpty && mv == v) ++q;
    }
    if (lane == 0) {
      float M = -INFINITY, S = 0.0f;
      uint32_t F = 0;
      for (int w = 0; w < kBeamWarps; ++w) {
        const float Mw = fmaxf(M, warp_parts[w].m);
        S = beam_rescale(S, M, Mw) + beam_rescale(warp_parts[w].s, warp_parts[w].m, Mw);
        M = Mw;
        F |= warp_parts[w].flags;
      }
      out->m = M;
      out->s = S;
      out->flags = F;
    }
  }
}

template <bool BF16, int CS>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(kBeamThreads)
    beam_topk_kernel(const void* __restrict__ logits, long long ld, long long vocab, long long slice, int n2k,
                     float* __restrict__ cand_z, uint32_t* __restrict__ cand_v, float* __restrict__ lse_out) {
  using T = typename std::conditional<BF16, __nv_bfloat16, float>::type;
  __shared__ float lists_z[kBeamThreads][kBeamList];
  __shared__ uint32_t lists_v[kBeamThreads][kBeamList];
  __shared__ BeamPartial warp_parts[kBeamWarps];
  __shared__ BeamPartial part;

  cg::cluster_group cluster = cg::this_cluster();
  const uint32_t rank = cluster.block_rank();
  const uint32_t row = blockIdx.x / CS;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long lo = (long long)rank * slice;
  const int n = (int)max(0LL, min(slice, vocab - lo));
  const T* src = reinterpret_cast<const T*>(logits) + (long long)row * ld + lo;

  pdl_prologue_late_trigger();
  float lz[kBeamList];
  uint32_t lv[kBeamList];
  float m, s;
  uint32_t flags;
  beam_scan<T>(src, n, (uint32_t)lo, 0, n2k, lz, lv, m, s, flags);
  beam_cta_reduce(lz, lv, m, s, flags, n2k, lists_z, lists_v, warp_parts, &part);
  cluster.sync();
  uint32_t gflags = 0;
  for (int r = 0; r < CS; ++r) gflags |= cluster.map_shared_rank(&part, r)->flags;
  if (gflags) {   // uniform over the cluster: the guarded pass (only rows with a NaN or an Inf)
    cluster.sync();   // every CTA has read the flags before `part` is rewritten
    beam_scan<T>(src, n, (uint32_t)lo, (gflags & 1u) ? 1 : 2, n2k, lz, lv, m, s, flags);
    beam_cta_reduce(lz, lv, m, s, flags, n2k, lists_z, lists_v, warp_parts, &part);
    cluster.sync();
  }
  if (rank == 0 && warp == 0) {
    // the cluster's lists, one per lane (lane r < CS reads rank r's shared memory)
    const BeamPartial* mine = cluster.map_shared_rank(&part, lane < CS ? lane : 0);
    int p = 0;
    for (int r = 0; r < n2k; ++r) {
      float z = -INFINITY;
      uint32_t v = kBeamEmpty;
      if (lane < CS && p < n2k) {
        z = mine->z[p];
        v = mine->v[p];
      }
      const uint32_t mv = v;
      beam_warp_first(z, v);
      if (lane == 0) {
        cand_z[(long long)row * n2k + r] = z;
        cand_v[(long long)row * n2k + r] = v;
      }
      if (v != kBeamEmpty && mv == v) ++p;   // the owner of the emitted entry
    }
    if (lane == 0) {
      float M = -INFINITY, S = 0.0f;
      for (int r = 0; r < CS; ++r) {
        const BeamPartial* q = cluster.map_shared_rank(&part, r);
        const float Mr = fmaxf(M, q->m);
        S = beam_rescale(S, M, Mr) + beam_rescale(q->s, q->m, Mr);
        M = Mr;
      }
      lse_out[row] = M + logf(S);
    }
  }
  cluster.sync();   // no CTA leaves while rank 0 still reads its shared memory
}

// candidate i before candidate j: c desc, z desc, flat index asc (flat indices are distinct)
__device__ __forceinline__ bool cand_before(float c1, float z1, long long f1, float c2, float z2, long long f2) {
  return c1 > c2 || (c1 == c2 && (z1 > z2 || (z1 == z2 && f1 < f2)));
}

// offer (score, len) to the finished set of one image held in shared memory; returns the slot or -1
__device__ __forceinline__ int hyp_offer(float score, int len, int K, float* hs, int* hl, int* hq, int& count) {
  const int filled = min(count, K);
  int slot = filled;
  if (filled == K) {
    int w = 0;
    for (int j = 1; j < K; ++j)
      if (hs[j] < hs[w] || (hs[j] == hs[w] && hq[j] < hq[w])) w = j;
    if (!(score > hs[w])) return -1;
    slot = w;
  }
  hs[slot] = score;
  hl[slot] = len;
  hq[slot] = count;
  count += 1;
  return slot;
}

__device__ __forceinline__ float length_norm(int n, float alpha) {
  return fminf(fmaxf(powf((float)n, alpha), FLT_MIN), FLT_MAX);
}

__global__ void __launch_bounds__(kSelThreads, 1)
    beam_select_kernel(const float* __restrict__ cand_z, const uint32_t* __restrict__ cand_v,
                       const float* __restrict__ lse, int K, int n2k, long long vocab, long long eos, float alpha,
                       int early_stopping, int t, const long long* __restrict__ ids, long long* __restrict__ ids_next,
                       long long ld_ids, long long* __restrict__ parents, b200b_beam_state st) {
  __shared__ float cc[kSelThreads], cz[kSelThreads];
  __shared__ long long cf[kSelThreads];
  __shared__ uint32_t cv[kSelThreads];
  __shared__ int order[kBeamList];
  __shared__ float hs[kBeamMaxK];
  __shared__ int hl[kBeamMaxK], hq[kBeamMaxK], pend[kBeamMaxK], par[kBeamMaxK];
  __shared__ long long tok[kBeamMaxK];
  __shared__ float news[kBeamMaxK];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int N = K * n2k;
  const long long row0 = (long long)b * K;

  pdl_prologue_late_trigger();
  const bool frozen = st.done[b] != 0;
  if (tid < N) {
    const int k = tid / n2k;
    const long long w = (row0 + k) * n2k + (tid - k * n2k);
    float z = cand_z[w];
    const uint32_t v = cand_v[w];
    float c;
    long long f;
    if (v == kBeamEmpty) {   // a row shorter than 2K: never before a token
      z = -INFINITY;
      c = -INFINITY;
      f = (long long)K * vocab + tid;
    } else {                 // s_k = -inf (a beam not yet live) gives c = -inf, never NaN: z - lse is finite
      c = __fadd_rn(st.beam_scores[row0 + k], __fsub_rn(z, lse[row0 + k]));
      if (c != c) c = -INFINITY;   // a NaN score left by a caller: rank it last, so the ranks stay a permutation
      f = (long long)k * vocab + v;
    }
    cc[tid] = c;
    cz[tid] = z;
    cf[tid] = f;
    cv[tid] = v;
  }
  __syncthreads();
  if (tid < N) {
    int rank = 0;
    for (int i = 0; i < N; ++i) rank += cand_before(cc[i], cz[i], cf[i], cc[tid], cz[tid], cf[tid]) ? 1 : 0;
    if (rank < n2k) order[rank] = tid;
  }
  __syncthreads();
  if (tid == 0) {
    const long long pad = eos >= 0 ? eos : 0;
    for (int k = 0; k < K; ++k) {
      pend[k] = -1;
      par[k] = k;
      tok[k] = pad;
    }
    if (!frozen) {
      int count = max(st.hyp_count[b], 0);
      for (int j = 0; j < K; ++j) {
        hs[j] = st.hyp_scores[row0 + j];
        hl[j] = st.hyp_lens[row0 + j];
        hq[j] = st.hyp_seq[row0 + j];
      }
      const float den = length_norm(t + 1, alpha);
      int nb = 0;
      for (int r = 0; r < n2k && nb < K; ++r) {
        const int ci = order[r];
        const int k = ci / n2k;   // the candidate's beam: in [0, K) since ci < N = K * n2k
        const long long v = cv[ci];
        if (v == eos) {
          if (r < K) {
            const int slot = hyp_offer(cc[ci] / den, t + 1, K, hs, hl, hq, count);
            if (slot >= 0) pend[slot] = k;
          }
          continue;
        }
        par[nb] = k;
        tok[nb] = v;
        news[nb] = cc[ci];
        ++nb;
      }
      // nb == K: the first 2K hold at most K EOS candidates (one per beam) and no empty slot (K * min(V, 2K)
      // >= 2K tokens for V >= 2)
      bool done = false;
      if (count >= K) {
        if (early_stopping) {
          done = true;
        } else {
          float worst = hs[0], best = -INFINITY;
          for (int j = 1; j < K; ++j) worst = fminf(worst, hs[j]);
          for (int k = 0; k < nb; ++k) best = fmaxf(best, news[k] / den);
          done = worst >= best;
        }
      }
      for (int k = 0; k < nb; ++k) st.beam_scores[row0 + k] = news[k];
      for (int j = 0; j < K; ++j) {
        st.hyp_scores[row0 + j] = hs[j];
        st.hyp_lens[row0 + j] = hl[j];
        st.hyp_seq[row0 + j] = hq[j];
      }
      st.hyp_count[b] = count;
      st.done[b] = done ? 1 : 0;
    }
  }
  __syncthreads();
  // ids rows of the new beams. par[k] is in [0, K) by construction (a candidate's beam index, or k itself for
  // a frozen image), so every row read below is row b*K + par[k] of this image.
  const int len = t + 1;
  for (int k = 0; k < K; ++k) {
    const long long* srow = ids + (row0 + par[k]) * ld_ids;
    long long* drow = ids_next + (row0 + k) * ld_ids;
    for (int j = tid; j < len; j += kSelThreads) drow[j] = srow[j];
    if (tid == 0) {
      drow[len] = tok[k];
      parents[row0 + k] = row0 + par[k];
    }
    // finished set, slot k: pend[k] is the parent (in [0, K)) of the slot's latest newcomer, -1 if none
    if (pend[k] >= 0) {
      const long long* hsrc = ids + (row0 + pend[k]) * ld_ids;
      long long* hdst = reinterpret_cast<long long*>(st.hyp_ids) + (row0 + k) * st.ld_hyp;
      for (int j = tid; j < len; j += kSelThreads) hdst[j] = hsrc[j];
      if (tid == 0) hdst[len] = eos;
    }
  }
}

// finished entry i of an image before entry j: score desc, then added first (seq asc)
__device__ __forceinline__ bool hyp_before(const float* hs, const int* hq, int i, int j) {
  return hs[i] > hs[j] || (hs[i] == hs[j] && hq[i] < hq[j]);
}

__global__ void __launch_bounds__(kSelThreads, 1)
    beam_finalize_kernel(int K, int N, long long eos, float alpha, int steps, const long long* __restrict__ ids,
                         long long ld_ids, b200b_beam_state st, long long* __restrict__ out_ids, long long ld_out,
                         long long* __restrict__ out_len, float* __restrict__ out_score) {
  __shared__ float hs[kBeamMaxK];
  __shared__ int hl[kBeamMaxK], hq[kBeamMaxK], src[kBeamMaxK];
  __shared__ int sel[kBeamMaxK];   // sel[r]: the slot of the r-th best hypothesis, in [0, K)
  const int b = blockIdx.x, tid = threadIdx.x;
  const long long row0 = (long long)b * K;

  pdl_prologue_late_trigger();
  if (tid == 0) {
    int count = max(st.hyp_count[b], 0);   // slots filled = min(count, K), never negative
    for (int j = 0; j < K; ++j) {
      hs[j] = st.hyp_scores[row0 + j];
      hl[j] = st.hyp_lens[row0 + j];
      hq[j] = st.hyp_seq[row0 + j];
      src[j] = j;   // finished hypothesis j
    }
    if (!st.done[b]) {
      const float den = length_norm(steps, alpha);
      for (int k = 0; k < K; ++k) {
        const int slot = hyp_offer(st.beam_scores[row0 + k] / den, steps + 1, K, hs, hl, hq, count);
        if (slot >= 0) src[slot] = K + k;   // running beam k
      }
    }
    // filled is K after the offers, and a done image holds K; clamped to [1, K] whatever the state holds. The N best
    // by selection (each pick is a slot not picked before, so sel is a list of distinct slots in [0, filled) for
    // N <= filled; a corrupt state with fewer filled slots repeats the last pick).
    const int filled = max(min(count, K), 1);
    unsigned used = 0;
    for (int r = 0; r < N; ++r) {
      int w = -1;
      for (int j = 0; j < filled; ++j)
        if (!(used >> j & 1u) && (w < 0 || hyp_before(hs, hq, j, w))) w = j;
      if (w < 0) w = sel[r - 1];   // r >= 1 here: filled >= 1 slots are free at r = 0
      used |= 1u << w;
      sel[r] = w;
      out_len[(long long)b * N + r] = hl[w];
      out_score[(long long)b * N + r] = hs[w];
    }
  }
  __syncthreads();
  const long long pad = eos >= 0 ? eos : 0;
  for (int r = 0; r < N; ++r) {
    // s < K: slot s of this image's finished set; else running beam s - K (in [0, K))
    const int s = src[sel[r]], len = hl[sel[r]];
    const long long* srow = s < K ? reinterpret_cast<const long long*>(st.hyp_ids) + (row0 + s) * st.ld_hyp
                                  : ids + (row0 + s - K) * ld_ids;
    long long* drow = out_ids + ((long long)b * N + r) * ld_out;
    for (int j = tid; j <= steps; j += kSelThreads) drow[j] = j < len ? srow[j] : pad;
  }
}

template <bool BF16, int CS>
static int beam_topk_launch(const void* logits, long long ld, long long rows, long long vocab, long long slice,
                            int n2k, float* cz, uint32_t* cv, float* lse, cudaStream_t stream) {
  cudaError_t e = launch_pdl(kPdlRows, beam_topk_kernel<BF16, CS>, dim3((unsigned)(rows * CS)), dim3(kBeamThreads), 0,
                             stream, logits, ld, vocab, slice, n2k, cz, cv, lse);
  if (e != cudaSuccess) {
    set_last_error("beam_step: top-k launch failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  return check_launch("beam_topk", stream);
}

struct BeamWs {
  float* cz;
  uint32_t* cv;
  float* lse;
  size_t bytes;
};

static BeamWs carve_beam_ws(long long rows, int n2k, void* base) {
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  BeamWs w;
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  w.cz = reinterpret_cast<float*>(p + off);
  off = up(off + (size_t)rows * n2k * sizeof(float));
  w.cv = reinterpret_cast<uint32_t*>(p + off);
  off = up(off + (size_t)rows * n2k * sizeof(uint32_t));
  w.lse = reinterpret_cast<float*>(p + off);
  off = up(off + (size_t)rows * sizeof(float));
  w.bytes = off;
  return w;
}

static bool state_ok(const b200b_beam_state* s) {
  return s && s->beam_scores && s->hyp_scores && s->hyp_lens && s->hyp_seq && s->hyp_count && s->done && s->hyp_ids;
}

}  // namespace b200b

using namespace b200b;

extern "C" size_t b200b_beam_step_workspace_bytes(int64_t batch, int num_beams) {
  if (batch < 1 || num_beams < 1 || num_beams > kBeamMaxK || batch > 0x7fffffffLL / kBeamMaxK) return 0;
  return carve_beam_ws(batch * num_beams, 2 * num_beams, nullptr).bytes;
}

extern "C" int b200b_beam_step(const void* logits, int dtype, int64_t ld, int64_t batch, int num_beams, int64_t vocab,
                               int64_t eos, float length_penalty, int early_stopping, int64_t step, const int64_t* ids,
                               int64_t* ids_next, int64_t ld_ids, int64_t* parents, const b200b_beam_state* state,
                               void* workspace, size_t workspace_bytes, void* stream_) {
  if (!logits || !ids || !ids_next || !parents || !workspace || !state_ok(state)) {
    set_last_error("beam_step: null pointer");
    return B200B_ERR_ARG;
  }
  if (ids == ids_next) {
    set_last_error("beam_step: ids and ids_next must be different buffers");
    return B200B_ERR_ARG;
  }
  if (dtype != 0 && dtype != 1) {
    set_last_error("beam_step: dtype must be 0 (f32) or 1 (bf16)");
    return B200B_ERR_ARG;
  }
  if (num_beams < 1 || num_beams > kBeamMaxK) {
    set_last_error("beam_step: num_beams must be in [1, %d]", kBeamMaxK);
    return B200B_ERR_ARG;
  }
  if (batch < 1) {
    set_last_error("beam_step: batch must be >= 1");
    return B200B_ERR_SHAPE;
  }
  if (vocab < 2) {
    set_last_error("beam_step: vocab must be >= 2");
    return B200B_ERR_SHAPE;
  }
  if (eos < -1 || eos >= vocab) {
    set_last_error("beam_step: eos must be -1 or in [0, vocab)");
    return B200B_ERR_ARG;
  }
  if (ld < vocab) {
    set_last_error("beam_step: ld < vocab");
    return B200B_ERR_ARG;
  }
  if (step < 0 || step > 0x7ffffffeLL - 2 || ld_ids < step + 2 || state->ld_hyp < step + 2) {
    set_last_error("beam_step: step must be >= 0 and ld_ids, ld_hyp >= step + 2");
    return B200B_ERR_ARG;
  }
  if (!isfinite(length_penalty)) {
    set_last_error("beam_step: length_penalty must be finite");
    return B200B_ERR_ARG;
  }
  if (early_stopping != 0 && early_stopping != 1) {
    set_last_error("beam_step: early_stopping must be 0 or 1");
    return B200B_ERR_ARG;
  }
  if (batch > 0x7fffffffLL / (kBeamMaxK * kBeamMaxK) || (long long)num_beams * vocab > 0x7fffffffLL) {
    set_last_error("beam_step: batch * K * 8 or K * vocab exceeds 2^31 - 1");
    return B200B_ERR_SHAPE;
  }
  const long long rows = batch * num_beams;
  const int n2k = 2 * num_beams;
  const int esz = dtype == 1 ? 2 : 4;
  long long slice = 0;
  if (sample_cluster_size(rows, vocab, esz, 1, &slice) == 0) {
    set_last_error("beam_step: vocab %lld exceeds the limit of %lld tokens for this dtype", (long long)vocab,
                   (long long)(8 * (176 * 1024 / esz)));
    return B200B_ERR_SHAPE;
  }
  const BeamWs ws = carve_beam_ws(rows, n2k, workspace);
  if (workspace_bytes < ws.bytes) {
    set_last_error("beam_step: workspace too small (%zu < %zu)", workspace_bytes, ws.bytes);
    return B200B_ERR_WORKSPACE;
  }
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc != B200B_OK) return rc;
  const int cs = sample_cluster_size(rows, vocab, esz, sms, &slice);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  rc = B200B_ERR_SHAPE;
#define BEAM_CASE(BF, C)                                                                                            \
  if (cs == C) rc = beam_topk_launch<BF, C>(logits, ld, rows, vocab, slice, n2k, ws.cz, ws.cv, ws.lse, stream);
  if (dtype == 1) {
    BEAM_CASE(true, 1) BEAM_CASE(true, 2) BEAM_CASE(true, 4) BEAM_CASE(true, 8)
  } else {
    BEAM_CASE(false, 1) BEAM_CASE(false, 2) BEAM_CASE(false, 4) BEAM_CASE(false, 8)
  }
#undef BEAM_CASE
  if (rc != B200B_OK) {
    if (rc == B200B_ERR_SHAPE) set_last_error("beam_step: no kernel for cluster size %d", cs);
    return rc;
  }
  cudaError_t e = launch_pdl(kPdlRows, beam_select_kernel, dim3((unsigned)batch), dim3(kSelThreads), 0, stream,
                             (const float*)ws.cz, (const uint32_t*)ws.cv, (const float*)ws.lse, num_beams, n2k,
                             (long long)vocab, (long long)eos, length_penalty, early_stopping, (int)step,
                             reinterpret_cast<const long long*>(ids), reinterpret_cast<long long*>(ids_next),
                             (long long)ld_ids, reinterpret_cast<long long*>(parents), *state);
  if (e != cudaSuccess) {
    set_last_error("beam_step: select launch failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  return check_launch("beam_select", stream);
}

extern "C" int b200b_beam_finalize_top(int64_t batch, int num_beams, int num_return, int64_t eos,
                                       float length_penalty, int64_t steps, const int64_t* ids, int64_t ld_ids,
                                       const b200b_beam_state* state, int64_t* out_ids, int64_t ld_out,
                                       int64_t* out_len, float* out_score, void* stream_) {
  if (!ids || !out_ids || !out_len || !out_score || !state_ok(state)) {
    set_last_error("beam_finalize: null pointer");
    return B200B_ERR_ARG;
  }
  if (num_beams < 1 || num_beams > kBeamMaxK) {
    set_last_error("beam_finalize: num_beams must be in [1, %d]", kBeamMaxK);
    return B200B_ERR_ARG;
  }
  if (num_return < 1 || num_return > num_beams) {
    set_last_error("beam_finalize: num_return must be in [1, num_beams]");
    return B200B_ERR_ARG;
  }
  if (batch < 1 || batch > 0x7fffffffLL / kBeamMaxK || steps < 1 || steps > 0x7ffffffeLL) {
    set_last_error("beam_finalize: batch and steps must be >= 1");
    return B200B_ERR_SHAPE;
  }
  if (eos < -1 || ld_ids < steps + 1 || state->ld_hyp < steps + 1 || ld_out < steps + 1) {
    set_last_error("beam_finalize: eos must be >= -1 and ld_ids, ld_hyp, ld_out >= steps + 1");
    return B200B_ERR_ARG;
  }
  if (!isfinite(length_penalty)) {
    set_last_error("beam_finalize: length_penalty must be finite");
    return B200B_ERR_ARG;
  }
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  cudaError_t e = launch_pdl(kPdlRows, beam_finalize_kernel, dim3((unsigned)batch), dim3(kSelThreads), 0, stream,
                             num_beams, num_return, (long long)eos, length_penalty, (int)steps,
                             reinterpret_cast<const long long*>(ids), (long long)ld_ids, *state,
                             reinterpret_cast<long long*>(out_ids), (long long)ld_out,
                             reinterpret_cast<long long*>(out_len), out_score);
  if (e != cudaSuccess) {
    set_last_error("beam_finalize: launch failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  return check_launch("beam_finalize", stream);
}

extern "C" int b200b_beam_finalize(int64_t batch, int num_beams, int64_t eos, float length_penalty, int64_t steps,
                                   const int64_t* ids, int64_t ld_ids, const b200b_beam_state* state,
                                   int64_t* out_ids, int64_t ld_out, int64_t* out_len, float* out_score,
                                   void* stream) {
  return b200b_beam_finalize_top(batch, num_beams, 1, eos, length_penalty, steps, ids, ld_ids, state, out_ids, ld_out,
                                 out_len, out_score, stream);
}
