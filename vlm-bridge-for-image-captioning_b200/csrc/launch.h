// Host-side helpers shared by the .cu translation units of libb200_bridge.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace b200b {

// records the message returned by b200b_last_error() (thread-local)
void set_last_error(const char* fmt, ...);
// cudaGetLastError() after a launch; bumps the process-wide launch counter on success. While a
// profile is open (b200b_profile_begin) it also records a CUDA event on `stream`, so that the time
// between consecutive events is attributed to the kernel named `what`.
int check_launch(const char* what, cudaStream_t stream);
// SM count of the current device (cached per device); fails on non-sm_100 devices
int device_sm_count(int* out);

// Tensor map of a bf16 row-major matrix [batch * rows, ld] read as per-head slices of `head_dim` columns:
// 4-D {head_dim, heads, rows, batch}, box {32 elements, 1, box_rows, 1}, 64-byte swizzle, out-of-range rows
// and columns read as zeros. A box lands in shared memory as [box_rows][64 B] (see common.cuh, "operand
// tiles of the training attention kernels"). Maps are cached by their arguments (the driver call costs
// about a microsecond and a step builds the same few dozen maps every time).
int make_tmap_heads_sw64(CUtensorMap* tm, const void* base, long long ld_elems, int head_dim, int heads, int rows,
                         int batch, int box_rows);

// How many CTAs (1, 2, 4 or 8; 0 if the row is too long) one vocabulary row of `vocab` elements of `esz` bytes is
// split over when `rows` rows run on `sms` SMs, and each CTA's slice (`*slice` tokens, a multiple of 8). Shared by
// the sampler (csrc/sampling.cu) and the beam step (csrc/beam.cu).
int sample_cluster_size(long long rows, long long vocab, int esz, int sms, long long* slice);

// Which kernel families are launched with programmatic stream serialization: bit mask from the
// environment variable B200B_PDL (1 = GEMMs, 2 = attention, 4 = row / column / cast kernels).
enum { kPdlGemm = 1, kPdlAttn = 2, kPdlRows = 4 };
int pdl_mask();

// Launch `kern` so that it may be scheduled while the previous kernel on `stream` is still running
// (programmatic dependent launch; also captured as a programmatic edge in CUDA graphs) when `family`
// is enabled. Only for kernels that call pdl_wait() / pdl_prologue() before their first
// global-memory access.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(int family, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg;
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (pdl_mask() & family) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// `stream` is the caller's dropout stream id: its B200B_SEED_INDIRECT bit says that `seed` is a device
// pointer to the 64-bit seed; the bit is cleared from `stream` here.
inline DropoutCfg make_dropout_cfg(float p, uint64_t seed, uint32_t* stream) {
  DropoutCfg d;
  d.seed_ptr = nullptr;
  if (stream != nullptr && (*stream & 0x80000000u)) {
    *stream &= 0x7fffffffu;
    d.seed_ptr = reinterpret_cast<const unsigned long long*>(static_cast<uintptr_t>(seed));
    seed = 0;
  }
  if (p > 0.0f) {
    uint32_t thr = (uint32_t)(p * 65536.0f + 0.5f);
    if (thr < 1) thr = 1;
    if (thr > 65535) thr = 65535;
    d.thr = thr;
    d.scale = 1.0f / (1.0f - p);
  } else {
    d.thr = 0;
    d.scale = 1.0f;
  }
  d.seed_lo = (uint32_t)seed;
  d.seed_hi = (uint32_t)(seed >> 32);
  return d;
}

}  // namespace b200b
