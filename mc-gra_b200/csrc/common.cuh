// Shared device helpers for libmcgra_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/mcgra.h"

#define TILE MCGRA_TILE
#define TILE_ELEMS (TILE * TILE)
#define HID MCGRA_HID

#define MCGRA_LAUNCH_CHECK()                         \
  do {                                               \
    cudaError_t e__ = cudaGetLastError();            \
    if (e__ != cudaSuccess) return (int)e__;         \
  } while (0)

__host__ __device__ __forceinline__ int64_t tri(int64_t I) { return I * (I + 1) / 2; }

// linear (global) tile index -> (I, J), J <= I
__device__ __forceinline__ void tile_coords(int64_t t, int& I, int& J) {
  int i = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (tri((int64_t)i + 1) <= t) ++i;
  while (tri((int64_t)i) > t) --i;
  I = i;
  J = (int)(t - tri((int64_t)i));
}

// b-th CTA of a shard of tile rows [tr0, tr1) -> tile (I, J) in an L2-friendly order: blocks of R tile rows are swept
// column by column, so the per-column operand block is re-used by R consecutive CTAs and the R per-row blocks stay
// resident for the whole sweep.  tix = storage index of the tile inside the shard (row-major triangle order).
__device__ __forceinline__ void tile_coords_blocked(int64_t b, int tr0, int tr1, int R, int& I, int& J, int64_t& tix) {
  int Ib, Jb;
  tile_coords(tri((int64_t)tr0) + b, Ib, Jb);
  const int I0 = tr0 + ((Ib - tr0) / R) * R;
  const int I1 = min(I0 + R, tr1);
  const int rows = I1 - I0;
  int64_t rb = b - (tri((int64_t)I0) - tri((int64_t)tr0));
  const int64_t full = (int64_t)(I0 + 1) * rows;        // columns 0..I0 hold all `rows` tiles
  if (rb < full) {
    J = (int)(rb / rows);
    I = I0 + (int)(rb % rows);
  } else {
    rb -= full;
    J = I0 + 1;
    while (rb >= I1 - J) { rb -= I1 - J; ++J; }         // triangular tail: column J holds rows J..I1-1
    I = J + (int)rb;
  }
  tix = tri((int64_t)I) + J - tri((int64_t)tr0);
}

// parameter view: value of the optimised parameter stored lazily as x' and mu (see mcgra.h)
// raw = 0: lazy projection (buffer = un-projected Adam output x', parameter = clamp(x' - mu, 0, 1))
// raw = 1: user-provided raw parameter (forward uses clamp(x, 0, 1) with the clamp's gradient mask)
// raw = 2: buffer already holds the parameter in [0, 1] (budget cannot bind: the fold kernel stored the clamped value)
struct ParamView {
  float mu;
  int raw;
  __device__ __forceinline__ float param(float xs) const {   // the parameter the optimiser holds
    return raw ? xs : fminf(fmaxf(xs - mu, 0.f), 1.f);
  }
  __device__ __forceinline__ float adj(float xs) const {     // entry of M = clamp(param, 0, 1)
    return raw == 2 ? xs : fminf(fmaxf(raw ? xs : xs - mu, 0.f), 1.f);
  }
  __device__ __forceinline__ float mask(float xs) const {    // d clamp / d param (closed interval)
    return (raw != 1 || (xs >= 0.f && xs <= 1.f)) ? 1.f : 0.f;
  }
};
__device__ __forceinline__ ParamView load_view(const float* mu, int raw) {
  ParamView v;
  v.mu = (mu != nullptr && !raw) ? *mu : 0.f;
  v.raw = raw;
  return v;
}

// order-preserving map float -> uint32 (ascending); shared by the AUC ranking and the top-k selection
__device__ __forceinline__ uint32_t fkey(float f) {
  uint32_t u = __float_as_uint(f + 0.0f);          // -0.0 -> +0.0: they compare equal, so they must share a key
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide double sum -> one atomicAdd per block.  `red` is shared scratch of >= 32 doubles.
__device__ __forceinline__ void block_atomic_add_d(double v, double* dst, double* red) {
  v = warp_sum_d(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  if (w == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    double s = lane < nw ? red[lane] : 0.0;
    s = warp_sum_d(s);
    if (lane == 0 && s != 0.0) atomicAdd(dst, s);
  }
}

__device__ __forceinline__ void atomic_min_f(float* addr, float v) {   // works for any sign
  if (v >= 0.f) atomicMin((int*)addr, __float_as_int(v));
  else atomicMax((unsigned int*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f(float* addr, float v) {
  if (v >= 0.f) atomicMax((int*)addr, __float_as_int(v));
  else atomicMin((unsigned int*)addr, __float_as_uint(v));
}

// entropy integrand of Info_entropy (topology_attack.py:44-47): q*log2(q), q = clamp(p,1e-4,1-1e-4),
// and its derivative w.r.t. p (zero outside the closed clamp interval).
#define ENT_LO 1e-4f
#define ENT_HI (1.f - 1e-4f)
#define INV_LN2 1.4426950408889634f
__device__ __forceinline__ float ent_val(float p) {
  float q = fminf(fmaxf(p, ENT_LO), ENT_HI);
  return q * log2f(q);
}
__device__ __forceinline__ float ent_grad(float p) {
  float q = fminf(fmaxf(p, ENT_LO), ENT_HI);
  return (p >= ENT_LO && p <= ENT_HI) ? (log2f(q) + INV_LN2) : 0.f;
}
