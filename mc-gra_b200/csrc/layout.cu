// Layout conversions between the reference's packed strict-lower-triangle vector / dense matrices and the
// tiled triangle the loop works on (see include/mcgra.h).  Replaces torch.tril_indices + index_put +
// m + m.t() + complementary*m (MC-GRA/topology_attack.py:365-379).
#include "common.cuh"

namespace {

__global__ void k_history_push(const double* __restrict__ row, double* __restrict__ hist, int64_t max_rows, int* step) {
  const int s = *step;
  if (s < max_rows && threadIdx.x < MCGRA_ACC_N) hist[(int64_t)s * MCGRA_ACC_N + threadIdx.x] = row[threadIdx.x];
  __syncwarp();
  if (threadIdx.x == 0) *step = s + 1;
}

// one CTA per tile, 256 threads, each thread handles float4 groups of a tile row
__global__ void k_tril_to_tiles(const float* __restrict__ packed, int64_t n, int64_t t0, float* __restrict__ tiles) {
  int I, J;
  const int64_t t = t0 + blockIdx.x;
  tile_coords(t, I, J);
  float* dst = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  for (int e = threadIdx.x; e < TILE_ELEMS; e += blockDim.x) {
    const int a = e >> 7, b = e & 127;
    const int64_t i = (int64_t)I * TILE + a, j = (int64_t)J * TILE + b;
    float v = 0.f;
    if (j < i && i < n) v = packed[i * (i - 1) / 2 + j];
    dst[e] = v;
  }
}

__global__ void k_tiles_to_tril(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
                                float* __restrict__ packed) {
  int I, J;
  const int64_t t = t0 + blockIdx.x;
  tile_coords(t, I, J);
  const ParamView pv = load_view(mu, raw);
  const float* src = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  for (int e = threadIdx.x; e < TILE_ELEMS; e += blockDim.x) {
    const int a = e >> 7, b = e & 127;
    const int64_t i = (int64_t)I * TILE + a, j = (int64_t)J * TILE + b;
    if (j < i && i < n) packed[i * (i - 1) / 2 + j] = pv.param(src[e]);
  }
}

__global__ void k_dense_to_tiles(const float* __restrict__ dense, int64_t ld, int64_t n, int64_t t0, int symmetrize,
                                 float* __restrict__ tiles, float* __restrict__ diag) {
  int I, J;
  const int64_t t = t0 + blockIdx.x;
  tile_coords(t, I, J);
  float* dst = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  for (int e = threadIdx.x; e < TILE_ELEMS; e += blockDim.x) {
    const int a = e >> 7, b = e & 127;
    const int64_t i = (int64_t)I * TILE + a, j = (int64_t)J * TILE + b;
    float v = 0.f;
    if (j < i && i < n) {
      v = dense[i * ld + j];
      if (symmetrize) v = 0.5f * (v + dense[j * ld + i]);
    }
    dst[e] = v;
    if (diag != nullptr && I == J && a == b && i < n) diag[i] = dense[i * ld + i];
  }
}

__global__ void k_tiles_to_dense(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
                                 float* __restrict__ dense, int64_t ld) {
  __shared__ float s[32][33];
  __shared__ unsigned char ok[32][33];
  int I, J;
  const int64_t t = t0 + blockIdx.x;
  tile_coords(t, I, J);
  const ParamView pv = load_view(mu, raw);
  const float* src = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  // direct part: rows of tile -> dense[i, j]; mirrored part through a 32x32 smem transpose
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 256 threads: 32 x 8
  for (int br = 0; br < TILE; br += 32) {
    for (int bc = 0; bc < TILE; bc += 32) {
      __syncthreads();
      for (int rr = ty; rr < 32; rr += 8) {
        const int a = br + rr, b = bc + tx;
        const int64_t i = (int64_t)I * TILE + a, j = (int64_t)J * TILE + b;
        float v = 0.f;
        const bool valid = (j < i && i < n);
        if (valid) {
          v = pv.param(src[a * TILE + b]);
          dense[i * ld + j] = v;
        }
        s[rr][tx] = v;
        ok[rr][tx] = valid ? 1 : 0;
      }
      __syncthreads();
      for (int rr = ty; rr < 32; rr += 8) {
        // element (a = br + tx, b = bc + rr) written to dense[j, i]
        const float v = s[tx][rr];
        const int a = br + tx, b = bc + rr;
        const int64_t i = (int64_t)I * TILE + a, j = (int64_t)J * TILE + b;
        if (ok[tx][rr]) dense[j * ld + i] = v;
      }
    }
  }
}

}  // namespace

extern "C" {

int mcgra_version(void) { return 2; }

int mcgra_history_push(const double* row, double* hist, int64_t max_rows, int* step, void* stream) {
  k_history_push<<<1, 32, 0, (cudaStream_t)stream>>>(row, hist, max_rows, step);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int64_t mcgra_tiles_in_rows(int tr0, int tr1) { return tri(tr1) - tri(tr0); }

int mcgra_tril_to_tiles(const float* packed, int64_t n, int tr0, int tr1, float* tiles, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_tril_to_tiles<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(packed, n, tri(tr0), tiles);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_tiles_to_tril(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, float* packed,
                        void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_tiles_to_tril<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, packed);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_dense_to_tiles(const float* dense, int64_t ld, int64_t n, int tr0, int tr1, int symmetrize, float* tiles,
                         float* diag, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_dense_to_tiles<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(dense, ld, n, tri(tr0), symmetrize, tiles, diag);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_tiles_to_dense(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, float* dense,
                         int64_t ld, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_tiles_to_dense<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, dense, ld);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
