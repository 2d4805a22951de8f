// Y = A_hat . B for a fixed sparse normalised adjacency held as CSR: the propagation of the defended GCN training
// (mcgpb_gcn.SparseAdjacency) on graphs whose n x n operand would not fit, forward and backward (A_hat is symmetric).
//
// A group of K lanes (a warp for K = 32, half a warp for K = 16) owns one row.  It is split into 4 sub-groups of K / 4
// lanes; sub-group s reads the row's entries s, s + 4, s + 8, ... and adds v * B[c, :] for each of them, every lane
// holding four columns of Y (one 16-byte load of B per entry and lane).  The four partial sums are then combined as
// (p0 + p1) + (p2 + p3) by two butterfly shuffles.  Every row is summed in this fixed order, without atomics, so a
// rerun is bit-identical.
#include "common.cuh"

namespace {

template <int K>
__global__ void __launch_bounds__(256)
k_spmm_csr(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ cols, const float* __restrict__ vals,
           int64_t n, const float* __restrict__ B, float* __restrict__ Y) {
  constexpr int L = K / 4;                 // lanes per row of B (4 columns each)
  const int lane = threadIdx.x & 31;
  const int sub = (lane % K) / L, c4 = lane % L;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / K;
  const bool live = i < n;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (live) {
    const int64_t e = rowptr[i + 1];
    for (int64_t p = rowptr[i] + sub; p < e; p += 4) {
      const float v = vals[p];
      const float4 b = __ldg(reinterpret_cast<const float4*>(B + (int64_t)cols[p] * K) + c4);
      acc.x = fmaf(v, b.x, acc.x);
      acc.y = fmaf(v, b.y, acc.y);
      acc.z = fmaf(v, b.z, acc.z);
      acc.w = fmaf(v, b.w, acc.w);
    }
  }
#pragma unroll
  for (int o = L; o < K; o <<= 1) {
    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
    acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o);
    acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
  }
  if (live && sub == 0) reinterpret_cast<float4*>(Y + i * K)[c4] = acc;
}

}  // namespace

extern "C" {

int mcgra_spmm_csr(const int64_t* rowptr, const int32_t* cols, const float* vals, int64_t n, const float* B, int K,
                   float* Y, void* stream) {
  if (n < 0 || (K != 16 && K != 32)) return -1;
  if ((reinterpret_cast<uintptr_t>(B) & 15) != 0 || (reinterpret_cast<uintptr_t>(Y) & 15) != 0) return -1;
  if (n == 0) return 0;
  const int64_t threads = n * K;
  const int64_t blocks = (threads + 255) / 256;
  if (blocks > 2147483647LL) return -3;
  if (K == 32)
    k_spmm_csr<32><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, cols, vals, n, B, Y);
  else
    k_spmm_csr<16><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, cols, vals, n, B, Y);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
