// --measure KDE: utils.MutualInformation(sigma = 0.4, num_bins = B) (MC-GRA/utils.py:980-1053), called on n x n operands
// with B = n for c1 / c2 and on n x 16 / n x c operands for c9 / c10 (topology_attack.py:199-201, 212-229, 246-269).
//
//   kv[i, j] = exp(-0.5 ((v_ij - bin_j) / s)^2),  s = 2 * 0.4^2,  bin_j = j B / (B - 1)      (marginalPdf, :995-1004)
//   p1 = mean_i kv1 / (sum + 1e-10),  pj = kv1^T kv2 / (sum + 1e-10)                           (jointPdf, :1006-1014)
//   MI = H1 + H2 - H12,  result = 2 MI / (H1 + H2)                                             (:1035-1045)
//
// On n x n operands the reference forms an n x n x n "joint pdf" GEMM, but its operands hold values in [0, 1] while bin_j
// ~ j: exp(-0.5 ((v - j) / 0.32)^2) underflows to exactly 0 in fp32 for j >= 6, so only the first columns of the two
// matrices take part (KDE_NB = 8 are kept).  Everything is therefore a function of weighted second moments of n x 8
// (n x 16, n x c) kernel-value slabs: mcgra_cross_moments forward, mcgra_cross_moments_bwd backward, plus the small
// kernels below; gradients w.r.t. the first 8 columns of A_hat / M1 go back to the tiled pipeline as gradient tiles.
#include "common.cuh"

namespace {

constexpr int KDE_MAXD = 32;
constexpr float KDE_SIGMA = 0.32f;          // 2 * 0.4^2 (utils.py:986)
constexpr double KDE_EPS = 1e-10;

__global__ void k_kde_kv(const float* __restrict__ V, int64_t ldv, int d, int64_t m, float bin_step, float* __restrict__ kv) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= m * d) return;
  const int64_t i = e / d;
  const int j = (int)(e % d);
  const float z = (V[i * ldv + j] - (float)j * bin_step) / KDE_SIGMA;
  kv[e] = expf(-0.5f * z * z);
}
// gV = gkv * kv * (-(v - bin) / s^2)
__global__ void k_kde_chain(const float* __restrict__ V, int64_t ldv, const float* __restrict__ kv, const float* __restrict__ gkv,
                            int d, int64_t m, float bin_step, float* __restrict__ gV, int accumulate) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= m * d) return;
  const int64_t i = e / d;
  const int j = (int)(e % d);
  const float z = (V[i * ldv + j] - (float)j * bin_step);
  const float g = gkv[e] * kv[e] * (-z / (KDE_SIGMA * KDE_SIGMA));
  gV[e] = accumulate ? gV[e] + g : g;
}

// mom = [s1 (d) | s2 (d) | Sxy (d*d) | Syy (d*d)] with weights summing to 1 (s = mean of the kernel values, Sxy = mean of
// the outer products); m = number of samples (the reference's joint pdf is a SUM over samples).
__global__ void k_kde_scalars(const double* __restrict__ mom, int d, double m, double weight, double* __restrict__ acc_slot,
                              double* __restrict__ gmom) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double* s1 = mom;
  const double* s2 = mom + d;
  const double* Sxy = mom + 2 * d;
  const double LN2 = 0.6931471805599453;
  auto fprime = [&](double p) { return -log2(p + KDE_EPS) - p / ((p + KDE_EPS) * LN2); };
  double N1 = KDE_EPS, N2 = KDE_EPS, NJ = KDE_EPS;
  for (int a = 0; a < d; ++a) { N1 += s1[a]; N2 += s2[a]; }
  for (int e = 0; e < d * d; ++e) NJ += m * Sxy[e];
  double H1 = 0, H2 = 0, H12 = 0, t1 = 0, t2 = 0, tj = 0;
  for (int a = 0; a < d; ++a) {
    const double p = s1[a] / N1, q = s2[a] / N2;
    H1 -= p * log2(p + KDE_EPS);
    H2 -= q * log2(q + KDE_EPS);
    t1 += fprime(p) * p;
    t2 += fprime(q) * q;
  }
  for (int e = 0; e < d * d; ++e) {
    const double p = m * Sxy[e] / NJ;
    H12 -= p * log2(p + KDE_EPS);
    tj += fprime(p) * p;
  }
  const double MI = H1 + H2 - H12, Hs = H1 + H2;
  const double value = 2.0 * MI / Hs;
  const double cH = 2.0 * H12 / (Hs * Hs), cJ = -2.0 / Hs;      // d value / dH1 = d value / dH2, d value / dH12
  for (int a = 0; a < d; ++a) {
    gmom[a] = weight * cH * (fprime(s1[a] / N1) - t1) / N1;
    gmom[d + a] = weight * cH * (fprime(s2[a] / N2) - t2) / N2;
  }
  for (int e = 0; e < d * d; ++e) {
    gmom[2 * d + e] = weight * cJ * m * (fprime(m * Sxy[e] / NJ) - tj) / NJ;
    gmom[2 * d + d * d + e] = 0.0;
  }
  *acc_slot += weight * value;
}

// first NB columns of A_hat from the tiled triangle (tile column 0): slab[i][j] += r_i M_ij r_j (+ r_i^2 on the diagonal).
// NOISY: M is the noisy estimate -- `tiles` is its L plane (values as stored, raw = 2), the mirrored entry A_hat_ji comes
// from the U plane (M_ji at (i, j)) and the diagonal is r_i^2 (1 + mdiag[i]) (mcgra_noise_stage)
template <bool NOISY>
__global__ void k_slab_ahat(const float* __restrict__ tiles, const float* __restrict__ Ut, const float* __restrict__ mdiag,
                            int64_t n, int tr0, const float* mu, int raw, const float* __restrict__ r, int NB,
                            float* __restrict__ slab) {
  const ParamView pv = load_view(mu, raw);
  const int I = tr0 + blockIdx.x;
  const int64_t toff = (tri((int64_t)I) - tri((int64_t)tr0)) * TILE_ELEMS;          // tile (I, 0)
  const float* t = tiles + toff;
  for (int e = threadIdx.x; e < TILE * NB; e += blockDim.x) {
    const int a = e / NB, b = e % NB;
    const int64_t i = (int64_t)I * TILE + a, j = b;
    if (i >= n || j >= n) continue;
    if (j < i) {
      const float v = r[i] * pv.adj(t[a * TILE + b]) * r[j];
      slab[i * NB + j] += v;
      if (i < NB)                                                 // mirrored entry (j, i), both < NB: tile (0, 0) only
        slab[j * NB + i] += NOISY ? (r[j] * Ut[toff + a * TILE + b]) * r[i] : v;
    } else if (i == j) {
      slab[i * NB + j] += NOISY ? (r[i] * (1.f + mdiag[i])) * r[i] : r[i] * r[i];
    }
  }
}
__global__ void k_slab_m1(const float* __restrict__ zhat, int64_t n, int NB, float* __restrict__ slab) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * NB) return;
  const int64_t i = e / NB;
  const int j = (int)(e % NB);
  float d = 0.f;
  if (j < n && i != j) {
#pragma unroll
    for (int k = 0; k < HID; ++k) d = fmaf(zhat[i * HID + k], zhat[(int64_t)j * HID + k], d);
    d = fmaxf(d, 0.f);
  }
  slab[e] = d;
}
// gradient slab G [n x NB] (dL/dX_ij for j < NB) -> tiles (I, 0) of G_ij + G_ji, diag[i] = G_ii (i < NB, else 0)
__global__ void k_slab_to_tiles(const float* __restrict__ G, int64_t n, int tr0, int NB, float* __restrict__ tiles,
                                float* __restrict__ diag) {
  const int I = tr0 + blockIdx.x;
  float* t = tiles + (tri((int64_t)I) - tri((int64_t)tr0)) * TILE_ELEMS;
  for (int e = threadIdx.x; e < TILE_ELEMS; e += blockDim.x) {
    const int a = e >> 7, b = e & 127;
    const int64_t i = (int64_t)I * TILE + a, j = b;
    float v = 0.f;
    if (j < i && i < n) {
      if (b < NB) v += G[i * NB + b];
      if (i < NB) v += G[j * NB + i];
    }
    t[e] = v;
  }
  if (diag != nullptr)
    for (int64_t i = (int64_t)I * TILE + threadIdx.x; i < min(n, (int64_t)(I + 1) * TILE); i += blockDim.x)
      diag[i] = i < NB ? G[i * NB + i] : 0.f;
}
// demd += (softmax backward of gp through p) Wl      (c10: gradient w.r.t. softmax(output2) back to the embedding)
__global__ void k_softmax_chain(const float* __restrict__ gp, const float* __restrict__ p, const float* __restrict__ Wl, int64_t n,
                                int c, float* __restrict__ demd) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float dot = 0.f;
  for (int l = 0; l < c; ++l) dot = fmaf(gp[i * c + l], p[i * c + l], dot);
  float g[HID];
#pragma unroll
  for (int k = 0; k < HID; ++k) g[k] = 0.f;
  for (int l = 0; l < c; ++l) {
    const float dz = p[i * c + l] * (gp[i * c + l] - dot);
#pragma unroll
    for (int k = 0; k < HID; ++k) g[k] = fmaf(dz, Wl[l * HID + k], g[k]);
  }
#pragma unroll
  for (int k = 0; k < HID; ++k) demd[i * HID + k] += g[k];
}
__global__ void k_softmax_rows(const float* __restrict__ em, const float* __restrict__ Wl, const float* __restrict__ bl, int64_t n,
                               int c, float* __restrict__ p2) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float z[KDE_MAXD];
  float mx = -INFINITY;
  for (int q = 0; q < c; ++q) {
    float s = bl[q];
#pragma unroll
    for (int k = 0; k < HID; ++k) s = fmaf(em[i * HID + k], Wl[q * HID + k], s);
    z[q] = s;
    mx = fmaxf(mx, s);
  }
  float den = 0.f;
  for (int q = 0; q < c; ++q) { z[q] = expf(z[q] - mx); den += z[q]; }
  for (int q = 0; q < c; ++q) p2[i * c + q] = z[q] / den;
}

// fp64 variant for two n x NB value slabs with the same bins (c1 / c2 on the noisy path): the kernel values are
// recomputed in fp64 and the moments accumulated from fp64 products.  MI is there a difference of entropies ~1e6 times
// larger than itself, and fp32 kernel values or fp32 products would already move it by ~1e-4 relative.
constexpr double KDE_S64 = 2.0 * 0.4 * 0.4;              // utils.py:986, as the fp64 reference evaluates it
constexpr int KR64 = 64;                                  // rows per CTA of k_kde_moments64
__device__ __forceinline__ double kde_kv64(float v, int j, double bin) {
  const double z = ((double)v - (double)j * bin) / KDE_S64;
  return exp(-0.5 * z * z);
}
// mom [s1 (d) | s2 (d) | Sxy (d*d)] += wt * sums over the rows (caller zero-fills; the Syy block is left untouched)
__global__ void __launch_bounds__(256)
k_kde_moments64(const float* __restrict__ X, const float* __restrict__ Y, int d, int64_t m, double bin, double wt,
                double* __restrict__ mom) {
  __shared__ double kx[KR64 * KDE_MAXD], ky[KR64 * KDE_MAXD];
  const int64_t i0 = (int64_t)blockIdx.x * KR64;
  for (int e = threadIdx.x; e < KR64 * d; e += blockDim.x) {
    const int64_t i = i0 + e / d;
    const int j = e % d;
    kx[e] = i < m ? kde_kv64(X[i * d + j], j, bin) : 0.0;
    ky[e] = i < m ? kde_kv64(Y[i * d + j], j, bin) : 0.0;
  }
  __syncthreads();
  for (int q = threadIdx.x; q < 2 * d + d * d; q += blockDim.x) {
    double s = 0.0;
    if (q < d) {
      for (int r = 0; r < KR64; ++r) s += kx[r * d + q];
    } else if (q < 2 * d) {
      for (int r = 0; r < KR64; ++r) s += ky[r * d + q - d];
    } else {
      const int a = (q - 2 * d) / d, b = (q - 2 * d) % d;
      for (int r = 0; r < KR64; ++r) s += kx[r * d + a] * ky[r * d + b];
    }
    if (s != 0.0) atomicAdd(mom + q, wt * s);
  }
}
// backward through the moments and the kernel to the values: with g = d loss / d mom (mcgra_kde_scalars)
//   gX[i][a] += wt (g_s1[a] + sum_b g_Sxy[a][b] kvy_b) kvx_a (-(x - bin_a) / s^2),  gY likewise with g_s2, g_Sxy^T
__global__ void k_kde_chain64(const float* __restrict__ X, const float* __restrict__ Y, int d, int64_t m, double bin,
                              double wt, const double* __restrict__ g, float* __restrict__ gX, float* __restrict__ gY) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= m * d) return;
  const int64_t i = e / d;
  const int a = (int)(e % d);
  const double* gJ = g + 2 * d;
  double sx = g[a], sy = g[d + a];
  for (int b = 0; b < d; ++b) {
    sx += gJ[a * d + b] * kde_kv64(Y[i * d + b], b, bin);
    sy += gJ[b * d + a] * kde_kv64(X[i * d + b], b, bin);
  }
  const double c = -wt / (KDE_S64 * KDE_S64);
  if (gX != nullptr) {
    const double zx = (double)X[e] - (double)a * bin;
    gX[e] = (float)((double)gX[e] + sx * kde_kv64(X[e], a, bin) * zx * c);
  }
  if (gY != nullptr) {
    const double zy = (double)Y[e] - (double)a * bin;
    gY[e] = (float)((double)gY[e] + sy * kde_kv64(Y[e], a, bin) * zy * c);
  }
}

}  // namespace

extern "C" {

int mcgra_kde_kv(const float* V, int64_t ldv, int d, int64_t m, float bin_step, float* kv, void* stream) {
  if (d < 1 || d > KDE_MAXD) return -1;
  if (m <= 0) return 0;
  k_kde_kv<<<(unsigned)((m * d + 255) / 256), 256, 0, (cudaStream_t)stream>>>(V, ldv, d, m, bin_step, kv);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_kde_chain(const float* V, int64_t ldv, const float* kv, const float* gkv, int d, int64_t m, float bin_step,
                    float* gV, int accumulate, void* stream) {
  if (d < 1 || d > KDE_MAXD) return -1;
  if (m <= 0) return 0;
  k_kde_chain<<<(unsigned)((m * d + 255) / 256), 256, 0, (cudaStream_t)stream>>>(V, ldv, kv, gkv, d, m, bin_step, gV, accumulate);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_kde_scalars(const double* mom, int d, double m, double weight, double* acc_slot, double* gmom, void* stream) {
  if (d < 1 || d > KDE_MAXD) return -1;
  k_kde_scalars<<<1, 32, 0, (cudaStream_t)stream>>>(mom, d, m, weight, acc_slot, gmom);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_slab_ahat(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* r, int NB,
                    float* slab, void* stream) {
  if (NB < 1 || NB > KDE_MAXD) return -1;
  if (tr1 > tr0)
    k_slab_ahat<false><<<(unsigned)(tr1 - tr0), 256, 0, (cudaStream_t)stream>>>(tiles, nullptr, nullptr, n, tr0, mu, raw,
                                                                              r, NB, slab);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_slab_ahat_noisy(const float* Lt, const float* Ut, const float* mdiag, int64_t n, int tr0, int tr1,
                          const float* r, int NB, float* slab, void* stream) {
  if (NB < 1 || NB > KDE_MAXD || Lt == nullptr || Ut == nullptr || mdiag == nullptr) return -1;
  if (tr1 > tr0)
    k_slab_ahat<true><<<(unsigned)(tr1 - tr0), 256, 0, (cudaStream_t)stream>>>(Lt, Ut, mdiag, n, tr0, nullptr, 2, r, NB,
                                                                             slab);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_kde_moments64(const float* X, const float* Y, int d, int64_t m, double bin_step, double wt, double* mom,
                        void* stream) {
  if (d < 1 || d > KDE_MAXD) return -1;
  if (m <= 0) return 0;
  k_kde_moments64<<<(unsigned)((m + KR64 - 1) / KR64), 256, 0, (cudaStream_t)stream>>>(X, Y, d, m, bin_step, wt, mom);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_kde_chain64(const float* X, const float* Y, int d, int64_t m, double bin_step, double wt, const double* gmom,
                      float* gX, float* gY, void* stream) {
  if (d < 1 || d > KDE_MAXD) return -1;
  if (m <= 0) return 0;
  k_kde_chain64<<<(unsigned)((m * d + 255) / 256), 256, 0, (cudaStream_t)stream>>>(X, Y, d, m, bin_step, wt, gmom, gX,
                                                                                 gY);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_slab_m1(const float* zhat, int64_t n, int NB, float* slab, void* stream) {
  if (NB < 1 || NB > KDE_MAXD) return -1;
  k_slab_m1<<<(unsigned)((n * NB + 255) / 256), 256, 0, (cudaStream_t)stream>>>(zhat, n, NB, slab);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_slab_to_tiles(const float* G, int64_t n, int tr0, int tr1, int NB, float* tiles, float* diag, void* stream) {
  if (NB < 1 || NB > KDE_MAXD) return -1;
  if (tr1 > tr0) k_slab_to_tiles<<<(unsigned)(tr1 - tr0), 256, 0, (cudaStream_t)stream>>>(G, n, tr0, NB, tiles, diag);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_softmax_rows(const float* em, const float* Wl, const float* bl, int64_t n, int c, float* p2, void* stream) {
  if (c < 1 || c > KDE_MAXD) return -1;
  k_softmax_rows<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(em, Wl, bl, n, c, p2);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_softmax_chain(const float* gp, const float* p, const float* Wl, int64_t n, int c, float* demd, void* stream) {
  if (c < 1 || c > KDE_MAXD) return -1;
  k_softmax_chain<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(gp, p, Wl, n, c, demd);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
