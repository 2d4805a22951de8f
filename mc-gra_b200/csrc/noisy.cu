// attack() with adjacency noise (--eps != 0): the reference adds a fresh, un-symmetrised Gaussian draw to the expanded
// estimate every iteration and clamps it (MC-GRA/topology_attack.py:165, 474-478):
//     M_ij = clamp(p_ij + N_ij * eps, 0, 1)  (i != j),    M_ii = clamp(N_ii * eps, 0, 1)
// so M is a general dense matrix: the two orientations of a stored entry differ, each has its own clamp mask, and the
// diagonal is not zero.  Everything else of the tiled pipeline stays: the two orientations are kept as tile planes Lt / Ut
// in the working layout and fed to the existing propagation kernels one product set at a time (mcgra_propagate_sel); the
// node kernels see M*B and M^T*B exactly where the symmetric path sees M*B, so only the degree gradient's diagonal changes
// (mcgra_node_rho_diag).  This file holds the stages whose algebra differs from the symmetric path:
//   k_noise_stage   x view + N -> Lt, Ut, degree row sums          (one CTA per stored tile)
//   k_noise_diag    M_ii and d_i = 1 + M_ii (ADD: d_i += 1 + M_ii)  (around k_noise_stage's row sums, see below)
//   k_noisy_terms   c1 / c2 (MSELoss) and c6 over both orientations, degree-gradient row + column parts, dzhat of c2
//   k_noisy_grad    dL/dx_ij = mask_ij dL/dM_ij + mask_ji dL/dM_ji into gradient tiles for mcgra_fold_adam (Gtiles)
// Both also take an upstream gradient of the first nb columns of A_hat (gslab, --measure KDE): it only reaches tiles of
// tile column 0, where it is added to e'_ij (column j < nb) and to e'_ji (row i < nb, i.e. tile (0, 0)).
// All are exact fp32 (FFMA) one-tile-per-CTA kernels.  The sums p + N*eps are formed as the reference forms them -- one
// rounded product, one rounded sum (no FMA) -- so the clamp masks agree with torch's on the same draw.
#include "common.cuh"

namespace {

constexpr int NT_LD = TILE + 1;        // padded row of a transposed noise block: column reads are conflict free

__device__ __forceinline__ float clamp01(float v) { return fminf(fmaxf(v, 0.f), 1.f); }
__device__ __forceinline__ float noisy_sum(float p, float nz, float eps) { return __fadd_rn(p, __fmul_rn(nz, eps)); }
__device__ __forceinline__ float box_mask(float v) { return (v >= 0.f && v <= 1.f) ? 1.f : 0.f; }   // torch.clamp's grad

// nt[b][a] = N[j0 + b][i0 + a]: the (J, I) block of the draw, i.e. N_ji of tile entry (a, b)
__device__ __forceinline__ void stage_noise_t(float* nt, const float* __restrict__ noise, int64_t n, int64_t i0, int64_t j0) {
  for (int e = threadIdx.x; e < TILE * TILE; e += blockDim.x) {
    const int b = e >> 7, a = e & (TILE - 1);
    const int64_t gj = j0 + b, gi = i0 + a;
    nt[b * NT_LD + a] = (gj < n && gi < n) ? noise[gj * n + gi] : 0.f;
  }
}

// ADD = false: d = 1 + M_ii before k_noise_stage adds one GPU's row sums; ADD = true: d += 1 + M_ii after the row sums of
// every shard were all-reduced (the diagonal is then counted once, not once per rank)
template <bool ADD>
__global__ void k_noise_diag(int64_t n, const float* __restrict__ noise, float eps, float* __restrict__ mdiag,
                             float* __restrict__ d) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float m = clamp01(__fmul_rn(noise[i * n + i], eps));     // 0 + N_ii * eps
  mdiag[i] = m;
  d[i] = ADD ? d[i] + (1.f + m) : 1.f + m;
}

__global__ void __launch_bounds__(256)
k_noise_stage(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
              const float* __restrict__ noise, float eps, float* __restrict__ Lt, float* __restrict__ Ut,
              float* __restrict__ d) {
  extern __shared__ float nt[];                        // [TILE][NT_LD]
  __shared__ float colacc[TILE];
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const int64_t base = (int64_t)blockIdx.x * TILE_ELEMS;
  if (tid < TILE) colacc[tid] = 0.f;
  stage_noise_t(nt, noise, n, i0, j0);
  __syncthreads();
  float col[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
  for (int a = warp; a < TILE; a += 8) {
    const int64_t gi = i0 + a;
    float rs = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int b = lane + 32 * k;
      const int64_t gj = j0 + b;
      const bool valid = (gj < gi) && (gi < n);
      float L = 0.f, U = 0.f;
      if (valid) {
        const float p = pv.param(tiles[base + a * TILE + b]);
        L = clamp01(noisy_sum(p, noise[gi * n + gj], eps));
        U = clamp01(noisy_sum(p, nt[b * NT_LD + a], eps));
      }
      Lt[base + a * TILE + b] = L;
      Ut[base + a * TILE + b] = U;
      rs += L;                                         // row i holds M_ij
      col[k] += U;                                     // row j holds M_ji
    }
    rs = warp_sum(rs);
    if (lane == 0 && gi < n && rs != 0.f) atomicAdd(d + gi, rs);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) atomicAdd(&colacc[lane + 32 * k], col[k]);
  __syncthreads();
  if (tid < TILE && j0 + tid < n && colacc[tid] != 0.f) atomicAdd(d + j0 + tid, colacc[tid]);
}

__global__ void k_diag_axpy(const float* __restrict__ mdiag, const float* __restrict__ B, int K, int64_t n,
                            float* __restrict__ Y) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * K) return;
  Y[e] += mdiag[e / K] * B[e];
}

// element-wise derivatives e'_ij, e'_ji of c1 / c2 / c6 at A_hat_ij = r_i M_ij r_j and A_hat_ji = r_j M_ji r_i (values
// added to v1, v2, v6 when `vals`); s = zhat_i . zhat_j (c2 only)
struct ElemOut {
  float eij, eji;
};
template <bool VALS>
__device__ __forceinline__ ElemOut elem_terms(const mcgra_noisy_args& a, float aij, float aji, float fij, float fji, float s,
                                              float& v1, float& v2, float& v6) {
  ElemOut o{0.f, 0.f};
  if (a.k1 != 0.f) {
    const float d1 = aij - fij, d2 = aji - fji;
    if (VALS) v1 += d1 * d1 + d2 * d2;
    o.eij += 2.f * a.k1 * d1;
    o.eji += 2.f * a.k1 * d2;
  }
  if (a.k6 != 0.f) {
    if (VALS) v6 += ent_val(aij) + ent_val(aji);
    o.eij += a.k6 * ent_grad(aij);
    o.eji += a.k6 * ent_grad(aji);
  }
  if (a.k2 != 0.f) {
    const float m1 = fmaxf(s, 0.f);
    const float d1 = aij - m1, d2 = aji - m1;
    if (VALS) v2 += d1 * d1 + d2 * d2;
    o.eij += 2.f * a.k2 * d1;
    o.eji += 2.f * a.k2 * d2;
  }
  return o;
}

// upstream dL/dA_hat of the first nb columns (slab [n x nb]) at the stored entry (i, j), i > j, of a tile of column 0:
// A_hat_ij is slab entry (i, j) when j < nb, A_hat_ji is slab entry (j, i) when i < nb
__device__ __forceinline__ void add_slab_grad(const mcgra_noisy_args& a, int64_t gi, int64_t gj, ElemOut& e) {
  if (gj < a.nb) e.eij += a.gslab[gi * a.nb + gj];
  if (gi < a.nb) e.eji += a.gslab[gj * a.nb + gi];
}

struct TermsSmem {
  float c[TILE][NT_LD];                  // dL/dS_ij of c2 (S = zhat zhat^T)
  float zI[TILE][HID + 1], zJ[TILE][HID + 1];
  float rI[TILE], rJ[TILE], colacc[TILE];
  double red[32];
};

__global__ void __launch_bounds__(256)
k_noisy_terms(mcgra_noisy_args na, int64_t t0) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TermsSmem& sm = *reinterpret_cast<TermsSmem*>(smem_raw);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n = na.n, i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const int64_t base = (int64_t)blockIdx.x * TILE_ELEMS;
  if (tid < TILE) {
    sm.rI[tid] = i0 + tid < n ? na.r[i0 + tid] : 0.f;
    sm.rJ[tid] = j0 + tid < n ? na.r[j0 + tid] : 0.f;
    sm.colacc[tid] = 0.f;
  }
  const bool c2 = na.k2 != 0.f;
  const bool slab = J == 0 && na.gslab != nullptr;
  if (c2) {
    for (int e = tid; e < TILE * HID; e += 256) {
      const int r = e >> 4, q = e & 15;
      sm.zI[r][q] = (i0 + r < n) ? na.zhat[(i0 + r) * HID + q] : 0.f;
      sm.zJ[r][q] = (j0 + r < n) ? na.zhat[(j0 + r) * HID + q] : 0.f;
    }
  }
  __syncthreads();
  float v1 = 0.f, v2 = 0.f, v6 = 0.f;
  float col[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
  for (int a = warp; a < TILE; a += 8) {
    const int64_t gi = i0 + a;
    const float ri = sm.rI[a];
    float rowp = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int b = lane + 32 * k;
      const int64_t gj = j0 + b;
      const bool valid = (gj < gi) && (gi < n);
      float cc = 0.f;
      if (valid) {
        const int64_t off = base + a * TILE + b;
        const float L = na.Lt[off], U = na.Ut[off];
        const float rj = sm.rJ[b];
        const float fij = na.FLt ? na.FLt[off] : 0.f, fji = na.FUt ? na.FUt[off] : 0.f;
        float s = 0.f;
        if (c2) {
#pragma unroll
          for (int q = 0; q < HID; ++q) s = fmaf(sm.zI[a][q], sm.zJ[b][q], s);
        }
        ElemOut e = elem_terms<true>(na, (ri * L) * rj, (rj * U) * ri, fij, fji, s, v1, v2, v6);
        if (slab) add_slab_grad(na, gi, gj, e);
        if (c2 && s > 0.f) cc = -2.f * na.k2 * ((((ri * L) * rj) - s) + (((rj * U) * ri) - s));
        const float t = e.eij * L + e.eji * U;         // row i: e'_ij M_ij r_j; row j: e'_ji M_ji r_i (+ column parts)
        rowp += t * rj;
        col[k] += t * ri;
      }
      if (c2) sm.c[a][b] = cc;
    }
    rowp = warp_sum(rowp);
    if (lane == 0 && gi < n && rowp != 0.f) atomicAdd(na.eps_row + gi, rowp);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (col[k] != 0.f) atomicAdd(&sm.colacc[lane + 32 * k], col[k]);
  __syncthreads();
  if (tid < TILE && j0 + tid < n && sm.colacc[tid] != 0.f) atomicAdd(na.eps_row + j0 + tid, sm.colacc[tid]);
  if (c2) {          // dzhat_i += sum_j C_ij zhat_j (threads 0-127, rows of I); dzhat_j += sum_i C_ij zhat_i (128-255)
    float g[HID];
#pragma unroll
    for (int q = 0; q < HID; ++q) g[q] = 0.f;
    const int u = tid & (TILE - 1);
    if (tid < TILE) {
#pragma unroll 4
      for (int b = 0; b < TILE; ++b) {
        const float cv = sm.c[u][b];
#pragma unroll
        for (int q = 0; q < HID; ++q) g[q] = fmaf(cv, sm.zJ[b][q], g[q]);
      }
    } else {
#pragma unroll 4
      for (int a = 0; a < TILE; ++a) {
        const float cv = sm.c[a][u];
#pragma unroll
        for (int q = 0; q < HID; ++q) g[q] = fmaf(cv, sm.zI[a][q], g[q]);
      }
    }
    const int64_t row = (tid < TILE ? i0 : j0) + u;
    if (row < n) {
#pragma unroll
      for (int q = 0; q < HID; ++q)
        if (g[q] != 0.f) atomicAdd(na.dzhat + row * HID + q, g[q]);
    }
  }
  if (na.k1 != 0.f) block_atomic_add_d((double)v1 * (double)na.k1, na.acc + MCGRA_ACC_C1, sm.red);
  if (c2) block_atomic_add_d((double)v2 * (double)na.k2, na.acc + MCGRA_ACC_C2, sm.red);
  if (na.k6 != 0.f) block_atomic_add_d((double)v6 * (double)na.k6, na.acc + MCGRA_ACC_C6, sm.red);
}

struct GradSmem {
  union {
    struct {
      float wi[64][TILE];
      float wj[64][TILE];
    } w;
    float nt[TILE * NT_LD];
  } u;
  float zI[TILE][HID + 1], zJ[TILE][HID + 1];
  float rI[TILE], rJ[TILE], rhoI[TILE], rhoJ[TILE];
};

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

// One CTA per stored tile, 256 threads, 8 x 8 entries per thread (the register tiling of k_fold_adam): the two rank-64
// products P_ij = U_i.V_j and P_ji = U_j.V_i are kept apart, then each orientation gets its element-wise part, its rho
// and its own clamp mask.
__global__ void __launch_bounds__(256, 1)
k_noisy_grad(mcgra_noisy_args na, int64_t t0) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GradSmem& sm = *reinterpret_cast<GradSmem*>(smem_raw);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(na.mu, na.raw);
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t n = na.n, np = na.npad, i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const int64_t base = (int64_t)blockIdx.x * TILE_ELEMS;
  const bool c2 = na.k2 != 0.f;
  const bool slab = J == 0 && na.gslab != nullptr;
  if (tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    sm.rI[tid] = gi < n ? na.r[gi] : 0.f;
    sm.rJ[tid] = gj < n ? na.r[gj] : 0.f;
    sm.rhoI[tid] = gi < n ? na.rho[gi] : 0.f;
    sm.rhoJ[tid] = gj < n ? na.rho[gj] : 0.f;
  }
  if (c2) {
    for (int e = tid; e < TILE * HID; e += 256) {
      const int r = e >> 4, q = e & 15;
      sm.zI[r][q] = (i0 + r < n) ? na.zhat[(i0 + r) * HID + q] : 0.f;
      sm.zJ[r][q] = (j0 + r < n) ? na.zhat[(j0 + r) * HID + q] : 0.f;
    }
  }
  // ---- acc[0] = U_I V_J^T (P_ij), acc[1] = V_I U_J^T (P_ji) ---------------------------------------------------------
  float acc[2][8][8];
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int p = 0; p < 8; ++p)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[h][p][q] = 0.f;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    __syncthreads();
    const int rowI = half == 0 ? 0 : 64, rowJ = half == 0 ? 64 : 0;
    for (int e = tid; e < 64 * 32; e += 256) {
      const int k = e >> 5, c4 = e & 31;
      reinterpret_cast<float4*>(&sm.u.w.wi[k][0])[c4] = ld4(na.Wt + (int64_t)(rowI + k) * np + i0 + c4 * 4);
      reinterpret_cast<float4*>(&sm.u.w.wj[k][0])[c4] = ld4(na.Wt + (int64_t)(rowJ + k) * np + j0 + c4 * 4);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < 64; ++k) {
      const float4 a0 = ld4(&sm.u.w.wi[k][ty * 4]);
      const float4 a1 = ld4(&sm.u.w.wi[k][64 + ty * 4]);
      const float4 b0 = ld4(&sm.u.w.wj[k][tx * 4]);
      const float4 b1 = ld4(&sm.u.w.wj[k][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int p = 0; p < 8; ++p)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[half][p][q] = fmaf(av[p], bv[q], acc[half][p][q]);
    }
  }
  __syncthreads();
  stage_noise_t(sm.u.nt, na.noise, n, i0, j0);
  __syncthreads();

  // ---- per entry: both orientations, masks, sum ------------------------------------------------------------------
  float dummy = 0.f;
#pragma unroll
  for (int p = 0; p < 8; ++p) {
    const int a = (p < 4) ? (ty * 4 + p) : (64 + ty * 4 + (p - 4));
    const int64_t gi = i0 + a;
    const float ri = sm.rI[a], rhoi = sm.rhoI[a];
#pragma unroll
    for (int cg = 0; cg < 2; ++cg) {
      const int b0 = cg * 64 + tx * 4;
      const int64_t off = base + a * TILE + b0;
      const float4 x4 = ld4(na.tiles + off);
      const float4 fl4 = na.FLt ? ld4(na.FLt + off) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 fu4 = na.FUt ? ld4(na.FUt + off) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
      const float fl[4] = {fl4.x, fl4.y, fl4.z, fl4.w};
      const float fu[4] = {fu4.x, fu4.y, fu4.z, fu4.w};
      float g[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int b = b0 + k;
        const int64_t gj = j0 + b;
        g[k] = 0.f;
        if ((gj < gi) && (gi < n)) {
          const float pr = pv.param(xs[k]);
          const float vl = noisy_sum(pr, na.noise[gi * n + gj], na.eps);
          const float vu = noisy_sum(pr, sm.u.nt[b * NT_LD + a], na.eps);
          const float L = clamp01(vl), U = clamp01(vu);
          const float rj = sm.rJ[b];
          float s = 0.f;
          if (c2) {
#pragma unroll
            for (int q = 0; q < HID; ++q) s = fmaf(sm.zI[a][q], sm.zJ[b][q], s);
          }
          ElemOut e = elem_terms<false>(na, (ri * L) * rj, (rj * U) * ri, fl[k], fu[k], s, dummy, dummy, dummy);
          if (slab) add_slab_grad(na, gi, gj, e);
          const float gij = acc[0][p][cg * 4 + k] + ri * rj * e.eij + rhoi;
          const float gji = acc[1][p][cg * 4 + k] + ri * rj * e.eji + sm.rhoJ[b];
          g[k] = box_mask(vl) * gij + box_mask(vu) * gji;
        }
      }
      *reinterpret_cast<float4*>(na.Gt + off) = make_float4(g[0], g[1], g[2], g[3]);
    }
  }
}

inline bool noisy_args_ok(const mcgra_noisy_args* a) {
  return a != nullptr && a->n > 0 && a->tiles != nullptr && a->noise != nullptr && a->r != nullptr &&
         (a->k1 == 0.f || (a->FLt != nullptr && a->FUt != nullptr)) && (a->k2 == 0.f || a->zhat != nullptr) &&
         (a->gslab == nullptr || (a->nb >= 1 && a->nb <= TILE));
}

}  // namespace

extern "C" {

int mcgra_noise_stage(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* noise,
                      float eps, float* Lt, float* Ut, float* mdiag, float* d, void* stream) {
  if (n <= 0 || noise == nullptr) return -1;
  k_noise_diag<false><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, noise, eps, mdiag, d);
  MCGRA_LAUNCH_CHECK();
  return mcgra_noise_tiles(tiles, n, tr0, tr1, mu, raw, noise, eps, Lt, Ut, d, stream);
}

int mcgra_noise_tiles(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* noise,
                      float eps, float* Lt, float* Ut, float* d, void* stream) {
  if (n <= 0 || noise == nullptr) return -1;
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  const size_t smem = (size_t)TILE * NT_LD * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(k_noise_stage, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_noise_stage<<<(unsigned)nt, 256, smem, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, noise, eps, Lt, Ut, d);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_noise_diag(int64_t n, const float* noise, float eps, float* mdiag, float* d, void* stream) {
  if (n <= 0 || noise == nullptr) return -1;
  k_noise_diag<true><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, noise, eps, mdiag, d);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_diag_axpy(const float* mdiag, const float* B, int K, int64_t n, float* Y, void* stream) {
  if (n <= 0) return 0;
  k_diag_axpy<<<(unsigned)((n * K + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mdiag, B, K, n, Y);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_noisy_terms(const mcgra_noisy_args* a, void* stream) {
  if (!noisy_args_ok(a) || a->Lt == nullptr || a->Ut == nullptr) return -1;
  const int64_t nt = tri(a->tr1) - tri(a->tr0);
  if (nt <= 0 || (a->k1 == 0.f && a->k2 == 0.f && a->k6 == 0.f && a->gslab == nullptr)) return 0;
  const size_t smem = sizeof(TermsSmem);
  cudaError_t e = cudaFuncSetAttribute(k_noisy_terms, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_noisy_terms<<<(unsigned)nt, 256, smem, (cudaStream_t)stream>>>(*a, tri(a->tr0));
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_noisy_grad(const mcgra_noisy_args* a, void* stream) {
  if (!noisy_args_ok(a) || a->Wt == nullptr || a->rho == nullptr || a->Gt == nullptr) return -1;
  const int64_t nt = tri(a->tr1) - tri(a->tr0);
  if (nt <= 0) return 0;
  const size_t smem = sizeof(GradSmem);
  cudaError_t e = cudaFuncSetAttribute(k_noisy_grad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_noisy_grad<<<(unsigned)nt, 256, smem, (cudaStream_t)stream>>>(*a, tri(a->tr0));
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
