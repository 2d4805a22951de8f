// Node-level stages of one PGD iteration: everything that is O(n * 16) -- the dense 16-wide halves of
// GraphConvolution.forward (MC-GRA/models/gcn.py:35-46), GCN.forward's relu / Linear / log_softmax
// (models/gcn.py:164-174), embedding_GCN.forward (models/gcn.py:71-76), F.nll_loss (topology_attack.py:326-336),
// F.normalize of dot_product_decode (topology_attack.py:415), the n x d measure terms c9 / c10
// (topology_attack.py:237-272) and the hand-derived backward of all of them, plus the degree gradient rho of
// utils.normalize_adj_tensor (MC-GRA/utils.py:211-230; SURVEY.md 8(a4)).  One thread per node; weights in smem.
#include "common.cuh"

namespace {

struct NodeW {
  float W2[HID * HID];
  float b1[HID], b2[HID];
  float Wl[MCGRA_MAXC * HID];
  float bl[MCGRA_MAXC];
};

__device__ __forceinline__ void load_weights(NodeW& w, const mcgra_node_args& a) {
  for (int e = threadIdx.x; e < HID * HID; e += blockDim.x) w.W2[e] = a.W2[e];
  for (int e = threadIdx.x; e < HID; e += blockDim.x) {
    w.b1[e] = a.b1[e];
    w.b2[e] = a.b2[e];
  }
  for (int e = threadIdx.x; e < a.nclass * HID; e += blockDim.x) w.Wl[e] = a.Wl[e];
  for (int e = threadIdx.x; e < a.nclass; e += blockDim.x) w.bl[e] = a.bl[e];
  __syncthreads();
}

__device__ __forceinline__ void ld16(const float* p, float* v) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 t = reinterpret_cast<const float4*>(p)[q];
    v[q * 4] = t.x; v[q * 4 + 1] = t.y; v[q * 4 + 2] = t.z; v[q * 4 + 3] = t.w;
  }
}
__device__ __forceinline__ void st16(float* p, const float* v) {
#pragma unroll
  for (int q = 0; q < 4; ++q)
    reinterpret_cast<float4*>(p)[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
}
__device__ __forceinline__ void zero16(float* p) {
#pragma unroll
  for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(p)[q] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// ---------------------------------------------------------------------------------------------------------
__global__ void k_node_pre(mcgra_node_args a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const float d = a.d[i];
  const float r = d > 0.f ? 1.0f / sqrtf(d) : 0.f;   // rowsum.pow(-1/2), inf -> 0 (utils.py:225-226)
  a.r[i] = r;
  float s1[HID], t[HID];
  ld16(a.S1 + i * HID, s1);
#pragma unroll
  for (int k = 0; k < HID; ++k) t[k] = r * s1[k];
  st16(a.B1 + i * 32, t);
  st16(a.B1 + i * 32 + HID, s1);
  zero16(a.Y1 + i * 32);
  zero16(a.Y1 + i * 32 + HID);
  a.eps_row[i] = 0.f;
}

__global__ void k_node_mid(mcgra_node_args a) {
  __shared__ NodeW w;
  load_weights(w, a);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const float r = a.r[i];
  float p1[HID], q1[HID], s1[HID], h1[HID], e1[HID], s2[HID], t2[HID];
  ld16(a.Y1 + i * 32, p1);
  ld16(a.Y1 + i * 32 + HID, q1);
  ld16(a.S1 + i * HID, s1);
  uint32_t mask = 0;
#pragma unroll
  for (int k = 0; k < HID; ++k) {
    const float z = r * (p1[k] + r * s1[k]) + w.b1[k];     // (A_hat S1)_i + b1
    h1[k] = fmaxf(z, 0.f);
    if (z > 0.f) mask |= (1u << k);
    const float q = q1[k] + w.b1[k];                       // (M S1)_i + b1
    e1[k] = fmaxf(q, 0.f);
    if (q > 0.f) mask |= (1u << (16 + k));
  }
#pragma unroll
  for (int c = 0; c < HID; ++c) {
    float s = 0.f, t = 0.f;
#pragma unroll
    for (int k = 0; k < HID; ++k) {
      s = fmaf(h1[k], w.W2[k * HID + c], s);
      t = fmaf(e1[k], w.W2[k * HID + c], t);
    }
    s2[c] = s;
    t2[c] = t;
  }
  a.masks[i] = mask;
  st16(a.S2 + i * HID, s2);
  st16(a.T2 + i * HID, t2);
#pragma unroll
  for (int k = 0; k < HID; ++k) s2[k] *= r;
  st16(a.B2 + i * 32, s2);
  st16(a.B2 + i * 32 + HID, t2);
  zero16(a.Y2 + i * 32);
  zero16(a.Y2 + i * 32 + HID);
}

// softmax over c entries in place; returns log-sum-exp
__device__ __forceinline__ float softmax_inplace(float* z, int c) {
  float mx = z[0];
  for (int k = 1; k < c; ++k) mx = fmaxf(mx, z[k]);
  float s = 0.f;
  for (int k = 0; k < c; ++k) {
    z[k] = expf(z[k] - mx);
    s += z[k];
  }
  const float inv = 1.f / s;
  for (int k = 0; k < c; ++k) z[k] *= inv;
  return mx + logf(s);
}

__global__ void k_node_head(mcgra_node_args a) {
  __shared__ NodeW w;
  __shared__ double red[32];
  load_weights(w, a);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < a.n;
  const int C = a.nclass;
  double v_nll = 0.0, v_c9 = 0.0, v_c10 = 0.0;
  if (live) {
    const float r = a.r[i];
    const float wi = a.wmult[i];
    float p2a[HID], q2a[HID], s2[HID], h2[HID], em[HID];
    ld16(a.Y2 + i * 32, p2a);
    ld16(a.Y2 + i * 32 + HID, q2a);
    ld16(a.S2 + i * HID, s2);
    uint32_t mask = 0;
#pragma unroll
    for (int k = 0; k < HID; ++k) {
      const float z = r * (p2a[k] + r * s2[k]) + w.b2[k];
      h2[k] = fmaxf(z, 0.f);
      if (z > 0.f) mask |= (1u << k);
      const float q = q2a[k] + w.b2[k];
      em[k] = fmaxf(q, 0.f);
      if (q > 0.f) mask |= (1u << (16 + k));
    }
    a.masks2[i] = mask;
    st16(a.H2 + i * HID, h2);
    if (a.em != nullptr) st16(a.em + i * HID, em);

    // ---- supervised head on the normalised branch (topology_attack.py:167,172) ----
    float lg[MCGRA_MAXC];
    for (int c = 0; c < C; ++c) {
      float s = w.bl[c];
#pragma unroll
      for (int k = 0; k < HID; ++k) s = fmaf(h2[k], w.Wl[c * HID + k], s);
      lg[c] = s;
    }
    const int y = (int)a.labels[i];
    const float ly = lg[y];
    const float lse = softmax_inplace(lg, C);
    v_nll = (double)(wi * (lse - ly));
    float dz2[HID];
#pragma unroll
    for (int k = 0; k < HID; ++k) dz2[k] = 0.f;
    if (wi != 0.f && a.weight_sup != 0.f) {
      for (int c = 0; c < C; ++c) {
        const float dl = a.weight_sup * wi * (lg[c] - (c == y ? 1.f : 0.f));
#pragma unroll
        for (int k = 0; k < HID; ++k) dz2[k] = fmaf(dl, w.Wl[c * HID + k], dz2[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < HID; ++k) dz2[k] = ((mask >> k) & 1u) ? dz2[k] : 0.f;
    st16(a.dZ2 + i * HID, dz2);

    // ---- raw branch: embedding, its row normalisation, second head (topology_attack.py:185-187,259) ----
    float nrm2 = 0.f;
#pragma unroll
    for (int k = 0; k < HID; ++k) nrm2 = fmaf(em[k], em[k], nrm2);
    const float inv = 1.f / fmaxf(sqrtf(nrm2), 1e-12f);
    float zh[HID];
#pragma unroll
    for (int k = 0; k < HID; ++k) zh[k] = em[k] * inv;
    st16(a.zhat + i * HID, zh);
    a.inv_norm[i] = inv;
    zero16(a.dzhat + i * HID);

    float dem[HID];
#pragma unroll
    for (int k = 0; k < HID; ++k) dem[k] = 0.f;
    const int meas = a.measure;
    if (a.w9 != 0.f && wi != 0.f) {
      float ha[HID];
      ld16(a.HA + i * HID, ha);
      if (meas == MCGRA_M_MSE) {                         // w9 * mean((H_A - em)^2)
        const float k9 = a.w9 / (float)HID;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < HID; ++k) {
          const float df = em[k] - ha[k];
          s = fmaf(df, df, s);
          dem[k] = fmaf(2.f * k9 * wi, df, dem[k]);
        }
        v_c9 = (double)(k9 * wi * s);
      } else if (meas == MCGRA_M_KL) {                   // batchmean KL(softmax(H_A) || softmax(em))
        float xs[HID], ys[HID];
#pragma unroll
        for (int k = 0; k < HID; ++k) { xs[k] = ha[k]; ys[k] = em[k]; }
        const float lx = softmax_inplace(xs, HID);
        const float ly2 = softmax_inplace(ys, HID);
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < HID; ++k) {
          if (xs[k] > 0.f) s += xs[k] * ((ha[k] - lx) - (em[k] - ly2));
          dem[k] = fmaf(a.w9 * wi, ys[k] - xs[k], dem[k]);
        }
        v_c9 = (double)(a.w9 * wi * s);
      }
    }
    if (a.w10 != 0.f && wi != 0.f && (meas == MCGRA_M_MSE || meas == MCGRA_M_KL)) {
      float p2[MCGRA_MAXC], dp[MCGRA_MAXC];
      for (int c = 0; c < C; ++c) {
        float s = w.bl[c];
#pragma unroll
        for (int k = 0; k < HID; ++k) s = fmaf(em[k], w.Wl[c * HID + k], s);
        p2[c] = s;
      }
      softmax_inplace(p2, C);                            // softmax(log_softmax(z)) == softmax(z)
      const float* ya = a.YA + i * C;
      float val = 0.f;
      if (meas == MCGRA_M_MSE) {                         // w10 * mean((Y_A - p2)^2), Y_A are log-probs (:264-271)
        const float k10 = a.w10 / (float)C;
        for (int c = 0; c < C; ++c) {
          const float df = p2[c] - ya[c];
          val = fmaf(df, df, val);
          dp[c] = 2.f * k10 * wi * df;
        }
        v_c10 = (double)(k10 * wi * val);
      } else {                                           // KL(softmax(Y_A) || softmax(p2))
        float xs[MCGRA_MAXC], ys[MCGRA_MAXC];
        for (int c = 0; c < C; ++c) { xs[c] = ya[c]; ys[c] = p2[c]; }
        const float lx = softmax_inplace(xs, C);
        const float ly2 = softmax_inplace(ys, C);
        for (int c = 0; c < C; ++c) {
          if (xs[c] > 0.f) val += xs[c] * ((ya[c] - lx) - (p2[c] - ly2));
          dp[c] = a.w10 * wi * (ys[c] - xs[c]);
        }
        v_c10 = (double)(a.w10 * wi * val);
      }
      float dot = 0.f;
      for (int c = 0; c < C; ++c) dot = fmaf(p2[c], dp[c], dot);
      for (int c = 0; c < C; ++c) {
        const float dl = p2[c] * (dp[c] - dot);          // softmax backward
#pragma unroll
        for (int k = 0; k < HID; ++k) dem[k] = fmaf(dl, w.Wl[c * HID + k], dem[k]);
      }
    }
    st16(a.demd + i * HID, dem);
  }
  block_atomic_add_d(v_nll, a.acc + MCGRA_ACC_NLL, red);
  block_atomic_add_d(v_c9, a.acc + MCGRA_ACC_C9, red);
  block_atomic_add_d(v_c10, a.acc + MCGRA_ACC_C10, red);
}

__global__ void k_node_bwd2(mcgra_node_args a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const float r = a.r[i];
  float dzh[HID], zh[HID], dem[HID], dz2[HID];
  ld16(a.dzhat + i * HID, dzh);
  ld16(a.zhat + i * HID, zh);
  ld16(a.demd + i * HID, dem);
  ld16(a.dZ2 + i * HID, dz2);
  const float inv = a.inv_norm[i];
  const uint32_t mask = a.masks2[i];
  float dot = 0.f;
#pragma unroll
  for (int k = 0; k < HID; ++k) dot = fmaf(zh[k], dzh[k], dot);
  float dq2[HID];
#pragma unroll
  for (int k = 0; k < HID; ++k) {
    const float g = dem[k] + (dzh[k] - zh[k] * dot) * inv;       // F.normalize backward
    dq2[k] = ((mask >> (16 + k)) & 1u) ? g : 0.f;
    dz2[k] *= r;
  }
  st16(a.dQ2 + i * HID, dq2);
  st16(a.B3 + i * 32, dz2);
  st16(a.B3 + i * 32 + HID, dq2);
  zero16(a.Y3 + i * 32);
  zero16(a.Y3 + i * 32 + HID);
}

__global__ void k_node_bwd1(mcgra_node_args a) {
  __shared__ NodeW w;
  load_weights(w, a);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const float r = a.r[i];
  float p3[HID], q3[HID], dz2[HID], ds2[HID], dz1[HID], dq1[HID];
  ld16(a.Y3 + i * 32, p3);
  ld16(a.Y3 + i * 32 + HID, q3);
  ld16(a.dZ2 + i * HID, dz2);
  const uint32_t mask = a.masks[i];
#pragma unroll
  for (int c = 0; c < HID; ++c) ds2[c] = r * (p3[c] + r * dz2[c]);   // A_hat dZ2
#pragma unroll
  for (int k = 0; k < HID; ++k) {
    float s = 0.f, t = 0.f;
#pragma unroll
    for (int c = 0; c < HID; ++c) {
      s = fmaf(ds2[c], w.W2[k * HID + c], s);
      t = fmaf(q3[c], w.W2[k * HID + c], t);
    }
    dz1[k] = ((mask >> k) & 1u) ? s : 0.f;
    dq1[k] = ((mask >> (16 + k)) & 1u) ? t : 0.f;
  }
  st16(a.dZ1 + i * HID, dz1);
  st16(a.dQ1 + i * HID, dq1);
#pragma unroll
  for (int k = 0; k < HID; ++k) dz1[k] *= r;
  st16(a.B4 + i * HID, dz1);
  zero16(a.Y4 + i * HID);
}

// DIAG: the estimate has a non-zero diagonal M_ii = mdiag[i] (noisy path): A_hat_ii = r^2 (1 + M_ii), and the diagonal
// entry enters rho's row and column parts with (M + I)_ii = 1 + M_ii
template <bool DIAG>
__global__ void k_node_rho(mcgra_node_args a, const float* __restrict__ mdiag) {
  __shared__ double red[32];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < a.n;
  double v1 = 0.0, v2 = 0.0, v6 = 0.0, v7 = 0.0;
  if (i == 0) {                               // reset the statistics the fold accumulates into
    for (int k = 0; k < MCGRA_ACC_N; ++k) a.acc_next[k] = 0.0;
    a.minmax[0] = INFINITY;
    a.minmax[1] = -INFINITY;
  }
  if (live) {
    a.d_next[i] = a.d_fill;
    const float r = a.r[i], d = a.d[i];
    float p1[HID], p2[HID], p3[HID], p4[HID], s1[HID], s2[HID], t2[HID], dz1[HID], dz2[HID], dq1[HID], dq2[HID];
    ld16(a.Y1 + i * 32, p1);
    ld16(a.Y2 + i * 32, p2);
    ld16(a.Y3 + i * 32, p3);
    ld16(a.Y4 + i * HID, p4);
    ld16(a.S1 + i * HID, s1);
    ld16(a.S2 + i * HID, s2);
    ld16(a.T2 + i * HID, t2);
    ld16(a.dZ1 + i * HID, dz1);
    ld16(a.dZ2 + i * HID, dz2);
    ld16(a.dQ1 + i * HID, dq1);
    ld16(a.dQ2 + i * HID, dq2);
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < HID; ++k) {
      t = fmaf(dz1[k], p1[k] + r * s1[k], t);
      t = fmaf(s1[k], p4[k] + r * dz1[k], t);
      t = fmaf(dz2[k], p2[k] + r * s2[k], t);
      t = fmaf(s2[k], p3[k] + r * dz2[k], t);
    }
    // diagonal entry A_hat_ii = r^2 of the element-wise terms
    const float mi1 = DIAG ? 1.f + mdiag[i] : 1.f;
    const float aii = DIAG ? (r * mi1) * r : r * r;
    float eii = 0.f;
    if (a.k1 != 0.f && a.measure_nn == MCGRA_M_MSE) {
      const float f = a.Fdiag ? a.Fdiag[i] : 0.f;
      eii += 2.f * a.k1 * (aii - f);
      v1 = (double)a.k1 * (double)((aii - f) * (aii - f));
    } else if (a.k1 != 0.f && a.measure_nn == MCGRA_M_KL) {
      const float f = a.Fdiag ? a.Fdiag[i] : 0.f;
      const float xii = expf(f - a.lseF[i]);
      const float lii = aii - a.lseA[i];
      eii += a.k1 * (expf(lii) - xii);
      v1 = (double)a.k1 * (double)(xii * ((f - aii) - a.dlse[i]));
    }
    if (a.measure_nn == MCGRA_M_PRE && a.Fdiag != nullptr) eii += a.Fdiag[i];
    if (a.k6 != 0.f) {
      eii += a.k6 * ent_grad(aii);
      v6 = (double)a.k6 * (double)ent_val(aii);
    }
    if (a.k2 != 0.f) {
      eii += 2.f * a.k2 * aii;
      v2 = (double)a.k2 * (double)(aii * aii);
    }
    if (a.k7 != 0.f) v7 = (double)a.k7 * (double)ent_val(0.f);
    const float tot = t + a.eps_row[i] + 2.f * eii * (DIAG ? mi1 * r : r);
    a.rho[i] = -0.5f * tot / (d * sqrtf(d));
    // fold factors, transposed: rows 0-63 U = [r dZ1 | r dZ2 | dQ1 | dQ2], rows 64-127 V = [r S1 | r S2 | S1 | T2]
    float* W = a.Wt + i;
    const int64_t np = a.npad;
#pragma unroll
    for (int k = 0; k < HID; ++k) {
      W[(int64_t)(k)*np] = r * dz1[k];
      W[(int64_t)(16 + k) * np] = r * dz2[k];
      W[(int64_t)(32 + k) * np] = dq1[k];
      W[(int64_t)(48 + k) * np] = dq2[k];
      W[(int64_t)(64 + k) * np] = r * s1[k];
      W[(int64_t)(80 + k) * np] = r * s2[k];
      W[(int64_t)(96 + k) * np] = s1[k];
      W[(int64_t)(112 + k) * np] = t2[k];
    }
  }
  block_atomic_add_d(v1, a.acc + MCGRA_ACC_C1D, red);
  block_atomic_add_d(v2, a.acc + MCGRA_ACC_C2D, red);
  block_atomic_add_d(v6, a.acc + MCGRA_ACC_C6D, red);
  block_atomic_add_d(v7, a.acc + MCGRA_ACC_C7D, red);
}

inline unsigned nblk(int64_t n) { return (unsigned)((n + 127) / 128); }

}  // namespace

extern "C" {

int mcgra_node_pre(const mcgra_node_args* a, void* stream) {
  k_node_pre<<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_node_mid(const mcgra_node_args* a, void* stream) {
  k_node_mid<<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_node_head(const mcgra_node_args* a, void* stream) {
  if (a->nclass > MCGRA_MAXC) return -2;
  k_node_head<<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_node_bwd2(const mcgra_node_args* a, void* stream) {
  k_node_bwd2<<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_node_bwd1(const mcgra_node_args* a, void* stream) {
  k_node_bwd1<<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_node_rho(const mcgra_node_args* a, void* stream) {
  k_node_rho<false><<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a, nullptr);
  MCGRA_LAUNCH_CHECK();
  return 0;
}
int mcgra_node_rho_diag(const mcgra_node_args* a, const float* mdiag, void* stream) {
  if (mdiag == nullptr) return -1;
  k_node_rho<true><<<nblk(a->n), 128, 0, (cudaStream_t)stream>>>(*a, mdiag);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
