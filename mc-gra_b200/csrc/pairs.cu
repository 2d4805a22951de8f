// Pair passes over n x 16 factors: the decode gram M1 = relu(zhat zhat^T) and everything that hangs off it.
//
// Reference work replaced: PGDAttack.dot_product_decode (MC-GRA/topology_attack.py:414-419),
// get_modified_adj_after (:381-395), Info_entropy(modified_adj1) = c7 (:233-236), MSELoss(adj_norm,
// modified_adj1) = c2 (:221-229) with their autograd, dot_product_decode2 (:421-467) and the final ensemble
// sum (:300-322).  The n x n gram is never stored: every tile of it is re-generated from the 16-wide factors.
#include "common.cuh"

namespace {

constexpr int CS_LD = TILE + 4;

struct PairSmem {
  float cs[TILE][CS_LD];          // coefficient tile dL/ds_ij (zero where invalid / relu inactive)
  float zI[TILE][HID + 1];
  float zJ[TILE][HID + 1];
  float rI[TILE], rJ[TILE];
  float rowacc[TILE], colacc[TILE];
  double red[32];
};

__global__ void __launch_bounds__(256, 2)
k_pairs(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
        const float* __restrict__ zhat, const float* __restrict__ r, float k7, float k2,
        const float* __restrict__ EAt, const float* __restrict__ Ct,
        float* __restrict__ dzhat, float* __restrict__ eps_row, double* __restrict__ acc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PairSmem& sm = *reinterpret_cast<PairSmem*>(smem_raw);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;

  for (int e = tid; e < TILE * HID; e += 256) {
    const int a = e >> 4, k = e & 15;
    sm.zI[a][k] = (i0 + a < n) ? zhat[(i0 + a) * HID + k] : 0.f;
    sm.zJ[a][k] = (j0 + a < n) ? zhat[(j0 + a) * HID + k] : 0.f;
  }
  if (tid < TILE) {
    sm.rI[tid] = (i0 + tid < n) ? r[i0 + tid] : 0.f;
    sm.rJ[tid] = (j0 + tid < n) ? r[j0 + tid] : 0.f;
    sm.rowacc[tid] = 0.f;
    sm.colacc[tid] = 0.f;
  }
  __syncthreads();

  // ---- s_ij = zhat_i . zhat_j on an 8x8 register tile ----
  float s[8][8];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int q = 0; q < 8; ++q) s[p][q] = 0.f;
#pragma unroll
  for (int k = 0; k < HID; ++k) {
    float av[8], bv[8];
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      av[p] = sm.zI[(p < 4) ? (ty * 4 + p) : (64 + ty * 4 + p - 4)][k];
      bv[p] = sm.zJ[(p < 4) ? (tx * 4 + p) : (64 + tx * 4 + p - 4)][k];
    }
#pragma unroll
    for (int p = 0; p < 8; ++p)
#pragma unroll
      for (int q = 0; q < 8; ++q) s[p][q] = fmaf(av[p], bv[q], s[p][q]);
  }

  // ---- element-wise stage: values, coefficient tile, c2's eps_row ----
  const float* xt = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  const float* eat = EAt ? EAt + (int64_t)blockIdx.x * TILE_ELEMS : nullptr;
  const float* ctt = Ct ? Ct + (int64_t)blockIdx.x * TILE_ELEMS : nullptr;
  const bool needx = (k2 != 0.f) || (eat != nullptr);
  float v7 = 0.f, v2 = 0.f;
  float colp[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) colp[q] = 0.f;
#pragma unroll
  for (int p = 0; p < 8; ++p) {
    const int a = (p < 4) ? (ty * 4 + p) : (64 + ty * 4 + p - 4);
    const int64_t gi = i0 + a;
    const float ri = sm.rI[a];
    float rowp = 0.f;
#pragma unroll
    for (int cg = 0; cg < 2; ++cg) {
      const int b0 = cg * 64 + tx * 4;
      float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f), e4 = x4, c4p = x4;
      if (needx) x4 = *reinterpret_cast<const float4*>(xt + a * TILE + b0);
      if (eat) e4 = *reinterpret_cast<const float4*>(eat + a * TILE + b0);
      if (ctt) c4p = *reinterpret_cast<const float4*>(ctt + a * TILE + b0);
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
      const float es[4] = {e4.x, e4.y, e4.z, e4.w};
      const float cp[4] = {c4p.x, c4p.y, c4p.z, c4p.w};
      float co[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int b = b0 + k;
        const int64_t gj = j0 + b;
        const bool valid = (gj < gi) && (gi < n);
        const float sv = s[p][cg * 4 + k];
        const float pm = fmaxf(sv, 0.f);
        float dp = 0.f;
        if (valid) {
          if (k7 != 0.f) {
            v7 += 2.f * ent_val(pm);
            dp += 2.f * k7 * ent_grad(pm);
          }
          if (k2 != 0.f) {
            const float M = pv.adj(xs[k]);
            const float rj = sm.rJ[b];
            const float df = ri * M * rj - pm;
            v2 += 2.f * df * df;
            dp -= 4.f * k2 * df;
            const float t = 4.f * k2 * df * M;      // (e'_ij + e'_ji) * M_ij
            rowp += t * rj;
            colp[cg * 4 + k] += t * ri;
          }
          if (eat) {
            const float t = es[k] * pv.adj(xs[k]);
            rowp += t * sm.rJ[b];
            colp[cg * 4 + k] += t * ri;
          }
          dp += cp[k];
        }
        co[k] = (valid && sv > 0.f) ? dp : 0.f;     // relu'(0) = 0
      }
      *reinterpret_cast<float4*>(&sm.cs[a][b0]) = make_float4(co[0], co[1], co[2], co[3]);
    }
    if (needx) {
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) rowp += __shfl_xor_sync(0xffffffffu, rowp, o);
      if (tx == 0) sm.rowacc[a] = rowp;
    }
  }
  if (needx) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int b = (q < 4) ? (tx * 4 + q) : (64 + tx * 4 + q - 4);
      if (colp[q] != 0.f) atomicAdd(&sm.colacc[b], colp[q]);
    }
  }
  __syncthreads();

  // ---- dzhat_I += C zhat_J (threads 0-127, one row each); dzhat_J += C^T zhat_I (threads 128-255) ----
  {
    const int u = tid & 127;
    float o[HID];
#pragma unroll
    for (int k = 0; k < HID; ++k) o[k] = 0.f;
    if (tid < 128) {
#pragma unroll 1
      for (int b = 0; b < TILE; b += 4) {
        const float4 c4 = *reinterpret_cast<const float4*>(&sm.cs[u][b]);
        const float cv[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int k = 0; k < HID; ++k) o[k] = fmaf(cv[q], sm.zJ[b + q][k], o[k]);
      }
    } else {
#pragma unroll 1
      for (int a = 0; a < TILE; ++a) {
        const float cv = sm.cs[a][u];
#pragma unroll
        for (int k = 0; k < HID; ++k) o[k] = fmaf(cv, sm.zI[a][k], o[k]);
      }
    }
    const int64_t g = (tid < 128 ? i0 : j0) + u;
    if (g < n) {
      float4* dst = reinterpret_cast<float4*>(dzhat + g * HID);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 val = make_float4(o[q * 4], o[q * 4 + 1], o[q * 4 + 2], o[q * 4 + 3]);
        if (val.x != 0.f || val.y != 0.f || val.z != 0.f || val.w != 0.f) atomicAdd(dst + q, val);
      }
    }
  }
  if (needx && tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    if (gi < n && sm.rowacc[tid] != 0.f) atomicAdd(eps_row + gi, sm.rowacc[tid]);
    if (gj < n && sm.colacc[tid] != 0.f) atomicAdd(eps_row + gj, sm.colacc[tid]);
  }
  if (k7 != 0.f) block_atomic_add_d((double)v7 * (double)k7, acc + MCGRA_ACC_C7, sm.red);
  if (k2 != 0.f) block_atomic_add_d((double)v2 * (double)k2, acc + MCGRA_ACC_C2, sm.red);
}


// ---------------------------------------------------------------------------------------------------------
// v2 engine: the three products of the pair pass on warp-level tensor-core MMA (mma.sync m16n8k8 tf32, 3xTF32):
//   S = zI zJ^T (128x128x16), then with the coefficient tile C = dL/dS:  dz_I += C zJ,  dz_J += C^T zI.
// Fragment loads are bank-conflict free by construction (strides / k-slot permutation noted at each array).
// ---------------------------------------------------------------------------------------------------------
constexpr int ZT_LD = TILE + 8;    // transposed factors [16][136]: phase-1 fragments, banks 8t+g
constexpr int ZJ_LD = 24;          // zJ [128][24]: direct-product B fragments, banks 24t+g == 8t'+g distinct
constexpr int ZI_LD = 20;          // zI [128][20]: mirrored-product B fragments with k slots 2t,2t+1: banks 8t+g

struct PairMmaSmem {
  float cs[TILE][CS_LD];           // coefficient tile; direct A fragments banks 4g+t, mirrored (slots 2t) 8t+g
  float zIt[HID][ZT_LD];
  float zJt[HID][ZT_LD];
  float zI[TILE][ZI_LD];
  float zJ[TILE][ZJ_LD];
  float rI[TILE], rJ[TILE];
  float rowacc[TILE], colacc[TILE];
  double red[32];
};

__device__ __forceinline__ void split_tf32p(float v, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(v) & 0xffffe000u;        // truncation split (2 ops): this kernel is ALU-bound on the splits;
  lo = __float_as_uint(v - __uint_as_float(hi));   // hi + lo == v exactly, bias of the dropped lo*lo term ~2^-22
}
__device__ __forceinline__ void mma_tf32p(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <bool K7, bool K2, bool DENSE>
__global__ void __launch_bounds__(256, 2)
k_pairs_mma(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
            const float* __restrict__ zhat, const float* __restrict__ r, float k7, float k2,
            const float* __restrict__ EAt, const float* __restrict__ Ct,
            float* __restrict__ dzhat, float* __restrict__ eps_row, double* __restrict__ acc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PairMmaSmem& sm = *reinterpret_cast<PairMmaSmem*>(smem_raw);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;

  for (int e = tid; e < TILE * HID; e += 256) {
    const int a = e >> 4, k = e & 15;
    const float vi = (i0 + a < n) ? zhat[(i0 + a) * HID + k] : 0.f;
    const float vj = (j0 + a < n) ? zhat[(j0 + a) * HID + k] : 0.f;
    sm.zIt[k][a] = vi; sm.zI[a][k] = vi;
    sm.zJt[k][a] = vj; sm.zJ[a][k] = vj;
  }
  if (tid < TILE) {
    sm.rI[tid] = (i0 + tid < n) ? r[i0 + tid] : 0.f;
    sm.rJ[tid] = (j0 + tid < n) ? r[j0 + tid] : 0.f;
    sm.rowacc[tid] = 0.f;
    sm.colacc[tid] = 0.f;
  }
  __syncthreads();

  // ---- phase 1: S tile, warp (wm, wn) owns rows [32 wm, +32) x cols [64 wn, +64) ----
  const int wm = warp >> 1, wn = warp & 1;
  float s[2][8][4];
#pragma unroll
  for (int mb = 0; mb < 2; ++mb)
#pragma unroll
    for (int nb = 0; nb < 8; ++nb)
#pragma unroll
      for (int q = 0; q < 4; ++q) s[mb][nb][q] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    const int k0 = ks * 8;
    uint32_t ahi[2][4], alo[2][4], bh[8][2], bl[8][2];
#pragma unroll
    for (int mb = 0; mb < 2; ++mb) {
      const int m0 = wm * 32 + mb * 16;
      split_tf32p(sm.zIt[k0 + t][m0 + g], ahi[mb][0], alo[mb][0]);
      split_tf32p(sm.zIt[k0 + t][m0 + g + 8], ahi[mb][1], alo[mb][1]);
      split_tf32p(sm.zIt[k0 + t + 4][m0 + g], ahi[mb][2], alo[mb][2]);
      split_tf32p(sm.zIt[k0 + t + 4][m0 + g + 8], ahi[mb][3], alo[mb][3]);
    }
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const int n0 = wn * 64 + nb * 8;
      split_tf32p(sm.zJt[k0 + t][n0 + g], bh[nb][0], bl[nb][0]);
      split_tf32p(sm.zJt[k0 + t + 4][n0 + g], bh[nb][1], bl[nb][1]);
    }
#pragma unroll
    for (int nb = 0; nb < 8; ++nb)
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) mma_tf32p(s[mb][nb], alo[mb], bh[nb][0], bh[nb][1]);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb)
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) mma_tf32p(s[mb][nb], ahi[mb], bl[nb][0], bl[nb][1]);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb)
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) mma_tf32p(s[mb][nb], ahi[mb], bh[nb][0], bh[nb][1]);
  }

  // ---- phase 2: the S tile goes through shared memory so that the element-wise stage is a compact loop (the fully
  // unrolled fragment form was instruction-fetch bound): warp w owns rows w, w+8, ..; lane = 4 consecutive columns.
  // S is overwritten in place by the coefficient tile dL/dS. ----
#pragma unroll
  for (int mb = 0; mb < 2; ++mb)
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const int a0 = wm * 32 + mb * 16 + g, b0 = wn * 64 + nb * 8 + 2 * t;
      *reinterpret_cast<float2*>(&sm.cs[a0][b0]) = make_float2(s[mb][nb][0], s[mb][nb][1]);
      *reinterpret_cast<float2*>(&sm.cs[a0 + 8][b0]) = make_float2(s[mb][nb][2], s[mb][nb][3]);
    }
  __syncthreads();
  const float* xt = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  const float* eat = (DENSE && EAt) ? EAt + (int64_t)blockIdx.x * TILE_ELEMS : nullptr;
  const float* ctt = (DENSE && Ct) ? Ct + (int64_t)blockIdx.x * TILE_ELEMS : nullptr;
  const bool needx = K2 || (eat != nullptr);
  const bool interior = (J < I) && (i0 + TILE <= n);
  float v7 = 0.f, v2 = 0.f;
  {
    const int c4 = lane * 4;
    const float4 rj4 = *reinterpret_cast<const float4*>(&sm.rJ[c4]);
    const float rj[4] = {rj4.x, rj4.y, rj4.z, rj4.w};
    const int gj0 = (int)(j0 + c4);
    float colp[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int it = 0; it < 16; ++it) {
      const int a = it * 8 + warp;
      const int gi = (int)(i0 + a);
      const float4 s4 = *reinterpret_cast<const float4*>(&sm.cs[a][c4]);
      float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f), e4 = x4, p4 = x4;
      if (needx) x4 = __ldg(reinterpret_cast<const float4*>(xt + a * TILE + c4));
      if (DENSE && eat) e4 = __ldg(reinterpret_cast<const float4*>(eat + a * TILE + c4));
      if (DENSE && ctt) p4 = __ldg(reinterpret_cast<const float4*>(ctt + a * TILE + c4));
      const float ri = sm.rI[a];
      const float sv4[4] = {s4.x, s4.y, s4.z, s4.w};
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
      const float es[4] = {e4.x, e4.y, e4.z, e4.w};
      const float cp[4] = {p4.x, p4.y, p4.z, p4.w};
      float co[4];
      float rowp = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const bool valid = interior || ((gj0 + k < gi) && (gi < n));
        const float sv = sv4[k];
        const float pm = fmaxf(sv, 0.f);
        float dp = 0.f;
        if (K7) {
          const float q = fminf(fmaxf(pm, ENT_LO), ENT_HI);
          const float lg = __log2f(q);
          v7 = valid ? fmaf(2.f * q, lg, v7) : v7;
          dp = (pm >= ENT_LO && pm <= ENT_HI) ? 2.f * k7 * (lg + INV_LN2) : 0.f;
        }
        if (K2 || DENSE) {
          const float M = valid ? pv.adj(xs[k]) : 0.f;      // M = 0 removes every contribution of an invalid entry
          float tt = 0.f;
          if (K2) {
            const float df = ri * M * rj[k] - pm;
            v2 = valid ? fmaf(2.f * df, df, v2) : v2;
            dp = fmaf(-4.f * k2, df, dp);
            tt = 4.f * k2 * df * M;                         // (e'_ij + e'_ji) * M_ij
          }
          if (DENSE) { tt = fmaf(es[k], M, tt); dp += cp[k]; }
          rowp = fmaf(tt, rj[k], rowp);
          colp[k] = fmaf(tt, ri, colp[k]);
        }
        co[k] = (valid && sv > 0.f) ? dp : 0.f;             // relu'(0) = 0
      }
      *reinterpret_cast<float4*>(&sm.cs[a][c4]) = make_float4(co[0], co[1], co[2], co[3]);
      if (K2 || DENSE) {
        rowp = warp_sum(rowp);
        if (lane == 0) sm.rowacc[a] = rowp;                 // every row is visited by exactly one warp iteration
      }
    }
    if (K2 || DENSE) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (colp[k] != 0.f) atomicAdd(&sm.colacc[c4 + k], colp[k]);
    }
  }
  __syncthreads();

  // ---- phase 3: warp w -> direct rows a in [16 w, +16) and mirrored rows b in [16 w, +16); N = 16 ----
  {
    float od[2][4], om[2][4];
#pragma unroll
    for (int nb = 0; nb < 2; ++nb)
#pragma unroll
      for (int q = 0; q < 4; ++q) od[nb][q] = om[nb][q] = 0.f;
    const int m0 = warp * 16;
#pragma unroll 2
    for (int ks = 0; ks < TILE / 8; ++ks) {
      const int k0 = ks * 8;
      uint32_t ah[4], al[4], mh[4], ml[4], bh[2][2], bl[2][2], ch[2][2], cl[2][2];
      split_tf32p(sm.cs[m0 + g][k0 + t], ah[0], al[0]);
      split_tf32p(sm.cs[m0 + g + 8][k0 + t], ah[1], al[1]);
      split_tf32p(sm.cs[m0 + g][k0 + t + 4], ah[2], al[2]);
      split_tf32p(sm.cs[m0 + g + 8][k0 + t + 4], ah[3], al[3]);
      split_tf32p(sm.cs[k0 + 2 * t][m0 + g], mh[0], ml[0]);
      split_tf32p(sm.cs[k0 + 2 * t][m0 + g + 8], mh[1], ml[1]);
      split_tf32p(sm.cs[k0 + 2 * t + 1][m0 + g], mh[2], ml[2]);
      split_tf32p(sm.cs[k0 + 2 * t + 1][m0 + g + 8], mh[3], ml[3]);
#pragma unroll
      for (int nb = 0; nb < 2; ++nb) {
        split_tf32p(sm.zJ[k0 + t][nb * 8 + g], bh[nb][0], bl[nb][0]);
        split_tf32p(sm.zJ[k0 + t + 4][nb * 8 + g], bh[nb][1], bl[nb][1]);
        split_tf32p(sm.zI[k0 + 2 * t][nb * 8 + g], ch[nb][0], cl[nb][0]);
        split_tf32p(sm.zI[k0 + 2 * t + 1][nb * 8 + g], ch[nb][1], cl[nb][1]);
      }
#pragma unroll
      for (int nb = 0; nb < 2; ++nb) { mma_tf32p(od[nb], al, bh[nb][0], bh[nb][1]); mma_tf32p(om[nb], ml, ch[nb][0], ch[nb][1]); }
#pragma unroll
      for (int nb = 0; nb < 2; ++nb) { mma_tf32p(od[nb], ah, bl[nb][0], bl[nb][1]); mma_tf32p(om[nb], mh, cl[nb][0], cl[nb][1]); }
#pragma unroll
      for (int nb = 0; nb < 2; ++nb) { mma_tf32p(od[nb], ah, bh[nb][0], bh[nb][1]); mma_tf32p(om[nb], mh, ch[nb][0], ch[nb][1]); }
    }
#pragma unroll
    for (int nb = 0; nb < 2; ++nb) {
      const int64_t ia = i0 + m0 + g, ib = ia + 8, ja = j0 + m0 + g, jb = ja + 8;
      const int c0 = nb * 8 + 2 * t;
      if (ia < n && (od[nb][0] != 0.f || od[nb][1] != 0.f))
        atomicAdd(reinterpret_cast<float2*>(dzhat + ia * HID + c0), make_float2(od[nb][0], od[nb][1]));
      if (ib < n && (od[nb][2] != 0.f || od[nb][3] != 0.f))
        atomicAdd(reinterpret_cast<float2*>(dzhat + ib * HID + c0), make_float2(od[nb][2], od[nb][3]));
      if (ja < n && (om[nb][0] != 0.f || om[nb][1] != 0.f))
        atomicAdd(reinterpret_cast<float2*>(dzhat + ja * HID + c0), make_float2(om[nb][0], om[nb][1]));
      if (jb < n && (om[nb][2] != 0.f || om[nb][3] != 0.f))
        atomicAdd(reinterpret_cast<float2*>(dzhat + jb * HID + c0), make_float2(om[nb][2], om[nb][3]));
    }
  }
  if (needx && tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    if (gi < n && sm.rowacc[tid] != 0.f) atomicAdd(eps_row + gi, sm.rowacc[tid]);
    if (gj < n && sm.colacc[tid] != 0.f) atomicAdd(eps_row + gj, sm.colacc[tid]);
  }
  if (k7 != 0.f) block_atomic_add_d((double)v7 * (double)k7, acc + MCGRA_ACC_C7, sm.red);
  if (k2 != 0.f) block_atomic_add_d((double)v2 * (double)k2, acc + MCGRA_ACC_C2, sm.red);
}

int g_ensemble_engine = 1;  // mcgra_set_engine(5, v): 0 one CTA per 64 x 64 block, 1 one CTA per block PAIR for the full matrix (default)
int g_pairs_engine = 2;     // 0 fp32 FFMA (exact), 1 mma.sync 3xTF32, 2 tcgen05 for the entropy-only configuration (else 1)

// x_final tiles = relu(z_i . z_j), j < i < n  (dot_product_decode of the last embedding, :300-301)
// Register-tiled: thread (tx, ty) owns rows 8 ty .. + 7 and columns 8 tx .. + 7 of the tile; factors staged transposed
// ([k][row], pitch 132) so that one k step is four 16-byte shared loads for 64 FMAs (the scalar form was LDS-bound:
// 9.4 ms for the 8.6 GB of tiles at n = 65 536).  The fmaf chain over k runs in the same order as before.
constexpr int DLD = TILE + 4;
__global__ void __launch_bounds__(256)
k_decode_to_tiles(const float* __restrict__ z, int64_t n, int64_t t0, float* __restrict__ tiles) {
  __shared__ __align__(16) float zIT[HID * DLD], zJT[HID * DLD];
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  for (int it = tid; it < 2 * TILE * (HID / 4); it += 256) {
    const int m = it >= TILE * (HID / 4) ? 1 : 0, idx = it - m * TILE * (HID / 4);
    const int a = idx >> 2, q4 = idx & 3;
    const int64_t row = (m ? j0 : i0) + a;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < n) {
      const float* zr = z + row * HID + 4 * q4;
      if ((reinterpret_cast<uintptr_t>(z) & 15) == 0) v = __ldg(reinterpret_cast<const float4*>(zr));
      else v = make_float4(zr[0], zr[1], zr[2], zr[3]);
    }
    float* dst = (m ? zJT : zIT) + (4 * q4) * DLD + a;
    dst[0] = v.x; dst[DLD] = v.y; dst[2 * DLD] = v.z; dst[3 * DLD] = v.w;
  }
  __syncthreads();
  float s[8][8];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int q = 0; q < 8; ++q) s[p][q] = 0.f;
#pragma unroll 4
  for (int k = 0; k < HID; ++k) {
    const float4 a0 = *reinterpret_cast<const float4*>(zIT + k * DLD + ty * 8);
    const float4 a1 = *reinterpret_cast<const float4*>(zIT + k * DLD + ty * 8 + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(zJT + k * DLD + tx * 8);
    const float4 b1 = *reinterpret_cast<const float4*>(zJT + k * DLD + tx * 8 + 4);
    const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int p = 0; p < 8; ++p)
#pragma unroll
      for (int q = 0; q < 8; ++q) s[p][q] = fmaf(av[p], bv[q], s[p][q]);
  }
  float* dst = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
#pragma unroll
  for (int p = 0; p < 8; ++p) {
    const int a = ty * 8 + p;
    const int64_t gi = i0 + a;
    float v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int64_t gj = j0 + tx * 8 + q;
      v[q] = (gj < gi && gi < n) ? fmaxf(s[p][q], 0.f) : 0.f;
    }
    float4* d4 = reinterpret_cast<float4*>(dst + a * TILE + tx * 8);
    d4[0] = make_float4(v[0], v[1], v[2], v[3]);
    d4[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
}

// rows [b0, b1) of the symmetric zero-diagonal expansion of the decode: out[(i - b0) ld + j] = relu(z_i . z_j) for j != i,
// 0 for j == i (what k_decode_to_tiles + k_tiles_to_dense give, as one write-only stream).  128 x 128 output block per CTA,
// register-tiled and staged exactly as k_decode_to_tiles, with the same fmaf chain over k: the product inside an fmaf is
// exact, so z_i . z_j above the diagonal is bit-equal to the z_j . z_i its mirrored tile entry holds.  Thread tx owns the
// columns 4 tx .. 4 tx + 3 and 64 + 4 tx .. 64 + 4 tx + 3 of its 8 rows: one 16-byte store instruction of a warp then fills
// two whole 256-byte row spans (the 8-consecutive-column split of k_decode_to_tiles left every 32-byte sector of a store
// half written: 0.85 ms instead of 0.64 ms for an 8 192-row band at n = 65 536 on a B200).
__global__ void __launch_bounds__(256)
k_decode_band(const float* __restrict__ z, int64_t n, int64_t b0, int64_t b1, float* __restrict__ out, int64_t ld,
              int vec) {
  __shared__ __align__(16) float zIT[HID * DLD], zJT[HID * DLD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t i0 = b0 + (int64_t)blockIdx.y * TILE, j0 = (int64_t)blockIdx.x * TILE;
  for (int it = tid; it < 2 * TILE * (HID / 4); it += 256) {
    const int m = it >= TILE * (HID / 4) ? 1 : 0, idx = it - m * TILE * (HID / 4);
    const int a = idx >> 2, q4 = idx & 3;
    const int64_t row = (m ? j0 : i0) + a;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < n) {
      const float* zr = z + row * HID + 4 * q4;
      if ((reinterpret_cast<uintptr_t>(z) & 15) == 0) v = __ldg(reinterpret_cast<const float4*>(zr));
      else v = make_float4(zr[0], zr[1], zr[2], zr[3]);
    }
    float* dst = (m ? zJT : zIT) + (4 * q4) * DLD + a;
    dst[0] = v.x; dst[DLD] = v.y; dst[2 * DLD] = v.z; dst[3 * DLD] = v.w;
  }
  __syncthreads();
  float s[8][8];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int q = 0; q < 8; ++q) s[p][q] = 0.f;
#pragma unroll 4
  for (int k = 0; k < HID; ++k) {
    const float4 a0 = *reinterpret_cast<const float4*>(zIT + k * DLD + ty * 8);
    const float4 a1 = *reinterpret_cast<const float4*>(zIT + k * DLD + ty * 8 + 4);
    const float4 c0 = *reinterpret_cast<const float4*>(zJT + k * DLD + tx * 4);
    const float4 c1 = *reinterpret_cast<const float4*>(zJT + k * DLD + 64 + tx * 4);
    const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float bv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
    for (int p = 0; p < 8; ++p)
#pragma unroll
      for (int q = 0; q < 8; ++q) s[p][q] = fmaf(av[p], bv[q], s[p][q]);
  }
#pragma unroll
  for (int p = 0; p < 8; ++p) {
    const int64_t gi = i0 + ty * 8 + p;
    if (gi >= b1) break;
    float* row = out + (gi - b0) * ld;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t jc = j0 + 64 * h + 4 * tx;
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) v[r] = (jc + r == gi) ? 0.f : fmaxf(s[p][4 * h + r], 0.f);
      if (vec && jc + 4 <= n) {
        *reinterpret_cast<float4*>(row + jc) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int r = 0; r < 4; ++r)
          if (jc + r < n) row[jc + r] = v[r];
      }
    }
  }
}

// sigmoid of dot_product_decode2 (:425) for v >= 0 (after the relu): MUFU ex2 + rcp, ~2e-7 relative (the IEEE expf + division
// form cost ~30 instructions per entry and term, more than the 16-step fmaf chain it follows).  ONE definition for the three
// kernels below, so that the fused ensemble stays bit-equal to the sequence of single-term kernels.
__device__ __forceinline__ float ens_sigmoid(float v) { return __fdividef(1.f, 1.f + __expf(-v)); }

// out[i, j] += f(Z_i . Z_j)   for i in [row0,row1), all j; 32x32 output block per CTA, d <= 32
__global__ void __launch_bounds__(256)
k_gram_accumulate(const float* __restrict__ Z, int d, int64_t n, int variant, const float* __restrict__ rownorm,
                  float* __restrict__ out, int64_t ld, int64_t row0, int64_t row1) {
  __shared__ float zi[32][33], zj[32][33];
  const int64_t bi = row0 + (int64_t)blockIdx.y * 32, bj = (int64_t)blockIdx.x * 32;
  const int tid = threadIdx.x;
  for (int e = tid; e < 32 * d; e += 256) {
    const int a = e / d, k = e % d;
    zi[a][k] = (bi + a < n) ? Z[(bi + a) * d + k] : 0.f;
    zj[a][k] = (bj + a < n) ? Z[(bj + a) * d + k] : 0.f;
  }
  __syncthreads();
  const int tx = tid & 31, ty = tid >> 5;
  for (int rr = ty; rr < 32; rr += 8) {
    const int64_t gi = bi + rr, gj = bj + tx;
    if (gi >= n || gj >= n || gi >= row1) continue;
    float s = 0.f;
    for (int k = 0; k < d; ++k) s = fmaf(zi[rr][k], zj[tx][k], s);
    if (variant == 2) s = s / fmaxf(rownorm[gi], 1e-12f);
    float v = (variant == 3) ? s : fmaxf(s - (gi == gj ? 1.f : 0.f), 0.f);
    if (variant == 4) v = (gi == gj) ? 0.f : fmaxf(s, 0.f);
    if (variant == 0) v = ens_sigmoid(v);
    out[gi * ld + gj] += v;
  }
}

// fused ensemble: 64 x 64 output block per CTA, thread (tx, ty) owns the 4 x 4 micro-tile rows 4 ty.., columns 4 tx..;
// the partial sums stay in registers across the terms and the block is written once.  Factors are staged transposed
// ([k][row]) so that one k step is two 16-byte shared loads for 16 FMAs (the 32 x 32 scalar form was LDS-bound).
// Per-element arithmetic (order of the fmaf chain over k, the variant transforms, the left-to-right sum of the terms)
// is exactly that of k_tiles_to_dense / k_gram_accumulate / k_dense_add / k_label_accumulate.
constexpr int EB = 64;
__global__ void __launch_bounds__(256)
k_ensemble(const float* __restrict__ tiles, int64_t n, mcgra_ensemble_args ea, float* __restrict__ out, int64_t ld,
           int64_t row0, int64_t row1) {
  __shared__ __align__(16) float buf[2 * 32 * EB + EB];       // M stage: [64][65]; gram stage: ziT[32][64] | zjT[32][64]
  const int64_t bi = row0 + (int64_t)blockIdx.y * EB, bj = (int64_t)blockIdx.x * EB;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[p][q] = 0.f;
  if (tiles != nullptr) {
    // stage the stored block (rows of the larger index, columns of the smaller one); entry (max, min) is read from it
    const int64_t br = bi >= bj ? bi : bj, bc = bi >= bj ? bj : bi;
    const float* tl = tiles + (tri(br / TILE) + bc / TILE) * (int64_t)TILE_ELEMS + (br % TILE) * TILE + (bc % TILE);
    for (int e = tid; e < EB * EB; e += 256) {
      const int rr = e >> 6, cc = e & 63;
      buf[rr * (EB + 1) + cc] = fminf(fmaxf(tl[rr * TILE + cc], 0.f), 1.f);
    }
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4 + q;
        const int a = (int)(gi > gj ? gi - br : gj - br), c = (int)(gi > gj ? gj - bc : gi - bc);
        acc[p][q] = (gi < n && gj < n && gi != gj) ? buf[a * (EB + 1) + c] : 0.f;
      }
    __syncthreads();
  }
  float* ziT = buf;
  float* zjT = buf + 32 * EB;
  for (int tm = 0; tm < ea.nterms; ++tm) {
    const mcgra_ensemble_term& T = ea.t[tm];
    if (T.kind == MCGRA_TERM_GRAM) {
      const int d = T.d;
      for (int e = tid; e < EB * d; e += 256) {
        const int a = e / d, k = e % d;
        ziT[k * EB + a] = (bi + a < n) ? T.Z[(bi + a) * d + k] : 0.f;
        zjT[k * EB + a] = (bj + a < n) ? T.Z[(bj + a) * d + k] : 0.f;
      }
      __syncthreads();
      float s[4][4];
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) s[p][q] = 0.f;
      for (int k = 0; k < d; ++k) {
        const float4 a4 = *reinterpret_cast<const float4*>(ziT + k * EB + ty * 4);
        const float4 b4 = *reinterpret_cast<const float4*>(zjT + k * EB + tx * 4);
        const float av[4] = {a4.x, a4.y, a4.z, a4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
          for (int q = 0; q < 4; ++q) s[p][q] = fmaf(av[p], bv[q], s[p][q]);
      }
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int64_t gi = bi + ty * 4 + p;
        const float rn = (T.variant == 2 && gi < n) ? fmaxf(T.rownorm[gi], 1e-12f) : 1.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int64_t gj = bj + tx * 4 + q;
          float sv = s[p][q];
          if (T.variant == 2) sv = sv / rn;
          float v = (T.variant == 3) ? sv : fmaxf(sv - (gi == gj ? 1.f : 0.f), 0.f);
          if (T.variant == 4) v = (gi == gj) ? 0.f : fmaxf(sv, 0.f);
          if (T.variant == 0) v = ens_sigmoid(v);
          acc[p][q] += v;
        }
      }
      __syncthreads();
    } else if (T.kind == MCGRA_TERM_DENSE) {
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4;
        if (gi >= n || gi >= row1) continue;
        if ((n & 3) == 0) {                       // rows are 16-byte aligned: one vector load (gj + 3 < n since n % 4 == 0)
          if (gj < n) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(T.dense + gi * n + gj));
            acc[p][0] += v.x; acc[p][1] += v.y; acc[p][2] += v.z; acc[p][3] += v.w;
          }
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (gj + q < n) acc[p][q] += T.dense[gi * n + gj + q];
        }
      }
    } else {
      int64_t lj[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) lj[q] = (bj + tx * 4 + q < n) ? T.labels[bj + tx * 4 + q] : -1;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int64_t gi = bi + ty * 4 + p;
        if (gi >= n || gi >= row1) continue;
        const int64_t li = T.labels[gi];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (bj + tx * 4 + q < n && li == lj[q]) acc[p][q] += 1.f;
      }
    }
  }
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4;
    if (gi >= n || gi >= row1) continue;
    if ((ld & 3) == 0 && gj + 3 < n && ((reinterpret_cast<uintptr_t>(out) & 15) == 0)) {
      *reinterpret_cast<float4*>(out + gi * ld + gj) = make_float4(acc[p][0], acc[p][1], acc[p][2], acc[p][3]);
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (gj + q < n) out[gi * ld + gj + q] = acc[p][q];
    }
  }
}

// Symmetric form of k_ensemble for the full matrix (row0 = 0, row1 = n): one CTA per PAIR of 64 x 64 blocks (I >= J).
// The stored block, the gram sums s_ij (the fmaf chain over k is the same for (i, j) and (j, i): the products commute)
// and their variant transforms (sigmoid: expf + division, the expensive part) are evaluated once and feed two
// accumulation chains -- the block (I, J) and its mirror (J, I) -- which differ only in the un-symmetric terms (dense
// operands, row norms of variant 2).  Element values are bit-for-bit those of k_ensemble: same chain order, same
// transforms, same left-to-right sum of the terms.  Factors are staged by 16-byte loads into a [k][row] layout with a
// 68-float pitch (2-way instead of 16-way bank conflicts on the transposing stores).
constexpr int ELD = EB + 4;
__device__ __forceinline__ float ens_transform(float sv, bool diag, int variant) {
  float v = (variant == 3) ? sv : fmaxf(sv - (diag ? 1.f : 0.f), 0.f);
  if (variant == 4) v = diag ? 0.f : fmaxf(sv, 0.f);
  if (variant == 0) v = ens_sigmoid(v);
  return v;
}

__global__ void __launch_bounds__(256, 3)
k_ensemble_sym(const float* __restrict__ tiles, int64_t n, mcgra_ensemble_args ea, float* __restrict__ out, int64_t ld) {
  __shared__ __align__(16) float buf[2 * 32 * ELD];       // M stage: [64][65]; gram stage: ziT[32][68] | zjT[32][68]
  int I, J;
  tile_coords((int64_t)blockIdx.x, I, J);                  // pair index -> (I, J), I >= J (same triangle enumeration)
  const int64_t bi = (int64_t)I * EB, bj = (int64_t)J * EB;
  const bool offdiag = I != J;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4], act[4][4];                               // act: the mirrored block, act[p][q] = out[gj + q][gi + p]
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[p][q] = act[p][q] = 0.f;
  if (tiles != nullptr) {
    const float* tl = tiles + (tri(bi / TILE) + bj / TILE) * (int64_t)TILE_ELEMS + (bi % TILE) * TILE + (bj % TILE);
    for (int e = tid; e < EB * EB; e += 256) {
      const int rr = e >> 6, cc = e & 63;
      buf[rr * (EB + 1) + cc] = fminf(fmaxf(tl[rr * TILE + cc], 0.f), 1.f);
    }
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4 + q;
        const int a = (int)(gi > gj ? gi - bi : gj - bi), c = (int)(gi > gj ? gj - bj : gi - bj);
        acc[p][q] = act[p][q] = (gi < n && gj < n && gi != gj) ? buf[a * (EB + 1) + c] : 0.f;
      }
    __syncthreads();
  }
  float* ziT = buf;
  float* zjT = buf + 32 * ELD;
  const bool vec_ok = (n & 3) == 0;
  for (int tm = 0; tm < ea.nterms; ++tm) {
    const mcgra_ensemble_term& T = ea.t[tm];
    if (T.kind == MCGRA_TERM_GRAM) {
      const int d = T.d;
      if ((d & 3) == 0 && (reinterpret_cast<uintptr_t>(T.Z) & 15) == 0) {
        const int dq = d >> 2, items = EB * dq;
        for (int it = tid; it < 2 * items; it += 256) {
          const int m = it >= items ? 1 : 0, idx = it - m * items;
          const int a = idx / dq, q4 = idx - a * dq;
          const int64_t row = (m ? bj : bi) + a;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (row < n) v = __ldg(reinterpret_cast<const float4*>(T.Z + row * d) + q4);
          float* dst = (m ? zjT : ziT) + (4 * q4) * ELD + a;
          dst[0] = v.x; dst[ELD] = v.y; dst[2 * ELD] = v.z; dst[3 * ELD] = v.w;
        }
      } else {
        for (int e = tid; e < EB * d; e += 256) {
          const int a = e / d, k = e % d;
          ziT[k * ELD + a] = (bi + a < n) ? T.Z[(bi + a) * d + k] : 0.f;
          zjT[k * ELD + a] = (bj + a < n) ? T.Z[(bj + a) * d + k] : 0.f;
        }
      }
      __syncthreads();
      float s[4][4];
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) s[p][q] = 0.f;
      for (int k = 0; k < d; ++k) {
        const float4 a4 = *reinterpret_cast<const float4*>(ziT + k * ELD + ty * 4);
        const float4 b4 = *reinterpret_cast<const float4*>(zjT + k * ELD + tx * 4);
        const float av[4] = {a4.x, a4.y, a4.z, a4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
          for (int q = 0; q < 4; ++q) s[p][q] = fmaf(av[p], bv[q], s[p][q]);
      }
      if (T.variant == 2) {                      // row-normalised gram: the two orientations divide by different norms
        float rni[4], rnj[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4 + p;
          rni[p] = gi < n ? fmaxf(T.rownorm[gi], 1e-12f) : 1.f;
          rnj[p] = gj < n ? fmaxf(T.rownorm[gj], 1e-12f) : 1.f;
        }
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const bool dg = (bi + ty * 4 + p) == (bj + tx * 4 + q);
            acc[p][q] += ens_transform(s[p][q] / rni[p], dg, 2);
            act[p][q] += ens_transform(s[p][q] / rnj[q], dg, 2);
          }
      } else {
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const bool dg = (bi + ty * 4 + p) == (bj + tx * 4 + q);
            const float v = ens_transform(s[p][q], dg, T.variant);
            acc[p][q] += v;
            act[p][q] += v;
          }
      }
      __syncthreads();
    } else if (T.kind == MCGRA_TERM_DENSE) {
#pragma unroll
      for (int p = 0; p < 4; ++p) {                         // block (I, J): row gi, columns gj .. gj + 3
        const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4;
        if (gi >= n) continue;
        if (vec_ok) {
          if (gj < n) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(T.dense + gi * n + gj));
            acc[p][0] += v.x; acc[p][1] += v.y; acc[p][2] += v.z; acc[p][3] += v.w;
          }
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (gj + q < n) acc[p][q] += T.dense[gi * n + gj + q];
        }
      }
      if (offdiag) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {                       // block (J, I): row gj, columns gi .. gi + 3
          const int64_t gj = bj + tx * 4 + q, gi = bi + ty * 4;
          if (gj >= n) continue;
          if (vec_ok) {
            if (gi < n) {
              const float4 v = __ldg(reinterpret_cast<const float4*>(T.dense + gj * n + gi));
              act[0][q] += v.x; act[1][q] += v.y; act[2][q] += v.z; act[3][q] += v.w;
            }
          } else {
#pragma unroll
            for (int p = 0; p < 4; ++p)
              if (gi + p < n) act[p][q] += T.dense[gj * n + gi + p];
          }
        }
      }
    } else {
      int64_t lj[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) lj[q] = (bj + tx * 4 + q < n) ? T.labels[bj + tx * 4 + q] : -1;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int64_t gi = bi + ty * 4 + p;
        if (gi >= n) continue;
        const int64_t li = T.labels[gi];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (bj + tx * 4 + q < n && li == lj[q]) { acc[p][q] += 1.f; act[p][q] += 1.f; }
      }
    }
  }
  const bool st_vec = (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const int64_t gi = bi + ty * 4 + p, gj = bj + tx * 4;
    if (gi >= n) continue;
    if (st_vec && gj + 3 < n) {
      *reinterpret_cast<float4*>(out + gi * ld + gj) = make_float4(acc[p][0], acc[p][1], acc[p][2], acc[p][3]);
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (gj + q < n) out[gi * ld + gj + q] = acc[p][q];
    }
  }
  if (offdiag) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t gj = bj + tx * 4 + q, gi = bi + ty * 4;
      if (gj >= n) continue;
      if (st_vec && gi + 3 < n) {
        *reinterpret_cast<float4*>(out + gj * ld + gi) = make_float4(act[0][q], act[1][q], act[2][q], act[3][q]);
      } else {
#pragma unroll
        for (int p = 0; p < 4; ++p)
          if (gi + p < n) out[gj * ld + gi + p] = act[p][q];
      }
    }
  }
}

__global__ void __launch_bounds__(256)
k_label_accumulate(const int64_t* __restrict__ labels, int64_t n, float* __restrict__ out, int64_t ld, int64_t row0,
                   int64_t row1) {
  const int64_t gj = (int64_t)blockIdx.x * 256 + threadIdx.x;
  const int64_t gi = row0 + blockIdx.y;
  if (gi >= row1 || gj >= n) return;
  if (labels[gi] == labels[gj]) out[gi * ld + gj] += 1.f;
}

__global__ void k_dense_add(float* __restrict__ out, const float* __restrict__ in, int64_t count) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += stride) out[e] += in[e];
}

// row p-norm normalisation (F.normalize(Z, p, dim=1), eps 1e-12); one thread per row
__global__ void k_row_normalize(const float* __restrict__ Z, int64_t n, int d, float p, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.f;
  for (int k = 0; k < d; ++k) {
    const float v = fabsf(Z[i * d + k]);
    acc += (p == 2.f) ? v * v : powf(v, p);
  }
  const float nrm = (p == 2.f) ? sqrtf(acc) : powf(acc, 1.f / p);
  const float inv = 1.f / fmaxf(nrm, 1e-12f);
  for (int k = 0; k < d; ++k) out[i * d + k] = Z[i * d + k] * inv;
}

template <bool K7, bool K2, bool DENSE>
int launch_pairs_mma(const float* tiles, int64_t n, int tr0, int64_t nt, const float* mu, int raw, const float* zhat,
                     const float* r, float k7, float k2, const float* EAt, const float* Ct, float* dzhat,
                     float* eps_row, double* acc, cudaStream_t st) {
  const size_t smem = sizeof(PairMmaSmem);
  cudaError_t e = cudaFuncSetAttribute(k_pairs_mma<K7, K2, DENSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_pairs_mma<K7, K2, DENSE><<<(unsigned)nt, 256, smem, st>>>(tiles, n, tri(tr0), mu, raw, zhat, r, k7, k2, EAt, Ct,
                                                             dzhat, eps_row, acc);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" {

int mcgra_set_pairs_engine_(int value) {
  if (value < 0 || value > 2) return -1;
  g_pairs_engine = value;
  return 0;
}
int mcgra_set_ensemble_engine_(int value) {
  if (value != 0 && value != 1) return -1;
  g_ensemble_engine = value;
  return 0;
}

int mcgra_pairs_tc_(int64_t n, int tr0, int tr1, const float* zhat, float k7, float* dzhat, double* acc, void* ws,
                    cudaStream_t st);

int mcgra_pairs(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* zhat,
                const float* r, float k7, float k2, const float* EAt, const float* Ct, float* dzhat, float* eps_row,
                double* acc, void* ws, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  // engine 2: the entropy-only configuration (README Cora profile) entirely on tcgen05, no HBM stream (pairs_tc.cu)
  if (g_pairs_engine == 2 && ws != nullptr && k7 != 0.f && k2 == 0.f && EAt == nullptr && Ct == nullptr)
    return mcgra_pairs_tc_(n, tr0, tr1, zhat, k7, dzhat, acc, ws, (cudaStream_t)stream);
  if (g_pairs_engine >= 1) {
    const bool f7 = k7 != 0.f, f2 = k2 != 0.f, fd = (EAt != nullptr) || (Ct != nullptr);
#define MCGRA_PAIRS_CASE(A, B, D)                                                                                  \
    if (f7 == A && f2 == B && fd == D)                                                                             \
      return launch_pairs_mma<A, B, D>(tiles, n, tr0, nt, mu, raw, zhat, r, k7, k2, EAt, Ct, dzhat, eps_row, acc,  \
                                       (cudaStream_t)stream);
    MCGRA_PAIRS_CASE(false, false, false) MCGRA_PAIRS_CASE(false, false, true)
    MCGRA_PAIRS_CASE(false, true, false) MCGRA_PAIRS_CASE(false, true, true)
    MCGRA_PAIRS_CASE(true, false, false) MCGRA_PAIRS_CASE(true, false, true)
    MCGRA_PAIRS_CASE(true, true, false) MCGRA_PAIRS_CASE(true, true, true)
#undef MCGRA_PAIRS_CASE
  }
  const size_t smem = sizeof(PairSmem);
  cudaError_t e = cudaFuncSetAttribute(k_pairs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_pairs<<<(unsigned)nt, 256, smem, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, zhat, r, k7, k2, EAt, Ct,
                                                              dzhat, eps_row, acc);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_decode_to_tiles(const float* zhat, int64_t n, int tr0, int tr1, float* tiles, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_decode_to_tiles<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(zhat, n, tri(tr0), tiles);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_decode_band(const float* z, int64_t n, int64_t b0, int64_t b1, float* out, int64_t ld, void* stream) {
  if (b0 < 0 || b1 > n || ld < n) return -1;
  if (b1 <= b0) return 0;
  dim3 grid((unsigned)((n + TILE - 1) / TILE), (unsigned)((b1 - b0 + TILE - 1) / TILE));
  if (grid.y > 65535) return -3;
  const int vec = (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  k_decode_band<<<grid, 256, 0, (cudaStream_t)stream>>>(z, n, b0, b1, out, ld, vec);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_gram_accumulate(const float* Z, int d, int64_t n, int variant, const float* rownorm, float* out, int64_t ld,
                          int64_t row0, int64_t row1, void* stream) {
  if (d > 32 || d < 1) return -1;
  if (row1 <= row0) return 0;
  dim3 grid((unsigned)((n + 31) / 32), (unsigned)((row1 - row0 + 31) / 32));
  if (grid.y > 65535) return -3;
  k_gram_accumulate<<<grid, 256, 0, (cudaStream_t)stream>>>(Z, d, n, variant, rownorm, out, ld, row0, row1);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_ensemble(const float* tiles, int64_t n, const mcgra_ensemble_args* args, float* out, int64_t ld,
                   int64_t row0, int64_t row1, void* stream) {
  if (args == nullptr || args->nterms < 0 || args->nterms > MCGRA_ENSEMBLE_MAX) return -1;
  if ((row0 & 63) != 0) return -1;
  for (int t = 0; t < args->nterms; ++t)
    if (args->t[t].kind == MCGRA_TERM_GRAM && (args->t[t].d < 1 || args->t[t].d > 32)) return -1;
  if (row1 <= row0) return 0;
  if (g_ensemble_engine == 1 && row0 == 0 && row1 >= n) {       // full matrix: block pairs (I >= J), both orientations per CTA
    const int64_t nb = (n + EB - 1) / EB, pairs = nb * (nb + 1) / 2;
    if (pairs > 2147483647LL) return -3;
    k_ensemble_sym<<<(unsigned)pairs, 256, 0, (cudaStream_t)stream>>>(tiles, n, *args, out, ld);
    MCGRA_LAUNCH_CHECK();
    return 0;
  }
  dim3 grid((unsigned)((n + EB - 1) / EB), (unsigned)((row1 - row0 + EB - 1) / EB));
  if (grid.y > 65535) return -3;
  k_ensemble<<<grid, 256, 0, (cudaStream_t)stream>>>(tiles, n, *args, out, ld, row0, row1);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_label_accumulate(const int64_t* labels, int64_t n, float* out, int64_t ld, int64_t row0, int64_t row1,
                           void* stream) {
  if (row1 <= row0) return 0;
  for (int64_t r = row0; r < row1; r += 65535) {
    const int64_t r1 = (r + 65535 < row1) ? r + 65535 : row1;
    dim3 grid((unsigned)((n + 255) / 256), (unsigned)(r1 - r));
    k_label_accumulate<<<grid, 256, 0, (cudaStream_t)stream>>>(labels, n, out, ld, r, r1);
    MCGRA_LAUNCH_CHECK();
  }
  return 0;
}

int mcgra_dense_add(float* out, const float* in, int64_t count, void* stream) {
  if (count <= 0) return 0;
  k_dense_add<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(out, in, count);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_row_normalize(const float* Z, int64_t n, int d, float p, float* out, void* stream) {
  if (n <= 0) return 0;
  k_row_normalize<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(Z, n, d, p, out);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
