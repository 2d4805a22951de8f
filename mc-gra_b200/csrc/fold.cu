// Gradient fold back to the triangle + Adam + box clamp, and the budget projection by bisection.
//
// Reference work replaced: loss.backward() (the n x n gradients of every propagation and element-wise term,
// autograd through utils.normalize_adj_tensor, the index_put / m+m.t() scatter back to the P-vector),
// torch.optim.Adam.step() and the clamp (MC-GRA/topology_attack.py:274-283); PGDAttack.projection / bisection
// (topology_attack.py:338-347, 397-412).
//
// The n x n gradient is never stored.  For entry (i,j), i > j, the gradient of the parameter is
//   g = mask * [ U_i.V_j + V_i.U_j  +  r_i r_j (e'_ij + e'_ji)  +  rho_i + rho_j ]  +  0.001 w_sup x / ||x||
// with U = [r dZ1 | r dZ2 | dQ1 | dQ2], V = [r S1 | r S2 | S1 | T2] (rank-64 factors built by the node kernels),
// e' the element-wise loss derivatives at A_hat_ij and rho the degree gradient (SURVEY.md 8(a4)).
// Engines (mcgra_set_engine(1, v)):
//   0  k_fold_adam  one CTA per tile, fp32 register-tiled FFMA product (exact; reference of the agreement tests)
//   2  k_fold_tc    one CTA per tile, tcgen05 kind::tf32 3xTF32 product (N = 256 [W_hi | W_lo] operands pre-formatted by
//                   k_prep_w, L2-friendly blocked tile order), every parameter view / measure
//   3  k_fold_rs    DEFAULT for "fast" launches (buffer holds the clamped parameter, MSE / precomputed / no c1 term):
//                   persistent row runs, A operand resident in tensor memory, bulk-copy rings for B and for x' / m / v / F,
//                   16 streaming warps; other launches run on k_fold_tc
// All read x', m, v (and feature_adj) once and write x', m, v once: 24 (+4) bytes per entry.
#include "common.cuh"
#include "tc_common.cuh"

namespace {

struct FoldSmem {
  float wi[64][TILE];
  float wj[64][TILE];
  float zI[TILE][HID + 1];
  float zJ[TILE][HID + 1];
  float rI[TILE], rJ[TILE], rhoI[TILE], rhoJ[TILE];
  float lseAI[TILE], lseAJ[TILE], lseFI[TILE], lseFJ[TILE];
  float rowacc[TILE], colacc[TILE];
  double red[32];
};

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

__global__ void __launch_bounds__(256, 2)
k_fold_adam(float* __restrict__ tiles, float* __restrict__ mbuf, float* __restrict__ vbuf, int64_t t0, const float* mu,
            int raw, mcgra_fold_args fa, float* __restrict__ minmax) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FoldSmem& sm = *reinterpret_cast<FoldSmem*>(smem_raw);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const int64_t n = fa.n, np = fa.npad;

  if (tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    sm.rI[tid] = gi < n ? fa.r[gi] : 0.f;
    sm.rJ[tid] = gj < n ? fa.r[gj] : 0.f;
    sm.rhoI[tid] = gi < n ? fa.rho[gi] : 0.f;
    sm.rhoJ[tid] = gj < n ? fa.rho[gj] : 0.f;
    if (fa.measure == MCGRA_M_KL) {
      sm.lseAI[tid] = gi < n ? fa.lseA[gi] : 0.f;
      sm.lseAJ[tid] = gj < n ? fa.lseA[gj] : 0.f;
      sm.lseFI[tid] = gi < n ? fa.lseF[gi] : 0.f;
      sm.lseFJ[tid] = gj < n ? fa.lseF[gj] : 0.f;
    }
    sm.colacc[tid] = 0.f;
    sm.rowacc[tid] = 0.f;
  }
  if (fa.k2 != 0.f) {
    for (int e = tid; e < TILE * HID; e += 256) {
      const int a = e >> 4, k = e & 15;
      sm.zI[a][k] = (i0 + a < n) ? fa.zhat[(i0 + a) * HID + k] : 0.f;
      sm.zJ[a][k] = (j0 + a < n) ? fa.zhat[(j0 + a) * HID + k] : 0.f;
    }
  }

  // ---- rank-128 product: acc[a][b] = U_i.V_j + V_i.U_j ----------------------------------------------------
  float acc[8][8];
#pragma unroll
  for (int p = 0; p < 8; ++p)
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[p][q] = 0.f;

#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    __syncthreads();
    const int rowI = half == 0 ? 0 : 64;     // U rows for I in half 0, V rows in half 1
    const int rowJ = half == 0 ? 64 : 0;
    for (int e = tid; e < 64 * 32; e += 256) {
      const int k = e >> 5, c4 = e & 31;
      reinterpret_cast<float4*>(&sm.wi[k][0])[c4] = ld4(fa.Wt + (int64_t)(rowI + k) * np + i0 + c4 * 4);
      reinterpret_cast<float4*>(&sm.wj[k][0])[c4] = ld4(fa.Wt + (int64_t)(rowJ + k) * np + j0 + c4 * 4);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < 64; ++k) {
      const float4 a0 = ld4(&sm.wi[k][ty * 4]);
      const float4 a1 = ld4(&sm.wi[k][64 + ty * 4]);
      const float4 b0 = ld4(&sm.wj[k][tx * 4]);
      const float4 b1 = ld4(&sm.wj[k][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int p = 0; p < 8; ++p)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[p][q] = fmaf(av[p], bv[q], acc[p][q]);
    }
  }

  // ---- streaming epilogue: element-wise terms, Adam, clamp statistics ------------------------------------
  const double sumsq_prev = fa.acc_prev[MCGRA_ACC_SUMSQ];
  const float inv_norm = sumsq_prev > 0.0 ? (float)(1.0 / sqrt(sumsq_prev)) : 0.f;
  const int adam_step = fa.step_ptr != nullptr ? (*fa.step_ptr + 1) : fa.step;
  const double bc1 = 1.0 - pow((double)fa.beta1, (double)adam_step);
  const double bc2 = 1.0 - pow((double)fa.beta2, (double)adam_step);
  const float step_size = (float)((double)fa.lr / bc1);
  const float sqrt_bc2 = (float)sqrt(bc2);
  const float omb1 = 1.f - fa.beta1, omb2 = 1.f - fa.beta2;

  float* xt = tiles + (int64_t)blockIdx.x * TILE_ELEMS;
  float* mt = mbuf + (int64_t)blockIdx.x * TILE_ELEMS;
  float* vt = vbuf + (int64_t)blockIdx.x * TILE_ELEMS;
  const float* ft = fa.Ftiles ? fa.Ftiles + (int64_t)blockIdx.x * TILE_ELEMS : nullptr;
  const float* gt_up = fa.Gtiles ? fa.Gtiles + (int64_t)blockIdx.x * TILE_ELEMS : nullptr;

  float s_clamp = 0.f, s_sq = 0.f, xmin = INFINITY, xmax = -INFINITY;
  float colp[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) colp[q] = 0.f;

#pragma unroll
  for (int p = 0; p < 8; ++p) {
    const int a = (p < 4) ? (ty * 4 + p) : (64 + ty * 4 + (p - 4));
    const int64_t gi = i0 + a;
    const float ri = sm.rI[a], rhoi = sm.rhoI[a];
    float rowp = 0.f;
#pragma unroll
    for (int cg = 0; cg < 2; ++cg) {
      const int b0 = cg * 64 + tx * 4;
      const int off = a * TILE + b0;
      const float4 x4 = ld4(xt + off);
      const float4 m4 = ld4(mt + off);
      const float4 v4 = ld4(vt + off);
      float4 f4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ft) f4 = ld4(ft + off);
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
      const float ms[4] = {m4.x, m4.y, m4.z, m4.w};
      const float vs[4] = {v4.x, v4.y, v4.z, v4.w};
      const float fs[4] = {f4.x, f4.y, f4.z, f4.w};
      float xo[4], mo[4], vo[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int b = b0 + k;
        const int64_t gj = j0 + b;
        const bool valid = (gj < gi) && (gi < n);
        const float p_ = pv.param(xs[k]);
        const float M = pv.adj(xs[k]);
        const float rj = sm.rJ[b];
        const float ah = ri * M * rj;
        float esym = 0.f;
        if (fa.measure == MCGRA_M_MSE) {
          esym += 4.f * fa.k1 * (ah - fs[k]);
        } else if (fa.measure == MCGRA_M_PRE) {
          esym += fs[k];
        } else if (fa.measure == MCGRA_M_KL) {
          const float xij = __expf(fs[k] - sm.lseFI[a]);
          const float xji = __expf(fs[k] - sm.lseFJ[b]);
          esym += fa.k1 * ((__expf(ah - sm.lseAI[a]) - xij) + (__expf(ah - sm.lseAJ[b]) - xji));
        }
        if (fa.k6 != 0.f) esym += 2.f * fa.k6 * ent_grad(ah);
        if (fa.k2 != 0.f) {
          float s = 0.f;
#pragma unroll
          for (int q = 0; q < HID; ++q) s = fmaf(sm.zI[a][q], sm.zJ[b][q], s);
          esym += 4.f * fa.k2 * (ah - fmaxf(s, 0.f));
        }
        float g = ri * rj * esym + rhoi + sm.rhoJ[b] + acc[p][cg * 4 + k];
        if (gt_up != nullptr) g += gt_up[off + k];
        g = pv.mask(xs[k]) * g + fa.norm_coef * p_ * inv_norm;
        const float mn = fa.beta1 * ms[k] + omb1 * g;
        const float vn = fa.beta2 * vs[k] + omb2 * g * g;
        const float denom = sqrtf(vn) / sqrt_bc2 + fa.adam_eps;
        const float xn = fa.plain_gd ? p_ - fa.lr * g : p_ - step_size * (mn / denom);
        const float c = fminf(fmaxf(xn, 0.f), 1.f);
        xo[k] = valid ? (fa.store_clamped ? c : xn) : 0.f;
        mo[k] = valid ? mn : 0.f;
        vo[k] = valid ? vn : 0.f;
        if (valid) {
          s_clamp += c;
          s_sq = fmaf(c, c, s_sq);
          xmin = fminf(xmin, xn);
          xmax = fmaxf(xmax, xn);
          rowp += c;
          colp[cg * 4 + k] += c;
        }
      }
      *reinterpret_cast<float4*>(xt + off) = make_float4(xo[0], xo[1], xo[2], xo[3]);
      *reinterpret_cast<float4*>(mt + off) = make_float4(mo[0], mo[1], mo[2], mo[3]);
      *reinterpret_cast<float4*>(vt + off) = make_float4(vo[0], vo[1], vo[2], vo[3]);
    }
    // row a is owned by the 16 threads of this ty: reduce over tx (half-warp)
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) rowp += __shfl_xor_sync(0xffffffffu, rowp, o);
    if (tx == 0) sm.rowacc[a] = rowp;
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int b = (q < 4) ? (tx * 4 + q) : (64 + tx * 4 + (q - 4));
    if (colp[q] != 0.f) atomicAdd(&sm.colacc[b], colp[q]);
  }
  __syncthreads();
  if (tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    if (gi < n && sm.rowacc[tid] != 0.f) atomicAdd(fa.d_next + gi, sm.rowacc[tid]);
    if (gj < n && sm.colacc[tid] != 0.f) atomicAdd(fa.d_next + gj, sm.colacc[tid]);
  }
  block_atomic_add_d((double)s_clamp, fa.acc_next + MCGRA_ACC_SUMCLAMP, sm.red);
  block_atomic_add_d((double)s_sq, fa.acc_next + MCGRA_ACC_SUMSQ, sm.red);
  xmin = warp_min(xmin);
  xmax = warp_max(xmax);
  if ((tid & 31) == 0) {
    if (xmin != INFINITY) atomic_min_f(minmax, xmin);
    if (xmax != -INFINITY) atomic_max_f(minmax + 1, xmax);
  }
}


constexpr int G_LD = TILE + 4;     // padded row stride of the parked product tile

struct EpiConst {
  float step_size, inv_sqrt_bc2, omb1, omb2, norm_scale;
};

// One 512 B tile row of the streaming epilogue (one warp; lane l owns columns 4l .. 4l+3): gradient assembly, Adam,
// clamp, running sums, stores.  FAST: the tile is interior (every entry valid) and the buffer already holds the parameter
// in [0,1] (raw == 2), no c2 term, MEAS is the compile-time c1 measure.  The generic instantiation handles everything else.
template <bool FAST, int MEAS, bool ENT, typename SM>
__device__ __forceinline__ void fold_row(SM& sm, const mcgra_fold_args& fa, const ParamView& pv, const EpiConst& ec,
                                         float* __restrict__ xt, float* __restrict__ mt, float* __restrict__ vt,
                                         const float* __restrict__ gt_up, int a, int b0, int64_t i0, int64_t j0,
                                         bool interior, const float4& x4, const float4& m4, const float4& v4,
                                         const float4& f4, const float* rj4, const float* rhoj4, float& s_clamp,
                                         float& s_sq, float& xmin, float& xmax, float* colp) {
  const int lane = threadIdx.x & 31;
  const int64_t n = fa.n;
  const int meas = FAST ? MEAS : fa.measure;
  const int off = a * TILE + b0;
  const int gi = (int)(i0 + a);
  const float ri = sm.rI[a], rhoi = sm.rhoI[a];
  const float4 g4 = ld4(&sm.u.gt[a][b0]);
  const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
  const float ms[4] = {m4.x, m4.y, m4.z, m4.w};
  const float vs[4] = {v4.x, v4.y, v4.z, v4.w};
  const float fs[4] = {f4.x, f4.y, f4.z, f4.w};
  const float gs[4] = {g4.x, g4.y, g4.z, g4.w};
  float sdot[4] = {0.f, 0.f, 0.f, 0.f};
  if (!FAST && fa.k2 != 0.f) {
#pragma unroll
    for (int q = 0; q < HID; ++q) {
      const float zi = sm.zI[a][q];
      const float4 zj = ld4(&sm.zJt[q][b0]);
      sdot[0] = fmaf(zi, zj.x, sdot[0]); sdot[1] = fmaf(zi, zj.y, sdot[1]);
      sdot[2] = fmaf(zi, zj.z, sdot[2]); sdot[3] = fmaf(zi, zj.w, sdot[3]);
    }
  }
  float xo[4], mo[4], vo[4];
  float rowp = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const bool valid = FAST ? true : (interior || (((int)(j0 + b0 + k) < gi) && (gi < n)));
    const float p_ = FAST ? xs[k] : pv.param(xs[k]);
    const float M = FAST ? xs[k] : pv.adj(xs[k]);
    const float rj = rj4[k];
    const float ah = ri * M * rj;
    float esym = 0.f;
    if (meas == MCGRA_M_MSE) {
      esym = 4.f * fa.k1 * (ah - fs[k]);
    } else if (meas == MCGRA_M_PRE) {
      esym = fs[k];
    } else if (meas == MCGRA_M_KL) {
      const float xij = __expf(fs[k] - sm.lseFI[a]);
      const float xji = __expf(fs[k] - sm.lseFJ[b0 + k]);
      esym = fa.k1 * ((__expf(ah - sm.lseAI[a]) - xij) + (__expf(ah - sm.lseAJ[b0 + k]) - xji));
    }
    if (ENT && fa.k6 != 0.f && ah >= ENT_LO && ah <= ENT_HI) esym = fmaf(2.f * fa.k6, __log2f(ah) + INV_LN2, esym);
    if (!FAST && fa.k2 != 0.f) esym = fmaf(4.f * fa.k2, ah - fmaxf(sdot[k], 0.f), esym);
    float gg = fmaf(ri * rj, esym, rhoi + rhoj4[k] + gs[k]);
    if (!FAST && gt_up != nullptr) gg += gt_up[off + k];
    if (!FAST) gg *= pv.mask(xs[k]);
    gg = fmaf(ec.norm_scale, p_, gg);
    const float mn = fmaf(ec.omb1, gg - ms[k], ms[k]);                 // beta1*m + (1-beta1)*g
    const float vn = fmaf(ec.omb2, gg * gg - vs[k], vs[k]);            // beta2*v + (1-beta2)*g^2
    // Adam: p - step * m / (sqrt(v)/sqrt(bc2) + eps); sqrt via rsqrt (1 MUFU), divide via rcp (1 MUFU)
    const float sq = vn > 0.f ? vn * rsqrtf(vn) : 0.f;
    const float denom = fmaf(sq, ec.inv_sqrt_bc2, fa.adam_eps);
    const float xn = (!FAST && fa.plain_gd) ? fmaf(-fa.lr, gg, p_) : fmaf(-ec.step_size, __fdividef(mn, denom), p_);
    const float c = fminf(fmaxf(xn, 0.f), 1.f);
    xo[k] = valid ? (fa.store_clamped ? c : xn) : 0.f;
    mo[k] = valid ? mn : 0.f;
    vo[k] = valid ? vn : 0.f;
    if (valid) {
      s_clamp += c;
      s_sq = fmaf(c, c, s_sq);
      xmin = fminf(xmin, xn);
      xmax = fmaxf(xmax, xn);
      rowp += c;
      colp[k] += c;
    }
  }
  *reinterpret_cast<float4*>(xt + off) = make_float4(xo[0], xo[1], xo[2], xo[3]);
  *reinterpret_cast<float4*>(mt + off) = make_float4(mo[0], mo[1], mo[2], mo[3]);
  *reinterpret_cast<float4*>(vt + off) = make_float4(vo[0], vo[1], vo[2], vo[3]);
  rowp = warp_sum(rowp);
  if (lane == 0 && gi < n && rowp != 0.f) atomicAdd(fa.d_next + gi, rowp);
}

// Constants of the persistent engine's inlined row arithmetic (same formulas as fold_row<true, ...> with the per-launch
// factors hoisted, sqrt / clamp as single instructions).
struct FastConst {
  float k1x4, k6x2, norm_scale, omb1, omb2, inv_sqrt_bc2, adam_eps, neg_step;
};
__device__ __forceinline__ float sqrt_approx(float v) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

// Streaming epilogue of a one-tile-per-CTA engine: 8 warps, UNR rows in flight per warp.
template <bool FAST, int MEAS, bool ENT, typename SM>
__device__ __forceinline__ void fold_stream(SM& sm, const mcgra_fold_args& fa, const ParamView& pv,
                                            const EpiConst& ec, int64_t tix, float* __restrict__ tiles,
                                            float* __restrict__ mbuf, float* __restrict__ vbuf, int I, int J,
                                            float& s_clamp, float& s_sq, float& xmin, float& xmax, float* colp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n = fa.n;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  float* xt = tiles + tix * TILE_ELEMS;
  float* mt = mbuf + tix * TILE_ELEMS;
  float* vt = vbuf + tix * TILE_ELEMS;
  const float* ft = fa.Ftiles ? fa.Ftiles + tix * TILE_ELEMS : nullptr;
  const float* gt_up = fa.Gtiles ? fa.Gtiles + tix * TILE_ELEMS : nullptr;
  const bool interior = (J < I) && (i0 + TILE <= n);
  const int b0 = lane * 4;
  const int meas = FAST ? MEAS : fa.measure;
  float rj4[4], rhoj4[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) { rj4[k] = sm.rJ[b0 + k]; rhoj4[k] = sm.rhoJ[b0 + k]; }
  constexpr int UNR = 4;
#pragma unroll 1
  for (int it = 0; it < TILE / (8 * UNR); ++it) {
    float4 x4[UNR], m4[UNR], v4[UNR], f4[UNR];
#pragma unroll
    for (int uu = 0; uu < UNR; ++uu) {
      const int a = (it * UNR + uu) * 8 + warp;
      const int off = a * TILE + b0;
      x4[uu] = ld4(xt + off);
      m4[uu] = ld4(mt + off);
      v4[uu] = ld4(vt + off);
      f4[uu] = (ft && meas != MCGRA_M_NONE) ? ld4(ft + off) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int uu = 0; uu < UNR; ++uu) {
      const int a = (it * UNR + uu) * 8 + warp;
      fold_row<FAST, MEAS, ENT>(sm, fa, pv, ec, xt, mt, vt, gt_up, a, b0, i0, j0, interior, x4[uu], m4[uu], v4[uu], f4[uu],
                                rj4, rhoj4, s_clamp, s_sq, xmin, xmax, colp);
    }
  }
}


// ---------------------------------------------------------------------------------------------------------
// v3 engine: the rank-128 factor product on tcgen05 (kind::tf32, 3xTF32, accumulator in TMEM).
// Operands come pre-formatted (k_prep_w): per 128-node block, 32 K-slabs of 4 factors, each slab =
// [hi: 16 row-groups x 128 B | lo: 16 row-groups x 128 B | 16 B pad] in the SWIZZLE_NONE K-major core layout, so the
// same block is the A operand (U|V order) and, read 16 slabs further, the B operand (V|U order); [hi|lo] adjacent
// gives the N = 256 concatenated B.   D[:, :128] = A_hi B_hi + A_lo B_hi,  D[:, 128:] = A_hi B_lo.
// One CTA per tile, 2 CTAs / SM (256 TMEM columns each), K processed in 4 quarters staged with cp.async; the product
// tile is then parked in shared memory (over the operand buffers) for the coalesced streaming epilogue.
// ---------------------------------------------------------------------------------------------------------
constexpr uint32_t WSLAB = 2 * 16 * 128 + 16;         // 4112 B per K-slab (hi | lo | pad)
constexpr uint32_t WBLOCK = 32 * WSLAB;               // per 128-node block

struct FoldTcSmem {
  union {
    struct { unsigned char a[8 * WSLAB]; unsigned char b[8 * WSLAB]; } op;
    float gt[TILE][G_LD];
  } u;
  float zI[TILE][HID + 1];
  float zJt[HID][TILE + 4];
  float rI[TILE], rJ[TILE], rhoI[TILE], rhoJ[TILE];
  float lseAI[TILE], lseAJ[TILE], lseFI[TILE], lseFJ[TILE];
  float colacc[TILE];
  double red[32];
  uint64_t bar;
  uint32_t tmem_base;
};

__global__ void k_prep_w(const float* __restrict__ Wt, int64_t npad, unsigned char* __restrict__ Wk) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;     // e = k * npad + node (coalesced reads)
  if (e >= npad * 128) return;
  const int k = (int)(e / npad);
  const int64_t node = e % npad;
  const float v = Wt[e];
  const float hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
  const int i = (int)(node & 127);
  unsigned char* p = Wk + (node >> 7) * (int64_t)WBLOCK + (uint32_t)(k >> 2) * WSLAB + (uint32_t)(i >> 3) * 128u +
                     (uint32_t)(i & 7) * 16u + (uint32_t)(k & 3) * 4u;
  *reinterpret_cast<float*>(p) = hi;
  *reinterpret_cast<float*>(p + 2048) = v - hi;
}

__global__ void __launch_bounds__(256, 2)
k_fold_tc(float* __restrict__ tiles, float* __restrict__ mbuf, float* __restrict__ vbuf, int tr0, int tr1, const float* mu,
          int raw, mcgra_fold_args fa, float* __restrict__ minmax, const unsigned char* __restrict__ Wk) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  FoldTcSmem& sm = *reinterpret_cast<FoldTcSmem*>(smem_raw);
  int I, J;
  int64_t tix;
  tile_coords_blocked(blockIdx.x, tr0, tr1, 8, I, J, tix);      // L2-friendly sweep: factor blocks are re-read from L2, not HBM
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const int64_t n = fa.n;

  if (warp == 0) tc::tmem_alloc(&sm.tmem_base, 256);
  if (tid == 0) tc::mbar_init(&sm.bar, 1);
  if (tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    sm.rI[tid] = gi < n ? fa.r[gi] : 0.f;
    sm.rJ[tid] = gj < n ? fa.r[gj] : 0.f;
    sm.rhoI[tid] = gi < n ? fa.rho[gi] : 0.f;
    sm.rhoJ[tid] = gj < n ? fa.rho[gj] : 0.f;
    if (fa.measure == MCGRA_M_KL) {
      sm.lseAI[tid] = gi < n ? fa.lseA[gi] : 0.f;
      sm.lseAJ[tid] = gj < n ? fa.lseA[gj] : 0.f;
      sm.lseFI[tid] = gi < n ? fa.lseF[gi] : 0.f;
      sm.lseFJ[tid] = gj < n ? fa.lseF[gj] : 0.f;
    }
    sm.colacc[tid] = 0.f;
  }
  if (fa.k2 != 0.f) {
    for (int e = tid; e < TILE * HID; e += 256) {
      const int a = e >> 4, k = e & 15;
      sm.zI[a][k] = (i0 + a < n) ? fa.zhat[(i0 + a) * HID + k] : 0.f;
      sm.zJt[k][a] = (j0 + a < n) ? fa.zhat[(j0 + a) * HID + k] : 0.f;
    }
  }
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tm = sm.tmem_base;

  // ---- rank-128 product: 4 K-quarters of 8 slabs (32 factors), 4 K-steps of 8 each ----
  const unsigned char* blkA = Wk + (int64_t)I * WBLOCK;
  const unsigned char* blkB = Wk + (int64_t)J * WBLOCK;
  uint32_t phase = 0;
#pragma unroll 1
  for (int qd = 0; qd < 4; ++qd) {
    if (qd > 0) {                              // tensor cores finished reading the previous quarter
      tc::mbar_wait(&sm.bar, phase);
      phase ^= 1;
      tc::fence_after();
    }
    const float4* sa = reinterpret_cast<const float4*>(blkA + (uint32_t)(8 * qd) * WSLAB);
    const float4* sb = reinterpret_cast<const float4*>(blkB + (uint32_t)((8 * qd + 16) & 31) * WSLAB);
    for (int e = tid; e < (int)(8 * WSLAB / 16); e += 256) {
      tc::cp_async16(reinterpret_cast<float4*>(sm.u.op.a) + e, sa + e);
      tc::cp_async16(reinterpret_cast<float4*>(sm.u.op.b) + e, sb + e);
    }
    tc::cp_async_wait_all();
    tc::fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      tc::fence_after();
      const uint32_t as = tc::smem_u32(sm.u.op.a), bs = tc::smem_u32(sm.u.op.b);
      const uint32_t id_cat = tc::make_idesc_tf32(128, 256, 0, 0);
      const uint32_t id_lo = tc::make_idesc_tf32(128, 128, 0, 0);
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const uint64_t a_hi = tc::make_desc(as + (uint32_t)ks * 2u * WSLAB, WSLAB, 128u);
        const uint64_t a_lo = tc::make_desc(as + (uint32_t)ks * 2u * WSLAB + 2048u, WSLAB, 128u);
        const uint64_t bd = tc::make_desc(bs + (uint32_t)ks * 2u * WSLAB, WSLAB, 128u);
        tc::mma_tf32(tm, a_hi, bd, id_cat, (qd > 0 || ks > 0) ? 1u : 0u);
        tc::mma_tf32(tm, a_lo, bd, id_lo, 1u);
      }
      tc::mma_commit(&sm.bar);
    }
  }
  tc::mbar_wait(&sm.bar, phase);
  tc::fence_after();
  __syncthreads();                             // operand buffers are dead (all threads observed the last commit)
  // ---- drain: D (TMEM) -> product tile in smem; warp w: lane quarter w % 4, column half w / 4 ----
  {
    const int qq = warp & 3, ch = warp >> 2;
    const int row = qq * 32 + lane;
    const uint32_t taddr = tm + ((uint32_t)(qq * 32) << 16) + (uint32_t)(ch * 64);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      float hi[32], lo[32];
      tc::tmem_ld32(taddr + c * 32, hi);
      tc::tmem_ld32(taddr + 128 + c * 32, lo);
#pragma unroll
      for (int u4 = 0; u4 < 8; ++u4)
        *reinterpret_cast<float4*>(&sm.u.gt[row][ch * 64 + c * 32 + u4 * 4]) =
            make_float4(hi[u4 * 4] + lo[u4 * 4], hi[u4 * 4 + 1] + lo[u4 * 4 + 1], hi[u4 * 4 + 2] + lo[u4 * 4 + 2],
                        hi[u4 * 4 + 3] + lo[u4 * 4 + 3]);
    }
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tm, 256);

  // ---- streaming epilogue (shared with the mma.sync engine) ----
  const double sumsq_prev = fa.acc_prev[MCGRA_ACC_SUMSQ];
  const float inv_norm = sumsq_prev > 0.0 ? (float)(1.0 / sqrt(sumsq_prev)) : 0.f;
  const int adam_step = fa.step_ptr != nullptr ? (*fa.step_ptr + 1) : fa.step;
  const double bc1 = 1.0 - pow((double)fa.beta1, (double)adam_step);
  const double bc2 = 1.0 - pow((double)fa.beta2, (double)adam_step);
  EpiConst ec;
  ec.step_size = (float)((double)fa.lr / bc1);
  ec.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  ec.omb1 = 1.f - fa.beta1;
  ec.omb2 = 1.f - fa.beta2;
  ec.norm_scale = fa.norm_coef * inv_norm;
  const bool interior = (J < I) && (i0 + TILE <= n);
  float s_clamp = 0.f, s_sq = 0.f, xmin = INFINITY, xmax = -INFINITY;
  float colp[4] = {0.f, 0.f, 0.f, 0.f};
  const bool fastview = (pv.raw == 2) && interior && fa.k2 == 0.f && fa.measure != MCGRA_M_KL && !fa.plain_gd && fa.Gtiles == nullptr;
  if (fastview) {
    if (fa.measure == MCGRA_M_MSE) {
      if (fa.k6 != 0.f) fold_stream<true, MCGRA_M_MSE, true>(sm, fa, pv, ec, tix, tiles, mbuf, vbuf, I, J, s_clamp, s_sq, xmin, xmax, colp);
      else fold_stream<true, MCGRA_M_MSE, false>(sm, fa, pv, ec, tix, tiles, mbuf, vbuf, I, J, s_clamp, s_sq, xmin, xmax, colp);
    } else if (fa.measure == MCGRA_M_PRE) {
      fold_stream<true, MCGRA_M_PRE, true>(sm, fa, pv, ec, tix, tiles, mbuf, vbuf, I, J, s_clamp, s_sq, xmin, xmax, colp);
    } else {
      fold_stream<true, MCGRA_M_NONE, true>(sm, fa, pv, ec, tix, tiles, mbuf, vbuf, I, J, s_clamp, s_sq, xmin, xmax, colp);
    }
  } else {
    fold_stream<false, -1, true>(sm, fa, pv, ec, tix, tiles, mbuf, vbuf, I, J, s_clamp, s_sq, xmin, xmax, colp);
  }
  const int b0 = lane * 4;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (colp[k] != 0.f) atomicAdd(&sm.colacc[b0 + k], colp[k]);
  __syncthreads();
  if (tid < TILE) {
    const int64_t gj = j0 + tid;
    if (gj < n && sm.colacc[tid] != 0.f) atomicAdd(fa.d_next + gj, sm.colacc[tid]);
  }
  block_atomic_add_d((double)s_clamp, fa.acc_next + MCGRA_ACC_SUMCLAMP, sm.red);
  block_atomic_add_d((double)s_sq, fa.acc_next + MCGRA_ACC_SUMSQ, sm.red);
  xmin = warp_min(xmin);
  xmax = warp_max(xmax);
  if (lane == 0) {
    if (xmin != INFINITY) atomic_min_f(minmax, xmin);
    if (xmax != -INFINITY) atomic_max_f(minmax + 1, xmax);
  }
}

// ---------------------------------------------------------------------------------------------------------
// v4 engine: persistent, warp-specialised, row-run schedule.  What bounds the one-tile-per-CTA engine is not HBM but the
// factor-operand traffic from L2 (2 x 131 KB per 64 KB tile; tools/stream7.cu: the same stream runs at 6.5 TB/s without it
// and at 4.9 TB/s with it), so this engine halves it and takes the staging off the streaming warps:
//   * every CTA walks a contiguous run of tiles in storage (row-major) order; the A operand (factor rows of tile row I,
//     [hi | lo] tf32 planes) stays RESIDENT IN TENSOR MEMORY (2 x 128 columns) for the whole run of that row, only the
//     B block of tile column J is staged per tile (cp.async.bulk, 2-stage ring of K-quarters)
//   * x', m, v, F reach the streaming warps through a 5-stage cp.async.bulk ring in shared memory (8 tile rows per
//     stage), so no registers are spent on prefetch and 16 streaming warps fit; results go back with coalesced stores
//   * the product of tile k + 1 is formed while tile k streams (single accumulator: it is free once drained)
//   warp 0 stream producer | warp 1 B producer | warp 2 MMA issuer + TMEM owner | warp 3 idle | warps 4-19 consumers
// Taken when the launch is "fast" (buffer holds the clamped parameter, clamped store, MSE / precomputed / no c1 term);
// everything else runs on k_fold_tc.
// ---------------------------------------------------------------------------------------------------------
constexpr int RS_S = 5;                        // stream ring stages
constexpr int RS_R = 8;                        // tile rows per stage
constexpr int RS_CH = RS_R * TILE;             // floats per array per stage
constexpr int RS_CW = 16;                      // consumer warps: warp cw -> row cw / 2 of a stage, column half cw % 2
constexpr int RS_THREADS = 128 + RS_CW * 32;   // 640
constexpr uint32_t RS_COL_AH = 256, RS_COL_AL = 384;   // TMEM columns: D [0, 256), A_hi [256, 384), A_lo [384, 512)

struct FoldRsSmem {
  float ring[RS_S][4][RS_CH];                  // x', m, v, F
  struct { float gt[TILE][G_LD]; } u;          // product tile (rank part of the gradient)
  unsigned char bop[2][8 * WSLAB];             // B operand ring: one K-quarter (8 slabs) per stage
  float rI[TILE], rJ[TILE], rhoI[TILE], rhoJ[TILE];
  float nxt[4][TILE];                          // the same four vectors of the next tile
  float rowacc[TILE], colacc[TILE];
  double dsum[2];
  uint64_t sfull[RS_S], sempty[RS_S], bfull[2], bempty[2], dfull, dempty;
  uint32_t tmem_base;
};

__device__ __forceinline__ void ws_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ws_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void ws_bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          tc::smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(tc::smem_u32(bar)), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// single-thread waits of the producer / MMA warps: back off between polls so that the spinning lane does not take issue
// slots from the streaming warps that share its scheduler
__device__ __forceinline__ void ws_wait_backoff(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}"
        : "=r"(done)
        : "r"(tc::smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(64);
  }
}
__device__ __forceinline__ void rs_cons_sync() { asm volatile("bar.sync 1, %0;" ::"n"(RS_CW * 32) : "memory"); }

// tile run iterator: storage (row-major triangle) order inside the shard of tile rows [tr0, tr1)
struct RunIter {
  int I, J;
  __device__ __forceinline__ void init(int tr0, int64_t tix) { tile_coords(tri((int64_t)tr0) + tix, I, J); }
  __device__ __forceinline__ void next() {
    if (++J > I) { ++I; J = 0; }
  }
};

// MEAS: MCGRA_M_MSE / MCGRA_M_PRE / MCGRA_M_NONE; ENT: entropy term on; LAZY: the buffer holds the un-projected Adam output
// x' (raw == 0: parameter = clamp(x' - mu, 0, 1) on read, un-clamped store, min / max tracked for the next bisection)
// instead of the clamped parameter itself (raw == 2)
template <int MEAS, bool ENT, bool LAZY>
__global__ void __launch_bounds__(RS_THREADS, 1)
k_fold_rs(float* __restrict__ tiles, float* __restrict__ mbuf, float* __restrict__ vbuf, int tr0, int64_t ntiles,
          const __grid_constant__ mcgra_fold_args fa, const unsigned char* __restrict__ Wk, const float* mu_ptr,
          float* __restrict__ minmax) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  FoldRsSmem& sm = *reinterpret_cast<FoldRsSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t t_begin = (int64_t)blockIdx.x * ntiles / gridDim.x;
  const int64_t t_end = (int64_t)(blockIdx.x + 1) * ntiles / gridDim.x;
  const int my_tiles = (int)(t_end - t_begin);
  constexpr bool USE_F = MEAS != MCGRA_M_NONE;
  constexpr uint32_t STAGE_BYTES = (USE_F ? 4u : 3u) * RS_CH * 4u;

  if (tid == 0) {
    for (int s = 0; s < RS_S; ++s) {
      tc::mbar_init(&sm.sfull[s], 1);
      tc::mbar_init(&sm.sempty[s], RS_CW);
    }
    for (int s = 0; s < 2; ++s) {
      tc::mbar_init(&sm.bfull[s], 1);
      tc::mbar_init(&sm.bempty[s], 1);
    }
    tc::mbar_init(&sm.dfull, 1);
    tc::mbar_init(&sm.dempty, RS_CW);
    sm.dsum[0] = 0.0;
    sm.dsum[1] = 0.0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) tc::tmem_alloc(&sm.tmem_base, 512);
  if (tid < TILE) { sm.colacc[tid] = 0.f; sm.rowacc[tid] = 0.f; }
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tm = sm.tmem_base;

  if (warp == 0) {
    // ================= stream producer: x', m, v, F rows of every tile of the run, 8 rows per stage =================
    if (lane == 0) {
      // the streamed arrays are touched once per launch: evict-first, so that the factor blocks (re-read by every CTA)
      // stay in L2
      const uint64_t pol = l2_policy_evict_first();
      uint32_t s = 0, ph = 0;
      for (int k = 0; k < my_tiles; ++k) {
        const int64_t base = (t_begin + k) * (int64_t)TILE_ELEMS;
#pragma unroll 1
        for (int ch = 0; ch < TILE / RS_R; ++ch) {
          ws_wait_backoff(&sm.sempty[s], ph ^ 1u);
          const int64_t o = base + (int64_t)ch * RS_CH;
          ws_expect_tx(&sm.sfull[s], STAGE_BYTES);
          ws_bulk_g2s_hint(sm.ring[s][0], tiles + o, RS_CH * 4u, &sm.sfull[s], pol);
          ws_bulk_g2s_hint(sm.ring[s][1], mbuf + o, RS_CH * 4u, &sm.sfull[s], pol);
          ws_bulk_g2s_hint(sm.ring[s][2], vbuf + o, RS_CH * 4u, &sm.sfull[s], pol);
          if (USE_F) ws_bulk_g2s_hint(sm.ring[s][3], fa.Ftiles + o, RS_CH * 4u, &sm.sfull[s], pol);
          if (++s == RS_S) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= B operand producer: factor block of tile column J, V|U order, one K-quarter per stage =========
    if (lane == 0) {
      RunIter it;
      it.init(tr0, t_begin);
      const uint64_t keep = tc::l2_policy_evict_last();      // every CTA of a tile column re-reads the block
      uint32_t cnt = 0;
      for (int k = 0; k < my_tiles; ++k, it.next()) {
        const unsigned char* blkB = Wk + (int64_t)it.J * WBLOCK;
#pragma unroll 1
        for (int qd = 0; qd < 4; ++qd, ++cnt) {
          const uint32_t s = cnt & 1u;
          ws_wait_backoff(&sm.bempty[s], ((cnt >> 1) & 1u) ^ 1u);
          ws_expect_tx(&sm.bfull[s], 8u * WSLAB);
          ws_bulk_g2s_hint(sm.bop[s], blkB + (uint32_t)((8 * qd + 16) & 31) * WSLAB, 8u * WSLAB, &sm.bfull[s], keep);
        }
      }
    }
  } else if (warp == 2) {
    // ================= MMA issuer: D = A (TMEM-resident factor rows of tile row I) x B^T =================
    if (lane == 0) {
      const uint32_t id_cat = tc::make_idesc_tf32(128, 256, 0, 0);
      const uint32_t id_lo = tc::make_idesc_tf32(128, 128, 0, 0);
      uint32_t cnt = 0;
      for (int k = 0; k < my_tiles; ++k) {
        // phase k of dempty: the consumers have drained tile k - 1 and (re)loaded A when the tile row changed
        ws_wait_backoff(&sm.dempty, (uint32_t)(k & 1));
        tc::fence_after();
#pragma unroll 1
        for (int qd = 0; qd < 4; ++qd, ++cnt) {
          const uint32_t s = cnt & 1u;
          ws_wait_backoff(&sm.bfull[s], (cnt >> 1) & 1u);
          tc::fence_after();
          const uint32_t bs = tc::smem_u32(sm.bop[s]);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t kk = (uint32_t)(qd * 4 + ks);
            const uint64_t bd = tc::make_desc(bs + (uint32_t)ks * 2u * WSLAB, WSLAB, 128u);
            tc::mma_tf32_ts(tm, tm + RS_COL_AH + kk * 8u, bd, id_cat, kk > 0 ? 1u : 0u);
            tc::mma_tf32_ts(tm, tm + RS_COL_AL + kk * 8u, bd, id_lo, 1u);
          }
          tc::mma_commit(&sm.bempty[s]);
        }
        tc::mma_commit(&sm.dfull);
      }
    }
  } else if (warp >= 4) {
    // ================= consumers =================
    const int cw = warp - 4, ct = tid - 128;
    const int64_t n = fa.n, np = fa.npad;
    FastConst fc;
    {
      const double sumsq_prev = fa.acc_prev[MCGRA_ACC_SUMSQ];
      const float inv_norm = sumsq_prev > 0.0 ? (float)(1.0 / sqrt(sumsq_prev)) : 0.f;
      const int adam_step = fa.step_ptr != nullptr ? (*fa.step_ptr + 1) : fa.step;
      const double bc1 = 1.0 - pow((double)fa.beta1, (double)adam_step);
      const double bc2 = 1.0 - pow((double)fa.beta2, (double)adam_step);
      fc.neg_step = -(float)((double)fa.lr / bc1);
      fc.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
      fc.omb1 = 1.f - fa.beta1;
      fc.omb2 = 1.f - fa.beta2;
      fc.norm_scale = fa.norm_coef * inv_norm;
      fc.k1x4 = 4.f * fa.k1;
      fc.k6x2 = 2.f * fa.k6;
      fc.adam_eps = fa.adam_eps;
    }
    const float mu = LAZY ? *mu_ptr : 0.f;
    float xmin = INFINITY, xmax = -INFINITY;
    const int qq = cw & 3;                               // TMEM lane quarter of this warp (= warp % 4)
    const int rw = cw >> 1, b0 = (cw & 1) * 64 + lane * 2;   // stage row / first column of this lane
    RunIter cur;
    cur.init(tr0, t_begin);

    // factor rows of tile row I -> TMEM [hi | lo] (lane = node, column = factor index); 4 warps per lane quarter split K
    auto load_A = [&](int I) {
      const int row = qq * 32 + lane;
      const float* src = fa.Wt + (int64_t)I * TILE + row;
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        const int k0 = (cw >> 2) * 32 + half * 16;
        uint32_t h[16], l[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float v = src[(int64_t)(k0 + j) * np];
          const uint32_t hb = (__float_as_uint(v) + 0x1000u) & 0xffffe000u;      // same split as k_prep_w
          h[j] = hb;
          l[j] = __float_as_uint(v - __uint_as_float(hb));
        }
        const uint32_t ta = tm + ((uint32_t)(qq * 32) << 16);
        tc::tmem_st16(ta + RS_COL_AH + (uint32_t)k0, h);
        tc::tmem_st16(ta + RS_COL_AL + (uint32_t)k0, l);
      }
      tc::tmem_st_wait();
    };
    auto load_consts = [&](const RunIter& t) {           // node vectors of a tile -> nxt (threads < 128)
      if (ct < TILE) {
        const int64_t gi = (int64_t)t.I * TILE + ct, gj = (int64_t)t.J * TILE + ct;
        sm.nxt[0][ct] = gi < n ? fa.r[gi] : 0.f;
        sm.nxt[1][ct] = gj < n ? fa.r[gj] : 0.f;
        sm.nxt[2][ct] = gi < n ? fa.rho[gi] : 0.f;
        sm.nxt[3][ct] = gj < n ? fa.rho[gj] : 0.f;
      }
    };
    if (my_tiles > 0) {
      load_A(cur.I);
      load_consts(cur);
    }
    tc::fence_before();
    __syncwarp();
    if (lane == 0) ws_arrive(&sm.dempty);                // phase 0: A of the first tile row is in place

    double d_sq = 0.0, d_clamp = 0.0;
    uint32_t s = 0, ph = 0;
    int Iprev = 0, Jprev = 0;
#pragma unroll 1
    for (int k = 0; k < my_tiles; ++k) {
      const bool has_next = k + 1 < my_tiles;
      RunIter nx = cur;
      nx.next();
      const int64_t i0 = (int64_t)cur.I * TILE, j0 = (int64_t)cur.J * TILE;
      tc::mbar_wait(&sm.dfull, (uint32_t)(k & 1));
      tc::fence_after();
      rs_cons_sync();                                    // A: every consumer finished streaming tile k - 1
      if (ct < TILE) {
        if (k > 0) {                                     // row / column sums of tile k - 1 -> next iteration's degrees
          const float rs = sm.rowacc[ct], cs = sm.colacc[ct];
          const int64_t gi = (int64_t)Iprev * TILE + ct, gj = (int64_t)Jprev * TILE + ct;
          if (rs != 0.f) atomicAdd(fa.d_next + gi, rs);
          if (cs != 0.f) atomicAdd(fa.d_next + gj, cs);
          sm.rowacc[ct] = 0.f;
          sm.colacc[ct] = 0.f;
        }
        sm.rI[ct] = sm.nxt[0][ct]; sm.rJ[ct] = sm.nxt[1][ct]; sm.rhoI[ct] = sm.nxt[2][ct]; sm.rhoJ[ct] = sm.nxt[3][ct];
      }
      {  // drain: TMEM lane quarter qq, 32-column group cw / 4; hi + lo, 16 columns at a time
        const int cg = cw >> 2;
        const int row = qq * 32 + lane;
        const uint32_t taddr = tm + ((uint32_t)(qq * 32) << 16) + (uint32_t)(cg * 32);
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {
          float hi[16], lo[16];
          tc::tmem_ld16(taddr + c * 16, hi);
          tc::tmem_ld16(taddr + 128 + c * 16, lo);
#pragma unroll
          for (int u4 = 0; u4 < 4; ++u4)
            *reinterpret_cast<float4*>(&sm.u.gt[row][cg * 32 + c * 16 + u4 * 4]) =
                make_float4(hi[u4 * 4] + lo[u4 * 4], hi[u4 * 4 + 1] + lo[u4 * 4 + 1], hi[u4 * 4 + 2] + lo[u4 * 4 + 2],
                            hi[u4 * 4 + 3] + lo[u4 * 4 + 3]);
        }
      }
      if (has_next && nx.I != cur.I) load_A(nx.I);       // (the MMAs that read the old rows completed before dfull)
      tc::fence_before();
      __syncwarp();
      if (lane == 0) ws_arrive(&sm.dempty);              // the MMA warp may form the product of tile k + 1
      rs_cons_sync();                                    // B: product tile + node vectors visible
      if (has_next) load_consts(nx);                     // (deferring the shared-memory stores to the end of the tile measured slower)

      float* xt = tiles + (t_begin + k) * (int64_t)TILE_ELEMS;
      float* mt = mbuf + (t_begin + k) * (int64_t)TILE_ELEMS;
      float* vt = vbuf + (t_begin + k) * (int64_t)TILE_ELEMS;
      const bool interior = (cur.J < cur.I) && (i0 + TILE <= n);
      const float rj[2] = {sm.rJ[b0], sm.rJ[b0 + 1]};
      const float rhoj[2] = {sm.rhoJ[b0], sm.rhoJ[b0 + 1]};
      float s_sq = 0.f;
      float colp[2] = {0.f, 0.f};
#pragma unroll 1
      for (int ch = 0; ch < TILE / RS_R; ++ch) {
        tc::mbar_wait(&sm.sfull[s], ph);
        const float* b = &sm.ring[s][0][rw * TILE + b0];
        const float2 X = *reinterpret_cast<const float2*>(b);
        const float2 M = *reinterpret_cast<const float2*>(b + RS_CH);
        const float2 V = *reinterpret_cast<const float2*>(b + 2 * RS_CH);
        const float2 F = USE_F ? *reinterpret_cast<const float2*>(b + 3 * RS_CH) : make_float2(0.f, 0.f);
        __syncwarp();
        if (lane == 0) ws_arrive(&sm.sempty[s]);         // this warp's part of the stage is in registers
        if (++s == RS_S) { s = 0; ph ^= 1u; }
        const int a = ch * RS_R + rw;
        const float ri = sm.rI[a], rhoi = sm.rhoI[a];
        const float2 G = *reinterpret_cast<const float2*>(&sm.u.gt[a][b0]);
        const float xr[2] = {X.x, X.y}, ms[2] = {M.x, M.y}, vs[2] = {V.x, V.y}, fs[2] = {F.x, F.y}, gs[2] = {G.x, G.y};
        const float xs[2] = {LAZY ? __saturatef(xr[0] - mu) : xr[0], LAZY ? __saturatef(xr[1] - mu) : xr[1]};
        float xo[2], mo[2], vo[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float rirj = ri * rj[e];
          const float ah = rirj * xs[e];
          float esym = 0.f;
          if (MEAS == MCGRA_M_MSE) esym = fc.k1x4 * (ah - fs[e]);
          else if (MEAS == MCGRA_M_PRE) esym = fs[e];
          if (ENT && ah >= ENT_LO && ah <= ENT_HI) esym = fmaf(fc.k6x2, __log2f(ah) + INV_LN2, esym);
          float gg = fmaf(rirj, esym, rhoi + rhoj[e] + gs[e]);
          gg = fmaf(fc.norm_scale, xs[e], gg);
          const float mn = fmaf(fc.omb1, gg - ms[e], ms[e]);
          const float vn = fmaf(fc.omb2, gg * gg - vs[e], vs[e]);
          const float denom = fmaf(sqrt_approx(vn), fc.inv_sqrt_bc2, fc.adam_eps);
          const float xn = fmaf(fc.neg_step, __fdividef(mn, denom), xs[e]);
          const float c = __saturatef(xn);
          // diagonal / last-row tiles: entries on or above the diagonal and beyond n stay zero
          const bool valid = interior || ((j0 + b0 + e) < (i0 + a) && (i0 + a) < n);
          const float cv = valid ? c : 0.f;
          xo[e] = LAZY ? (valid ? xn : 0.f) : cv;
          mo[e] = valid ? mn : 0.f;
          vo[e] = valid ? vn : 0.f;
          s_sq = fmaf(cv, cv, s_sq);
          colp[e] += cv;
          if (LAZY && valid) { xmin = fminf(xmin, xn); xmax = fmaxf(xmax, xn); }
        }
        const float rowc = LAZY ? (__saturatef(xo[0]) + __saturatef(xo[1])) : (xo[0] + xo[1]);
        const int off = a * TILE + b0;
        // streaming (.cs) stores: nothing in this launch reads x', m, v back (with the two load policies: 10.54 -> 10.18 ms)
        __stcs(reinterpret_cast<float2*>(xt + off), make_float2(xo[0], xo[1]));
        __stcs(reinterpret_cast<float2*>(mt + off), make_float2(mo[0], mo[1]));
        __stcs(reinterpret_cast<float2*>(vt + off), make_float2(vo[0], vo[1]));
        const float rp = warp_sum(rowc);
        if (lane == 0 && rp != 0.f) atomicAdd(&sm.rowacc[a], rp);
      }
      if (colp[0] != 0.f) atomicAdd(&sm.colacc[b0], colp[0]);
      if (colp[1] != 0.f) atomicAdd(&sm.colacc[b0 + 1], colp[1]);
      d_sq += (double)s_sq;
      d_clamp += (double)(colp[0] + colp[1]);
      Iprev = cur.I; Jprev = cur.J;
      cur = nx;
    }
    rs_cons_sync();
    if (ct < TILE && my_tiles > 0) {
      const float rs = sm.rowacc[ct], cs = sm.colacc[ct];
      const int64_t gi = (int64_t)Iprev * TILE + ct, gj = (int64_t)Jprev * TILE + ct;
      if (rs != 0.f) atomicAdd(fa.d_next + gi, rs);
      if (cs != 0.f) atomicAdd(fa.d_next + gj, cs);
    }
    d_clamp = warp_sum_d(d_clamp);
    d_sq = warp_sum_d(d_sq);
    if (lane == 0) {
      atomicAdd(&sm.dsum[0], d_clamp);
      atomicAdd(&sm.dsum[1], d_sq);
    }
    rs_cons_sync();
    if (ct == 0) {
      if (sm.dsum[0] != 0.0) atomicAdd(fa.acc_next + MCGRA_ACC_SUMCLAMP, sm.dsum[0]);
      if (sm.dsum[1] != 0.0) atomicAdd(fa.acc_next + MCGRA_ACC_SUMSQ, sm.dsum[1]);
    }
    if (LAZY) {
      xmin = warp_min(xmin);
      xmax = warp_max(xmax);
      if (lane == 0) {
        if (xmin != INFINITY) atomic_min_f(minmax, xmin);
        if (xmax != -INFINITY) atomic_max_f(minmax + 1, xmax);
      }
    }
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tm, 512);
}

int g_fold_engine = 3;     // 0 = exact fp32 FFMA (reference of the agreement tests), 2 = tcgen05 one tile per CTA (k_fold_tc: every
                           // parameter view / measure), 3 = persistent row-run tcgen05 (k_fold_rs) for fast launches, k_fold_tc otherwise

// ---------------------------------------------------------------------------------------------------------
// Bisection on device.  state: [0]=a [1]=b [2]=mu(last midpoint) [3]=done [4]=active
// One pass evaluates the 7 midpoints of a depth-3 bisection tree rooted at (a,b); the update walks the tree
// with the reference's decision rule (func(miu)*func(a) < 0 -> b = miu else a = miu, func(a) > 0 invariant).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void bisect_candidates(float a, float b, float* c) {
  // heap order: c[0] root; children of node k are 2k+1 (left: (a, c_k)), 2k+2 (right: (c_k, b))
  float lo[7], hi[7];
  lo[0] = a; hi[0] = b;
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    c[k] = (lo[k] + hi[k]) / 2;          // fp32, same expression as the reference (:403)
    if (2 * k + 2 < 7) {
      lo[2 * k + 1] = lo[k]; hi[2 * k + 1] = c[k];
      lo[2 * k + 2] = c[k];  hi[2 * k + 2] = hi[k];
    }
  }
}

__global__ void k_bisect_init(const double* acc, const float* minmax, double budget, float* state, float* mu) {
  const bool active = acc[MCGRA_ACC_SUMCLAMP] > budget;       // :339
  state[0] = minmax[0] - 1.f;                                  // left  = (x-1).min()  (:340)
  state[1] = minmax[1];                                        // right = x.max()      (:341)
  state[2] = state[0];                                         // miu = a              (:401)
  state[3] = active ? 0.f : 1.f;
  state[4] = active ? 1.f : 0.f;
  *mu = 0.f;
}

__global__ void __launch_bounds__(256)
k_bisect_pass(const float* __restrict__ tiles, int64_t n, int64_t t0, float epsilon, const float* __restrict__ state,
              double* __restrict__ cand_sums) {
  __shared__ double red[32];
  if (state[3] != 0.f) return;                                 // done / inactive: nothing to read
  if (!((state[1] - state[0]) >= epsilon)) return;
  float c[7];
  bisect_candidates(state[0], state[1], c);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const float4* src = reinterpret_cast<const float4*>(tiles + (int64_t)blockIdx.x * TILE_ELEMS);
  float s[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const bool interior = (J < I) && (i0 + TILE <= n);
  // 16 float4 per thread, loaded in two batches of 8 before any arithmetic (the pass is otherwise latency / issue bound)
#pragma unroll 1
  for (int hb = 0; hb < 2; ++hb) {
    float4 xq[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) xq[u] = src[(hb * 8 + u) * 256 + threadIdx.x];
    if (interior) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const float xv[4] = {xq[u].x, xq[u].y, xq[u].z, xq[u].w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int q = 0; q < 7; ++q) s[q] += __saturatef(xv[k] - c[q]);
      }
    } else {
#pragma unroll 1
      for (int u = 0; u < 8; ++u) {
        const int e = (hb * 8 + u) * 256 + threadIdx.x;
        const int row = e >> 5, c4 = e & 31;
        const int64_t gi = i0 + row, gj = j0 + c4 * 4;
        const float4 x4 = src[e];
        const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if ((gj + k < gi) && (gi < n)) {
#pragma unroll
            for (int q = 0; q < 7; ++q) s[q] += __saturatef(xv[k] - c[q]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 7; ++q) block_atomic_add_d((double)s[q], cand_sums + q, red);
}

__global__ void k_bisect_update(double budget, float epsilon, float* state, double* cand_sums, float* mu) {
  if (state[3] == 0.f) {
    float a = state[0], b = state[1], miu = state[2];
    float c[7];
    bisect_candidates(a, b, c);
    int k = 0;
    bool done = false;
    for (int lvl = 0; lvl < 3; ++lvl) {
      if (!((b - a) >= epsilon)) { done = true; break; }      // while ((b - a) >= epsilon)  (:402)
      miu = c[k];
      const double f = cand_sums[k] - budget;                  // func(miu)            (:399)
      if (f == 0.0) { done = true; break; }                    // (:405)
      if (f < 0.0) { b = miu; k = 2 * k + 1; }                 // func(miu)*func(a) < 0 with func(a) > 0  (:408)
      else { a = miu; k = 2 * k + 2; }
    }
    if (!done && !((b - a) >= epsilon)) done = true;
    state[0] = a; state[1] = b; state[2] = miu;
    *mu = miu;               // always the last visited midpoint: an unfinished search still projects (never mu = 0)
    if (done) state[3] = 1.f;
  }
  for (int q = 0; q < 7; ++q) cand_sums[q] = 0.0;
}

// after the bisection: statistics of the projected parameter clamp(x' - mu, 0, 1)
__global__ void __launch_bounds__(256)
k_bisect_finish(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* __restrict__ state,
                const float* __restrict__ mu, double* __restrict__ acc_next, float* __restrict__ d_next) {
  __shared__ float colacc[TILE];
  __shared__ float rowpart[TILE][33];                          // per-lane row sums, summed once per tile
  __shared__ double red[32];
  if (state[4] == 0.f) return;                                 // projection inactive: fold's statistics stand
  const float m = *mu;
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const float4* src = reinterpret_cast<const float4*>(tiles + (int64_t)blockIdx.x * TILE_ELEMS);
  if (tid < TILE) colacc[tid] = 0.f;
  const bool interior = (J < I) && (i0 + TILE <= n);
  float col[4] = {0.f, 0.f, 0.f, 0.f};
  float ssq = 0.f;
#pragma unroll 1
  for (int hb = 0; hb < 2; ++hb) {                             // rows (hb * 8 + u) * 8 + warp, 8 loads in flight per thread
    float4 xq[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) xq[u] = src[((hb * 8 + u) * 8 + warp) * 32 + lane];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int row = (hb * 8 + u) * 8 + warp;
      const int64_t gi = i0 + row, gj = j0 + lane * 4;
      const float xv[4] = {xq[u].x, xq[u].y, xq[u].z, xq[u].w};
      float rs = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (interior || ((gj + k < gi) && (gi < n))) {
          const float c = __saturatef(xv[k] - m);
          rs += c;
          col[k] += c;
          ssq = fmaf(c, c, ssq);
        }
      }
      rowpart[row][lane] = rs;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (col[k] != 0.f) atomicAdd(&colacc[lane * 4 + k], col[k]);
  if (tid < TILE) {
    float rs = 0.f;
#pragma unroll 8
    for (int l = 0; l < 32; ++l) rs += rowpart[tid][l];
    if (i0 + tid < n && rs != 0.f) atomicAdd(d_next + i0 + tid, rs);
  }
  __syncthreads();
  if (tid < TILE && j0 + tid < n && colacc[tid] != 0.f) atomicAdd(d_next + j0 + tid, colacc[tid]);
  block_atomic_add_d((double)ssq, acc_next + MCGRA_ACC_SUMSQ, red);
}

__global__ void k_bisect_reset(int64_t n, const float* state, double* acc_next, float* d_next) {
  if (state[4] == 0.f) return;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d_next[i] = 1.f;
  if (i == 0) acc_next[MCGRA_ACC_SUMSQ] = 0.0;
}

}  // namespace

extern "C" {

int g_fold_ws_grid = 0;     // test knob: cap on the persistent grid (0 = one CTA per SM), mcgra_set_engine(1, 100 + cap)
int mcgra_set_fold_engine_(int value) {
  if (value >= 100 && value < 1000) g_fold_ws_grid = value - 100;
  else if (value == 0 || value == 2 || value == 3) g_fold_engine = value;
  else return -1;
  return 0;
}

int64_t mcgra_fold_ws_bytes(int64_t n) { return ((n + TILE - 1) / TILE) * (int64_t)WBLOCK + 256; }

int mcgra_fold_adam(float* tiles, float* m, float* v, int tr0, int tr1, const float* mu, int raw,
                    const mcgra_fold_args* a, float* minmax, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  const bool lazy = raw == 0 && !a->store_clamped;        // un-projected buffer + mu (the budget may bind)
  const bool fastable = ((raw == 2 && a->store_clamped) || lazy) && a->k2 == 0.f && a->measure != MCGRA_M_KL && !a->plain_gd &&
                        a->Gtiles == nullptr && !(a->measure != MCGRA_M_NONE && a->Ftiles == nullptr);
  if (g_fold_engine == 3 && a->Wk != nullptr && fastable) {
    const int64_t np = a->npad;
    k_prep_w<<<(unsigned)((np * 128 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a->Wt, np, (unsigned char*)a->Wk);
    static int sms = 0;
    if (sms == 0) {
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    const int cap = g_fold_ws_grid > 0 ? g_fold_ws_grid : sms;
    const unsigned grid = (unsigned)(nt < cap ? nt : cap);
    const size_t smem4 = sizeof(FoldRsSmem) + 1024;
    const unsigned char* wk = (const unsigned char*)a->Wk;
    cudaError_t e4 = cudaSuccess;
#define MCGRA_FOLD_RS_(MEAS, ENT, LZ)                                                                                 \
  e4 = cudaFuncSetAttribute(k_fold_rs<MEAS, ENT, LZ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4);       \
  if (e4 != cudaSuccess) return (int)e4;                                                                              \
  k_fold_rs<MEAS, ENT, LZ><<<grid, RS_THREADS, smem4, (cudaStream_t)stream>>>(tiles, m, v, tr0, nt, *a, wk, mu, minmax)
#define MCGRA_FOLD_RS(MEAS, ENT)                                                                                      \
  if (lazy) { MCGRA_FOLD_RS_(MEAS, ENT, true); } else { MCGRA_FOLD_RS_(MEAS, ENT, false); }
    if (a->measure == MCGRA_M_MSE) {
      if (a->k6 != 0.f) { MCGRA_FOLD_RS(MCGRA_M_MSE, true); } else { MCGRA_FOLD_RS(MCGRA_M_MSE, false); }
    } else if (a->measure == MCGRA_M_PRE) {
      if (a->k6 != 0.f) { MCGRA_FOLD_RS(MCGRA_M_PRE, true); } else { MCGRA_FOLD_RS(MCGRA_M_PRE, false); }
    } else {
      if (a->k6 != 0.f) { MCGRA_FOLD_RS(MCGRA_M_NONE, true); } else { MCGRA_FOLD_RS(MCGRA_M_NONE, false); }
    }
#undef MCGRA_FOLD_RS
#undef MCGRA_FOLD_RS_
    MCGRA_LAUNCH_CHECK();
    return 0;
  }
  if (g_fold_engine >= 2 && a->Wk != nullptr) {
    const int64_t np = a->npad;
    k_prep_w<<<(unsigned)((np * 128 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a->Wt, np, (unsigned char*)a->Wk);
    const size_t smem3 = sizeof(FoldTcSmem) + 1024;
    cudaError_t e3 = cudaFuncSetAttribute(k_fold_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3);
    if (e3 != cudaSuccess) return (int)e3;
    k_fold_tc<<<(unsigned)nt, 256, smem3, (cudaStream_t)stream>>>(tiles, m, v, tr0, tr1, mu, raw, *a, minmax,
                                                                  (const unsigned char*)a->Wk);
    MCGRA_LAUNCH_CHECK();
    return 0;
  }
  const size_t smem = sizeof(FoldSmem);
  cudaError_t e = cudaFuncSetAttribute(k_fold_adam, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_fold_adam<<<(unsigned)nt, 256, smem, (cudaStream_t)stream>>>(tiles, m, v, tri(tr0), mu, raw, *a, minmax);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_bisect_init(const double* acc, const float* minmax, double budget, float* state, float* mu, void* stream) {
  k_bisect_init<<<1, 1, 0, (cudaStream_t)stream>>>(acc, minmax, budget, state, mu);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_bisect_pass(const float* tiles, int64_t n, int tr0, int tr1, float epsilon, const float* state,
                      double* cand_sums, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_bisect_pass<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), epsilon, state, cand_sums);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_bisect_update(double budget, float epsilon, float* state, double* cand_sums, float* mu, void* stream) {
  k_bisect_update<<<1, 1, 0, (cudaStream_t)stream>>>(budget, epsilon, state, cand_sums, mu);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_bisect_finish(const float* tiles, int64_t n, int tr0, int tr1, const float* state, const float* mu,
                        double* acc_next, float* d_next, int reset, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (reset) {
    k_bisect_reset<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, state, acc_next, d_next);
    MCGRA_LAUNCH_CHECK();
  }
  if (nt <= 0) return 0;
  k_bisect_finish<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), state, mu, acc_next, d_next);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
