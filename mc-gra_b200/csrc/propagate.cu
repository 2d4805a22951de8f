// Propagation over the tiled symmetric adjacency estimate: degree, Y += M*B, row sum-exp.
//
// Reference work replaced: GraphConvolution.forward's torch.spmm(adj, support) (MC-GRA/models/gcn.py:42) and its
// transposed product in autograd, the row sums of utils.normalize_adj_tensor (MC-GRA/utils.py:224-225), and the
// element-wise loss terms c1 (MSE/KL vs feature_adj) and c6 (Info_entropy) over A_hat
// (MC-GRA/topology_attack.py:212-232, 44-47), computed by a stand-alone streaming pass ahead of the first propagation.
//
// Tile-symmetric schedule: one CTA per 128x128 tile (I,J) of the lower triangle.  The tile is read from HBM once
// and used twice:  Y[I rows] += T * B[J rows]  and  Y[J rows] += T^T * B[I rows].  The unnormalised / normalised
// n x n matrices are never materialised: the D^-1/2 scaling lives in the B operand (prologue, node kernels) and in
// the consumers of Y (epilogue, node kernels).
//
// Engines (mcgra_set_engine(0, v); DESIGN.md 3.1), all with HBM traffic = one read of the tile shard (4 bytes per stored
// entry) + O(n K):
//   0  k_propagate        fp32 FFMA, 2 x K register tile per thread (exact fp32; the reference of the agreement tests)
//   5  k_propagate_h      both products on tcgen05 kind::f16 from ONE fp16x2 image per tile (K-major for the direct,
//                         MN-major for the mirrored product); DEFAULT
// plus k_elem_stats (the element-wise terms as a stand-alone streaming pass), k_degree, k_row_sumexp.
#include <cuda_fp16.h>
#include <type_traits>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

constexpr int XS_LD = TILE + 4;   // padded row stride (floats): LDS.128 along a row is conflict free

template <int KC>
struct PropSmem {
  float xs[TILE][XS_LD];
  float bj[TILE][KC];
  float bi[TILE][KC];
};

template <int KC>
__global__ void __launch_bounds__(128, 2)
k_propagate(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
            const float* __restrict__ B, float* __restrict__ Y, int products) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PropSmem<KC>& sm = *reinterpret_cast<PropSmem<KC>*>(smem_raw);
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const float4* src = reinterpret_cast<const float4*>(tiles + (int64_t)blockIdx.x * TILE_ELEMS);

  // ---- stage B rows of both sides -------------------------------------------------------------------------
  for (int e = tid; e < TILE * KC / 4; e += 128) {
    const int row = e / (KC / 4), c4 = e % (KC / 4);
    float4 vj = make_float4(0.f, 0.f, 0.f, 0.f), vi = vj;
    if (j0 + row < n) vj = reinterpret_cast<const float4*>(B + (j0 + row) * KC)[c4];
    if (i0 + row < n) vi = reinterpret_cast<const float4*>(B + (i0 + row) * KC)[c4];
    reinterpret_cast<float4*>(&sm.bj[row][0])[c4] = vj;
    reinterpret_cast<float4*>(&sm.bi[row][0])[c4] = vi;
  }

  // ---- stage the tile (one warp = one 512 B row per step) ------------------------------------------------
#pragma unroll 4
  for (int it = 0; it < 32; ++it) {
    const int row = it * 4 + warp;
    const float4 raw4 = src[row * 32 + lane];
    const int64_t gi = i0 + row;
    const int64_t gj = j0 + lane * 4;
    float xv[4] = {raw4.x, raw4.y, raw4.z, raw4.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) xv[k] = ((gj + k < gi) && (gi < n)) ? pv.adj(xv[k]) : 0.f;
    *reinterpret_cast<float4*>(&sm.xs[row][lane * 4]) = make_float4(xv[0], xv[1], xv[2], xv[3]);
  }
  __syncthreads();

  // ---- compute: warps 0-1 direct product (rows of I), warps 2-3 mirrored product (rows of J) -------------
  const int u = tid & 63;
  // product selector (MCGRA_PROD_*): warps 0-1 carry the direct product, warps 2-3 the mirrored one
  if (!(products & (warp < 2 ? MCGRA_PROD_DIRECT : MCGRA_PROD_MIRRORED))) return;
  float acc0[KC], acc1[KC];
#pragma unroll
  for (int c = 0; c < KC; ++c) acc0[c] = acc1[c] = 0.f;

  if (warp < 2) {
    // Y[i0+u], Y[i0+u+64] += sum_b xs[u][b] * bj[b][:]
#pragma unroll 1
    for (int b = 0; b < TILE; b += 4) {
      const float4 xa = *reinterpret_cast<const float4*>(&sm.xs[u][b]);
      const float4 xb = *reinterpret_cast<const float4*>(&sm.xs[u + 64][b]);
      const float xa_[4] = {xa.x, xa.y, xa.z, xa.w};
      const float xb_[4] = {xb.x, xb.y, xb.z, xb.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int c4 = 0; c4 < KC / 4; ++c4) {
          const float4 bv = *reinterpret_cast<const float4*>(&sm.bj[b + k][c4 * 4]);
          acc0[c4 * 4 + 0] = fmaf(xa_[k], bv.x, acc0[c4 * 4 + 0]);
          acc0[c4 * 4 + 1] = fmaf(xa_[k], bv.y, acc0[c4 * 4 + 1]);
          acc0[c4 * 4 + 2] = fmaf(xa_[k], bv.z, acc0[c4 * 4 + 2]);
          acc0[c4 * 4 + 3] = fmaf(xa_[k], bv.w, acc0[c4 * 4 + 3]);
          acc1[c4 * 4 + 0] = fmaf(xb_[k], bv.x, acc1[c4 * 4 + 0]);
          acc1[c4 * 4 + 1] = fmaf(xb_[k], bv.y, acc1[c4 * 4 + 1]);
          acc1[c4 * 4 + 2] = fmaf(xb_[k], bv.z, acc1[c4 * 4 + 2]);
          acc1[c4 * 4 + 3] = fmaf(xb_[k], bv.w, acc1[c4 * 4 + 3]);
        }
      }
    }
  } else {
    // Y[j0+u], Y[j0+u+64] += sum_a xs[a][u] * bi[a][:]
#pragma unroll 1
    for (int a = 0; a < TILE; a += 4) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float xa = sm.xs[a + k][u];
        const float xb = sm.xs[a + k][u + 64];
#pragma unroll
        for (int c4 = 0; c4 < KC / 4; ++c4) {
          const float4 bv = *reinterpret_cast<const float4*>(&sm.bi[a + k][c4 * 4]);
          acc0[c4 * 4 + 0] = fmaf(xa, bv.x, acc0[c4 * 4 + 0]);
          acc0[c4 * 4 + 1] = fmaf(xa, bv.y, acc0[c4 * 4 + 1]);
          acc0[c4 * 4 + 2] = fmaf(xa, bv.z, acc0[c4 * 4 + 2]);
          acc0[c4 * 4 + 3] = fmaf(xa, bv.w, acc0[c4 * 4 + 3]);
          acc1[c4 * 4 + 0] = fmaf(xb, bv.x, acc1[c4 * 4 + 0]);
          acc1[c4 * 4 + 1] = fmaf(xb, bv.y, acc1[c4 * 4 + 1]);
          acc1[c4 * 4 + 2] = fmaf(xb, bv.z, acc1[c4 * 4 + 2]);
          acc1[c4 * 4 + 3] = fmaf(xb, bv.w, acc1[c4 * 4 + 3]);
        }
      }
    }
  }

  // ---- flush: vector reductions into Y ---------------------------------------------------------------------
  {
    const int64_t base = (warp < 2) ? i0 : j0;
    const int64_t r0 = base + u, r1 = base + u + 64;
    if (r0 < n) {
      float4* dst = reinterpret_cast<float4*>(Y + r0 * KC);
#pragma unroll
      for (int c4 = 0; c4 < KC / 4; ++c4)
        atomicAdd(dst + c4, make_float4(acc0[c4 * 4], acc0[c4 * 4 + 1], acc0[c4 * 4 + 2], acc0[c4 * 4 + 3]));
    }
    if (r1 < n) {
      float4* dst = reinterpret_cast<float4*>(Y + r1 * KC);
#pragma unroll
      for (int c4 = 0; c4 < KC / 4; ++c4)
        atomicAdd(dst + c4, make_float4(acc1[c4 * 4], acc1[c4 * 4 + 1], acc1[c4 * 4 + 2], acc1[c4 * 4 + 3]));
    }
  }
}

// degree: one CTA per tile, 128 threads, row sums through warp shuffles, column sums in registers
__global__ void __launch_bounds__(128)
k_degree(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw, float* __restrict__ d) {
  __shared__ float colacc[TILE];
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const float4* src = reinterpret_cast<const float4*>(tiles + (int64_t)blockIdx.x * TILE_ELEMS);
  colacc[tid] = 0.f;
  __syncthreads();
  float col[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
  for (int it = 0; it < 32; ++it) {
    const int row = it * 4 + warp;
    const float4 raw4 = src[row * 32 + lane];
    const int64_t gi = i0 + row, gj = j0 + lane * 4;
    const float xv[4] = {raw4.x, raw4.y, raw4.z, raw4.w};
    float rs = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float a = ((gj + k < gi) && (gi < n)) ? pv.adj(xv[k]) : 0.f;
      rs += a;
      col[k] += a;
    }
    rs = warp_sum(rs);
    if (lane == 0 && gi < n && rs != 0.f) atomicAdd(d + gi, rs);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) atomicAdd(&colacc[lane * 4 + k], col[k]);
  __syncthreads();
  if (j0 + tid < n && colacc[tid] != 0.f) atomicAdd(d + j0 + tid, colacc[tid]);
}

// sumexp[i] += sum_{j != i, valid} exp(r_i M_ij r_j)   (both orientations of every stored entry)
__global__ void __launch_bounds__(128)
k_row_sumexp(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw,
             const float* __restrict__ r, float* __restrict__ sumexp) {
  __shared__ float colacc[TILE], rI[TILE], rJ[TILE];
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  const float4* src = reinterpret_cast<const float4*>(tiles + (int64_t)blockIdx.x * TILE_ELEMS);
  colacc[tid] = 0.f;
  rI[tid] = i0 + tid < n ? r[i0 + tid] : 0.f;
  rJ[tid] = j0 + tid < n ? r[j0 + tid] : 0.f;
  __syncthreads();
  float col[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
  for (int it = 0; it < 32; ++it) {
    const int row = it * 4 + warp;
    const float4 raw4 = src[row * 32 + lane];
    const int64_t gi = i0 + row, gj = j0 + lane * 4;
    const float xv[4] = {raw4.x, raw4.y, raw4.z, raw4.w};
    float rs = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if ((gj + k < gi) && (gi < n)) {
        const float e = __expf(rI[row] * pv.adj(xv[k]) * rJ[lane * 4 + k]);
        rs += e;
        col[k] += e;
      }
    }
    rs = warp_sum(rs);
    if (lane == 0 && gi < n && rs != 0.f) atomicAdd(sumexp + gi, rs);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) atomicAdd(&colacc[lane * 4 + k], col[k]);
  __syncthreads();
  if (j0 + tid < n && colacc[tid] != 0.f) atomicAdd(sumexp + j0 + tid, colacc[tid]);
}


// ---------------------------------------------------------------------------------------------------------
// v5 engine: both products on tcgen05 kind::f16 from ONE staged image per tile, no transposition pass.
//
// Measured on B200 (tools/umma_rate.cu): one tcgen05.mma costs a fixed ~110-140 clk for kind::tf32 (K = 8) and ~60 clk for
// kind::f16 (K = 16) for every N <= 128, so the tf32 engines are bound by their 64 MMA instructions per tile
// (~6-8k clk against an HBM floor of 2.8k clk per tile).  16-bit operands need a quarter of that, and -- unlike tf32 --
// 16-bit operands may be MN-major without swizzle, so the SAME shared-memory image serves the direct product as a
// K-major A operand (M = tile row, K = tile column) and the mirrored product as an MN-major A operand (M = tile
// column, K = tile row) (tools/umma_test16.cu).
//
// Precision (fp16 x 2 on both sides, fp32 accumulation, ~2^-22 like 3xTF32):
//   tile entry  x in [0, 1]:   h0 = fp16(x),  h1 = fp16((x - h0) * 2^11)
//   feature     f (column c):  g = f * s_c (s_c = power of two with max_c |g| < 2^14),  g0 = fp16(g), g1 = fp16((g - g0) * 2^11)
//   D[:, 0:2KC] += h0 * [g0 | g1]      D[:, 2KC:3KC] += h1 * g0       y_c = (d0 + (d1 + d2) * 2^-11) / s_c
// (mixed f16 x bf16 operands are rejected by the hardware; bf16 x 3 would need 3 planes and 48 MMAs per tile).
//
// Plane image: element (i, j) at (j/8)*H_SJ + (i/8)*128 + (i%8)*16 + (j%8)*2, two planes per tile, two tile buffers.
// Warps 0-7 convert their prefetched registers into the planes, arrive on ready[b], prefetch the tile after next and
// flush the mirrored result of the previous tile; warp 8 (one lane) issues the 32 MMAs of a tile and nothing else -- a
// clock64 trace showed its serial instruction stream to be the bound of the kernel (2.6 k clk of MMA issue + 1.9 k clk of
// cp.async B-block loading per tile for an HBM time of 2.7 k clk) -- and warp 9 (one lane) streams the pre-formatted B[J]
// blocks with one cp.async.bulk each into a ring of three.  With the issuer freed, the converters' own chain (convert +
// flush of the previous tile, 3-3.4 k clk) became the bound, so the flush moved to warps 8-11; registers are re-partitioned
// with setmaxnreg (converters keep two prefetched tiles in registers, everything else needs few).  TMEM columns: D1 (even tiles) [0, 3KC) | D1 (odd tiles) [96, 96+3KC) | D2[0] [192, 192+3KC) | D2[1] [288, 288+3KC).
// ---------------------------------------------------------------------------------------------------------
constexpr int H_RUN = 64;
constexpr uint32_t H_SJ = 16 * 128 + 16;           // stride between 8-column groups of a plane (padded: conflict-free stores)
constexpr uint32_t H_PLANE = 16 * H_SJ;

template <int KC>
struct PropHSmem {
  unsigned char tile[2][2][H_PLANE];               // [buffer][plane h0 / h1]
  unsigned char bkJ[3][16 * (2 * KC) * 16];        // 16 K-groups x (2KC rows [g0 | g1] x 16 B); ring of 3
  unsigned char bkI[16 * (2 * KC) * 16];
  uint64_t ready[2], tile_done[2], flushed[2];
  uint64_t bfull[3], bfree[3], bIfull;           // B-block ring (bulk copies by the loader warp)
  float inv_s[32];
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N, int a_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                          // D = F32; A = B = F16 (format 0)
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}

// column scales: maxbits[c] = bits of max_i |B[i][c]|
template <int KC>
__global__ void k_colmax(const float* __restrict__ B, int64_t n, unsigned int* __restrict__ maxbits) {
  const int c = threadIdx.x % KC;
  float m = 0.f;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n * KC; e += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(B[e]));
  if (m > 0.f) atomicMax(maxbits + c, __float_as_uint(m));
}
__device__ __forceinline__ float h_col_scale(unsigned int maxbits) {     // power of two s with max * s < 2^14
  if (maxbits == 0u) return 1.f;
  int e = (int)((maxbits >> 23) & 0xffu) - 127;                          // max < 2^(e+1)
  int se = 13 - e;
  se = se > 126 ? 126 : (se < -126 ? -126 : se);
  return __uint_as_float((uint32_t)(se + 127) << 23);
}
// B (n x KC fp32) -> per node tile a K-major [g0 | g1] fp16 block; scale[0:KC] = s_c, scale[KC:2KC] = 1 / s_c
template <int KC>
__global__ void k_prep_b16(const float* __restrict__ B, int64_t n, int64_t npad, const unsigned int* __restrict__ maxbits,
                           unsigned char* __restrict__ Bk, float* __restrict__ scale) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= npad * KC) return;
  const int64_t node = e / KC;
  const int c = (int)(e % KC);
  const float s = h_col_scale(maxbits[c]);
  if (node == 0) { scale[c] = s; scale[KC + c] = 1.f / s; }
  const float g = node < n ? B[e] * s : 0.f;
  const __half g0 = __float2half_rn(g);
  const __half g1 = __float2half_rn((g - __half2float(g0)) * 2048.f);
  const int k = (int)(node & 127);
  unsigned char* blk = Bk + (node >> 7) * (int64_t)(16 * (2 * KC) * 16) + (uint32_t)(k >> 3) * (uint32_t)((2 * KC) * 16) + (uint32_t)(k & 7) * 2u;
  *reinterpret_cast<__half*>(blk + (uint32_t)(c >> 3) * 128u + (uint32_t)(c & 7) * 16u) = g0;
  const int c2 = c + KC;
  *reinterpret_cast<__half*>(blk + (uint32_t)(c2 >> 3) * 128u + (uint32_t)(c2 & 7) * 16u) = g1;
}

// one chunk (4 consecutive tile columns of a row) -> 8 bytes of each fp16 plane
__device__ __forceinline__ void h_convert_store(float x0, float x1, float x2, float x3, unsigned char* p0, unsigned char* p1) {
  const __half2 a01 = __floats2half2_rn(x0, x1), a23 = __floats2half2_rn(x2, x3);
  const float2 f01 = __half22float2(a01), f23 = __half22float2(a23);
  const __half2 r01 = __floats2half2_rn((x0 - f01.x) * 2048.f, (x1 - f01.y) * 2048.f);
  const __half2 r23 = __floats2half2_rn((x2 - f23.x) * 2048.f, (x3 - f23.y) * 2048.f);
  *reinterpret_cast<uint2*>(p0) = make_uint2(*reinterpret_cast<const uint32_t*>(&a01), *reinterpret_cast<const uint32_t*>(&a23));
  *reinterpret_cast<uint2*>(p1) = make_uint2(*reinterpret_cast<const uint32_t*>(&r01), *reinterpret_cast<const uint32_t*>(&r23));
}
// register-array element by run-time index without local memory (rolled generic path)
__device__ __forceinline__ float4 h_pick(const float4 (&a)[16], int it) {
  float4 v = a[0];
#pragma unroll
  for (int u = 1; u < 16; ++u) if (it == u) v = a[u];
  return v;
}

// y[row][c0 + 0..15] += (d0 + (d1 + d2) * 2^-11) * inv_s   for 16 feature columns of one accumulator
template <int KC>
__device__ __forceinline__ void h_flush(float* __restrict__ Y, int64_t n, int64_t row, uint32_t taddr, int c0, const float* inv_s) {
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    uint32_t d0[8], d1[8], d2[8];
    const int c = c0 + half * 8;
    tc::tmem_ld8_nowait(taddr + c, d0);
    tc::tmem_ld8_nowait(taddr + KC + c, d1);
    tc::tmem_ld8_nowait(taddr + 2 * KC + c, d2);
    tc::tmem_ld_wait();
    if (row < n) {
      float4* dst = reinterpret_cast<float4*>(Y + row * KC + c);
      const float* is = inv_s + half * 8;
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u)
        v[u] = (__uint_as_float(d0[u]) + (__uint_as_float(d1[u]) + __uint_as_float(d2[u])) * (1.f / 2048.f)) * is[u];
      atomicAdd(dst, make_float4(v[0], v[1], v[2], v[3]));
      atomicAdd(dst + 1, make_float4(v[4], v[5], v[6], v[7]));
    }
  }
}

constexpr int H_THREADS = 512;      // 4 warpgroups: converters (2), flushers, MMA issuer + B loader (+ 2 idle warps)
// the same for the sum of two accumulators (the run's direct result is split over the two MMA-issuing lanes)
template <int KC>
__device__ __forceinline__ void h_flush2(float* __restrict__ Y, int64_t n, int64_t row, uint32_t ta, uint32_t tb, int c0, const float* inv_s) {
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    uint32_t a0[8], a1[8], a2[8], b0[8], b1[8], b2[8];
    const int c = c0 + half * 8;
    tc::tmem_ld8_nowait(ta + c, a0);
    tc::tmem_ld8_nowait(ta + KC + c, a1);
    tc::tmem_ld8_nowait(ta + 2 * KC + c, a2);
    tc::tmem_ld8_nowait(tb + c, b0);
    tc::tmem_ld8_nowait(tb + KC + c, b1);
    tc::tmem_ld8_nowait(tb + 2 * KC + c, b2);
    tc::tmem_ld_wait();
    if (row < n) {
      float4* dst = reinterpret_cast<float4*>(Y + row * KC + c);
      const float* is = inv_s + half * 8;
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u)
        v[u] = ((__uint_as_float(a0[u]) + __uint_as_float(b0[u])) +
                ((__uint_as_float(a1[u]) + __uint_as_float(b1[u])) + (__uint_as_float(a2[u]) + __uint_as_float(b2[u]))) * (1.f / 2048.f)) * is[u];
      atomicAdd(dst, make_float4(v[0], v[1], v[2], v[3]));
      atomicAdd(dst + 1, make_float4(v[4], v[5], v[6], v[7]));
    }
  }
}

template <int KC>
__global__ void __launch_bounds__(H_THREADS, 1)
k_propagate_h(const float* __restrict__ tiles, int64_t n, int tr0, const float* mu, int raw,
              const unsigned char* __restrict__ Bk, const float* __restrict__ scale, float* __restrict__ Y,
              int products) {
  const int I = tr0 + (int)blockIdx.y;
  const int Jbeg = (int)blockIdx.x * H_RUN;
  if (Jbeg > I) return;
  const int Jend = min(I + 1, Jbeg + H_RUN);
  const int nt = Jend - Jbeg;
  // the tiles of a run are visited in a rotated order (start depends on the tile row) so that concurrently resident
  // CTAs of neighbouring tile rows do not add their mirrored results to the same rows of Y at the same time
  const int rot = (I * 5) % nt;
  auto tile_of = [&](int k) { const int r = k + rot; return Jbeg + (r >= nt ? r - nt : r); };
  extern __shared__ __align__(128) unsigned char smem_raw[];
  PropHSmem<KC>& sm = *reinterpret_cast<PropHSmem<KC>*>(smem_raw);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE;
  constexpr uint32_t LBO_B = (2 * KC) * 16;
  constexpr uint32_t BLK = 16 * LBO_B;
  constexpr uint32_t COL_D1 = 0, COL_D2 = 192;    // D1 of the even / odd tiles at 0 / 96, D2[b] at 192 + 96 b
  const bool tcwarp = warp == 12 || warp == 14;   // two issuing lanes: even / odd tiles of the run
  const bool rows_ok = (i0 + TILE <= n) && (pv.raw == 2);
  const bool do_dir = (products & MCGRA_PROD_DIRECT) != 0, do_mir = (products & MCGRA_PROD_MIRRORED) != 0;
  const int64_t tix0 = tri((int64_t)I) - tri((int64_t)tr0);

  if (warp == 0) tc::tmem_alloc(&sm.tmem_base, 512);
  if (tid == 0) {
    tc::mbar_init(&sm.ready[0], 256); tc::mbar_init(&sm.ready[1], 256);
    tc::mbar_init(&sm.tile_done[0], 1); tc::mbar_init(&sm.tile_done[1], 1);
    tc::mbar_init(&sm.flushed[0], 128); tc::mbar_init(&sm.flushed[1], 128);
    for (int r = 0; r < 3; ++r) { tc::mbar_init(&sm.bfull[r], 1); tc::mbar_init(&sm.bfree[r], 1); }
    tc::mbar_init(&sm.bIfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid >= 32 && tid < 32 + KC) sm.inv_s[tid - 32] = scale[KC + tid - 32];
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tm = sm.tmem_base;

  if (warp >= 12) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(48));
  if (warp == 13) {
    // =================================== B-block loader ===================================
    if (lane == 0) {
      tc::mbar_expect_tx(&sm.bIfull, BLK);
      tc::bulk_g2s(sm.bkI, Bk + (int64_t)I * BLK, BLK, &sm.bIfull);
      for (int k = 0; k < nt; ++k) {
        const int r = k % 3;
        if (k >= 3) tc::mbar_wait_backoff(&sm.bfree[r], (uint32_t)((k / 3 - 1) & 1));     // MMAs of tile k-3 have read slot r
        tc::mbar_expect_tx(&sm.bfull[r], BLK);
        tc::bulk_g2s(sm.bkJ[r], Bk + (int64_t)tile_of(k) * BLK, BLK, &sm.bfull[r]);
      }
    }
  } else if (tcwarp) {
    // =================================== MMA issuers ===================================
    // Two lanes (warps 12 and 14) take the even / odd tiles of the run: the barrier round trips of one overlap the MMA issue
    // of the other (a single lane spent ~0.75 k clk per tile in them next to ~3 k clk of issue).  Each accumulates the direct
    // result of its tiles in its own D1 (summed by the final flush); D2[b] belongs to parity b anyway.
    if (lane == 0) {
      const int par = (warp - 12) >> 1;
      const uint32_t id_cat = make_idesc_f16(128, 2 * KC, 0), id_one = make_idesc_f16(128, KC, 0);
      const uint32_t id_cat_t = make_idesc_f16(128, 2 * KC, 1), id_one_t = make_idesc_f16(128, KC, 1);
      const uint64_t bI0 = tc::make_desc(tc::smem_u32(sm.bkI), LBO_B, 128u);
      const uint32_t d1 = tm + COL_D1 + (uint32_t)par * 96u, d2 = tm + COL_D2 + (uint32_t)par * 96u;
      tc::mbar_wait(&sm.bIfull, 0u);
      for (int k = par; k < nt; k += 2) {
        const int b = par, r = k % 3;
        tc::mbar_wait(&sm.bfull[r], (uint32_t)((k / 3) & 1));
        tc::mbar_wait(&sm.ready[b], (uint32_t)((k >> 1) & 1));
        if (k >= 2) tc::mbar_wait(&sm.flushed[b], (uint32_t)(((k - 2) >> 1) & 1));   // D2[b] of tile k-2 has been read
        tc::fence_after();
        const uint32_t p0 = tc::smem_u32(sm.tile[b][0]), p1 = tc::smem_u32(sm.tile[b][1]);
        const uint64_t bJ0 = tc::make_desc(tc::smem_u32(sm.bkJ[r]), LBO_B, 128u);
#pragma unroll 2
        for (int ks = 0; ks < TILE / 16; ++ks) {
          const uint64_t db = (uint64_t)((uint32_t)ks * ((2u * LBO_B) >> 4));
          const uint32_t acc1 = (k > par || ks > 0) ? 1u : 0u, acc2 = ks > 0 ? 1u : 0u;
          // direct: A K-major (M = row: SBO 128 between 8-row groups; K = column: LBO H_SJ between 8-column groups)
          if (do_dir) {
            mma_f16(d1, tc::make_desc(p0 + (uint32_t)ks * 2u * H_SJ, H_SJ, 128u), bJ0 + db, id_cat, acc1);
            mma_f16(d1 + 2 * KC, tc::make_desc(p1 + (uint32_t)ks * 2u * H_SJ, H_SJ, 128u), bJ0 + db, id_one, acc1);
          }
          // mirrored: the same image as an MN-major A operand (M = column: SBO H_SJ; K = row: LBO 128)
          if (do_mir) {
            mma_f16(d2, tc::make_desc(p0 + (uint32_t)ks * 256u, 128u, H_SJ), bI0 + db, id_cat_t, acc2);
            mma_f16(d2 + 2 * KC, tc::make_desc(p1 + (uint32_t)ks * 256u, 128u, H_SJ), bI0 + db, id_one_t, acc2);
          }
        }
        tc::mma_commit(&sm.tile_done[b]);
        tc::mma_commit(&sm.bfree[r]);
      }
    }
  } else if (warp >= 8 && warp < 12) {
    // =================================== flusher warps ===================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(72));
    const int q = warp & 3;                              // TMEM lane quarter (= warp % 4)
    const int ltid = q * 32 + lane;
    const uint32_t tlane = tm + ((uint32_t)(q * 32) << 16);
    for (int k = 0; k < nt; ++k) {
      const int b = k & 1;
      tc::mbar_wait(&sm.tile_done[b], (uint32_t)((k >> 1) & 1));
      tc::fence_after();
      if (do_mir) {
#pragma unroll
        for (int cg = 0; cg < KC / 16; ++cg)
          h_flush<KC>(Y, n, (int64_t)tile_of(k) * TILE + ltid, tlane + COL_D2 + (uint32_t)b * 96u, cg * 16, sm.inv_s + cg * 16);
      }
      tc::fence_before();
      mbar_arrive(&sm.flushed[b]);
    }
    if (do_dir) {                                        // the run's direct result (complete with the last tile_done)
#pragma unroll
      for (int cg = 0; cg < KC / 16; ++cg) {
        if (nt >= 2) h_flush2<KC>(Y, n, i0 + ltid, tlane + COL_D1, tlane + COL_D1 + 96u, cg * 16, sm.inv_s + cg * 16);
        else h_flush<KC>(Y, n, i0 + ltid, tlane + COL_D1, cg * 16, sm.inv_s + cg * 16);
      }
    }
  } else if (warp < 8) {
    // =================================== converter warps ===================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(192));     // 2 x 128 x 192 + 128 x 72 + 128 x 48 <= 64 K registers
    auto fetch = [&](int J, float4 (&dst)[16]) {
      const float4* src = reinterpret_cast<const float4*>(tiles + (tix0 + J) * TILE_ELEMS);
#pragma unroll
      for (int it = 0; it < 16; ++it) dst[it] = src[(it * 8 + warp) * 32 + lane];
    };
    auto step = [&](int k, float4 (&cur)[16], float4 (&nxt)[16]) {
      const int J = tile_of(k), b = k & 1;
      const int64_t j0 = (int64_t)J * TILE;
      if (k >= 2) tc::mbar_wait(&sm.tile_done[b], (uint32_t)(((k - 2) >> 1) & 1));   // MMAs of tile k-2 released buffer b
      // this thread's 16 chunks: row = it * 8 + warp, columns 4 * lane .. + 3  ->  8 bytes per plane at
      // (lane/2) * H_SJ + it * 128 + warp * 16 + (lane%2) * 8
      unsigned char* pl0 = sm.tile[b][0] + (uint32_t)(lane >> 1) * H_SJ + (uint32_t)warp * 16u + (uint32_t)(lane & 1) * 8u;
      unsigned char* pl1 = pl0 + H_PLANE;
      if (rows_ok && J < I) {
#pragma unroll
        for (int it = 0; it < 16; ++it) h_convert_store(cur[it].x, cur[it].y, cur[it].z, cur[it].w, pl0 + it * 128, pl1 + it * 128);
      } else if ((J < I) && (i0 + TILE <= n)) {   // interior tile of a lazily projected / raw parameter: apply the view
#pragma unroll
        for (int it = 0; it < 16; ++it)
          h_convert_store(pv.adj(cur[it].x), pv.adj(cur[it].y), pv.adj(cur[it].z), pv.adj(cur[it].w), pl0 + it * 128,
                          pl1 + it * 128);
      } else {                                 // diagonal / last tile row: validity mask + view
        const bool interior = false;
        const int gj = (int)(j0 + lane * 4);
#pragma unroll 1
        for (int it = 0; it < 16; ++it) {
          const int gi = (int)(i0 + it * 8 + warp);
          const float4 v = h_pick(cur, it);
          float xv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const bool ok = interior || ((gj + c < gi) && (gi < n));
            xv[c] = ok ? pv.adj(xv[c]) : 0.f;
          }
          h_convert_store(xv[0], xv[1], xv[2], xv[3], pl0 + it * 128, pl1 + it * 128);
        }
      }
      tc::fence_async_smem();
      mbar_arrive(&sm.ready[b]);
      if (k + 2 < nt) fetch(tile_of(k + 2), cur);   // two tiles ahead, into the registers just consumed
    };
    float4 ra[16], rb[16];
    fetch(tile_of(0), ra);
    if (nt > 1) fetch(tile_of(1), rb);
    for (int k = 0; k < nt; k += 2) {
      step(k, ra, rb);
      if (k + 1 < nt) step(k + 1, rb, ra);
    }
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tm, 512);
}

inline int64_t prop_ws_bk_bytes(int64_t n, int K) {
  const int64_t T = (n + TILE - 1) / TILE;
  return (T * 32 * ((2 * K) * 16 + 16) + 255) / 256 * 256;
}

template <int KC>
int launch_prop_h(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* B, float* Y,
                  void* ws, cudaStream_t st, int products) {
  const int64_t npad = (n + TILE - 1) / TILE * TILE;
  unsigned char* Bk = reinterpret_cast<unsigned char*>(ws);
  float* scale = reinterpret_cast<float*>(Bk + prop_ws_bk_bytes(n, KC));        // [s_c | 1/s_c | max bits]
  unsigned int* maxbits = reinterpret_cast<unsigned int*>(scale + 2 * KC);
  cudaError_t e = cudaMemsetAsync(maxbits, 0, KC * sizeof(unsigned int), st);
  if (e != cudaSuccess) return (int)e;
  k_colmax<KC><<<(unsigned)min((int64_t)592, (n * KC + 255) / 256), 256, 0, st>>>(B, n, maxbits);
  k_prep_b16<KC><<<(unsigned)((npad * KC + 255) / 256), 256, 0, st>>>(B, n, npad, maxbits, Bk, scale);
  const size_t smem = sizeof(PropHSmem<KC>);
  e = cudaFuncSetAttribute(k_propagate_h<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  if (tr1 - tr0 > 65535) return -3;
  dim3 grid((unsigned)((tr1 + H_RUN - 1) / H_RUN), (unsigned)(tr1 - tr0));
  k_propagate_h<KC><<<grid, H_THREADS, smem, st>>>(tiles, n, tr0, mu, raw, Bk, scale, Y, products);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

// 0 = exact fp32 FFMA (reference of the engine-agreement tests), 5 = tcgen05 kind::f16 on the fp16x2 image (default).
// (Engines 1-4 of rounds 1-2 -- mma.sync 3xTF32, the tcgen05 tf32 hybrids -- are gone; their measurements are in
// profiles/history and profiles/r01_umma_rate.txt.)
int g_prop_engine = 5;
int g_elem_engine = 1;     // mcgra_set_engine(4, v): 0 = k_elem_stats everywhere, 1 = bulk-staged persistent k_elem_rs for the steady state
int g_elem_grid = 0;       // test knob: cap on the persistent grid (mcgra_set_engine(4, 100 + cap); 0 = one CTA per SM)


// ---------------------------------------------------------------------------------------------------------
// Stand-alone element-wise pass (c1 MSE/KL against feature_adj, c6 entropy; values + degree-gradient row sums).
// A pure streaming kernel (x and F tiles read once, 8 bytes per entry) that runs at full occupancy; the propagation
// passes then all use the plain tensor-core kernels.
// ---------------------------------------------------------------------------------------------------------
// Streaming structure: a warp owns rows warp, warp + 8, ...; the loads of EIGHT rows (x and F: 16 LDG.128 per thread)
// are issued before any arithmetic, and the per-row degree-gradient sums go to shared memory instead of one global
// atomic per row -- with the atomic inside the loop the compiler could not hoist the next rows' loads above it
// (eps_row may alias), and the kernel was latency-bound at 0.57 of the HBM roofline (61 % long-scoreboard stalls).
__global__ void __launch_bounds__(256, 2)
k_elem_stats(const float* __restrict__ tiles, int64_t n, int64_t t0, const float* mu, int raw, mcgra_elem_args ea) {
  __shared__ float rI[TILE], rJ[TILE], lseAI[TILE], lseAJ[TILE], lseFI[TILE], lseFJ[TILE], dlI[TILE], dlJ[TILE];
  __shared__ float colacc[TILE], rowacc[TILE];
  __shared__ double red[32];
  int I, J;
  tile_coords(t0 + blockIdx.x, I, J);
  const ParamView pv = load_view(mu, raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
  if (tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    rI[tid] = gi < n ? ea.r[gi] : 0.f;
    rJ[tid] = gj < n ? ea.r[gj] : 0.f;
    if (ea.measure == MCGRA_M_KL) {
      lseAI[tid] = gi < n ? ea.lseA[gi] : 0.f;  lseAJ[tid] = gj < n ? ea.lseA[gj] : 0.f;
      lseFI[tid] = gi < n ? ea.lseF[gi] : 0.f;  lseFJ[tid] = gj < n ? ea.lseF[gj] : 0.f;
      dlI[tid] = gi < n ? ea.dlse[gi] : 0.f;    dlJ[tid] = gj < n ? ea.dlse[gj] : 0.f;
    }
    colacc[tid] = 0.f;
    rowacc[tid] = 0.f;
  }
  __syncthreads();
  const float4* src = reinterpret_cast<const float4*>(tiles + (int64_t)blockIdx.x * TILE_ELEMS);
  const float4* fsrc = ea.Ftiles ? reinterpret_cast<const float4*>(ea.Ftiles + (int64_t)blockIdx.x * TILE_ELEMS) : nullptr;
  const bool interior = (J < I) && (i0 + TILE <= n);
  float rj4[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) rj4[k] = rJ[lane * 4 + k];
  float col_e[4] = {0.f, 0.f, 0.f, 0.f};
  float v1 = 0.f, v6 = 0.f;
  // one row (4 consecutive entries per lane): FAST = interior tile whose buffer already holds the clamped parameter and
  // the MSE measure (the steady state of the headline profile) -- no validity tests, no measure dispatch
  auto row_step = [&](auto fast_tag, int it, const float4 raw4, const float4 f4) {
    constexpr bool FAST = decltype(fast_tag)::value;
    const int row = it * 8 + warp;
    const int gi = (int)(i0 + row), gj = (int)(j0 + lane * 4);
    const float xr[4] = {raw4.x, raw4.y, raw4.z, raw4.w};
    const float fv[4] = {f4.x, f4.y, f4.z, f4.w};
    const float ri = rI[row];
    float row_e = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (!FAST && !(interior || ((gj + k < gi) && (gi < n)))) continue;
      const float xv = FAST ? xr[k] : pv.adj(xr[k]);
      const float rj = rj4[k];
      const float ah = ri * xv * rj;
      float esym = 0.f;   // e'_ij + e'_ji
      if (FAST || ea.measure == MCGRA_M_MSE) {
        const float df = ah - fv[k];
        v1 = fmaf(2.f * df, df, v1);
        esym = 4.f * ea.k1 * df;
      } else if (ea.measure == MCGRA_M_KL) {
        const float xij = __expf(fv[k] - lseFI[row]);
        const float xji = __expf(fv[k] - lseFJ[lane * 4 + k]);
        const float lij = ah - lseAI[row];
        const float lji = ah - lseAJ[lane * 4 + k];
        v1 += xij * ((fv[k] - ah) - dlI[row]) + xji * ((fv[k] - ah) - dlJ[lane * 4 + k]);
        esym = ea.k1 * ((__expf(lij) - xij) + (__expf(lji) - xji));
      }
      if (ea.k6 != 0.f) {
        const float q = fminf(fmaxf(ah, ENT_LO), ENT_HI);
        const float lg = __log2f(q);
        v6 = fmaf(2.f * q, lg, v6);
        if (ah >= ENT_LO && ah <= ENT_HI) esym = fmaf(2.f * ea.k6, lg + INV_LN2, esym);
      }
      const float tt = esym * xv;
      row_e = fmaf(tt, rj, row_e);
      col_e[k] = fmaf(tt, ri, col_e[k]);
    }
    row_e = warp_sum(row_e);
    if (lane == 0) rowacc[row] = row_e;              // every row is visited by exactly one warp iteration
  };
  const bool fast = interior && pv.raw == 2 && ea.measure == MCGRA_M_MSE && fsrc != nullptr;
#pragma unroll 1
  for (int hb = 0; hb < 2; ++hb) {
    float4 xq[8], fq[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int row = (hb * 8 + u) * 8 + warp;
      xq[u] = src[row * 32 + lane];
      fq[u] = fsrc != nullptr ? fsrc[row * 32 + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (fast) {
#pragma unroll
      for (int u = 0; u < 8; ++u) row_step(std::true_type{}, hb * 8 + u, xq[u], fq[u]);
    } else {
#pragma unroll
      for (int u = 0; u < 8; ++u) row_step(std::false_type{}, hb * 8 + u, xq[u], fq[u]);
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) atomicAdd(&colacc[lane * 4 + k], col_e[k]);
  __syncthreads();
  if (tid < TILE) {
    const int64_t gi = i0 + tid, gj = j0 + tid;
    if (gi < n && rowacc[tid] != 0.f) atomicAdd(ea.eps_row + gi, rowacc[tid]);
    if (gj < n && colacc[tid] != 0.f) atomicAdd(ea.eps_row + gj, colacc[tid]);
  }
  if (ea.measure != MCGRA_M_NONE) block_atomic_add_d((double)v1 * (double)ea.k1, ea.acc + MCGRA_ACC_C1, red);
  if (ea.k6 != 0.f) block_atomic_add_d((double)v6 * (double)ea.k6, ea.acc + MCGRA_ACC_C6, red);
}

// ---------------------------------------------------------------------------------------------------------
// k_elem_rs: the same pass as k_elem_stats for the steady state of the headline profile (buffer holds the clamped
// parameter, MSE against feature_adj, optional entropy term), persistent and bulk-staged: every CTA walks a contiguous run
// of tiles in storage order; one producer lane streams x' and F rows (16 rows per stage) through a cp.async.bulk ring in
// shared memory, 16 warps consume one row each per stage.  Row / column sums, node vectors and the tile switch are double
// buffered by tile parity: one consumer barrier per tile.
// ---------------------------------------------------------------------------------------------------------
constexpr int ES_S = 4;                        // ring stages
constexpr int ES_R = 32;                       // rows per stage: warp cw takes rows cw and cw + 16 of a stage
constexpr int ES_CH = ES_R * TILE;             // floats per array per stage
constexpr int ES_CW = 16;                      // consumer warps
constexpr int ES_THREADS = 32 + ES_CW * 32;

struct ElemRsSmem {
  float ring[ES_S][2][ES_CH];                  // x', F
  float rI[2][TILE], rJ[2][TILE];              // by tile parity
  float rowpart[2][TILE][33];                  // per-lane row sums (summed once per tile instead of a shuffle chain per row)
  float colacc[2][TILE];
  double dsum[2];
  uint64_t full[ES_S], empty[ES_S];
};

// LAZY: the buffer holds the un-projected Adam output (raw == 0): entry = clamp(x' - mu, 0, 1) on read
template <bool LAZY>
__global__ void __launch_bounds__(ES_THREADS, 1)
k_elem_rs(const float* __restrict__ tiles, int64_t n, int tr0, int64_t ntiles, const __grid_constant__ mcgra_elem_args ea,
          const float* mu_ptr) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  ElemRsSmem& sm = *reinterpret_cast<ElemRsSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t t_begin = (int64_t)blockIdx.x * ntiles / gridDim.x;
  const int64_t t_end = (int64_t)(blockIdx.x + 1) * ntiles / gridDim.x;
  const int my_tiles = (int)(t_end - t_begin);
  if (tid == 0) {
    for (int s = 0; s < ES_S; ++s) {
      tc::mbar_init(&sm.full[s], 1);
      tc::mbar_init(&sm.empty[s], ES_CW);
    }
    sm.dsum[0] = 0.0;
    sm.dsum[1] = 0.0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < 2 * TILE) (&sm.colacc[0][0])[tid] = 0.f;
  __syncthreads();

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      for (int k = 0; k < my_tiles; ++k) {
        const int64_t base = (t_begin + k) * (int64_t)TILE_ELEMS;
#pragma unroll 1
        for (int ch = 0; ch < TILE / ES_R; ++ch) {
          tc::mbar_wait_backoff(&sm.empty[s], ph ^ 1u);
          const int64_t o = base + (int64_t)ch * ES_CH;
          tc::mbar_expect_tx(&sm.full[s], 2u * ES_CH * 4u);
          tc::bulk_g2s(sm.ring[s][0], tiles + o, ES_CH * 4u, &sm.full[s]);
          tc::bulk_g2s(sm.ring[s][1], ea.Ftiles + o, ES_CH * 4u, &sm.full[s]);
          if (++s == ES_S) { s = 0; ph ^= 1u; }
        }
      }
    }
    return;
  }
  const int cw = warp - 1, ct = tid - 32;
  const int b0 = lane * 4;
  int I, J;
  tile_coords(tri((int64_t)tr0) + t_begin, I, J);
  if (my_tiles > 0 && ct < TILE) {
    const int64_t gi = (int64_t)I * TILE + ct, gj = (int64_t)J * TILE + ct;
    sm.rI[0][ct] = gi < n ? ea.r[gi] : 0.f;
    sm.rJ[0][ct] = gj < n ? ea.r[gj] : 0.f;
  }
  const float k1x4 = 4.f * ea.k1, k6x2 = 2.f * ea.k6;
  const bool ent = ea.k6 != 0.f;
  const float mu = LAZY ? *mu_ptr : 0.f;
  double d1 = 0.0, d6 = 0.0;
  uint32_t s = 0, ph = 0;
  int Iprev = 0, Jprev = 0;
  auto flush = [&](int p, int Ix, int Jx) {          // sums of a finished tile (parity p) -> eps_row (threads < 128)
    float rs = 0.f;
#pragma unroll 8
    for (int l = 0; l < 32; ++l) rs += sm.rowpart[p][ct][l];
    const float cs = sm.colacc[p][ct];
    const int64_t gi = (int64_t)Ix * TILE + ct, gj = (int64_t)Jx * TILE + ct;
    if (gi < n && rs != 0.f) atomicAdd(ea.eps_row + gi, rs);
    if (gj < n && cs != 0.f) atomicAdd(ea.eps_row + gj, cs);
    sm.colacc[p][ct] = 0.f;
  };
#pragma unroll 1
  for (int k = 0; k < my_tiles; ++k) {
    const int p = k & 1;
    int In = I, Jn = J + 1;
    if (Jn > In) { ++In; Jn = 0; }
    asm volatile("bar.sync 1, %0;" ::"n"(ES_CW * 32) : "memory");   // tile k - 1 complete everywhere; r[p] visible
    // node vectors of tile k + 1: loads issued now, parked in shared memory after the stream (no stall on their latency)
    float nrI = 0.f, nrJ = 0.f;
    if (k + 1 < my_tiles && ct < TILE) {
      const int64_t gi = (int64_t)In * TILE + ct, gj = (int64_t)Jn * TILE + ct;
      nrI = gi < n ? ea.r[gi] : 0.f;
      nrJ = gj < n ? ea.r[gj] : 0.f;
    }
    if (k > 0 && ct < TILE) flush(p ^ 1, Iprev, Jprev);            // while tile k streams
    const int64_t i0 = (int64_t)I * TILE, j0 = (int64_t)J * TILE;
    const bool interior = (J < I) && (i0 + TILE <= n);
    float rj4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) rj4[q] = sm.rJ[p][b0 + q];
    float col_e[4] = {0.f, 0.f, 0.f, 0.f};
    float v1 = 0.f, v6 = 0.f;
#pragma unroll 1
    for (int ch = 0; ch < TILE / ES_R; ++ch) {
      tc::mbar_wait(&sm.full[s], ph);
      float4 X[2], F[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        X[h] = *reinterpret_cast<const float4*>(&sm.ring[s][0][(h * 16 + cw) * TILE + b0]);
        F[h] = *reinterpret_cast<const float4*>(&sm.ring[s][1][(h * 16 + cw) * TILE + b0]);
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive1(&sm.empty[s]);
      if (++s == ES_S) { s = 0; ph ^= 1u; }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int a = ch * ES_R + h * 16 + cw;
        const float ri = sm.rI[p][a];
        const float fs[4] = {F[h].x, F[h].y, F[h].z, F[h].w};
        const float xs[4] = {LAZY ? __saturatef(X[h].x - mu) : X[h].x, LAZY ? __saturatef(X[h].y - mu) : X[h].y,
                             LAZY ? __saturatef(X[h].z - mu) : X[h].z, LAZY ? __saturatef(X[h].w - mu) : X[h].w};
        float row_e = 0.f;
        if (interior) {                            // every entry valid: ~16 instructions per entry
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float ah = (ri * rj4[q]) * xs[q];
            const float df = ah - fs[q];
            v1 = fmaf(df, df, v1);                 // (x 2 below)
            float esym = k1x4 * df;
            if (ent) {
              const float qc = fminf(fmaxf(ah, ENT_LO), ENT_HI);
              const float lg = __log2f(qc);
              v6 = fmaf(qc, lg, v6);               // (x 2 below)
              if (qc == ah) esym = fmaf(k6x2, lg + INV_LN2, esym);
            }
            const float tt = esym * xs[q];
            row_e = fmaf(tt, rj4[q], row_e);
            col_e[q] = fmaf(tt, ri, col_e[q]);
          }
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const bool valid = ((j0 + b0 + q) < (i0 + a) && (i0 + a) < n);
            if (!valid) continue;
            const float ah = (ri * rj4[q]) * xs[q];
            const float df = ah - fs[q];
            v1 = fmaf(df, df, v1);
            float esym = k1x4 * df;
            if (ent) {
              const float qc = fminf(fmaxf(ah, ENT_LO), ENT_HI);
              const float lg = __log2f(qc);
              v6 = fmaf(qc, lg, v6);
              if (qc == ah) esym = fmaf(k6x2, lg + INV_LN2, esym);
            }
            const float tt = esym * xs[q];
            row_e = fmaf(tt, rj4[q], row_e);
            col_e[q] = fmaf(tt, ri, col_e[q]);
          }
        }
        sm.rowpart[p][a][lane] = row_e;            // every row is visited by exactly one warp per tile
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (col_e[q] != 0.f) atomicAdd(&sm.colacc[p][b0 + q], col_e[q]);
    if (k + 1 < my_tiles && ct < TILE) { sm.rI[p ^ 1][ct] = nrI; sm.rJ[p ^ 1][ct] = nrJ; }   // (last read by tile k - 1)
    d1 += 2.0 * (double)v1;
    d6 += 2.0 * (double)v6;
    Iprev = I; Jprev = J;
    I = In; J = Jn;
  }
  asm volatile("bar.sync 1, %0;" ::"n"(ES_CW * 32) : "memory");
  if (ct < TILE && my_tiles > 0) flush((my_tiles - 1) & 1, Iprev, Jprev);
  d1 = warp_sum_d(d1);
  d6 = warp_sum_d(d6);
  if (lane == 0) {
    atomicAdd(&sm.dsum[0], d1);
    atomicAdd(&sm.dsum[1], d6);
  }
  asm volatile("bar.sync 1, %0;" ::"n"(ES_CW * 32) : "memory");
  if (ct == 0) {
    if (sm.dsum[0] != 0.0) atomicAdd(ea.acc + MCGRA_ACC_C1, sm.dsum[0] * (double)ea.k1);
    if (ent && sm.dsum[1] != 0.0) atomicAdd(ea.acc + MCGRA_ACC_C6, sm.dsum[1] * (double)ea.k6);
  }
}

template <int KC>
int launch_prop(const float* tiles, int64_t n, int64_t t0, int64_t nt, const float* mu, int raw, const float* B,
                float* Y, cudaStream_t st, int products) {
  const size_t smem = sizeof(PropSmem<KC>);
  cudaError_t e = cudaFuncSetAttribute(k_propagate<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  k_propagate<KC><<<(unsigned)nt, 128, smem, st>>>(tiles, n, t0, mu, raw, B, Y, products);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" {

int mcgra_set_fold_engine_(int value);
int mcgra_set_pairs_engine_(int value);
int mcgra_set_ensemble_engine_(int value);
int mcgra_set_auc_engine_(int value);
int mcgra_set_engine(int which, int value) {
  switch (which) {
    case 0:
      if (value != 0 && value != 5) return -1;
      g_prop_engine = value;
      return 0;
    case 1: return mcgra_set_fold_engine_(value);
    case 2: return mcgra_set_pairs_engine_(value);
    case 4:
      if (value >= 100 && value < 1000) g_elem_grid = value - 100;
      else if (value == 0 || value == 1) g_elem_engine = value;
      else return -1;
      return 0;
    case 5: return mcgra_set_ensemble_engine_(value);
    case 6: return mcgra_set_auc_engine_(value);
    default: return -1;
  }
}

int mcgra_degree(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, float* d, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_degree<<<(unsigned)nt, 128, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, d);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_row_sumexp(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* r,
                     float* sumexp, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0) return 0;
  k_row_sumexp<<<(unsigned)nt, 128, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, r, sumexp);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_elem_stats(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                     const mcgra_elem_args* elem, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (nt <= 0 || elem == nullptr) return 0;
  if (g_elem_engine == 1 && (raw == 2 || raw == 0) && elem->measure == MCGRA_M_MSE && elem->Ftiles != nullptr) {
    static int sms = 0;
    if (sms == 0) {
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    const size_t smem = sizeof(ElemRsSmem) + 128;
    const int cap = g_elem_grid > 0 ? g_elem_grid : sms;
    const unsigned grid = (unsigned)(nt < cap ? nt : cap);
    cudaError_t e;
    if (raw == 0) {
      e = cudaFuncSetAttribute(k_elem_rs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      k_elem_rs<true><<<grid, ES_THREADS, smem, (cudaStream_t)stream>>>(tiles, n, tr0, nt, *elem, mu);
    } else {
      e = cudaFuncSetAttribute(k_elem_rs<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      k_elem_rs<false><<<grid, ES_THREADS, smem, (cudaStream_t)stream>>>(tiles, n, tr0, nt, *elem, mu);
    }
    MCGRA_LAUNCH_CHECK();
    return 0;
  }
  k_elem_stats<<<(unsigned)nt, 256, 0, (cudaStream_t)stream>>>(tiles, n, tri(tr0), mu, raw, *elem);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int64_t mcgra_propagate_ws_bytes(int64_t n, int K) {
  const int64_t npad = (n + TILE - 1) / TILE * TILE;
  return prop_ws_bk_bytes(n, K) + npad * 2 * K * (int64_t)sizeof(float) + 256;
}

int mcgra_propagate_sel(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* B, int K,
                        float* Y, void* ws, int products, void* stream) {
  const int64_t nt = tri(tr1) - tri(tr0);
  if (products < MCGRA_PROD_DIRECT || products > MCGRA_PROD_BOTH) return -1;
  if (nt <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t t0 = tri(tr0);
  if (ws != nullptr && g_prop_engine == 5) {
    if (K == 32) return launch_prop_h<32>(tiles, n, tr0, tr1, mu, raw, B, Y, ws, st, products);
    if (K == 16) return launch_prop_h<16>(tiles, n, tr0, tr1, mu, raw, B, Y, ws, st, products);
    return -1;
  }
  if (K == 32) return launch_prop<32>(tiles, n, t0, nt, mu, raw, B, Y, st, products);
  if (K == 16) return launch_prop<16>(tiles, n, t0, nt, mu, raw, B, Y, st, products);
  return -1;
}

int mcgra_propagate(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* B, int K,
                    float* Y, void* ws, void* stream) {
  return mcgra_propagate_sel(tiles, n, tr0, tr1, mu, raw, B, K, Y, ws, MCGRA_PROD_BOTH, stream);
}

}  // extern "C"
