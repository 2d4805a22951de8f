// Pair pass on tcgen05 for the entropy term of the decode gram (engine 2 of mcgra_pairs; the K7-only instantiation:
// Info_entropy(modified_adj1) = c7 and its autograd through dot_product_decode, topology_attack.py:233-236, 414-419).
//
// Per tile (I, J) of the triangle:   S = zhat_I zhat_J^T   (128 x 128 x 16)              -> tcgen05, D in TMEM
//                                    C = dL/dS = 2 k7 (log2 q + 1/ln 2) [q in range]     -> CUDA cores, from TMEM to smem
//                                    dz_I += C zhat_J,  dz_J += C^T zhat_I  (128 x 16 x 128) -> tcgen05, D in TMEM
// i.e. the propagate engine v5 (propagate.cu) with the tile GENERATED on chip instead of streamed from HBM: the kernel
// has no HBM stream at all (0 algorithmic bytes), it is bound by the element-wise stage (one MUFU log2 per pair).
//
// Precision: fp16 x 2 on both sides, fp32 accumulation (same class as 3xTF32):
//   S operands   zs = 2^10 z:  hi = fp16(zs), lo = fp16(zs - hi);  S 2^20 = hi hi^T + hi lo^T + lo hi^T  (one accumulator)
//   C planes     cs = s_c C:   h0 = fp16(cs), h1 = fp16((cs - h0) 2^11)                 (s_c: power of two, |cs| < 2^14)
//   zhat blocks  g = s_f z:    g0, g1 likewise per feature column f;   D[:, 0:32] += h0 [g0 | g1],  D[:, 32:48] += h1 g0,
//                dz = (d0 + (d1 + d2) 2^-11) / (s_f s_c)
// Pipeline (320 threads, 1 CTA / SM, runs of up to 32 tiles of one tile row): warp 9 (one lane) streams the pre-formatted
// operand blocks (ring of 4, two cp.async.bulk per tile); warp 8 (one lane) only issues MMAs -- its serial instruction
// stream is what bounds this family of kernels (propagate.cu) -- the S product of tile k+1 and then the 32 skinny MMAs of
// tile k;
// warps 0-7 read S[k] from TMEM (lane = row), write the two fp16 planes of C (the same image is the K-major A operand of
// the direct product and the MN-major A operand of the mirrored one) and flush the mirrored result of tile k-1.
// TMEM columns: D1 [0,48) | D2[0] [48,96) | D2[1] [96,144) | S[0] [256,384) | S[1] [384,512).
#include <cuda_fp16.h>
#include <type_traits>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

constexpr uint32_t ZB_LBO = tc::GBlock<HID>::LBO;   // [g0 | g1] block of 128 nodes (tc_common.cuh)
constexpr uint32_t ZB_BLK = tc::GBlock<HID>::BYTES;
constexpr uint32_t ZA_LBO = 16 * 128;                // node x feature image: 16 row groups x 128 B per 8-feature K group
constexpr uint32_t ZA_PLANE = 2 * ZA_LBO;            // 4096 B (hi), + 4096 B (lo)
constexpr uint32_t ZA_BLK = 2 * ZA_PLANE;
constexpr int RING = 4;
constexpr uint32_t COL_D1 = 0, COL_D2 = 48, COL_S = 256;

struct PairTcSmem {
  unsigned char tile[2][2][tc::PLANE_BYTES];         // [buffer][plane h0 / h1]
  unsigned char zbJ[RING][ZB_BLK];
  unsigned char zaJ[RING][ZA_BLK];
  unsigned char zbI[ZB_BLK];
  unsigned char zaI[ZA_BLK];
  uint64_t ready[2], tile_done[2], s_ready[2], s_free[2];
  uint64_t bfull[RING], bfree[RING], bIfull;         // operand-block ring (loader warp)
  float inv_s[16];
  double red[32];
  uint32_t tmem_base;
};

// ---- operand preparation (once per call) ----
__global__ void k_ptc_prep(const float* __restrict__ Z, int64_t n, int64_t npad, const unsigned int* __restrict__ maxbits,
                           unsigned char* __restrict__ Zb, unsigned char* __restrict__ Za, float* __restrict__ scale) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= npad * HID) return;
  const int64_t node = e / HID;
  const int c = (int)(e % HID);
  const float z = node < n ? Z[e] : 0.f;
  const int k = (int)(node & 127);
  {
    const float s = tc::col_scale(maxbits[c]);
    if (node == 0) { scale[c] = s; scale[HID + c] = 1.f / s; }
    tc::store_gblock<HID>(Zb, node, c, z * s);
  }
  // node x feature image, K = feature: (c/8) * ZA_LBO + (k/8) * 128 + (k%8) * 16 + (c%8) * 2; hi plane, then lo plane
  {
    const float zs = z * 1024.f;
    const __half hi = __float2half_rn(zs);
    const __half lo = __float2half_rn(zs - __half2float(hi));
    unsigned char* blk = Za + (node >> 7) * (int64_t)ZA_BLK + (uint32_t)(c >> 3) * ZA_LBO + (uint32_t)(k >> 3) * 128u +
                         (uint32_t)(k & 7) * 16u + (uint32_t)(c & 7) * 2u;
    *reinterpret_cast<__half*>(blk) = hi;
    *reinterpret_cast<__half*>(blk + ZA_PLANE) = lo;
  }
}

// dz[row][c0 .. c0+15] += (d0 + (d1 + d2) 2^-11) inv_s[c] inv_sc
__device__ __forceinline__ void ptc_flush(float* __restrict__ dz, int64_t n, int64_t row, uint32_t taddr, const float* inv_s,
                                          float inv_sc) {
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    uint32_t d0[8], d1[8], d2[8];
    const int c = half * 8;
    tc::tmem_ld8_nowait(taddr + c, d0);
    tc::tmem_ld8_nowait(taddr + HID + c, d1);
    tc::tmem_ld8_nowait(taddr + 2 * HID + c, d2);
    tc::tmem_ld_wait();
    if (row < n) {
      float v[8];
      bool any = false;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        v[u] = (__uint_as_float(d0[u]) + (__uint_as_float(d1[u]) + __uint_as_float(d2[u])) * (1.f / 2048.f)) * inv_s[c + u] * inv_sc;
        any |= v[u] != 0.f;
      }
      if (any) {
        float4* dst = reinterpret_cast<float4*>(dz + row * HID + c);
        atomicAdd(dst, make_float4(v[0], v[1], v[2], v[3]));
        atomicAdd(dst + 1, make_float4(v[4], v[5], v[6], v[7]));
      }
    }
  }
}

__global__ void __launch_bounds__(320, 1)
k_pairs_tc(int64_t n, int tr0, const unsigned char* __restrict__ Zb, const unsigned char* __restrict__ Za,
           const float* __restrict__ scale, float k7, float sc, float* __restrict__ dzhat, double* __restrict__ acc) {
  tc::TileRun run;
  if (!run.init(tr0)) return;
  const int I = run.I, nt = run.nt;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  PairTcSmem& sm = *reinterpret_cast<PairTcSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t i0 = (int64_t)I * TILE;

  if (warp == 0) tc::tmem_alloc(&sm.tmem_base, 512);
  if (tid == 0) {
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&sm.ready[b], 256);
      tc::mbar_init(&sm.tile_done[b], 1);
      tc::mbar_init(&sm.s_ready[b], 1);
      tc::mbar_init(&sm.s_free[b], 256);
    }
    for (int r = 0; r < RING; ++r) { tc::mbar_init(&sm.bfull[r], 1); tc::mbar_init(&sm.bfree[r], 1); }
    tc::mbar_init(&sm.bIfull, 1);
    tc::fence_mbar_init();
  }
  if (tid >= 32 && tid < 32 + HID) sm.inv_s[tid - 32] = scale[HID + tid - 32];
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tm = sm.tmem_base;

  if (warp == 9) {
    // =================================== operand-block loader ===================================
    if (lane == 0) {
      tc::mbar_expect_tx(&sm.bIfull, ZB_BLK + ZA_BLK);
      tc::bulk_g2s(sm.zbI, Zb + (int64_t)I * ZB_BLK, ZB_BLK, &sm.bIfull);
      tc::bulk_g2s(sm.zaI, Za + (int64_t)I * ZA_BLK, ZA_BLK, &sm.bIfull);
      for (int k = 0; k < nt; ++k) {
        const int r = k % RING;
        if (k >= RING) tc::mbar_wait_backoff(&sm.bfree[r], (uint32_t)((k / RING - 1) & 1));   // MMAs of tile k - RING are done
        const int J = run.tile_of(k);
        tc::mbar_expect_tx(&sm.bfull[r], ZB_BLK + ZA_BLK);
        tc::bulk_g2s(sm.zbJ[r], Zb + (int64_t)J * ZB_BLK, ZB_BLK, &sm.bfull[r]);
        tc::bulk_g2s(sm.zaJ[r], Za + (int64_t)J * ZA_BLK, ZA_BLK, &sm.bfull[r]);
      }
    }
  } else if (warp == 8) {
    // =================================== MMA issuer ===================================
    if (lane == 0) {
      const uint32_t id_s = tc::make_idesc_f16(128, 128, 0);
      const uint32_t id_cat = tc::make_idesc_f16(128, 2 * HID, 0), id_one = tc::make_idesc_f16(128, HID, 0);
      const uint32_t id_cat_t = tc::make_idesc_f16(128, 2 * HID, 1), id_one_t = tc::make_idesc_f16(128, HID, 1);
      const uint32_t zaI = tc::smem_u32(sm.zaI);
      const uint64_t aIh = tc::make_desc(zaI, ZA_LBO, 128u), aIl = tc::make_desc(zaI + ZA_PLANE, ZA_LBO, 128u);
      const uint64_t bI0 = tc::make_desc(tc::smem_u32(sm.zbI), ZB_LBO, 128u);
      auto issue_s = [&](int k) {                     // S[k & 1] = zhat_I zhat_J(k)^T, three K = 16 MMAs
        const int b = k & 1;
        tc::mbar_wait(&sm.bfull[k % RING], (uint32_t)((k / RING) & 1));      // blocks of tile k have landed
        if (k >= 2) tc::mbar_wait(&sm.s_free[b], (uint32_t)(((k - 2) >> 1) & 1));
        tc::fence_after();
        const uint32_t zaJ = tc::smem_u32(sm.zaJ[k % RING]);
        const uint64_t bJh = tc::make_desc(zaJ, ZA_LBO, 128u), bJl = tc::make_desc(zaJ + ZA_PLANE, ZA_LBO, 128u);
        const uint32_t d = tm + COL_S + (uint32_t)b * 128u;
        tc::mma_f16(d, aIh, bJh, id_s, 0u);
        tc::mma_f16(d, aIh, bJl, id_s, 1u);
        tc::mma_f16(d, aIl, bJh, id_s, 1u);
        tc::mma_commit(&sm.s_ready[b]);
      };
      tc::mbar_wait(&sm.bIfull, 0u);
      issue_s(0);
      for (int k = 0; k < nt; ++k) {
        const int b = k & 1;
        if (k + 1 < nt) issue_s(k + 1);               // next tile's gram first: the converters never wait for it
        tc::mbar_wait(&sm.ready[b], (uint32_t)((k >> 1) & 1));
        tc::fence_after();
        const uint32_t p0 = tc::smem_u32(sm.tile[b][0]), p1 = tc::smem_u32(sm.tile[b][1]);
        const uint64_t bJ0 = tc::make_desc(tc::smem_u32(sm.zbJ[k % RING]), ZB_LBO, 128u);
        const uint32_t d2 = tm + COL_D2 + (uint32_t)b * 48u;
#pragma unroll 2
        for (int ks = 0; ks < TILE / 16; ++ks) {
          const uint64_t db = (uint64_t)((uint32_t)ks * ((2u * ZB_LBO) >> 4));
          const uint32_t acc1 = (k > 0 || ks > 0) ? 1u : 0u, acc2 = ks > 0 ? 1u : 0u;
          // direct: C as a K-major A operand (M = row, K = column)
          tc::mma_f16(tm + COL_D1, tc::make_desc(p0 + (uint32_t)ks * 2u * tc::PLANE_SJ, tc::PLANE_SJ, 128u), bJ0 + db, id_cat, acc1);
          tc::mma_f16(tm + COL_D1 + 2 * HID, tc::make_desc(p1 + (uint32_t)ks * 2u * tc::PLANE_SJ, tc::PLANE_SJ, 128u), bJ0 + db, id_one, acc1);
          // mirrored: the same image as an MN-major A operand (M = column, K = row)
          tc::mma_f16(d2, tc::make_desc(p0 + (uint32_t)ks * 256u, 128u, tc::PLANE_SJ), bI0 + db, id_cat_t, acc2);
          tc::mma_f16(d2 + 2 * HID, tc::make_desc(p1 + (uint32_t)ks * 256u, 128u, tc::PLANE_SJ), bI0 + db, id_one_t, acc2);
        }
        tc::mma_commit(&sm.tile_done[b]);
        tc::mma_commit(&sm.bfree[k % RING]);
      }
    }
  } else if (warp < 8) {
    // =================================== converter warps ===================================
    const int q = warp & 3, ch = warp >> 2;         // TMEM lane quarter; column half [64 ch, +64)
    const int row = q * 32 + lane;
    const uint32_t tlane = tm + ((uint32_t)(q * 32) << 16);
    const bool flusher = ch == 0;
    const int64_t gi = i0 + row;
    const float k7s2 = 2.f * k7 * sc, k7s2_ln = k7s2 * INV_LN2;
    float v7 = 0.f;
    for (int k = 0; k < nt; ++k) {
      const int J = run.tile_of(k), b = k & 1;
      const int64_t j0 = (int64_t)J * TILE;
      const bool interior = (J < I) && (i0 + TILE <= n);
      tc::mbar_wait(&sm.s_ready[b], (uint32_t)((k >> 1) & 1));
      if (k >= 2) tc::mbar_wait(&sm.tile_done[b], (uint32_t)(((k - 2) >> 1) & 1));   // planes of buffer b are free
      tc::fence_after();
      unsigned char* pl0 = sm.tile[b][0] + (uint32_t)(row >> 3) * 128u + (uint32_t)(row & 7) * 16u;
      unsigned char* pl1 = pl0 + tc::PLANE_BYTES;
      // the element-wise stage is the bound of this kernel (one MUFU log2 + ~12 ALU ops per pair): interior tiles take
      // the mask-free instantiation, 32-bit indices everywhere
      auto convert = [&](auto interior_tag) {
        constexpr bool INTERIOR = decltype(interior_tag)::value;
        const int rel = (int)(gi - j0);             // column c of the tile is valid iff c < rel (and the row exists)
        const bool row_ok = gi < n;
#pragma unroll 1
        for (int cc = 0; cc < 2; ++cc) {
          const int c0 = ch * 64 + cc * 32;
          float s[32];
          tc::tmem_ld32(tlane + COL_S + (uint32_t)b * 128u + (uint32_t)c0, s);
#pragma unroll
          for (int g8 = 0; g8 < 4; ++g8) {
            float co[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float sv = s[g8 * 8 + u] * (1.f / 1048576.f);
              const float qq = fminf(fmaxf(sv, ENT_LO), ENT_HI);      // = clamp(relu(sv)): ENT_LO > 0
              const float lg = __log2f(qq);
              const float dp = fmaf(k7s2, lg, k7s2_ln);               // 2 k7 s_c (log2 q + 1/ln 2)
              if (INTERIOR) {
                v7 = fmaf(qq, lg, v7);
                co[u] = (qq == sv) ? dp : 0.f;                         // inside the clamp interval <=> q == s
              } else {
                const bool valid = row_ok && (c0 + g8 * 8 + u < rel);
                v7 = valid ? fmaf(qq, lg, v7) : v7;
                co[u] = (valid && qq == sv) ? dp : 0.f;
              }
            }
            uint32_t hi[4], lo[4];
            tc::split_pairs<4>(co, hi, lo);
            const uint32_t off = (uint32_t)((c0 >> 3) + g8) * tc::PLANE_SJ;
            *reinterpret_cast<uint4*>(pl0 + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(pl1 + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
      };
      if (interior) convert(std::true_type{}); else convert(std::false_type{});
      tc::fence_before();
      tc::mbar_arrive1(&sm.s_free[b]);                   // S[b] has been read
      tc::fence_async_smem();
      tc::mbar_arrive1(&sm.ready[b]);                    // planes of tile k are in shared memory
      if (k >= 1) {                                 // flush the mirrored result of the previous tile
        tc::mbar_wait(&sm.tile_done[b ^ 1], (uint32_t)(((k - 1) >> 1) & 1));
        tc::fence_after();
        if (flusher) ptc_flush(dzhat, n, (int64_t)run.tile_of(k - 1) * TILE + row, tlane + COL_D2 + (uint32_t)(b ^ 1) * 48u, sm.inv_s, 1.f / sc);
        tc::fence_before();
      }
    }
    const int bl = (nt - 1) & 1;
    tc::mbar_wait(&sm.tile_done[bl], (uint32_t)(((nt - 1) >> 1) & 1));
    tc::fence_after();
    if (flusher) {
      ptc_flush(dzhat, n, (int64_t)run.tile_of(nt - 1) * TILE + row, tlane + COL_D2 + (uint32_t)bl * 48u, sm.inv_s, 1.f / sc);
      ptc_flush(dzhat, n, i0 + row, tlane + COL_D1, sm.inv_s, 1.f / sc);
    }
    // c7 value: sum 2 q log2 q over valid pairs, scaled by k7 (one atomic per CTA); 256 converter threads
    double v = (double)v7 * 2.0 * (double)k7;
    v = warp_sum_d(v);
    if (lane == 0) sm.red[warp] = v;
    tc::bar_sync_named<256>();
    if (warp == 0) {
      double s = lane < 8 ? sm.red[lane] : 0.0;
      s = warp_sum_d(s);
      if (lane == 0 && s != 0.0) atomicAdd(acc + MCGRA_ACC_C7, s);
    }
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tm, 512);
}

}  // namespace

extern "C" {

int64_t mcgra_pairs_ws_bytes(int64_t n) {
  const int64_t T = (n + TILE - 1) / TILE;
  return T * (int64_t)(ZB_BLK + ZA_BLK) + 1024;
}

// engine 2 of mcgra_pairs for the entropy-only configuration (k7 != 0, k2 == 0, no upstream tiles)
int mcgra_pairs_tc_(int64_t n, int tr0, int tr1, const float* zhat, float k7, float* dzhat, double* acc, void* ws,
                    cudaStream_t st) {
  const int64_t T = (n + TILE - 1) / TILE;
  const int64_t npad = T * TILE;
  unsigned char* Zb = reinterpret_cast<unsigned char*>(ws);
  unsigned char* Za = Zb + T * (int64_t)ZB_BLK;
  float* scale = reinterpret_cast<float*>(Za + T * (int64_t)ZA_BLK);         // [s_f | 1/s_f | max bits]
  unsigned int* maxbits = reinterpret_cast<unsigned int*>(scale + 2 * HID);
  cudaError_t e = cudaMemsetAsync(maxbits, 0, HID * sizeof(unsigned int), st);
  if (e != cudaSuccess) return (int)e;
  k_colmax<HID><<<(unsigned)min((int64_t)592, (n * HID + 255) / 256), 256, 0, st>>>(zhat, n, maxbits);
  k_ptc_prep<<<(unsigned)((npad * HID + 255) / 256), 256, 0, st>>>(zhat, n, npad, maxbits, Zb, Za, scale);
  // coefficient scale: |dL/dS| <= 2 |k7| (|log2 1e-4| + 1/ln 2) = 29.5 |k7|;  s_c = 2^floor(log2(2^14 / bound))
  const double bound = 29.5 * fabs((double)k7);
  int ex = 0;
  frexp(16384.0 / bound, &ex);                      // 16384 / bound = m 2^ex, m in [0.5, 1)
  ex = ex - 1;
  ex = ex > 100 ? 100 : (ex < -100 ? -100 : ex);
  const float sc = (float)ldexp(1.0, ex);
  const size_t smem = sizeof(PairTcSmem);
  e = cudaFuncSetAttribute(k_pairs_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  if (tr1 - tr0 > tc::RUN_MAX_ROWS) return -3;
  k_pairs_tc<<<tc::run_grid(tr0, tr1), 320, smem, st>>>(n, tr0, Zb, Za, scale, k7, sc, dzhat, acc);
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
