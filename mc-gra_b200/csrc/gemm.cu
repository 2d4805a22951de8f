// K6: the dense n x n x n contraction of the HSIC / CKA / DP measures on two n x n operands
// (CudaCKA.linear_HSIC / linear_CKA, utils.py:1060-1091; PGDAttack.dot_product, topology_attack.py:480-481; call sites
// topology_attack.py:190-229) as ONE generic TMA-fed tcgen05 kernel:
//
//        C[M x N]  =  beta * C  +  alpha * ( A[M x K] * B[N x K]^T  -  coef * u_i v_j )        (+ fused reductions)
//
// Operands are fp16x2 IMAGES of fp32 matrices (dense.cu builds them): row i of X is stored as two fp16 planes
//        hi = fp16(s_i x),   lo = fp16(s_i x - hi),      s_i = a power of two with max_j |s_i x_ij| <= 2^14,
// i.e. 4 bytes per element like fp32, ~2^-23 relative to the row maximum.  The product keeps the three leading terms
//        acc += A_hi B_hi + A_hi B_lo + A_lo B_hi        (three tcgen05.mma kind::f16, fp32 accumulation in TMEM)
// which is the same error class as 3xTF32 at twice its tensor-pipe rate (kind::f16 runs K = 16 per instruction where
// kind::tf32 runs K = 8); the epilogue removes the row / column scales exactly (powers of two).
//
// Kernel shape (DESIGN.md 3.4): one CTA PAIR (cluster of 2, tcgen05 cta_group::2) per 256 x 256 output tile, UMMA
// M = 256, N = 256, K = 16; each CTA holds 128 rows of A and 128 rows (its half of N) of B per K-block of 64 halves
// (128-byte rows, SWIZZLE_128B, K-major), hi and lo planes -> 64 KB per stage, ring of 3 stages filled by TMA
// (cp.async.bulk.tensor.2d.cta_group::2, both CTAs signal the leader's mbarrier); warp 0 = TMA producer, warp 1 = MMA
// issuer (leader CTA only, one thread) and TMEM owner, warps 2-9 = epilogue (tcgen05.ld -> scale -> rank-1 correction
// -> reductions -> global).
//
// Accumulation: the tensor core adds every MMA into its fp32 TMEM accumulator with TRUNCATION -- measured here on
// all-positive operands: a relative bias of -4.2e-8 per MMA, i.e. -1.3e-4 at K = 16 384 and -4.2e-4 at K = 65 536 when one
// accumulator runs over the whole K (tests/test_gpu_gemm.py::test_gemm_large_k), above the 1e-4 loss budget.  The K loop is
// therefore cut into CHUNKS of 16 K-blocks (192 MMAs, bias <= 8e-6; 8 K-blocks cost ~15 % at n = 65 536 because the drains
// compete with the MMAs for TMEM bandwidth, 32 K-blocks cost nothing): the MMA warp alternates between two TMEM accumulators
// (2 x 256 columns) and the eight epilogue warps drain each finished chunk into fp32 REGISTERS (round-to-nearest adds, 128
// per thread) while the next chunk is being accumulated; the epilogue proper then runs from the registers.
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

constexpr int G_BK = 64;                       // halves per K-block = one 128-byte swizzle row
constexpr int G_PLANE = 128 * 128;             // bytes of one 128-row x 128-byte plane
constexpr int G_STAGE = 4 * G_PLANE;           // A_hi | A_lo | B_hi | B_lo
constexpr int G_STAGES = 3;
constexpr int G_SMEM = G_STAGES * G_STAGE + 1024 /* alignment slack */ + 256 /* barriers */;
constexpr int G_CHUNK = 16;                    // K-blocks per TMEM accumulation chunk (see header)
constexpr int G_THREADS = 320;                 // producer warp, MMA warp, 8 epilogue warps
constexpr int G_GROUP = 8;                     // tile rasterisation: sweep groups of 8 tile rows (L2 reuse)
constexpr int G_BT = 256;                      // tile edge of the CTA pair

struct GemmParams {
  int64_t M, N, K;              // C is M x N (rows of A image x rows of B image), K = common column count
  int64_t row0;                 // first row of C / A computed by this launch (row panel)
  int64_t rows;                 // number of rows of the panel
  const float* inv_sa;          // [M] 1 / s_i of A's rows
  const float* inv_sb;          // [N]
  float* C;
  int64_t ldc;
  float alpha, beta;
  const float* alpha_dev;       // optional device scalars multiplying alpha / beta
  const float* beta_dev;
  const float* u;               // rank-1 correction coef * u_i * v_j (u == NULL: u_i = 1); v == NULL: none
  const float* v;
  float coef;
  double* sumsq;                // += sum (acc - rank1)^2
  double* dot;                  // += sum (acc - rank1) * E_ij, E = image (Eh + El) * inv_se[i]
  const __half* Eh;
  const __half* El;
  const float* inv_se;
  int64_t lde;
  int tiles_m, tiles_n;
};

// ---- PTX wrappers (cluster, cta_group::2) ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t mbar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
          "r"(dst), "l"((uint64_t)map), "r"(mbar), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void mma_f16_cg(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// arrive on the mbarrier (same shared-memory offset in both CTAs of the pair) when all MMAs issued so far are complete
__device__ __forceinline__ void mma_commit_cg(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          tc::smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}

__device__ __forceinline__ void tmem_alloc_cg(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc::smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// K-major SWIZZLE_128B operand: rows of 128 bytes, 8-row groups 1024 bytes apart (TMA box {64 halves, 128 rows})
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr) {
  return tc::make_desc_sw(saddr, 16, 1024, 2);
}

// ---- the kernel ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive_rank(uint64_t* bar, uint32_t rank, bool remote) {
  if (remote) {
    const uint32_t a = mapa_rank(tc::smem_u32(bar), rank);
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(a) : "memory");
  } else {
    tc::mbar_arrive1(bar);
  }
}

__global__ void __launch_bounds__(G_THREADS, 1)
k_gemm3(const __grid_constant__ CUtensorMap mapAh, const __grid_constant__ CUtensorMap mapAl,
        const __grid_constant__ CUtensorMap mapBh, const __grid_constant__ CUtensorMap mapBl, const GemmParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + G_STAGES * G_STAGE);
  uint64_t* empty = full + G_STAGES;
  uint64_t* acc_full = empty + G_STAGES;       // [2] chunk accumulator b complete (MMA -> epilogue warps)
  uint64_t* acc_empty = acc_full + 2;          // [2] chunk accumulator b drained (epilogue warps of the pair -> MMA)
  uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  constexpr uint32_t NCOLS = G_BT;             // accumulator columns per CTA
  constexpr int NPT = (int)NCOLS / 2;          // accumulator columns per epilogue thread

  // grouped rasterisation of the pair's tile
  const int64_t tid = (int64_t)blockIdx.x / 2;
  const int64_t per_group = (int64_t)G_GROUP * p.tiles_n;
  const int first_m = (int)(tid / per_group) * G_GROUP;
  const int gsz = min(p.tiles_m - first_m, G_GROUP);
  const int tm = first_m + (int)((tid % per_group) % gsz);
  const int tn = (int)((tid % per_group) / gsz);

  const int64_t m_cta = p.row0 + (int64_t)tm * G_BT + (int64_t)cta_rank * 128;   // A rows / accumulator rows of this CTA
  const int64_t nb_cta = (int64_t)tn * G_BT + (int64_t)cta_rank * 128;           // B rows this CTA stages
  const int64_t n0 = (int64_t)tn * G_BT;                                         // first output column of the tile
  const int num_kb = (int)((p.K + G_BK - 1) / G_BK);
  const int num_ch = (num_kb + G_CHUNK - 1) / G_CHUNK;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < G_STAGES; ++s) {
      tc::mbar_init(&full[s], 1);
      tc::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&acc_full[b], 1);
      tc::mbar_init(&acc_empty[b], 16);        // one arrival per epilogue warp of both CTAs of the pair
    }
    tc::fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_cg(tmem_slot, 2 * NCOLS);
  tc::fence_before();
  __syncthreads();                             // CTA-level order for tmem_slot / the barriers (and for racecheck, which
  cluster_sync_all();                          // does not model barrier.cluster); the pair then syncs across CTAs
  tc::fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % G_STAGES;
        const uint32_t ph = (uint32_t)(kb / G_STAGES) & 1u;
        tc::mbar_wait(&empty[s], ph ^ 1u);
        if (cta_rank == 0) tc::mbar_expect_tx(&full[s], (uint32_t)(2 * G_STAGE));
        const uint32_t bar = mapa_rank(tc::smem_u32(&full[s]), 0);
        const uint32_t base = tc::smem_u32(smem + s * G_STAGE);
        const int k0 = kb * G_BK;
        tma_load_2d(base, &mapAh, k0, (int)m_cta, bar);
        tma_load_2d(base + G_PLANE, &mapAl, k0, (int)m_cta, bar);
        tma_load_2d(base + 2 * G_PLANE, &mapBh, k0, (int)nb_cta, bar);
        tma_load_2d(base + 3 * G_PLANE, &mapBl, k0, (int)nb_cta, bar);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA, one thread) =====
    if (cta_rank == 0 && lane == 0) {
      const uint32_t idesc = tc::make_idesc_f16(G_BT, G_BT, 0);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % G_STAGES;
        const uint32_t ph = (uint32_t)(kb / G_STAGES) & 1u;
        const int ch = kb / G_CHUNK, kc = kb % G_CHUNK, b = ch & 1;
        if (kc == 0 && ch >= 2) {              // accumulator b was last used by chunk ch - 2: wait until it is drained
          tc::mbar_wait(&acc_empty[b], (uint32_t)(((ch - 2) >> 1) & 1));
          tc::fence_after();
        }
        tc::mbar_wait(&full[s], ph);
        tc::fence_after();
        const uint32_t base = tc::smem_u32(smem + s * G_STAGE);
        const uint32_t d = tmem + (uint32_t)b * NCOLS;
#pragma unroll
        for (int k = 0; k < G_BK / 16; ++k) {
          const uint64_t ah = desc_sw128(base + k * 32), al = desc_sw128(base + G_PLANE + k * 32);
          const uint64_t bh = desc_sw128(base + 2 * G_PLANE + k * 32), bl = desc_sw128(base + 3 * G_PLANE + k * 32);
          mma_f16_cg(d, ah, bh, idesc, (kc | k) ? 1u : 0u);
          mma_f16_cg(d, ah, bl, idesc, 1u);
          mma_f16_cg(d, al, bh, idesc, 1u);
        }
        mma_commit_cg(&empty[s]);          // frees the stage in both CTAs once these MMAs have read it
        if (kc == G_CHUNK - 1 || kb == num_kb - 1) mma_commit_cg(&acc_full[b]);   // chunk complete -> epilogue warps
      }
    }
  } else {
    // ===== epilogue warps 2..9: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4 =====
    const int q = warp & 3, half = (warp - 2) >> 2;
    float acc[NPT];
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * NPT);
    for (int ch = 0; ch < num_ch; ++ch) {
      const int b = ch & 1;
      tc::mbar_wait(&acc_full[b], (uint32_t)((ch >> 1) & 1));
      tc::fence_after();
#pragma unroll
      for (int g = 0; g < NPT / 32; ++g) {
        float a[32];
        tc::tmem_ld32(tl + (uint32_t)b * NCOLS + (uint32_t)(g * 32), a);
        if (ch == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[g * 32 + j] = a[j];
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[g * 32 + j] += a[j];
        }
      }
      tc::fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_rank(&acc_empty[b], 0, cta_rank != 0);
    }
    const int64_t row = m_cta + q * 32 + lane;
    const bool row_ok = row < p.row0 + p.rows && row < p.M;
    const float isa = row_ok ? p.inv_sa[row] : 0.f;
    const float ui = (row_ok && p.v != nullptr) ? (p.u != nullptr ? p.u[row] : 1.f) * p.coef : 0.f;
    const float alpha = p.alpha * (p.alpha_dev != nullptr ? *p.alpha_dev : 1.f);
    const float beta = p.beta * (p.beta_dev != nullptr ? *p.beta_dev : 1.f);
    const float ise = (row_ok && p.dot != nullptr) ? p.inv_se[row] : 0.f;
    double ssq = 0.0, sdot = 0.0;
    float* crow = (p.C != nullptr && row_ok) ? p.C + row * p.ldc : nullptr;
    const int64_t cbase = n0 + half * NPT;
    if (row_ok && cbase < p.N) {
#pragma unroll
      for (int g = 0; g < NPT / 32; ++g) {
        float fsq = 0.f, fdot = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int64_t col = cbase + g * 32 + j;
          if (col < p.N) {
            float val = acc[g * 32 + j] * isa * __ldg(p.inv_sb + col);
            if (p.v != nullptr) val = fmaf(-ui, __ldg(p.v + col), val);
            fsq = fmaf(val, val, fsq);
            if (p.dot != nullptr) {
              const float e = (__half2float(p.Eh[row * p.lde + col]) + __half2float(p.El[row * p.lde + col])) * ise;
              fdot = fmaf(val, e, fdot);
            }
            if (crow != nullptr) {
              float o = alpha * val;
              if (beta != 0.f) o = fmaf(beta, crow[col], o);
              crow[col] = o;
            }
          }
        }
        ssq += (double)fsq;
        sdot += (double)fdot;
      }
    }
    if (p.sumsq != nullptr) {
      ssq = warp_sum_d(ssq);
      if (lane == 0 && ssq != 0.0) atomicAdd(p.sumsq, ssq);
    }
    if (p.dot != nullptr) {
      sdot = warp_sum_d(sdot);
      if (lane == 0 && sdot != 0.0) atomicAdd(p.dot, sdot);
    }
  }

  tc::fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_cg(tmem, 2 * NCOLS);
}

// ---- host side: tensor maps ------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

// fp16 plane [rows x cols], leading dimension ld (halves, multiple of 8), boxes of 64 halves x 128 rows, 128-byte swizzle
int make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld) {
  EncodeTiledFn enc = encode_fn();
  if (enc == nullptr) return -20;
  if ((ld & 7) != 0 || ((uintptr_t)base & 15) != 0) return -21;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)G_BK, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -22;
}

int launch_gemm(const CUtensorMap* maps, GemmParams& p, cudaStream_t st) {
  p.tiles_m = (int)((p.rows + G_BT - 1) / G_BT);
  p.tiles_n = (int)((p.N + G_BT - 1) / G_BT);
  const int64_t groups = (int64_t)p.tiles_m * p.tiles_n;
  if (groups <= 0) return 0;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(k_gemm3, cudaFuncAttributeMaxDynamicSharedMemorySize, G_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr_done = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(groups * 2));
  cfg.blockDim = dim3(G_THREADS);
  cfg.dynamicSmemBytes = G_SMEM;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, k_gemm3, maps[0], maps[1], maps[2], maps[3], p);
  if (e != cudaSuccess) return (int)e;
  return 0;
}

}  // namespace

extern "C" {

int mcgra_gemm_nt(const mcgra_image* A, const mcgra_image* B, const mcgra_gemm_epilogue* e, void* stream) {
  if (A == nullptr || B == nullptr || e == nullptr) return -1;
  if (A->cols != B->cols) return -2;
  GemmParams p = {};
  p.M = A->rows;
  p.N = B->rows;
  p.K = A->cols;
  p.row0 = e->row0;
  p.rows = (e->row1 > e->row0 ? e->row1 : p.M) - e->row0;
  if (p.row0 < 0 || p.row0 + p.rows > p.M) return -3;
  p.inv_sa = A->inv_scale;
  p.inv_sb = B->inv_scale;
  p.C = e->C;
  p.ldc = e->ldc;
  p.alpha = e->alpha;
  p.beta = e->beta;
  p.alpha_dev = e->alpha_dev;
  p.beta_dev = e->beta_dev;
  p.u = e->u;
  p.v = e->v;
  p.coef = e->coef;
  p.sumsq = e->sumsq;
  p.dot = e->dot;
  if (e->dot != nullptr) {
    if (e->dot_with == nullptr) return -4;
    p.Eh = (const __half*)e->dot_with->hi;
    p.El = (const __half*)e->dot_with->lo;
    p.inv_se = e->dot_with->inv_scale;
    p.lde = e->dot_with->ld;
  }
  CUtensorMap maps[4];
  int rc;
  if ((rc = make_map(&maps[0], A->hi, A->rows, A->cols, A->ld)) != 0) return rc;
  if ((rc = make_map(&maps[1], A->lo, A->rows, A->cols, A->ld)) != 0) return rc;
  if ((rc = make_map(&maps[2], B->hi, B->rows, B->cols, B->ld)) != 0) return rc;
  if ((rc = make_map(&maps[3], B->lo, B->rows, B->cols, B->ld)) != 0) return rc;
  return launch_gemm(maps, p, (cudaStream_t)stream);
}

}  // extern "C"
