// tcgen05 / TMEM / mbarrier PTX wrappers (sm_100a) used by the tensor-core engines, and (at the end) the fp16 x 2 split
// operand format shared by the kind::f16 engines.
// Operand tiles are written by CUDA threads in the SWIZZLE_NONE ("interleaved") canonical core-matrix layouts, so no
// TMA descriptor is needed:
//   K-major  (element (r, k), r = M/N index):  (r%8)*16 B + (r/8)*SBO + (k%4)*4 B + (k/4)*LBO       [tf32: 4 elem / 16 B]
//   MN-major (element (mn, k)):                (mn%4)*4 B + (mn/4)*SBO + (k%8)*16 B + (k/8)*LBO
// (cute/arch/mma_sm100_desc.hpp canonical layouts "INTERLEAVE").  One tcgen05.mma kind::tf32 consumes K = 8.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 64-bit shared-memory matrix descriptor, SWIZZLE_NONE, descriptor version 1 (sm_100)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;                // version
  return d;                              // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}

// same, with an explicit layout type (0 none, 1 SWIZZLE_128B_BASE32B, 2 SWIZZLE_128B, 4 SWIZZLE_64B, 6 SWIZZLE_32B)
__device__ __forceinline__ uint64_t make_desc_sw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  return make_desc(saddr, lbo_bytes, sbo_bytes) | ((uint64_t)(layout_type & 7u) << 61);
}

// 32-bit instruction descriptor: D = F32, A = B = TF32, dense, no negate
__device__ __forceinline__ uint32_t make_idesc_tf32(int M, int N, int a_mn_major, int b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                          // c_format = F32
  d |= 2u << 7;                          // a_format = TF32
  d |= 2u << 10;                         // b_format = TF32
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(b_mn_major & 1) << 16;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}
// the same for D = F32, A = B = F16 (format 0), B K-major
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N, int a_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                          // c_format = F32
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {      // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {        // one full warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// makes the initialised barriers visible to the async proxy (bulk copies, MMA commits) before they are used
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand in tensor memory (lane = M index, one 32-bit column per K element)
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem] with fp16 operands (K = 16); issued by ONE thread
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 16 consecutive columns from registers (thread t -> lane base + t)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// arrive on an mbarrier when all previously issued MMAs of this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 consecutive columns: thread t of the warp receives lane (lane_base + t), columns col..col+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// 16-byte asynchronous global -> shared copy (LDGSTS) and its completion wait
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
// same with an L2 eviction policy (createpolicy): operands that every CTA re-reads should outlive the streamed tiles
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
// for data touched once per launch, so that it does not push the re-read operands out of L2
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void cp_async16_hint(void* smem_dst, const void* gsrc, uint64_t policy) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int NPEND>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(NPEND) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// 32 lanes x 16 consecutive columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 8 consecutive columns, asynchronous: the registers are valid after tmem_ld_wait()
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 8 consecutive columns
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- bulk-async (TMA, 1-D) global -> shared copies completing on an mbarrier ----
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive1(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// same with an L2 eviction policy (l2_policy_evict_*)
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
// single-thread wait with back-off (producer / issuer lanes must not take issue slots from the working warps)
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(64);
  }
}

// named barrier 1 for the NTHREADS threads of the working warps of a warp-specialised kernel (the producer / issuer warps
// do not take part)
template <int NTHREADS>
__device__ __forceinline__ void bar_sync_named() { asm volatile("bar.sync 1, %0;" ::"n"(NTHREADS) : "memory"); }

// ==== fp16 x 2 split operands (DESIGN.md 3.1, 3.3) ==============================================================================
// The operand format of k_propagate_h (propagate.cu) and k_pairs_tc (pairs_tc.cu).  An fp32 value x of the 128 x 128 A operand
// is carried by two fp16 planes,  h0 = fp16(x),  h1 = fp16((x - h0) 2^11);  a column c of the n x KC B operand is scaled by a
// power of two s_c with max |B[:, c]| s_c < 2^14, and g = B s_c by g0 = fp16(g), g1 = fp16((g - g0) 2^11) in one K-major block
// [g0 | g1] per 128 nodes.  Then  D[:, 0:2KC] += h0 [g0 | g1],  D[:, 2KC:3KC] += h1 g0,  y_c = (d0 + (d1 + d2) 2^-11) / s_c.

// plane image: element (i, j) at (j/8) PLANE_SJ + (i/8) 128 + (i%8) 16 + (j%8) 2
constexpr uint32_t PLANE_SJ = 16 * 128 + 16;       // stride between 8-column groups (padded: conflict-free stores)
constexpr uint32_t PLANE_BYTES = 16 * PLANE_SJ;

// [g0 | g1] block: element (node k, row r) at (k/8) LBO + (r/8) 128 + (r%8) 16 + (k%8) 2, rows 0 .. KC-1 g0, KC .. 2KC-1 g1
template <int KC>
struct GBlock {
  static constexpr uint32_t LBO = (2 * KC) * 16;
  static constexpr uint32_t BYTES = 16 * LBO;
};

// s_c from maxbits = bits of max_i |B[i][c]| (k_colmax)
__device__ __forceinline__ float col_scale(unsigned int maxbits) {
  if (maxbits == 0u) return 1.f;
  int e = (int)((maxbits >> 23) & 0xffu) - 127;                          // max < 2^(e+1)
  int se = 13 - e;
  se = se > 126 ? 126 : (se < -126 ? -126 : se);
  return __uint_as_float((uint32_t)(se + 127) << 23);
}

// g = B[node][c] s_c (0 for the padding nodes of the last block) into the blocks starting at Bk
template <int KC>
__device__ __forceinline__ void store_gblock(unsigned char* Bk, int64_t node, int c, float g) {
  const __half g0 = __float2half_rn(g);
  const __half g1 = __float2half_rn((g - __half2float(g0)) * 2048.f);
  const int k = (int)(node & 127);
  unsigned char* blk = Bk + (node >> 7) * (int64_t)GBlock<KC>::BYTES + (uint32_t)(k >> 3) * GBlock<KC>::LBO + (uint32_t)(k & 7) * 2u;
  *reinterpret_cast<__half*>(blk + (uint32_t)(c >> 3) * 128u + (uint32_t)(c & 7) * 16u) = g0;
  const int c2 = c + KC;
  *reinterpret_cast<__half*>(blk + (uint32_t)(c2 >> 3) * 128u + (uint32_t)(c2 & 7) * 16u) = g1;
}

// x[0 .. 2NP) -> the h0 words hi[0 .. NP) and the h1 words lo[0 .. NP) of 2NP consecutive plane elements
template <int NP>
__device__ __forceinline__ void split_pairs(const float (&x)[2 * NP], uint32_t (&hi)[NP], uint32_t (&lo)[NP]) {
  __half2 a[NP];
  float2 f[NP];
#pragma unroll
  for (int p = 0; p < NP; ++p) a[p] = __floats2half2_rn(x[2 * p], x[2 * p + 1]);
#pragma unroll
  for (int p = 0; p < NP; ++p) f[p] = __half22float2(a[p]);
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    const __half2 r = __floats2half2_rn((x[2 * p] - f[p].x) * 2048.f, (x[2 * p + 1] - f[p].y) * 2048.f);
    hi[p] = *reinterpret_cast<const uint32_t*>(&a[p]);
    lo[p] = *reinterpret_cast<const uint32_t*>(&r);
  }
}

// Run schedule: CTA (x, y) takes the run of up to RUN tiles Jbeg = RUN x .. of tile row I = tr0 + y.  The tiles of a run are
// visited in a rotated order (the start depends on the tile row) so that concurrently resident CTAs of neighbouring tile rows
// do not add their mirrored results to the same rows at the same time.
constexpr int RUN = 64;
constexpr int RUN_MAX_ROWS = 65535;                // tile rows per launch (gridDim.y)
struct TileRun {
  int I, Jbeg, nt, rot;
  // false for a CTA whose run lies right of the diagonal
  __device__ __forceinline__ bool init(int tr0) {
    I = tr0 + (int)blockIdx.y;
    Jbeg = (int)blockIdx.x * RUN;
    if (Jbeg > I) return false;
    nt = min(I + 1, Jbeg + RUN) - Jbeg;
    rot = (I * 5) % nt;
    return true;
  }
  __device__ __forceinline__ int tile_of(int k) const { const int r = k + rot; return Jbeg + (r >= nt ? r - nt : r); }
};
// the grid over tile rows [tr0, tr1), at most RUN_MAX_ROWS of them
inline dim3 run_grid(int tr0, int tr1) { return dim3((unsigned)((tr1 + RUN - 1) / RUN), (unsigned)(tr1 - tr0)); }

}  // namespace tc

// internal linkage, like the other kernels: every translation unit that launches it compiles its own copy
namespace {

// column maxima: maxbits[c] = bits of max_i |B[i][c]| (maxbits zeroed by the caller)
template <int KC>
__global__ void k_colmax(const float* __restrict__ B, int64_t n, unsigned int* __restrict__ maxbits) {
  const int c = threadIdx.x % KC;
  float m = 0.f;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n * KC; e += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(B[e]));
  if (m > 0.f) atomicMax(maxbits + c, __float_as_uint(m));
}

}  // namespace
