// Top-k node pairs of a dense score matrix: the k largest S[i, j] over the strict upper triangle (i < j), ordered by
// score descending and, among equal scores, by the row-major index i * n + j ascending.
//
// Method: MSB radix select on the order-preserving 32-bit key (fkey), streamed over the row-major matrix or a row band
// of it (rows [row0, row0 + rows), leading dimension n).  Only the columns j > i of a row are read.
//   levels 0 / 1 / 2   histogram of the candidates whose key matches the prefix found so far: 2^11 / 2^11 / 2^10 bins of
//                      key bits 31..21 / 20..10 / 9..0 (CTA-private shared-memory bins, one flush per CTA, 64-bit global
//                      counts); a one-block select picks the bin that holds the remaining-th largest key.  After level 2
//                      the threshold key tau is known, and t = the number of candidates equal to tau still to take.
//   count              per work item (a fixed chunk of columns of one row) the candidates with key > tau and == tau, then an
//                      exclusive scan over the items in row-major order.
//   write              every candidate with key > tau, and the first t with key == tau in index order, to its slot
//                      (slot = #selected before it in index order), so the k slots are in index order.
// The caller then sorts the k values with the stable mcgra_argsort_desc: (score desc, index asc).
// Workspace: 256 B control + 2 049 histogram words + two int64 words per work item; never O(n^2).
#include "common.cuh"

namespace {

constexpr int TK_CW = 8192;                // columns per work item
constexpr int TK_THREADS = 256;
constexpr int TK_BINS = 2048;
constexpr int TK_HIST_WORDS = TK_BINS + 1;   // bins, then the NaN count (level 0)
constexpr int TK_SCAN_SEG = 8;             // items per thread and round of the single-block scan

// control words (int64 at byte 0 of the workspace)
enum { C_PREFIX = 0, C_REMAIN = 1, C_GT = 2, C_EQ = 3, C_SHORT = 4 };

inline int64_t tk_align(int64_t b) { return (b + 255) / 256 * 256; }
inline int64_t tk_nc(int64_t n) { return (n + TK_CW - 1) / TK_CW; }

struct Band {
  const float* s;     // row row0 of the matrix, leading dimension n
  int64_t row0, rows, n, nc;
};

// work item w = (local row r, column chunk c) -> candidate columns [c0, c1) of that row; false when empty
__device__ __forceinline__ bool item_range(const Band& b, int64_t w, int64_t& r, int64_t& c0, int64_t& c1) {
  r = w / b.nc;
  const int64_t c = w - r * b.nc;
  const int64_t gi = b.row0 + r;
  c0 = max(c * TK_CW, gi + 1);
  c1 = min((c + 1) * TK_CW, b.n);
  return c0 < c1;
}

__device__ __forceinline__ int lvl_shift(int level) { return level == 0 ? 21 : level == 1 ? 10 : 0; }
__device__ __forceinline__ uint32_t lvl_mask(int level) {      // key bits fixed by the levels before `level`
  return level == 0 ? 0u : level == 1 ? 0xFFE00000u : 0xFFFFFC00u;
}
__device__ __forceinline__ uint32_t lvl_bins(int level) { return level == 2 ? 1024u : 2048u; }

// The four columns j0 .. j0 + 3 of one row that a thread visits: one 16-byte load when the rows are 16-byte aligned
// (j0 is then a multiple of 4 and j0 + 3 < c1), scalar loads otherwise.
template <bool VEC>
__device__ __forceinline__ void load4(const float* __restrict__ row, int64_t j0, int64_t c1, float (&v)[4]) {
  if (VEC) {
    const float4 q = *reinterpret_cast<const float4*>(row + j0);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = j0 + e < c1 ? row[j0 + e] : 0.f;
  }
}

// Histogram of one level.  A thread merges runs of equal bins before it updates the shared bins: tied scores (exact zeros,
// quantised values) would otherwise serialise on one shared-memory address.
template <bool VEC>
__global__ void __launch_bounds__(TK_THREADS)
k_tk_hist(Band b, int level, const int64_t* __restrict__ ctrl, unsigned long long* __restrict__ ghist) {
  __shared__ uint32_t h[TK_BINS];
  __shared__ uint32_t hnan;
  for (int e = threadIdx.x; e < TK_BINS; e += TK_THREADS) h[e] = 0;
  if (threadIdx.x == 0) hnan = 0;
  __syncthreads();
  const uint32_t mask = lvl_mask(level);
  const uint32_t prefix = level == 0 ? 0u : (uint32_t)ctrl[C_PREFIX];
  const int shift = lvl_shift(level);
  const uint32_t bmask = lvl_bins(level) - 1;
  uint32_t cur = 0, run = 0, nan = 0;
  auto visit = [&](float v) {
    if (isnan(v)) { ++nan; return; }
    const uint32_t key = fkey(v);
    if ((key & mask) != prefix) return;
    const uint32_t bin = (key >> shift) & bmask;
    if (bin == cur) {
      ++run;
    } else {
      if (run) atomicAdd(&h[cur], run);
      cur = bin;
      run = 1;
    }
  };
  const int64_t nitems = b.rows * b.nc;
  constexpr int64_t STEP = 4 * TK_THREADS;
  for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x) {
    int64_t r, c0, c1;
    if (!item_range(b, w, r, c0, c1)) continue;
    const float* row = b.s + r * b.n;
    const int64_t base = VEC ? (c0 & ~(int64_t)3) : c0;
    for (int64_t j = base + 4 * threadIdx.x; j < c1; j += 2 * STEP) {       // two loads in flight per thread
      float v[4], u[4];
      const bool second = j + STEP < c1;
      load4<VEC>(row, j, c1, v);
      if (second) load4<VEC>(row, j + STEP, c1, u);
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (j + e >= c0 && j + e < c1) visit(v[e]);
      if (second) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (j + STEP + e < c1) visit(u[e]);
      }
    }
  }
  if (run) atomicAdd(&h[cur], run);
  if (level == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nan += __shfl_xor_sync(0xffffffffu, nan, o);
    if ((threadIdx.x & 31) == 0 && nan) atomicAdd(&hnan, nan);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < (int)lvl_bins(level); e += TK_THREADS)
    if (h[e]) atomicAdd(ghist + e, (unsigned long long)h[e]);
  if (threadIdx.x == 0 && hnan) atomicAdd(ghist + TK_BINS, (unsigned long long)hnan);
}

// inclusive block scan of one int64 per thread (blockDim.x == 1024); `ws` is shared scratch of 32 words
__device__ __forceinline__ int64_t block_incl_scan(int64_t v, int64_t* ws) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int64_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0) {
    const int64_t s = ws[lane];
    int64_t si = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t t = __shfl_up_sync(0xffffffffu, si, o);
      if (lane >= o) si += t;
    }
    ws[lane] = si - s;
  }
  __syncthreads();
  const int64_t r = inc + ws[w];
  __syncthreads();
  return r;
}

// One block of 1024 threads: bins in descending order (thread t holds positions 2t, 2t + 1), the first position where
// the running count reaches the remaining count is the bin of the remaining-th largest key.
__global__ void __launch_bounds__(1024)
k_tk_select(int level, int64_t k, int64_t* __restrict__ ctrl, const unsigned long long* __restrict__ ghist) {
  __shared__ int64_t ws[32];
  const int64_t nb = lvl_bins(level);
  const int64_t remain = level == 0 ? k : ctrl[C_REMAIN];
  const uint32_t prefix = level == 0 ? 0u : (uint32_t)ctrl[C_PREFIX];
  const int64_t b0 = nb - 1 - 2 * (int64_t)threadIdx.x, b1 = b0 - 1;
  const int64_t h0 = b0 >= 0 ? (int64_t)ghist[b0] : 0, h1 = b1 >= 0 ? (int64_t)ghist[b1] : 0;
  const int64_t incl = block_incl_scan(h0 + h1, ws);
  const int64_t excl = incl - h0 - h1;
  int64_t bin = -1, above = 0;
  if (h0 > 0 && excl < remain && excl + h0 >= remain) { bin = b0; above = excl; }
  else if (h1 > 0 && excl + h0 < remain && incl >= remain) { bin = b1; above = excl + h0; }
  if (bin >= 0) {
    ctrl[C_PREFIX] = (int64_t)(prefix | ((uint32_t)bin << lvl_shift(level)));
    ctrl[C_REMAIN] = remain - above;
  }
  if (threadIdx.x == 1023 && incl < remain) ctrl[C_SHORT] = 1;    // fewer candidates than asked for (NaNs, bad reduce)
}

// candidates > tau and == tau of every work item
template <bool VEC>
__global__ void __launch_bounds__(TK_THREADS)
k_tk_count(Band b, const int64_t* __restrict__ ctrl, int64_t* __restrict__ gtc, int64_t* __restrict__ eqc) {
  __shared__ uint32_t sg, se;
  if (threadIdx.x == 0) { sg = 0; se = 0; }
  __syncthreads();
  const uint32_t tau = (uint32_t)ctrl[C_PREFIX];
  const int64_t nitems = b.rows * b.nc;
  constexpr int64_t STEP = 4 * TK_THREADS;
  for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x) {
    int64_t r, c0, c1;
    if (!item_range(b, w, r, c0, c1)) {
      if (threadIdx.x == 0) { gtc[w] = 0; eqc[w] = 0; }
      continue;
    }
    const float* row = b.s + r * b.n;
    const int64_t base = VEC ? (c0 & ~(int64_t)3) : c0;
    uint32_t ng = 0, ne = 0;
    for (int64_t j = base + 4 * threadIdx.x; j < c1; j += STEP) {
      float v[4];
      load4<VEC>(row, j, c1, v);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (j + e >= c0 && j + e < c1 && !isnan(v[e])) {
          const uint32_t key = fkey(v[e]);
          ng += key > tau ? 1u : 0u;
          ne += key == tau ? 1u : 0u;
        }
      }
    }
    ng = __reduce_add_sync(0xffffffffu, ng);
    ne = __reduce_add_sync(0xffffffffu, ne);
    if ((threadIdx.x & 31) == 0) {
      if (ng) atomicAdd(&sg, ng);
      if (ne) atomicAdd(&se, ne);
    }
    __syncthreads();
    if (threadIdx.x == 0) { gtc[w] = sg; eqc[w] = se; sg = 0; se = 0; }
    __syncthreads();
  }
}

// in-place exclusive scan of both count arrays over the items; totals to ctrl[C_GT], ctrl[C_EQ].  One block of 1024.
__global__ void __launch_bounds__(1024)
k_tk_scan(int64_t nitems, int64_t* __restrict__ gtc, int64_t* __restrict__ eqc, int64_t* __restrict__ ctrl) {
  __shared__ int64_t wsg[32], wse[32], tot[2];
  int64_t carry_g = 0, carry_e = 0;
  for (int64_t base = 0; base < nitems; base += 1024 * TK_SCAN_SEG) {
    const int64_t i0 = base + (int64_t)threadIdx.x * TK_SCAN_SEG;
    int64_t g[TK_SCAN_SEG], e[TK_SCAN_SEG], sg = 0, se = 0;
#pragma unroll
    for (int q = 0; q < TK_SCAN_SEG; ++q) {
      const bool in = i0 + q < nitems;
      g[q] = in ? gtc[i0 + q] : 0;
      e[q] = in ? eqc[i0 + q] : 0;
      sg += g[q];
      se += e[q];
    }
    const int64_t ig = block_incl_scan(sg, wsg);
    const int64_t ie = block_incl_scan(se, wse);
    int64_t xg = carry_g + ig - sg, xe = carry_e + ie - se;
#pragma unroll
    for (int q = 0; q < TK_SCAN_SEG; ++q) {
      if (i0 + q < nitems) { gtc[i0 + q] = xg; eqc[i0 + q] = xe; }
      xg += g[q];
      xe += e[q];
    }
    if (threadIdx.x == 1023) { tot[0] = ig; tot[1] = ie; }      // block totals: the last thread's inclusive values
    __syncthreads();
    carry_g += tot[0];
    carry_e += tot[1];
    __syncthreads();
  }
  if (threadIdx.x == 0) { ctrl[C_GT] = carry_g; ctrl[C_EQ] = carry_e; }
}

// exclusive block scan of one uint32 per thread (blockDim.x == TK_THREADS); returns the exclusive value, *total the sum
__device__ __forceinline__ uint32_t block_excl_scan_u32(uint32_t v, uint32_t* ws, uint32_t* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0) {
    const uint32_t s = lane < TK_THREADS / 32 ? ws[lane] : 0u;
    uint32_t si = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, si, o);
      if (lane >= o) si += t;
    }
    if (lane < TK_THREADS / 32) ws[lane] = si - s;
    if (lane == TK_THREADS / 32 - 1) ws[TK_THREADS / 32] = si;
  }
  __syncthreads();
  const uint32_t r = ws[w] + inc - v;
  *total = ws[TK_THREADS / 32];
  __syncthreads();
  return r;
}

// Ordered write.  A candidate's slot is off + (#> tau before it) + min(#== tau before it, quota) in this band's index
// order; items holding nothing to write are skipped without reading them.  A thread visits four consecutive columns per
// step, so the block scan of the per-thread counts (packed: > tau in the high half, == tau in the low half) gives the
// index order.
template <bool VEC>
__global__ void __launch_bounds__(TK_THREADS)
k_tk_write(Band b, const int64_t* __restrict__ ctrl, const int64_t* __restrict__ gto, const int64_t* __restrict__ eqo,
           int64_t off, int64_t quota, int64_t cap, int64_t* __restrict__ oidx, float* __restrict__ oval) {
  __shared__ uint32_t ws[TK_THREADS / 32 + 1];
  const uint32_t tau = (uint32_t)ctrl[C_PREFIX];
  const int64_t nitems = b.rows * b.nc;
  const int64_t tot_g = ctrl[C_GT], tot_e = ctrl[C_EQ];
  constexpr int64_t STEP = 4 * TK_THREADS;
  for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x) {
    const int64_t G0 = gto[w], E0 = eqo[w];
    const int64_t ng_item = (w + 1 < nitems ? gto[w + 1] : tot_g) - G0;
    const int64_t ne_item = (w + 1 < nitems ? eqo[w + 1] : tot_e) - E0;
    if (ng_item == 0 && (ne_item == 0 || E0 >= quota)) continue;
    int64_t r, c0, c1;
    item_range(b, w, r, c0, c1);
    const float* row = b.s + r * b.n;
    const int64_t gidx0 = (b.row0 + r) * b.n;
    const int64_t base = VEC ? (c0 & ~(int64_t)3) : c0;
    int64_t Grun = G0, Erun = E0;
    for (int64_t js = base; js < c1; js += STEP) {
      const int64_t j = js + 4 * threadIdx.x;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      bool gt[4], eq[4];
      uint32_t lg = 0, le = 0;
      if (j < c1) load4<VEC>(row, j, c1, v);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool in = j + e >= c0 && j + e < c1 && !isnan(v[e]);
        const uint32_t key = in ? fkey(v[e]) : 0u;
        gt[e] = in && key > tau;
        eq[e] = in && key == tau;
        lg += gt[e] ? 1u : 0u;
        le += eq[e] ? 1u : 0u;
      }
      uint32_t total;
      const uint32_t x = block_excl_scan_u32((lg << 16) | le, ws, &total);
      int64_t pg = Grun + (x >> 16), pe = Erun + (x & 0xffffu);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        int64_t slot = -1;
        if (gt[e]) slot = off + pg + min(pe, quota);
        else if (eq[e] && pe < quota) slot = off + pg + pe;
        if (slot >= 0 && slot < cap) {
          oidx[slot] = gidx0 + j + e;
          oval[slot] = v[e];
        }
        pg += gt[e] ? 1 : 0;
        pe += eq[e] ? 1 : 0;
      }
      Grun += total >> 16;
      Erun += total & 0xffffu;
    }
  }
}

// persistent grid: as many CTAs of `kern` as are resident at once, at most one per work item
template <typename K>
unsigned tk_grid(K kern, int64_t nitems) {
  int dev = 0, sms = 148, per = 1;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kern, TK_THREADS, 0);
  const int64_t g = (int64_t)sms * (per > 0 ? per : 1);
  return (unsigned)(nitems < g ? (nitems > 0 ? nitems : 1) : g);
}

}  // namespace

extern "C" {

// [control 256 B][histogram (TK_BINS + 1) x int64][> tau per item x int64][== tau per item x int64]
int64_t mcgra_topk_workspace_bytes(int64_t rows, int64_t n, int64_t k) {
  (void)k;
  const int64_t nitems = (rows > 0 ? rows : 0) * tk_nc(n > 0 ? n : 1);
  return 256 + tk_align(TK_HIST_WORDS * 8) + 2 * tk_align((nitems > 0 ? nitems : 1) * 8);
}

int mcgra_topk_stage(int stage, const float* scores, int64_t row0, int64_t rows, int64_t n, int64_t k, void* ws,
                     int64_t out_offset, int64_t tie_quota, int64_t* out_idx, float* out_val, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (stage < 0 || stage > 7 || n < 2 || k < 1 || rows < 0 || row0 < 0 || row0 + rows > n || ws == nullptr) return -1;
  if (rows > 0 && scores == nullptr) return -1;
  char* p = (char*)ws;
  int64_t* ctrl = (int64_t*)p;
  unsigned long long* hist = (unsigned long long*)(p + 256);
  const int64_t nc = tk_nc(n);
  const int64_t nitems = rows * nc;
  int64_t* gtc = (int64_t*)(p + 256 + tk_align(TK_HIST_WORDS * 8));
  int64_t* eqc = (int64_t*)((char*)gtc + tk_align((nitems > 0 ? nitems : 1) * 8));
  const Band b{scores, row0, rows, n, nc};
  const bool vec = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(scores) & 15) == 0);
  if (stage == 0 || stage == 2 || stage == 4) {
    const int level = stage / 2;
    cudaError_t e = level == 0 ? cudaMemsetAsync(ws, 0, 256 + TK_HIST_WORDS * 8, st)
                               : cudaMemsetAsync(hist, 0, TK_HIST_WORDS * 8, st);
    if (e != cudaSuccess) return (int)e;
    if (nitems > 0) {
      if (vec) k_tk_hist<true><<<tk_grid(k_tk_hist<true>, nitems), TK_THREADS, 0, st>>>(b, level, ctrl, hist);
      else k_tk_hist<false><<<tk_grid(k_tk_hist<false>, nitems), TK_THREADS, 0, st>>>(b, level, ctrl, hist);
    }
  } else if (stage == 1 || stage == 3 || stage == 5) {
    k_tk_select<<<1, 1024, 0, st>>>(stage / 2, k, ctrl, hist);
  } else if (stage == 6) {
    if (nitems > 0) {
      if (vec) k_tk_count<true><<<tk_grid(k_tk_count<true>, nitems), TK_THREADS, 0, st>>>(b, ctrl, gtc, eqc);
      else k_tk_count<false><<<tk_grid(k_tk_count<false>, nitems), TK_THREADS, 0, st>>>(b, ctrl, gtc, eqc);
    }
    k_tk_scan<<<1, 1024, 0, st>>>(nitems, gtc, eqc, ctrl);
  } else {
    if (out_offset < 0 || tie_quota < 0) return -1;
    if (nitems > 0) {
      if (out_idx == nullptr || out_val == nullptr) return -1;
      if (vec) k_tk_write<true><<<tk_grid(k_tk_write<true>, nitems), TK_THREADS, 0, st>>>(b, ctrl, gtc, eqc, out_offset,
                                                                                 tie_quota, k, out_idx, out_val);
      else k_tk_write<false><<<tk_grid(k_tk_write<false>, nitems), TK_THREADS, 0, st>>>(b, ctrl, gtc, eqc, out_offset,
                                                                                 tie_quota, k, out_idx, out_val);
    }
  }
  MCGRA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
