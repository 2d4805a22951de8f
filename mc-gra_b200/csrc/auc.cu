// ROC-AUC / average precision over N (score, label) pairs and a stable descending arg-sort, on the GPU.
//
// Reference work replaced: main.metric_pool (MC-GRA/main.py:66-75: .cpu() of two n^2 vectors + sklearn roc_curve
// + auc) and the AP of gcn_parameterized.metric (MC-GRA/gcn_parameterized.py:55-65).  sklearn semantics (stable
// descending sort, thresholds at distinct scores, trapezoid => ties contribute 1/2; AP = sum_k (R_k - R_{k-1}) P_k).
//
// Method: positives are few (true edges), negatives are ~n^2.  The positives' keys are radix-sorted (LSD, 8-bit
// digits, stable); every negative is then ranked against them by binary search:
//     2*AUC*P*N = sum_neg ( 2 * #pos_above + #pos_tied )            (exact integers, uint64)
// and a histogram of the negatives' upper-bound positions gives fp(>= v) for every distinct positive score v,
// from which AP follows in float64.  The same radix sort with an index payload gives the full ranking.
#include "common.cuh"

namespace {

constexpr int CHUNK = 4096;   // elements per single-warp block

__global__ void k_hist(const uint32_t* __restrict__ keys, int64_t N, int shift, uint32_t* __restrict__ hist /*[256][nb]*/,
                       int64_t nb) {
  __shared__ uint32_t h[256];
  for (int e = threadIdx.x; e < 256; e += blockDim.x) h[e] = 0;
  __syncthreads();
  const int64_t b0 = (int64_t)blockIdx.x * CHUNK;
  for (int e = threadIdx.x; e < CHUNK; e += blockDim.x) {
    const int64_t g = b0 + e;
    if (g < N) atomicAdd(&h[(keys[g] >> shift) & 255u], 1u);
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 256; e += blockDim.x) hist[(int64_t)e * nb + blockIdx.x] = h[e];
}

// exclusive scan of hist (bin-major, block-minor) into 64-bit offsets; single block, sequential over chunks
__global__ void k_scan(const uint32_t* __restrict__ hist, int64_t total, int64_t* __restrict__ offs) {
  __shared__ int64_t carry;
  __shared__ int64_t wsum[32];
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t base = 0; base < total; base += blockDim.x) {
    const int64_t g = base + threadIdx.x;
    int64_t v = g < total ? (int64_t)hist[g] : 0;
    int64_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
      int64_t s = lane < (int)(blockDim.x >> 5) ? wsum[lane] : 0;
      int64_t si = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, si, o);
        if (lane >= o) si += t;
      }
      wsum[lane] = si - s;   // exclusive warp offsets
    }
    __syncthreads();
    const int64_t excl = carry + wsum[w] + inc - v;
    if (g < total) offs[g] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = excl + v;
    __syncthreads();
  }
}

// stable scatter: one warp per chunk, elements visited in order, match_any gives the in-warp rank
template <typename PAY>
__global__ void __launch_bounds__(32)
k_scatter(const uint32_t* __restrict__ kin, const PAY* __restrict__ pin, int64_t N, int shift,
          const int64_t* __restrict__ offs, int64_t nb, uint32_t* __restrict__ kout, PAY* __restrict__ pout) {
  __shared__ int64_t pos[256];
  const int lane = threadIdx.x;
  for (int e = lane; e < 256; e += 32) pos[e] = offs[(int64_t)e * nb + blockIdx.x];
  __syncwarp();
  const int64_t b0 = (int64_t)blockIdx.x * CHUNK;
  for (int it = 0; it < CHUNK / 32; ++it) {
    const int64_t g = b0 + it * 32 + lane;
    const bool ok = g < N;
    const uint32_t k = ok ? kin[g] : 0xffffffffu;
    const uint32_t dg = ok ? ((k >> shift) & 255u) : 256u + lane;   // inactive lanes never match anything
    const unsigned peers = __match_any_sync(0xffffffffu, dg);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    int64_t base = 0;
    if (ok) base = pos[dg];
    __syncwarp();
    if (ok) {
      kout[base + rank] = k;
      if (pin != nullptr) pout[base + rank] = pin[g];
      if (rank == __popc(peers) - 1) pos[dg] = base + rank + 1;
    }
    __syncwarp();
  }
}

__global__ void k_compact_pos(const float* __restrict__ scores, const uint8_t* __restrict__ labels, int64_t N,
                              uint32_t* __restrict__ poskeys, int64_t cap, unsigned long long* __restrict__ counter) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < N; g += stride) {
    if (labels[g]) {
      const unsigned long long s = atomicAdd(counter, 1ull);
      if ((int64_t)s < cap) poskeys[s] = fkey(scores[g]);
    }
  }
}

__device__ __forceinline__ int64_t upper_bound(const uint32_t* a, int64_t n, uint32_t k) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] <= k) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// every negative against the sorted positives.  A 1024-entry sample of the sorted keys sits in shared memory: the
// search does ~10 steps there and only log2(npos / 1024) steps in global memory; upper_bound continues from lower_bound
// only when a positive has the same key, so a negative costs ~10 global loads instead of 2 * log2(npos).
constexpr int RANK_TAB = 1024;
__global__ void __launch_bounds__(256)
k_rank_negatives(const float* __restrict__ scores, const uint8_t* __restrict__ labels, int64_t N,
                 const uint32_t* __restrict__ pos, const unsigned long long* __restrict__ counter,
                 unsigned long long* __restrict__ hist /*[npos+1]*/, unsigned long long* __restrict__ sums /*[2]*/) {
  __shared__ uint32_t tab[RANK_TAB];
  const int npos = (int)*counter;
  const int step = (npos + RANK_TAB - 1) / RANK_TAB > 0 ? (npos + RANK_TAB - 1) / RANK_TAB : 1;
  const int ntab = (npos + step - 1) / step;               // tab[t] = pos[t * step]
  for (int t = threadIdx.x; t < ntab; t += blockDim.x) tab[t] = pos[(int64_t)t * step];
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned long long twice = 0, nneg = 0;
  const int lane = threadIdx.x & 31;
  const int64_t nround = (N + stride - 1) / stride;
  for (int64_t rd = 0; rd < nround; ++rd) {
    const int64_t g = rd * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool neg = (g < N) && !labels[g];
    int ub = -1 - lane;         // unique sentinel so inactive lanes do not aggregate
    if (neg) {
      const uint32_t k = fkey(scores[g]);
      // first sample >= k in the table: lower_bound(pos, k) lies in ((t-1) * step, t * step]
      int lo = 0, hi = ntab;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tab[mid] < k) lo = mid + 1; else hi = mid;
      }
      int l = lo == 0 ? 0 : (lo - 1) * step + 1;
      int h = lo == ntab ? npos : lo * step;
      while (l < h) {
        const int mid = (l + h) >> 1;
        if (pos[mid] < k) l = mid + 1; else h = mid;
      }
      const int lb = l;
      ub = (lb < npos && pos[lb] == k) ? (int)upper_bound(pos, npos, k) : lb;    // ties with a positive are rare
      twice += 2ull * (unsigned long long)(npos - ub) + (unsigned long long)(ub - lb);
      nneg += 1;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, ub);
    if (neg && lane == (__ffs(peers) - 1)) atomicAdd(hist + ub, (unsigned long long)__popc(peers));
  }
  // block reduce
  __shared__ unsigned long long r0[8], r1[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    twice += __shfl_xor_sync(0xffffffffu, twice, o);
    nneg += __shfl_xor_sync(0xffffffffu, nneg, o);
  }
  if (lane == 0) { r0[threadIdx.x >> 5] = twice; r1[threadIdx.x >> 5] = nneg; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long a = 0, b = 0;
    for (int w = 0; w < 8; ++w) { a += r0[w]; b += r1[w]; }
    if (a) atomicAdd(sums, a);
    if (b) atomicAdd(sums + 1, b);
  }
}

// Ranking against the DISTINCT positive keys, search table in dynamic shared memory.
//
// What bounds k_rank_negatives (measured, profiles/r02_auc_ablation.txt, 4.3e9 negatives): not the histogram updates (5 ms) but the
// searches (87 of 119 ms) -- after its 1024-sample table every lane walks the sorted array in its own 128-byte line, and a
// negative that ties with a positive is searched twice (lower and upper bound).  The scores of the reference's ensemble
// (sums of sigmoids of clamped grams + integer label terms) are heavily tied: 2 055 distinct values among 294 878 positives at
// the bench size.  So the sorted positives are first reduced to their distinct keys U[0 .. nU) with C[u] = number of positives
// below U[u] (C[nU] = npos; k_unique_pos), and a negative needs ONE search over U: lb = C[u], ub = C[u + 1] if U[u] ties with
// it, else lb.  U and C both live in shared memory while 2 nU + 1 <= 57 344 words; beyond that U is sampled (57 344 samples,
// the remaining log2(nU / 57 344) levels in global memory) and C is read from global memory.  The search has a uniform trip
// count (branch-free halving), and a thread ranks 4 consecutive pairs per round (16-byte score / 4-byte label loads, the next
// round's loaded before the current one is ranked).
extern __shared__ uint32_t dyn_tab[];

// distinct keys of the sorted positives; single block (npos is a few 1e5: < 1 ms)
__global__ void __launch_bounds__(1024)
k_unique_pos(const uint32_t* __restrict__ pos, unsigned long long* __restrict__ counter, int64_t npos_max,
             uint32_t* __restrict__ U, uint32_t* __restrict__ Cidx) {
  __shared__ int carry;
  __shared__ int wsum[32];
  const int64_t np64 = (int64_t)counter[0];
  const int npos = (int)(np64 < npos_max ? np64 : npos_max);
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < npos; base += 1024) {
    const int t = base + threadIdx.x;
    const int flag = (t < npos && (t == 0 || pos[t] != pos[t - 1])) ? 1 : 0;
    int inc = flag;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += v;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
      const int sv = wsum[lane];
      int si = sv;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, si, o);
        if (lane >= o) si += v;
      }
      wsum[lane] = si - sv;
    }
    __syncthreads();
    const int excl = carry + wsum[w] + inc - flag;
    if (flag) { U[excl] = pos[t]; Cidx[excl] = (uint32_t)t; }
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + flag;
    __syncthreads();
  }
  if (threadIdx.x == 0) { Cidx[carry] = (uint32_t)npos; counter[3] = (unsigned long long)carry; }
}

// Sampled mode with <= 3 distinct keys per sample: segment t -> one aligned 32-byte block
//   [U[t step .. t step + step) | C[t step .. t step + step]]   (keys beyond nU = +inf, indices clamped to C[nU] = npos)
// so that a negative needs one sector of global memory instead of a walk over U plus two reads of C (each divergent
// global access costs ~15 ms per 4.3e9 negatives: 32 L1 wavefronts per warp).
__global__ void k_build_blocks(const uint32_t* __restrict__ U, const uint32_t* __restrict__ Cidx,
                               const unsigned long long* __restrict__ counter, int tab_cap, uint32_t* __restrict__ blocks) {
  const int nU = (int)counter[3];
  if (2 * (int64_t)nU + 1 <= (int64_t)tab_cap) return;
  const int step = (nU + tab_cap - 1) / tab_cap;
  if (step > 3) return;
  const int ntab = (nU + step - 1) / step;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < ntab; t += gridDim.x * blockDim.x) {
    uint32_t* w = blocks + 8 * (int64_t)t;
    for (int i = 0; i < 8; ++i) {
      uint32_t v = 0xffffffffu;
      if (i < step) {
        const int idx = t * step + i;
        if (idx < nU) v = U[idx];
      } else if (i <= 2 * step) {
        const int idx = t * step + (i - step);
        v = Cidx[idx < nU ? idx : nU];
      }
      w[i] = v;
    }
  }
}

constexpr int RK_E = 4;       // pairs per thread and round
__global__ void __launch_bounds__(1024, 1)
k_rank_negatives_tab(const float* __restrict__ scores, const uint8_t* __restrict__ labels, int64_t N,
                     const uint32_t* __restrict__ U, const uint32_t* __restrict__ Cidx, const uint4* __restrict__ blocks,
                     const unsigned long long* __restrict__ counter, unsigned long long* __restrict__ hist /*[npos+1]*/,
                     unsigned long long* __restrict__ sums /*[2]*/, int tab_cap) {
  uint32_t* tab = dyn_tab;
  const int npos = (int)counter[0];
  const int nU = (int)counter[3];
  const bool both = 2 * (int64_t)nU + 1 <= (int64_t)tab_cap;      // keys and start indices in shared memory
  const bool hsm = 3 * (int64_t)nU + 2 <= (int64_t)tab_cap;       // ... and a CTA-private histogram over the nU + 1 possible ub
  const int step = both ? 1 : (nU + tab_cap - 1) / tab_cap;
  const int ntab = both ? nU : (nU + step - 1) / step;             // tab[t] = U[t * step]
  uint32_t* Cs = tab + ntab;
  uint32_t* Hs = Cs + nU + 1;
  const bool ident = nU == npos;
  const bool blocked = !both && step <= 3;                          // sampled table + one 32-byte block per segment (k_build_blocks)
  for (int t = threadIdx.x; t < ntab; t += blockDim.x) tab[t] = U[(int64_t)t * step];
  if (both)
    for (int t = threadIdx.x; t <= nU; t += blockDim.x) Cs[t] = Cidx[t];
  if (hsm)
    for (int t = threadIdx.x; t <= nU; t += blockDim.x) Hs[t] = 0u;
  __syncthreads();
  const bool vec = ((reinterpret_cast<uintptr_t>(scores) & 15) == 0) && ((reinterpret_cast<uintptr_t>(labels) & 3) == 0);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * RK_E;
  const int64_t nround = (N + stride - 1) / stride;
  const int lane = threadIdx.x & 31;
  unsigned long long twice = 0, nneg = 0;

  auto load = [&](int64_t g, float (&sc)[RK_E], bool (&neg)[RK_E]) {
    if (vec && g + RK_E <= N) {
      const float4 s4 = *reinterpret_cast<const float4*>(scores + g);
      const uchar4 l4 = *reinterpret_cast<const uchar4*>(labels + g);
      sc[0] = s4.x; sc[1] = s4.y; sc[2] = s4.z; sc[3] = s4.w;
      neg[0] = !l4.x; neg[1] = !l4.y; neg[2] = !l4.z; neg[3] = !l4.w;
    } else {
#pragma unroll
      for (int e = 0; e < RK_E; ++e) {
        const bool in = g + e < N;
        neg[e] = in && !labels[in ? g + e : 0];
        sc[e] = in ? scores[g + e] : 0.f;
      }
    }
  };

  int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * RK_E;
  float sc[RK_E], scn[RK_E];
  bool neg[RK_E], negn[RK_E];
#pragma unroll
  for (int e = 0; e < RK_E; ++e) { sc[e] = scn[e] = 0.f; neg[e] = negn[e] = false; }
  if (g < N) load(g, sc, neg);
  for (int64_t rd = 0; rd < nround; ++rd) {
    const int64_t gn = g + stride;
#pragma unroll
    for (int e = 0; e < RK_E; ++e) negn[e] = false;
    if (rd + 1 < nround && gn < N) load(gn, scn, negn);
    {                                                   // rounds further ahead: into L2 (no registers)
      const int64_t gp = g + 4 * stride;
      if (gp + RK_E <= N) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(scores + gp));
        if ((lane & 3) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(labels + gp));
      }
    }
    uint32_t k[RK_E];
    int u[RK_E];
    int lb[RK_E], ub[RK_E], vb[RK_E];     // vb: ub in the space of distinct keys (ub = C[vb])
#pragma unroll
    for (int e = 0; e < RK_E; ++e) { k[e] = fkey(sc[e]); u[e] = 0; lb[e] = ub[e] = vb[e] = 0; }
    if (blocked) {
      // segment t = [t * step, (t + 1) * step) of the distinct keys, tab[t] = its first key.  t = last sample <= k; then
      // the keys below k, a tie and the start indices C[u], C[u + 1] all come from the segment's 32-byte block.
      int base[RK_E];
#pragma unroll
      for (int e = 0; e < RK_E; ++e) base[e] = 0;
      int len = ntab;
      while (len > 1) {
        const int half = len >> 1;
#pragma unroll
        for (int e = 0; e < RK_E; ++e) base[e] += (tab[base[e] + half - 1] <= k[e]) ? half : 0;
        len -= half;
      }
#pragma unroll
      for (int pr = 0; pr < RK_E; pr += 2) {           // two blocks in flight (register budget of 1024 threads)
        uint32_t w[2][8];
        int t[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int e = pr + q;
          t[q] = base[e] + ((tab[base[e]] <= k[e]) ? 1 : 0) - 1;
          const uint4* bp = blocks + 2 * (int64_t)(t[q] < 0 ? 0 : t[q]);
          // one 256-bit load (LDG.E.256): a divergent access costs its L1 wavefronts per instruction, not per byte
          asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                       : "=r"(w[q][0]), "=r"(w[q][1]), "=r"(w[q][2]), "=r"(w[q][3]), "=r"(w[q][4]), "=r"(w[q][5]),
                         "=r"(w[q][6]), "=r"(w[q][7])
                       : "l"(bp));
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int e = pr + q;
          const uint32_t w0 = w[q][0], w1 = w[q][1], w2 = w[q][2], w3 = w[q][3];
          const uint32_t w4 = w[q][4], w5 = w[q][5], w6 = w[q][6], w7 = w[q][7];
          const uint32_t kk = k[e];
          const bool s1 = step > 1, s2 = step > 2;
          const int m = (w0 < kk ? 1 : 0) + ((s1 && w1 < kk) ? 1 : 0) + ((s2 && w2 < kk) ? 1 : 0);
          const bool tied = (w0 == kk) || (s1 && w1 == kk) || (s2 && w2 == kk);
          const int ci = step + m;                       // C[u] sits at word step + m of the block, C[u + 1] behind it
          const uint32_t c0 = ci == 1 ? w1 : ci == 2 ? w2 : ci == 3 ? w3 : ci == 4 ? w4 : ci == 5 ? w5 : w6;
          const uint32_t c1 = ci == 1 ? w2 : ci == 2 ? w3 : ci == 3 ? w4 : ci == 4 ? w5 : ci == 5 ? w6 : w7;
          lb[e] = t[q] < 0 ? 0 : (int)c0;
          ub[e] = t[q] < 0 ? 0 : (tied ? (int)c1 : (int)c0);
        }
      }
    } else {
    if (ntab > 0) {
      // RK_E interleaved searches with one trip count
      int base[RK_E];
#pragma unroll
      for (int e = 0; e < RK_E; ++e) base[e] = 0;
      int len = ntab;
      while (len > 1) {
        const int half = len >> 1;
#pragma unroll
        for (int e = 0; e < RK_E; ++e) base[e] += (tab[base[e] + half - 1] < k[e]) ? half : 0;
        len -= half;
      }
#pragma unroll
      for (int e = 0; e < RK_E; ++e) u[e] = base[e] + ((tab[base[e]] < k[e]) ? 1 : 0);
      if (step > 1) {
        // u = first SAMPLE not below k: the distinct key sought lies in ((u - 1) * step, u * step]  (u == ntab: up to nU).
        // The RK_E segment searches run interleaved with one trip count (segments are <= step long; entries beyond a
        // segment's end count as +inf), so that their global loads overlap instead of forming one dependent chain.
        int l[RK_E], h[RK_E];
#pragma unroll
        for (int e = 0; e < RK_E; ++e) {
          l[e] = u[e] == 0 ? 0 : (u[e] - 1) * step + 1;
          h[e] = u[e] == ntab ? nU : u[e] * step;
        }
        int len2 = step;
        while (len2 > 1) {
          const int half = len2 >> 1;
#pragma unroll
          for (int e = 0; e < RK_E; ++e) {
            const int idx = l[e] + half - 1;
            const uint32_t v = idx < h[e] ? U[idx] : 0xffffffffu;
            l[e] += (v < k[e]) ? half : 0;
          }
          len2 -= half;
        }
#pragma unroll
        for (int e = 0; e < RK_E; ++e) {
          const uint32_t v = l[e] < h[e] ? U[l[e]] : 0xffffffffu;
          u[e] = l[e] + ((v < k[e]) ? 1 : 0);
        }
      }
    } else {
#pragma unroll
      for (int e = 0; e < RK_E; ++e) u[e] = 0;
    }
#pragma unroll
    for (int e = 0; e < RK_E; ++e) {
      if (both) {
        const bool tied = u[e] < nU && tab[u[e]] == k[e];
        lb[e] = (int)Cs[u[e]];
        vb[e] = u[e] + (tied ? 1 : 0);
        ub[e] = tied ? (int)Cs[vb[e]] : lb[e];
      } else {
        const bool tied = u[e] < nU && U[u[e]] == k[e];
        vb[e] = u[e] + (tied ? 1 : 0);
        if (ident) { lb[e] = u[e]; ub[e] = vb[e]; }       // all positives distinct: C[u] = u
        else { lb[e] = (int)Cidx[u[e]]; ub[e] = tied ? (int)Cidx[vb[e]] : lb[e]; }
      }
    }
    }      // !blocked
    unsigned int tw32 = 0;
#pragma unroll
    for (int e = 0; e < RK_E; ++e) {
      if (neg[e]) {
        tw32 += 2u * (unsigned)(npos - ub[e]) + (unsigned)(ub[e] - lb[e]);      // 12 npos < 2^32: npos < 2^28 checked by the host
        nneg += 1;
      }
      const int sent = -1 - lane;         // unique sentinel so inactive lanes do not aggregate
      if (hsm) {
        // few distinct values = hot bins: global updates of the same ~nU addresses serialise in L2 (90 of 120 ms measured)
        const unsigned peers = __match_any_sync(0xffffffffu, neg[e] ? vb[e] : sent);
        if (neg[e] && lane == (__ffs(peers) - 1)) atomicAdd(Hs + vb[e], (unsigned)__popc(peers));
      } else {
        const unsigned peers = __match_any_sync(0xffffffffu, neg[e] ? ub[e] : sent);
        if (neg[e] && lane == (__ffs(peers) - 1)) atomicAdd(hist + ub[e], (unsigned long long)__popc(peers));
      }
    }
    twice += (unsigned long long)tw32;
    g = gn;
#pragma unroll
    for (int e = 0; e < RK_E; ++e) { sc[e] = scn[e]; neg[e] = negn[e]; }
  }
  __shared__ unsigned long long r0[32], r1[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    twice += __shfl_xor_sync(0xffffffffu, twice, o);
    nneg += __shfl_xor_sync(0xffffffffu, nneg, o);
  }
  if (lane == 0) { r0[threadIdx.x >> 5] = twice; r1[threadIdx.x >> 5] = nneg; }
  __syncthreads();
  if (hsm) {
    for (int t = threadIdx.x; t <= nU; t += blockDim.x) {
      const uint32_t c = Hs[t];
      if (c) atomicAdd(hist + Cs[t], (unsigned long long)c);
    }
  }
  if (threadIdx.x == 0) {
    unsigned long long a = 0, b = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += r0[w]; b += r1[w]; }
    if (a) atomicAdd(sums, a);
    if (b) atomicAdd(sums + 1, b);
  }
}

int g_auc_engine = 1;      // mcgra_set_engine(6, v): 0 k_rank_negatives (1024-sample table), 1 k_rank_negatives_tab (default)
constexpr int TAB_CAP_MAX = 57344;      // 224 KB of dynamic shared memory

// suffix sums of hist -> fp(>= pos[t]) = sum_{j > t} hist[j]; AP over distinct positive values.  Single block.
__global__ void __launch_bounds__(1024)
k_ap_finish(const uint32_t* __restrict__ pos, const unsigned long long* __restrict__ counter,
            unsigned long long* __restrict__ hist, const unsigned long long* __restrict__ sums,
            double* __restrict__ out) {
  const int64_t npos = (int64_t)*counter;
  __shared__ unsigned long long carry;
  __shared__ unsigned long long wsum[32];
  __shared__ double red[32];
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  // in-place inclusive suffix scan over j = npos .. 0 : after it hist[j] = sum_{q >= j} hist[q]
  for (int64_t base = npos; base >= 0; base -= blockDim.x) {
    const int64_t j = base - threadIdx.x;
    unsigned long long v = j >= 0 ? hist[j] : 0ull;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    if (w == 0) {
      unsigned long long s = wsum[lane], si = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, si, o);
        if (lane >= o) si += t;
      }
      wsum[lane] = si - s;
    }
    __syncthreads();
    const unsigned long long tot = carry + wsum[w] + inc;
    if (j >= 0) hist[j] = tot;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = tot;
    __syncthreads();
  }
  // AP = (1/npos) sum over first occurrences t of a distinct value: cnt * tp / (tp + fp),
  //   tp = npos - t (positives >= v), fp = hist[t+1] (negatives with upper_bound > t), cnt = run length
  double ap = 0.0;
  for (int64_t t = threadIdx.x; t < npos; t += blockDim.x) {
    if (t == 0 || pos[t] != pos[t - 1]) {
      int64_t e = t + 1;
      while (e < npos && pos[e] == pos[t]) ++e;
      const double tp = (double)(npos - t), fp = (double)hist[t + 1];
      ap += (double)(e - t) * tp / (tp + fp);
    }
  }
  ap = warp_sum_d(ap);
  if (lane == 0) red[w] = ap;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) s += red[q];
    const double P = (double)npos, Nn = (double)sums[1];
    out[0] = (P > 0 && Nn > 0) ? (double)sums[0] / (2.0 * P * Nn) : 0.0;   // AUC
    out[1] = P > 0 ? s / P : 0.0;                                          // AP
    out[2] = P;
    out[3] = Nn;
  }
}

__global__ void k_make_keys_desc(const float* __restrict__ scores, int64_t N, uint32_t* __restrict__ keys,
                                 int64_t* __restrict__ idx) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < N; g += stride) {
    keys[g] = ~fkey(scores[g]);     // ascending sort of ~key == descending score; LSD stability keeps index order
    idx[g] = g;
  }
}

inline int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }
constexpr int64_t TAB_CAP_MAX_WS = 57344;      // = TAB_CAP_MAX: one 32-byte block per table sample

// LSD radix sort of `keys` (and payload) in place using `tmp` buffers; 4 passes of 8 bits
template <typename PAY>
int radix_sort(uint32_t* keys, PAY* pay, uint32_t* keys_tmp, PAY* pay_tmp, int64_t N, uint32_t* hist, int64_t* offs,
               cudaStream_t st) {
  if (N <= 0) return 0;
  const int64_t nb = (N + CHUNK - 1) / CHUNK;
  uint32_t* kin = keys; uint32_t* kout = keys_tmp;
  PAY* pin = pay; PAY* pout = pay_tmp;
  for (int pass = 0; pass < 4; ++pass) {
    k_hist<<<(unsigned)nb, 256, 0, st>>>(kin, N, pass * 8, hist, nb);
    k_scan<<<1, 1024, 0, st>>>(hist, nb * 256, offs);
    k_scatter<PAY><<<(unsigned)nb, 32, 0, st>>>(kin, pin, N, pass * 8, offs, nb, kout, pout);
    uint32_t* tk = kin; kin = kout; kout = tk;
    PAY* tp = pin; pin = pout; pout = tp;
  }
  MCGRA_LAUNCH_CHECK();
  return 0;   // after 4 passes the result is back in `keys` / `pay`
}

}  // namespace

extern "C" {

int mcgra_set_auc_engine_(int value) {
  if (value != 0 && value != 1) return -1;
  g_auc_engine = value;
  return 0;
}

// workspace layout (bytes): [counter+sums 256][poskeys cap*4][poskeys_tmp cap*4][hist_sort][offs_sort][hist cap+1 u64]
// [start indices of the distinct keys cap+1 u32][segment blocks 57 344 x 32 B]   (counter block: [0] npos, [1..2] sums, [3] number of distinct keys)
int64_t mcgra_auc_workspace_bytes(int64_t N, int64_t npos_max) {
  (void)N;
  const int64_t nb = (npos_max + CHUNK - 1) / CHUNK + 1;
  return 256 + 2 * align256(npos_max * 4) + align256(nb * 256 * 4) + align256(nb * 256 * 8) +
         align256((npos_max + 2) * 8) + align256((npos_max + 2) * 4) + TAB_CAP_MAX_WS * 32;
}

// The three stages of mcgra_auc_ap, callable separately so that the n^2 pairs can be split over ranks by row bands:
//   stage 0  compact the positives' keys of the local pairs (ws: counter[0] = count, pos[0 .. count))
//            -- the caller may then replace pos / counter[0] by the GLOBAL positives (all-gather)
//   stage 1  sort the positives, rank the local negatives against them (ws: hist, sums)
//            -- the caller may then sum hist / sums over ranks (all-reduce)
//   stage 2  AUC / AP from the counts.
// Workspace byte offsets: counter 0, sums 8, pos 256, hist = mcgra_auc_hist_offset(npos_max).
int64_t mcgra_auc_hist_offset(int64_t npos_max) {
  const int64_t nb = (npos_max + CHUNK - 1) / CHUNK + 1;
  return 256 + 2 * align256(npos_max * 4) + align256(nb * 256 * 4) + align256(nb * 256 * 8);
}

int mcgra_auc_stage(int stage, const float* scores, const uint8_t* labels, int64_t N, int64_t npos_max, void* ws,
                    double* out, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (npos_max <= 0 || stage < 0 || stage > 2) return -1;
  char* p = (char*)ws;
  unsigned long long* counter = (unsigned long long*)p;       // [0] npos, [1..2] sums
  unsigned long long* sums = counter + 1;
  p += 256;
  uint32_t* pos = (uint32_t*)p; p += align256(npos_max * 4);
  uint32_t* pos_tmp = (uint32_t*)p; p += align256(npos_max * 4);
  const int64_t nb = (npos_max + CHUNK - 1) / CHUNK + 1;
  uint32_t* hs = (uint32_t*)p; p += align256(nb * 256 * 4);
  int64_t* offs = (int64_t*)p; p += align256(nb * 256 * 8);
  unsigned long long* hist = (unsigned long long*)p;
  if (stage == 0) {
    cudaError_t e = cudaMemsetAsync(ws, 0, 256, st);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemsetAsync(hist, 0, (npos_max + 2) * 8, st);
    if (e != cudaSuccess) return (int)e;
    // keys of unused slots sort to the top and are ignored (counter gives the true count); fill with 0xff
    e = cudaMemsetAsync(pos, 0xff, npos_max * 4, st);
    if (e != cudaSuccess) return (int)e;
    if (N > 0) k_compact_pos<<<148 * 8, 256, 0, st>>>(scores, labels, N, pos, npos_max, counter);
  } else if (stage == 1) {
    int rc = radix_sort<uint32_t>(pos, nullptr, pos_tmp, nullptr, npos_max, hs, offs, st);
    if (rc) return rc;
    if (N > 0 && g_auc_engine == 1 && npos_max < (1LL << 28)) {      // (per-round 32-bit partial sums: 12 npos < 2^32)
      // distinct keys into the (now free) sort buffer, start indices behind the histogram
      uint32_t* Cidx = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(hist) + align256((npos_max + 2) * 8));
      k_unique_pos<<<1, 1024, 0, st>>>(pos, counter, npos_max, pos_tmp, Cidx);
      // table capacity (32-bit words): keys + start indices + private histogram of all distinct values when they fit, else
      // what fits of them (the kernel decides from the number of distinct keys), at least the largest sample
      const int64_t want = 3 * npos_max + 2;
      const int cap = (int)(want < TAB_CAP_MAX ? (want > 1024 ? want : 1024) : TAB_CAP_MAX);
      const size_t smem = (size_t)cap * 4;
      static bool attr_set = false;
      if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(k_rank_negatives_tab, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             TAB_CAP_MAX * 4);
        if (e != cudaSuccess) return (int)e;
        attr_set = true;
      }
      uint32_t* blocks = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(Cidx) + align256((npos_max + 2) * 4));
      if (want > cap) k_build_blocks<<<64, 256, 0, st>>>(pos_tmp, Cidx, counter, cap, blocks);
      k_rank_negatives_tab<<<148, 1024, smem, st>>>(scores, labels, N, pos_tmp, Cidx, reinterpret_cast<const uint4*>(blocks),
                                                    counter, hist, sums, cap);
    } else if (N > 0) {
      k_rank_negatives<<<148 * 8, 256, 0, st>>>(scores, labels, N, pos, counter, hist, sums);
    }
  } else {
    k_ap_finish<<<1, 1024, 0, st>>>(pos, counter, hist, sums, out);
  }
  MCGRA_LAUNCH_CHECK();
  return 0;
}

int mcgra_auc_ap(const float* scores, const uint8_t* labels, int64_t N, int64_t npos_max, void* ws, double* out,
                 void* stream) {
  if (N <= 0 || npos_max <= 0) return -1;
  for (int stage = 0; stage < 3; ++stage) {
    const int rc = mcgra_auc_stage(stage, scores, labels, N, npos_max, ws, out, stream);
    if (rc) return rc;
  }
  return 0;
}

// workspace: [keys N*4][keys_tmp N*4][idx_tmp N*8][hist][offs]
int64_t mcgra_sort_workspace_bytes(int64_t N) {
  const int64_t nb = (N + CHUNK - 1) / CHUNK + 1;
  return 2 * align256(N * 4) + align256(N * 8) + align256(nb * 256 * 4) + align256(nb * 256 * 8);
}

int mcgra_argsort_desc(const float* scores, int64_t N, int64_t* order, void* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (N <= 0) return 0;
  char* p = (char*)ws;
  uint32_t* keys = (uint32_t*)p; p += align256(N * 4);
  uint32_t* keys_tmp = (uint32_t*)p; p += align256(N * 4);
  int64_t* idx_tmp = (int64_t*)p; p += align256(N * 8);
  const int64_t nb = (N + CHUNK - 1) / CHUNK + 1;
  uint32_t* hs = (uint32_t*)p; p += align256(nb * 256 * 4);
  int64_t* offs = (int64_t*)p;
  k_make_keys_desc<<<148 * 8, 256, 0, st>>>(scores, N, keys, order);
  return radix_sort<int64_t>(keys, order, keys_tmp, idx_tmp, N, hs, offs, st);
}

}  // extern "C"
