/*
 * mcgra.h -- C ABI of libmcgra_b200.so: hand-written sm_100a CUDA kernels for the MC-GRA PGD attack
 * inner loop (reference: /root/reference/MC-GRA/topology_attack.py:161-324 and the helpers it calls).
 *
 * The reference has no FFI of its own (it is pure PyTorch); each entry point below replaces the ATen
 * call sequence of the reference lines it cites.  The Python host (mc-gra_b200/) binds these with ctypes.
 *
 * Conventions
 *   - extern "C"; every function returns int: 0 ok, >0 a cudaError_t, <0 an argument error.
 *   - never allocates, never synchronises, never throws: the caller owns every buffer, all work is
 *     enqueued on the cudaStream_t passed as `void* stream`.
 *   - fp32 data, int64 sizes, device pointers unless a parameter says "host".
 *   - PACKED vector  : reference layout, strict lower triangle row-major, k = i(i-1)/2 + j, i > j
 *                      (topology_attack.py:372-374).
 *   - TILED triangle : working layout of the loop.  T = ceil(n/128) tile rows; tile (I,J), J <= I, is a
 *                      contiguous row-major 128x128 fp32 block at element offset
 *                      (I(I+1)/2 + J - tr0(tr0+1)/2) * 16384 of a buffer that holds tile rows [tr0,tr1)
 *                      (one rank's shard).  Entry (a,b) of the tile is element (i,j) = (128I+a, 128J+b);
 *                      it is "valid" iff j < i < n, every other entry is kept at 0.
 *   - PARAMETER VIEW : the optimised parameter is stored lazily as the un-projected Adam output x'
 *                      together with a device scalar mu; the parameter value is clamp(x' - mu, 0, 1)
 *                      (topology_attack.py:338-347).  raw != 0 means "the buffer is a user-provided raw
 *                      parameter": value = x', forward uses clamp(x',0,1) with the clamp's gradient mask
 *                      (topology_attack.py:474-478).  raw == 2: the buffer already holds the parameter in [0,1]
 *                      (mcgra_fold_adam with store_clamped, used when the edge budget can never bind).
 */
#ifndef MCGRA_H
#define MCGRA_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MCGRA_TILE 128
#define MCGRA_HID 16            /* GCN hidden width, hard-coded in the reference (main.py:175) */
#define MCGRA_MAXC 32           /* max classes handled by the node kernels */

/* measures for the n x n terms c1/c2 and the n x d terms c9/c10 (topology_attack.py:190-208) */
enum { MCGRA_M_NONE = 0, MCGRA_M_MSE = 1, MCGRA_M_KL = 2, MCGRA_M_HSIC = 3, MCGRA_M_CKA = 4, MCGRA_M_DP = 5,
       MCGRA_M_PRE = 6 /* element-wise gradient of the n x n terms supplied as tiles (Ftiles = dL/dA_ij + dL/dA_ji,
                          Fdiag = dL/dA_ii): used for measures whose n x n contraction is computed upstream */,
       MCGRA_M_KDE = 7 /* host-side tag only (csrc/kde.cu stages hand MCGRA_M_PRE tiles over; the node kernels treat it as NONE) */ };

/* slots of the per-iteration double-precision accumulator block `acc` (32 doubles).
 * Slots 0-15 are accumulated by the tile kernels over one rank's shard (all-reduced across ranks);
 * slots 16-31 by the node kernels, which every rank runs redundantly (NOT reduced).                 */
enum {
  MCGRA_ACC_C1 = 1,       /* c1 term, off-diagonal part, fully scaled (w1 * 1000 * 100 * measure)  */
  MCGRA_ACC_C2 = 2,
  MCGRA_ACC_C6 = 3,
  MCGRA_ACC_C7 = 4,
  MCGRA_ACC_SUMCLAMP = 8, /* sum clamp(x',0,1) after the Adam step (budget test, :339)            */
  MCGRA_ACC_SUMSQ = 9,    /* sum of squares of the projected parameter (for 0.001*||x||, :172)    */
  MCGRA_ACC_NLL = 16,     /* sum_i w_i * -log p(y_i)   (w_i already divided by |idx|)             */
  MCGRA_ACC_C9 = 17,
  MCGRA_ACC_C10 = 18,
  MCGRA_ACC_C1D = 19,     /* diagonal (A_hat_ii = r_i^2) parts of the element-wise terms           */
  MCGRA_ACC_C2D = 20,
  MCGRA_ACC_C6D = 21,
  MCGRA_ACC_C7D = 22,
  MCGRA_ACC_N = 32
};

int mcgra_version(void);
/* engine selection for A/B validation; the engines 0 are the exact references of the agreement tests:
 *   which 0 = propagate:    0 exact fp32 FFMA, 5 both products on tcgen05 kind::f16 from one fp16x2 image per tile [default]
 *   which 1 = fold:         0 exact fp32 FFMA, 2 tcgen05 one tile per CTA (every parameter view / measure), 3 persistent
 *                           row runs with the A operand resident in tensor memory for the clamped and the lazily projected
 *                           view, engine 2 otherwise [default]; 100 + cap (0 <= cap < 900) caps the persistent grid at
 *                           cap CTAs (0 = one per SM, the default)
 *   which 2 = pairs:        0 FFMA, 1 mma.sync 3xTF32, 2 tcgen05 for the entropy-only configuration + 1 otherwise [default]
 *   which 4 = element-wise pass: 0 one tile per CTA, 1 persistent bulk-staged kernel for MSE on the clamped / lazily
 *                           projected view, 0 otherwise [default]; 100 + cap as for which 1
 *   which 5 = mcgra_ensemble: 0 one CTA per 64 x 64 block, 1 one CTA per block PAIR (I, J) / (J, I) when the full matrix is
 *                           written (symmetric terms evaluated once), 0 for row bands [default]
 *   which 6 = mcgra_auc_ap: 0 1024-sample search table over the sorted positives, 1 the DISTINCT positive keys with their
 *                           start indices (and a CTA-private histogram while they fit) in up to 224 KB of shared memory,
 *                           sampled keys + one 32-byte block per segment beyond that [default]
 * Returns 0, or -1 (and changes nothing) for any other selector or value.                                              */
int mcgra_set_engine(int which, int value);
int64_t mcgra_tiles_in_rows(int tr0, int tr1);           /* number of tiles in tile rows [tr0,tr1) */

/* ---- layout (replaces torch.tril_indices + index_put + m+m.t(), topology_attack.py:365-379) ---- */
int mcgra_tril_to_tiles(const float* packed, int64_t n, int tr0, int tr1, float* tiles, void* stream);
int mcgra_tiles_to_tril(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                        float* packed, void* stream);
/* lower triangle of a dense row-major matrix (leading dimension ld) -> tiles; symmetrize!=0 stores
 * (F_ij+F_ji)/2; diag (may be NULL) receives F_ii for the rows of [tr0,tr1).                        */
int mcgra_dense_to_tiles(const float* dense, int64_t ld, int64_t n, int tr0, int tr1, int symmetrize,
                         float* tiles, float* diag, void* stream);
/* symmetric dense expansion with zero diagonal (get_modified_adj, :365-379); writes rows AND mirrored
 * columns of the owned tile rows into dense[n x ld]; caller zero-fills dense first.                 */
int mcgra_tiles_to_dense(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                         float* dense, int64_t ld, void* stream);

/* ---- degree: d[i] += sum_j M_ij over the shard (utils.py:224-225); caller pre-fills d with 1 ---- */
int mcgra_degree(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, float* d,
                 void* stream);

/* ---- propagation Y += M * B (GraphConvolution.forward's spmm, models/gcn.py:42, and its transpose
 *      in backward); M symmetric zero-diagonal from the tiles; B,Y row-major [n x K], K in {16,32}.
 *      Caller zero-fills Y.                                                                          */
/* ws (optional, may be NULL): device scratch of mcgra_propagate_ws_bytes(n, K) bytes; with it the tcgen05 engine
 * pre-formats B once per call (tf32 hi/lo split, K-major core-matrix layout) instead of once per tile.          */
int64_t mcgra_propagate_ws_bytes(int64_t n, int K);
int mcgra_propagate(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                    const float* B, int K, float* Y, void* ws, void* stream);
/* the same with a product selector: with L the stored strict lower triangle (entry (i,j), i > j, at tile (I,J)),
 * DIRECT adds L*B, MIRRORED adds L^T*B, BOTH (= mcgra_propagate) their sum.  The noisy path (mcgra_noise_stage) keeps
 * the two orientations of a non-symmetric M in two tile planes and forms M*B / M^T*B from one product of each.   */
enum { MCGRA_PROD_DIRECT = 1, MCGRA_PROD_MIRRORED = 2, MCGRA_PROD_BOTH = 3 };
int mcgra_propagate_sel(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                        const float* B, int K, float* Y, void* ws, int products, void* stream);

/* ---- element-wise terms of the layer-1 pass (c1 MSE/KL against feature_adj, c6 entropy;
 *      topology_attack.py:212-232,44-47) as a streaming pass over the shard (x and F tiles read once):
 *      values into elem->acc, the row sums eps_row[i] += sum_j (e'_ij+e'_ji) M_ij r_j needed by the
 *      degree gradient (SURVEY 8(a4)) into elem->eps_row.                                           */
typedef struct {
  const float* r;         /* [n] D^-1/2                                                              */
  const float* Ftiles;    /* tiled feature_adj (same shard) or NULL                                  */
  const float* lseA;      /* [n] log sum_j exp(A_hat_ij)  (KL only)                                   */
  const float* lseF;      /* [n] log sum_j exp(F_ij)      (KL only)                                   */
  int measure;            /* MCGRA_M_NONE / MCGRA_M_MSE / MCGRA_M_KL for c1                           */
  float k1;               /* c1 scale: w1*1e5/n^2 (MSE) or w1*1e5/n (KL); sign included               */
  float k6;               /* c6 scale: -w6*1000/n^2, 0 = off                                          */
  double* acc;            /* accumulator block (slots C1, C6)                                         */
  float* eps_row;         /* [n]                                                                      */
  const float* dlse;      /* [n] lseF - lseA evaluated in fp64 (KL value: log-ratio without cancellation)     */
} mcgra_elem_args;
int mcgra_elem_stats(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                     const mcgra_elem_args* elem, void* stream);
/* row log-sum-exp of A_hat over the shard: sumexp[i] += sum_{j != i} exp(r_i M_ij r_j) (KL measure) */
int mcgra_row_sumexp(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                     const float* r, float* sumexp, void* stream);

/* ---- node-level stages (n x 16 work of GCN.forward / embedding_GCN.forward, models/gcn.py:71-76,
 *      164-174, their hand-derived backward, nll (:326-336) and the n x d measure terms c9/c10) ---- */
typedef struct {
  int64_t n;
  int nclass;
  const float *W2, *b1, *b2, *Wl, *bl;   /* victim weights: W2[16x16], Wl[c x 16] (nn.Linear layout)  */
  const float* S1;                       /* X W1 [n x 16] (constant)                                   */
  const int64_t* labels;                 /* [n]                                                        */
  const float* wmult;                    /* [n] multiplicity of node i in idx_attack / |idx_attack|    */
  const float* HA;                       /* H_A target [n x 16]                                        */
  const float* YA;                       /* Y_A target [n x c] (log-probabilities, :264-271)           */
  float* d;                              /* [n] degree (1 + row sum)                                   */
  float* r;                              /* [n]                                                        */
  float *B1, *Y1, *B2, *Y2, *B3, *Y3;    /* [n x 32] operands / results of the three 32-wide passes    */
  float *B4, *Y4;                        /* [n x 16] operand / result of the degree-gradient pass      */
  float *S2, *T2, *H2, *dZ2, *dZ1, *dQ1, *dQ2, *demd, *zhat, *dzhat;   /* [n x 16]                   */
  float* inv_norm;                       /* [n] 1/max(||em||,1e-12)                                    */
  uint32_t* masks;                       /* [n] relu masks: bits 0-15 H1>0, 16-31 E1>0                 */
  uint32_t* masks2;                      /* [n] bits 0-15 Z2>0, 16-31 em>0                             */
  float* eps_row;                        /* [n] element-wise degree-gradient row sums                  */
  float* rho;                            /* [n] degree gradient                                        */
  float* Wt;                             /* [128 x npad] transposed fold factors [U|V]                 */
  const float* Fdiag;                    /* [n] diagonal of feature_adj (or NULL)                      */
  double* acc;                           /* accumulator block                                          */
  int measure;                           /* measure for c1 (diag part) and c9/c10                      */
  float weight_sup;
  float k1, k2, k6, k7;                  /* scaled weights of the n x n element-wise terms             */
  float w9, w10;                         /* raw weights of c9 / c10 (sign for HSIC included)           */
  int64_t npad;
  /* state reset done by mcgra_node_rho for the fold that follows it */
  float* d_next;                         /* [n] filled with d_fill (1 on rank 0, 0 elsewhere)          */
  float d_fill;
  double* acc_next;                      /* [MCGRA_ACC_N] zeroed                                       */
  float* minmax;                         /* [2] set to {+inf, -inf}                                    */
  const float* lseA;                     /* KL: [n] log sum_j exp(A_hat_ij) incl. diagonal (or NULL)   */
  const float* lseF;                     /* KL: [n] log sum_j exp(F_ij)                                */
  float* em;                             /* [n x 16] raw-branch embedding (kept for upstream measure stages)  */
  const float* dlse;                     /* KL: [n] lseF - lseA (fp64-evaluated)                              */
  int measure_nn;                        /* measure of the n x n terms (diagonal part in mcgra_node_rho);
                                            `measure` above is the one of the n x d terms c9 / c10           */
} mcgra_node_args;
int mcgra_node_pre(const mcgra_node_args* a, void* stream);    /* r = d^-1/2 ; B1 = [r*S1 | S1]       */
int mcgra_node_mid(const mcgra_node_args* a, void* stream);    /* after pass 1: H1,E1,S2,T2,B2        */
int mcgra_node_head(const mcgra_node_args* a, void* stream);   /* after pass 2: heads, losses, dZ2... */
int mcgra_node_bwd2(const mcgra_node_args* a, void* stream);   /* dQ2, B3                              */
int mcgra_node_bwd1(const mcgra_node_args* a, void* stream);   /* after pass 3: dZ1,dQ1,B4             */
int mcgra_node_rho(const mcgra_node_args* a, void* stream);    /* after pass 4: rho, fold factors Wt   */
/* mcgra_node_rho for an estimate with a non-zero diagonal M_ii = mdiag[i] (the noisy path): the diagonal entry of
 * A_hat is r_i^2 (1 + M_ii) in the element-wise terms and in rho.                                                    */
int mcgra_node_rho_diag(const mcgra_node_args* a, const float* mdiag, void* stream);

/* ---- pair pass over the decode gram M1 = relu(zhat zhat^T) (dot_product_decode :414-419,
 *      get_modified_adj_after :381-395): c7 entropy (:233-236) and c2 MSE (:221-229) values, their
 *      gradient w.r.t. zhat (dzhat, caller zero-fills) and c2's eps_row contribution.              */
/* Optional precomputed inputs (MCGRA_M_PRE measures): EAt = tiles of dL/dA_ij + dL/dA_ji (their eps_row
 * contribution is accumulated here), Ct = tiles of dL/dM1_ij + dL/dM1_ji (added to the coefficient tile).     */
/* ws (may be NULL): device scratch of mcgra_pairs_ws_bytes(n) bytes; with it the entropy-only configuration (k7 != 0,
 * k2 == 0, no upstream tiles) runs entirely on tcgen05 (pairs_tc.cu: gram, coefficient planes and both skinny products
 * on chip, no HBM stream).                                                                                       */
int64_t mcgra_pairs_ws_bytes(int64_t n);
int mcgra_pairs(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw,
                const float* zhat, const float* r, float k7, float k2, const float* EAt, const float* Ct,
                float* dzhat, float* eps_row, double* acc, void* ws, void* stream);

/* ---- gradient fold + Adam + box clamp (loss.backward()+optimizer.step()+clamp, :274-283) ---- */
typedef struct {
  int64_t n;
  int64_t npad;
  const float* Wt;        /* [128 x npad] fold factors                                               */
  const float* r;         /* [n]                                                                      */
  const float* rho;       /* [n]                                                                      */
  const float* Ftiles;    /* tiled feature_adj or NULL                                                */
  const float* lseA;      /* KL */
  const float* lseF;      /* KL */
  const float* zhat;      /* [n x 16] (c2 only) or NULL                                               */
  int measure;            /* c1 measure                                                               */
  float k1, k6, k2;       /* element-wise scales as above                                             */
  float norm_coef;        /* weight_sup * 0.001                                                       */
  float lr, beta1, beta2, adam_eps;
  int step;               /* 1-based Adam step                                                        */
  const double* acc_prev; /* accumulator block of the state the gradient was taken at (SUMSQ)         */
  double* acc_next;       /* receives SUMCLAMP, SUMSQ, XMIN, XMAX of the new x'                       */
  float* d_next;          /* [n] += row/col sums of clamp(x',0,1) (caller pre-fills with 1)           */
  int store_clamped;      /* != 0: the budget cannot bind -> store clamp(x',0,1) (readers then use raw = 2)   */
  void* Wk;               /* scratch of mcgra_fold_ws_bytes(n) bytes for the tcgen05 engine (NULL: mma.sync)   */
  const int* step_ptr;    /* optional: device counter of completed iterations; Adam step = *step_ptr + 1 (overrides
                             `step`) so that the launch carries no per-iteration host scalar (CUDA-graph replay) */
  int plain_gd;           /* != 0: x <- x - lr * g instead of Adam (MC-GPB/topology_attack.py:66-70: adj_changes +=
                             lr * (-grad), lr = 0.1); m, v still receive Adam's moment update, which the step ignores */
  const float* Gtiles;    /* optional tiles of dL/dM_ij + dL/dM_ji computed upstream (feature smoothing of the GraphMI
                             attack, MC-GPB/topology_attack.py:57-61), added to the gradient as is; NULL = none      */
} mcgra_fold_args;
int64_t mcgra_fold_ws_bytes(int64_t n);
/* minmax: device float[2] = {min x', max x'} (bisection bracket, :340-341); reset by mcgra_node_rho          */
int mcgra_fold_adam(float* tiles, float* m, float* v, int tr0, int tr1, const float* mu, int raw,
                    const mcgra_fold_args* a, float* minmax, void* stream);

/* ---- budget projection by bisection on device (projection/bisection, :338-347, 397-412) ----
 * state[8] floats on device: a, b, mu, done, active, ... ; one call = 3 halvings evaluated in one
 * pass over x' (7 candidate midpoints, the same fp32 midpoints the scalar loop would visit).       */
int mcgra_bisect_init(const double* acc, const float* minmax, double budget, float* state, float* mu,
                      void* stream);
int mcgra_bisect_pass(const float* tiles, int64_t n, int tr0, int tr1, float epsilon, const float* state,
                      double* cand_sums /* device [7], zero on entry */, void* stream);
int mcgra_bisect_update(double budget, float epsilon, float* state, double* cand_sums, float* mu,
                        void* stream);
/* after the last pass: recompute SUMSQ and the degree of the projected parameter (only if active);
 * reset != 0 first discards the fold's mu = 0 statistics (d_next = 1, SUMSQ = 0).                   */
int mcgra_bisect_finish(const float* tiles, int64_t n, int tr0, int tr1, const float* state,
                        const float* mu, double* acc_next, float* d_next, int reset, void* stream);

/* hist[*step][0:MCGRA_ACC_N] = row; (*step)++  -- one tiny launch at the end of an iteration: the accumulator rows can
 * then be a fixed ring of two and the Adam step a device counter, which makes the whole iteration replayable as a CUDA
 * graph (the launch-bound regime of small graphs).  No-op beyond max_rows.                                        */
int mcgra_history_push(const double* row, double* hist, int64_t max_rows, int* step, void* stream);

/* ---- finalisation (topology_attack.py:300-322) ---- */
/* x_final tiles = relu(zf_i . zf_j) for j<i (dot_product_decode of the last embedding)              */
int mcgra_decode_to_tiles(const float* zhat, int64_t n, int tr0, int tr1, float* tiles, void* stream);
/* rows [b0, b1) of the expanded decode, written (not accumulated) row-major: out[(i - b0) * ld + j] = relu(z_i . z_j) for
 * j != i and 0 for j == i, z n x 16 as given (row-normalised or raw).  Every entry is bit-equal to what
 * mcgra_decode_to_tiles followed by mcgra_tiles_to_dense (raw = 1) produce: same 16-term fmaf order, no clamp.
 * The GraphMI attacks' modified_adj on a row band (baseline.py, mcgpb_attack.py with world > 1). 0 <= b0, b1 <= n <= ld. */
int mcgra_decode_band(const float* zhat, int64_t n, int64_t b0, int64_t b1, float* out, int64_t ld, void* stream);
/* one gram term of the ensemble: out[i,j] (+)= f(Z_i . Z_j) with the dataset's decode2 variant
 * (dot_product_decode2, :421-467): variant 0 sigmoid(relu(g - I)), 1 relu(g - I),
 * 2 relu(g/rownorm_i - I) (rownorm = ||row i of ZZ^T||, given), 3 plain g (gcn_parameterized.py:406-416),
 * 4 relu(g) with a zero diagonal (the symmetric expansion of dot_product_decode: get_modified_adj, :365-379, 414-419,
 * used when the row band of an ensemble is computed on a rank that does not hold the mirrored tiles).
 * The sigmoid of variant 0 is evaluated as 1 / (1 + 2^(-v log2 e)) on the MUFU ex2 / rcp units (~2e-7 relative; v >= 0),
 * with the same definition in mcgra_ensemble.                                                                       */
int mcgra_gram_accumulate(const float* Z, int d, int64_t n, int variant, const float* rownorm,
                          float* out, int64_t ld, int64_t row0, int64_t row1, void* stream);
/* out[i,j] += (labels[i]==labels[j])                                                                */
int mcgra_label_accumulate(const int64_t* labels, int64_t n, float* out, int64_t ld, int64_t row0,
                           int64_t row1, void* stream);

/* The whole ensemble sum of :300-322 in ONE pass over the n x n result (each term above re-reads and re-writes it):
 * out[i,j] = M_ij (symmetric zero-diagonal expansion of `tiles`, skipped when tiles == NULL: out starts from 0)
 *            + term_0 + term_1 + ... added left to right in fp32, so the value equals the sequence of
 * mcgra_tiles_to_dense / mcgra_gram_accumulate / mcgra_dense_add / mcgra_label_accumulate calls bit for bit.       */
#define MCGRA_ENSEMBLE_MAX 8
enum { MCGRA_TERM_GRAM = 0, MCGRA_TERM_DENSE = 1, MCGRA_TERM_LABEL = 2 };
typedef struct {
  int kind;                 /* MCGRA_TERM_*                                                            */
  int d;                    /* gram: factor width (<= 32)                                              */
  int variant;              /* gram: as mcgra_gram_accumulate                                          */
  int pad_;
  const float* Z;           /* gram: n x d factors                                                     */
  const float* rownorm;     /* gram variant 2                                                          */
  const float* dense;       /* dense: n x n row-major addend (leading dimension n)                     */
  const int64_t* labels;    /* label: adds (labels[i] == labels[j])                                    */
} mcgra_ensemble_term;
typedef struct {
  int nterms;
  int pad_;
  mcgra_ensemble_term t[MCGRA_ENSEMBLE_MAX];
} mcgra_ensemble_args;
int mcgra_ensemble(const float* tiles, int64_t n, const mcgra_ensemble_args* args, float* out, int64_t ld,
                   int64_t row0, int64_t row1, void* stream);

/* out += in (dense, `count` floats); F.normalize(Z, p, dim=1) with eps 1e-12                          */
int mcgra_dense_add(float* out, const float* in, int64_t count, void* stream);
int mcgra_row_normalize(const float* Z, int64_t n, int d, float p, float* out, void* stream);

/* ---- HSIC / CKA family on m x d samples (hsic.py; utils.py:803-822, 1056-1097) ----
 * One fused pass over the m^2 pairs, no m x m kernel stored:  K = exp(-gx |xi-xj|^2), L = exp(-gy |yi-yj|^2);
 * rowK[i] += sum_j K_ij, rowL[i] += sum_j L_ij (caller zero-fills), out[0] += sum K.L, out[1] += sum K,
 * out[2] += sum L (device double[3], zero on entry).  tr(KHLH) = out0 - (2/m) rowK.rowL + out1*out2/m^2.       */
int mcgra_gauss_stats(const float* X, int dx, const float* Y, int dy, int64_t m, float gx, float gy,
                      float* rowK, float* rowL, double* out, void* stream);
/* dense pair matrix out[m1 x m2]: mode 0 = |xi - zj|^2 (hsic.distmat), mode 1 = exp(-gamma |xi - zj|^2)        */
int mcgra_pair_dense(const float* X, int d, int64_t m1, const float* Z, int64_t m2, int mode, float gamma,
                     float* out, void* stream);
/* weighted raw moments of two factor matrices (w NULL = 1): out (device double, zero on entry) =
 * [sum w x (dx) | sum w y (dy) | sum w x y^T (dx*dy) | sum w y y^T (dy*dy)]; linear HSIC/CKA in O(n d d')     */
int mcgra_cross_moments(const float* X, int dx, const float* Y, int dy, const float* w, int64_t n,
                        double* out, void* stream);

/* ---- dense n x n contractions of the HSIC / CKA / DP measures on two n x n operands (K6) ----
 * (CudaCKA.centering / linear_HSIC / linear_CKA, utils.py:1060-1091; PGDAttack.dot_product, topology_attack.py:480-481;
 *  call sites topology_attack.py:190-229.)  The reference evaluates linear_HSIC(X, Y) with six n^3 GEMMs through dense
 *  centring matrices; here every measure is a short sequence of mcgra_gemm_nt calls with closed-form gradients:
 *     c1  HSIC(F, A) = sum (Kf A) o A,           Kf = H F F^T H  (constant),         d/dA = 2 Kf A
 *     c2  HSIC(A, M) = || T ||_F^2,  T = A Hc M = A M - (A 1)(M 1 / n)^T,            d/dA = 2 (Hc M) T^T, d/dM = 2 (Hc A) T
 *  (A, M symmetric; Hc = H for HSIC / CKA, I for DP; CKA adds the self terms S = A Hc A, d/dA = 4 Hc A S.)
 *
 * An IMAGE is the tensor-core operand form of an fp32 matrix: two fp16 planes hi = fp16(s_i x), lo = fp16(s_i x - hi)
 * per row i with a power-of-two row scale s_i (max_j |s_i x_ij| <= 2^14), 4 bytes per element like fp32, ~2^-23 of the
 * row maximum.  ld (in halves) must be a multiple of 8 and the planes 16-byte aligned (TMA).                         */
typedef struct {
  void* hi;                 /* fp16 [rows x ld]                                                        */
  void* lo;                 /* fp16 [rows x ld]                                                        */
  float* inv_scale;         /* [rows] 1 / s_i                                                          */
  int64_t rows, cols, ld;
} mcgra_image;

typedef struct {
  float* C;                 /* [M x ldc] fp32 output or NULL (reductions only)                         */
  int64_t ldc;
  float alpha, beta;        /* C = beta * C + alpha * (A B^T - coef * u_i v_j)                          */
  const float* alpha_dev;   /* optional device scalars that multiply alpha / beta                      */
  const float* beta_dev;
  const float* u;           /* [M] or NULL (= 1); ignored when v is NULL                               */
  const float* v;           /* [N] or NULL (no rank-1 correction)                                      */
  float coef;
  double* sumsq;            /* device: += sum (A B^T - coef u v^T)^2 over the computed rows, or NULL    */
  double* dot;              /* device: += sum (A B^T - coef u v^T) o E, E = dot_with (M x N image)      */
  const mcgra_image* dot_with;
  int64_t row0, row1;       /* row panel [row0, row1) of C computed by this call (row1 <= row0: all)    */
} mcgra_gemm_epilogue;

/* C[M x N] = A[M x K] * B[N x K]^T on tcgen05 (kind::f16, three MMAs per K step, TMEM accumulators, TMA-fed,
 * cta_group::2); M = A->rows, N = B->rows, K = A->cols = B->cols.                                                  */
int mcgra_gemm_nt(const mcgra_image* A, const mcgra_image* B, const mcgra_gemm_epilogue* e, void* stream);

/* image of a dense fp32 matrix src[rows x cols] (leading dimension ld); transpose != 0 builds the image of src^T
 * (cols x rows).  ws: device scratch of max(rows, cols) uint32.                                                      */
int mcgra_image_from_dense(const float* src, int64_t rows, int64_t cols, int64_t ld, int transpose,
                           const mcgra_image* out, void* ws, void* stream);
/* image of A_hat = D^-1/2 (M + I) D^-1/2 (utils.py:211-230) from the FULL tiled triangle (tile rows [0, T)) and
 * r = d^-1/2; rowsum[i] (device double, zero on entry) += sum_j A_hat_ij.                                            */
int mcgra_image_ahat(const float* tiles, int64_t n, const float* mu, int raw, const float* r, const mcgra_image* out,
                     double* rowsum, void* stream);
/* image of M1 = relu(zhat zhat^T) with zero diagonal (dot_product_decode + get_modified_adj_after, :381-395, 414-419);
 * rowsum as above.                                                                                                   */
int mcgra_image_m1(const float* zhat, int64_t n, const mcgra_image* out, double* rowsum, void* stream);
/* X <- H X H (CudaCKA.centering, utils.py:1060-1065) in place on a dense symmetric fp32 matrix; ws: n doubles + 1     */
int mcgra_center_dense(float* X, int64_t n, int64_t ld, double* ws, void* stream);
/* out[j] += scale * sum_k w[k] X[k][j] (transpose == 0) or scale * sum_k X[j][k] w[k] (transpose != 0); X is
 * rows x cols fp32; w, out device double (caller zero-fills out).                                                    */
int mcgra_dense_gemv(const float* X, int64_t rows, int64_t cols, int64_t ld, const double* w, double scale,
                     int transpose, double* out, void* stream);
/* out[0] += sum X_ij^2 (device double)                                                                               */
int mcgra_dense_sumsq(const float* X, int64_t rows, int64_t cols, int64_t ld, double* out, void* stream);
/* tiles of (G_ij + G_ji) * scale (* *scale_dev) for the tile rows [tr0, tr1) and, when diag != NULL, diag[i] =
 * G_ii * scale for ALL i (every rank holds the full G).                                                              */
int mcgra_sym_to_tiles(const float* G, int64_t ld, int64_t n, int tr0, int tr1, float scale, const float* scale_dev,
                       float* tiles, float* diag, void* stream);
/* scalars of the dense measures: in = device double[8] {S1, hAM, hAA, hMM, hFF, -, -, -}; writes the loss values
 * c1, c2 (fully scaled, sign NOT applied) to acc[MCGRA_ACC_C1D], acc[MCGRA_ACC_C2D] (+=) and the gradient scales
 * alpha[8] (device float): {a1: G1 -> dL/dA, a2: (Hc M) T^T -> dL/dA, a3: (Hc A) S_A -> dL/dA, a4: (Hc A) T -> dL/dM,
 * a5: (Hc M) S_M -> dL/dM}; sign = -1 for HSIC (topology_attack.py:215-229).                                           */
int mcgra_dense_scalars(int measure, const double* in, double k1c, double k2c, double sign, double* acc, float* alpha,
                        void* stream);
/* out[i] = (float)(in[i] * scale)                                                                                    */
int mcgra_d2f(const double* in, int64_t count, double scale, float* out, void* stream);

/* ---- KL measure on two n x n operands (PGDAttack.calc_kl, topology_attack.py:483-487; c1 / c2 at :212-229) as
 * three passes over the tiled triangle (csrc/kl2.cu); the gram M1 is regenerated per tile from zhat.  Row statistics
 * (seA, seM, klrow, c1row: float [n], zero on entry of the pass that accumulates them) are all-reduced across ranks by
 * the caller between passes.  Pass 2 writes the tiles EAt = dL/dA_ij + dL/dA_ji and Ct = dL/dM1_ij + dL/dM1_ji that
 * mcgra_pairs / mcgra_fold_adam consume as MCGRA_M_PRE.                                                               */
typedef struct {
  const float* tiles;       /* x' shard (tile rows [tr0, tr1))                                          */
  const float* mu;
  int raw;
  int tr0, tr1;
  int64_t n;
  const float* Ftiles;      /* tiled feature_adj (same shard) or NULL when c1 is off                    */
  const float* Fdiag_feat;  /* [n] diagonal of feature_adj                                              */
  const float* lseF;        /* [n] row log-sum-exp of feature_adj                                       */
  const float* zhat;        /* [n x 16]                                                                 */
  const float* r;           /* [n]                                                                      */
  float *seA, *seM;         /* [n] pass 0 accumulators                                                  */
  float *lseA, *lseM;       /* [n] written by node stage 0                                              */
  float *klrow, *c1row;     /* [n] pass 1 accumulators                                                  */
  float *EAt, *Ct;          /* pass 2 outputs (shard tiles)                                             */
  double k1c, k2c;          /* fully scaled term weights (w1 * 1000 * 100, w2 * 100 * 1000); 0 = off    */
} mcgra_kl2_args;
int mcgra_kl2_pass(int pass, const mcgra_kl2_args* k, void* stream);
/* stage 0: lseA / lseM from the exp sums; stage 1: KL_i, loss values into acc[C1D], acc[C2D], Fdiag = dL/dA_ii        */
int mcgra_kl2_node(int stage, const mcgra_kl2_args* k, float* Fdiag, double* acc, void* stream);

/* ---- the n x d prior terms c9 / c10 under HSIC / CKA / DP (topology_attack.py:237-272), forward and backward from
 * weighted second moments in O(n d d') (csrc/ndmeasure.cu).  Adds the gradient w.r.t. the raw-branch embedding to
 * demd and the signed term values to acc[MCGRA_ACC_C9], acc[MCGRA_ACC_C10].                                         */
typedef struct {
  int64_t n;
  int nclass;
  int measure;              /* MCGRA_M_HSIC / MCGRA_M_CKA / MCGRA_M_DP                                  */
  const float* em;          /* [n x 16] embedding(X, M) (variable)                                      */
  const float* HA;          /* [n x 16] target H_A                                                      */
  const float* YA;          /* [n x c] target Y_A (log-probabilities)                                   */
  const float* Wl;          /* [c x 16] linear head                                                     */
  const float* bl;          /* [c]                                                                      */
  const float* wmult;       /* [n] multiplicity of node i in idx_attack / |idx_attack|                  */
  double m;                 /* |idx_attack|                                                             */
  float w9, w10;            /* signed term weights; 0 = off                                             */
  float* p2;                /* scratch [n x c]                                                          */
  double* mom;              /* scratch, mcgra_nd_scratch_doubles(c) doubles                             */
  float* coef;              /* scratch, mcgra_nd_scratch_floats(c) floats                               */
  float* demd;              /* [n x 16] +=                                                              */
  double* acc;
} mcgra_nd_args;
int64_t mcgra_nd_scratch_doubles(int nclass);
int64_t mcgra_nd_scratch_floats(int nclass);
int mcgra_nd_measure(const mcgra_nd_args* a, void* stream);

/* ---- stand-alone helpers of the class surface ----
 * M <- clamp(M + eps * noise, 0, 1) (PGDAttack.adding_noise, topology_attack.py:474-478; noise = the caller's N(0,1) draw) */
int mcgra_noise_clamp(float* M, const float* noise, float eps, int64_t count, void* stream);

/* ---- attack() with adjacency noise (--eps != 0, topology_attack.py:165, 474-478), MSELoss / KDE ----
 * Per iteration M = clamp(p + N*eps, 0, 1) with a fresh dense n x n N (row-major fp32) and p the parameter view of
 * the tiles (off the diagonal; the diagonal is clamp(N_ii*eps, 0, 1)).  M is not symmetric: its two orientations are
 * kept as tile planes Lt (M_ij at (i,j), i > j) and Ut (M_ji at (i,j)), read by mcgra_propagate_sel with raw = 2:
 *     M B = DIRECT(Lt) + MIRRORED(Ut) + diag(mdiag) B,     M^T B = DIRECT(Ut) + MIRRORED(Lt) + diag(mdiag) B.
 * The clamp masks are not stored: the gradient pass recomputes p + N*eps with the same two roundings.             */
int mcgra_noise_stage(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* noise,
                      float eps, float* Lt, float* Ut, float* mdiag, float* d, void* stream);   /* d = 1 + row sums of M */
/* The same stage split for tile-row shards (world > 1), where d must be all-reduced between the two halves:
 *   mcgra_noise_tiles: Lt, Ut of tile rows [tr0, tr1) and d += this shard's part of the row sums (d is not initialised);
 *   mcgra_noise_diag:  mdiag = M_ii and d += 1 + M_ii, once, after the all-reduce of d.
 * mcgra_noise_stage = k_noise_diag (d = 1 + M_ii) + mcgra_noise_tiles. */
int mcgra_noise_tiles(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* noise,
                      float eps, float* Lt, float* Ut, float* d, void* stream);
int mcgra_noise_diag(int64_t n, const float* noise, float eps, float* mdiag, float* d, void* stream);
/* Y[i, :] += mdiag[i] * B[i, :]  (B, Y row-major [n x K]) */
int mcgra_diag_axpy(const float* mdiag, const float* B, int K, int64_t n, float* Y, void* stream);
typedef struct {
  int64_t n, npad;
  int tr0, tr1;
  const float* tiles;      /* parameter tiles and their view (mu, raw) as given to mcgra_noise_stage        */
  const float* mu;
  int raw;
  const float* noise;      /* [n x n] this iteration's draw                                                 */
  float eps;
  const float *Lt, *Ut;    /* the two orientations written by mcgra_noise_stage                             */
  const float *FLt, *FUt;  /* feature_adj: F_ij and F_ji at (i,j) (mcgra_dense_to_tiles of F and F^T), or NULL */
  const float* zhat;       /* [n x 16] row-normalised embedding (c2: M1 = relu(zhat zhat^T))                */
  const float* r;          /* [n] D^-1/2                                                                    */
  const float* rho;        /* [n] degree gradient (mcgra_node_rho_diag)                                     */
  const float* Wt;         /* [128 x npad] factors U, V (mcgra_node_rho_diag)                               */
  float k1, k2, k6;        /* as in mcgra_node_args (c1 and c2 under MSELoss, c6)                           */
  double* acc;             /* slots C1, C2, C6 (+=)                                                         */
  float* eps_row;          /* [n] += row and column parts of the element-wise degree gradient               */
  float* dzhat;            /* [n x 16] += gradient of c2 through M1                                         */
  float* Gt;               /* gradient tiles: dL/dx_ij (consumed by mcgra_fold_adam as Gtiles)              */
  const float* gslab;      /* [n x nb] dL/dA_hat_ij for j < nb computed upstream (--measure KDE), or NULL;
                              added to e'_ij (j < nb) and e'_ji (i < nb) of the stored entries                 */
  int nb;                  /* columns of gslab, 1 <= nb <= MCGRA_TILE when gslab != NULL                     */
} mcgra_noisy_args;
/* c1 (MSE), c2 (MSE, both orientations of A_hat against the symmetric M1) and c6 over the off-diagonal entries:
 * values, eps_row, dzhat; gslab's part of eps_row.  Launches when any of k1, k2, k6 is non-zero or gslab != NULL. */
int mcgra_noisy_terms(const mcgra_noisy_args* a, void* stream);
/* dL/dx_ij = mask_ij dL/dM_ij + mask_ji dL/dM_ji with dL/dM_ij = U_i.V_j + r_i r_j e'_ij + rho_i, written to Gt */
int mcgra_noisy_grad(const mcgra_noisy_args* a, void* stream);
/* out[0] += sum_rows KL(softmax(X_i) || softmax(Y_i)) (PGDAttack.calc_kl, :483-487; divide by rows for batchmean)      */
int mcgra_row_kl(const float* X, const float* Y, int64_t rows, int64_t cols, int64_t ldx, int64_t ldy, double* out,
                 void* stream);

/* ---- feature smoothing of the GraphMI attack (MC-GPB/topology_attack.py:57-61, 163-177): coef * tr(X^T L~ X) ----
 * Gfeat = tiled X X^T (same shard), gdiag[i] = |x_i|^2, d = the engine's degree (1 + row sum).  mcgra_smooth writes the
 * element-wise gradient tiles Gt (consumed by mcgra_fold_adam as Gtiles) and the row sums trow (all-reduced by the caller
 * across ranks); mcgra_smooth_node then adds the degree part to rho and coef * value to *acc_slot.                      */
int mcgra_smooth(const float* tiles, const float* Gfeat, const float* gdiag, int64_t n, int tr0, int tr1, const float* mu,
                 int raw, const float* d, float coef, float* rt, float* trow, float* Gt, void* stream);
int mcgra_smooth_node(int64_t n, const float* d, const float* rt, const float* trow, const float* gdiag, float coef,
                      float* rho, double* acc_slot, void* stream);

/* backward of mcgra_cross_moments: g = d loss / d out (device double, same layout); writes dX [n x dx] and dY [n x dy]
 * (either may be NULL).  With it every linear HSIC / CKA / DP penalty on factor grams is differentiable in O(n d d')
 * (MC-GPB/models/gcn.py:400-417, utils.py:774-797).                                                                 */
int mcgra_cross_moments_bwd(const float* X, int dx, const float* Y, int dy, const float* w, int64_t n, const double* g,
                            float* dX, float* dY, void* stream);

/* ---- --measure KDE: utils.MutualInformation(sigma 0.4, num_bins B) (MC-GRA/utils.py:980-1053; call sites
 * topology_attack.py:199-201, 212-229, 246-269) from weighted second moments of kernel-value slabs (csrc/kde.cu):
 * kv = exp(-0.5 ((v - j * bin_step) / 0.32)^2) per column j; moments by mcgra_cross_moments(kvX, kvY, w) with sum w = 1;
 * mcgra_kde_scalars adds weight * 2 MI / (H1 + H2) to *acc_slot and writes d/d moments (same layout) for
 * mcgra_cross_moments_bwd; mcgra_kde_chain takes the gradient through the kernel back to the values.  On n x n operands
 * only the first columns take part (bin_j ~ j, values in [0,1]: the kernel underflows to 0 for j >= 6): the slab helpers
 * extract the first NB columns of A_hat / M1 and return the gradient as tiles of tile column 0.                        */
int mcgra_kde_kv(const float* V, int64_t ldv, int d, int64_t m, float bin_step, float* kv, void* stream);
int mcgra_kde_chain(const float* V, int64_t ldv, const float* kv, const float* gkv, int d, int64_t m, float bin_step,
                    float* gV, int accumulate, void* stream);
int mcgra_kde_scalars(const double* mom, int d, double m, double weight, double* acc_slot, double* gmom, void* stream);
/* slab [n x NB] += first NB columns of A_hat from this rank's tile rows (caller zero-fills; all-reduce across ranks)     */
int mcgra_slab_ahat(const float* tiles, int64_t n, int tr0, int tr1, const float* mu, int raw, const float* r, int NB,
                    float* slab, void* stream);
/* the same for the noisy estimate (mcgra_noise_stage): A_hat_ij = r_i Lt_ij r_j below the diagonal, the entry above it
 * (i < j < NB) from the U orientation of the stored entry (j, i), and A_hat_jj = r_j^2 (1 + mdiag[j])                    */
int mcgra_slab_ahat_noisy(const float* Lt, const float* Ut, const float* mdiag, int64_t n, int tr0, int tr1,
                          const float* r, int NB, float* slab, void* stream);
/* fp64 MI of two value slabs X, Y [m x d] that share the bins j * bin_step (c1 / c2 on the noisy path, where MI is ~1e-6
 * of the entropies it is the difference of): mcgra_kde_moments64 recomputes the kernel values in fp64 and adds
 * wt * [sum kvX (d) | sum kvY (d) | sum kvX kvY^T (d*d)] to mom (caller zero-fills; layout of mcgra_kde_scalars, whose
 * Syy block it leaves untouched); mcgra_kde_chain64 adds the gradient w.r.t. the values, given gmom = d loss / d mom,
 * to gX and gY (either may be NULL).                                                                                    */
int mcgra_kde_moments64(const float* X, const float* Y, int d, int64_t m, double bin_step, double wt, double* mom,
                        void* stream);
int mcgra_kde_chain64(const float* X, const float* Y, int d, int64_t m, double bin_step, double wt, const double* gmom,
                      float* gX, float* gY, void* stream);
int mcgra_slab_m1(const float* zhat, int64_t n, int NB, float* slab, void* stream);
/* gradient slab G [n x NB] -> tiles (I, 0), I in [tr0, tr1), of G_ij + G_ji; diag[i] = G_ii for the rows of those tiles */
int mcgra_slab_to_tiles(const float* G, int64_t n, int tr0, int tr1, int NB, float* tiles, float* diag, void* stream);
/* p2 = softmax(em Wl^T + bl) and its backward into demd (the second head of c10, topology_attack.py:259-271)           */
int mcgra_softmax_rows(const float* em, const float* Wl, const float* bl, int64_t n, int c, float* p2, void* stream);
int mcgra_softmax_chain(const float* gp, const float* p, const float* Wl, int64_t n, int c, float* demd, void* stream);

/* ---- AUC / AP (main.metric_pool, main.py:66-75; gcn_parameterized.py:55-65) ----
 * scores [N] fp32, labels [N] uint8 (non-zero = positive).  The positives' keys are radix-sorted on the GPU and
 * reduced to their distinct values; every negative is ranked against them; exact integer counts => sklearn's trapezoid AUC with ties, and
 * sklearn's average precision.  npos_max bounds the number of positives (workspace size).
 * out: device double[4] = {auc, ap, npos, nneg}.                                                     */
int64_t mcgra_auc_workspace_bytes(int64_t N, int64_t npos_max);
int mcgra_auc_ap(const float* scores, const uint8_t* labels, int64_t N, int64_t npos_max, void* ws,
                 double* out, void* stream);
/* the three stages of mcgra_auc_ap, callable separately so that the n^2 pairs can be split over ranks by row bands:
 * stage 0 compacts the positives' keys of the local pairs (ws: u64 count at byte 0, u32 keys from byte 256); the caller
 * may replace them by the global positives (all-gather); stage 1 sorts the positives and ranks the local negatives
 * (ws: u64 sums[2] at byte 8, u64 hist[npos_max + 2] at mcgra_auc_hist_offset(npos_max)); the caller may sum hist / sums
 * over ranks (all-reduce); stage 2 writes out[4] = {auc, ap, npos, nneg}.                                          */
int64_t mcgra_auc_hist_offset(int64_t npos_max);
int mcgra_auc_stage(int stage, const float* scores, const uint8_t* labels, int64_t N, int64_t npos_max, void* ws,
                    double* out, void* stream);
/* stable descending arg-sort (LSD radix sort, key = score, payload = index): the recovered-edge ranking */
int64_t mcgra_sort_workspace_bytes(int64_t N);
int mcgra_argsort_desc(const float* scores, int64_t N, int64_t* order, void* ws, void* stream);

/* ---- top-k recovered edges ----
 * The k largest S[i, j] over the strict upper triangle (i < j) of a dense row-major n x n fp32 score matrix, or of the
 * row band scores = rows [row0, row0 + rows) of it (leading dimension n), in row-major index order i * n + j.  Sorting
 * the k values with the stable mcgra_argsort_desc then gives (score descending, index ascending).  fkey order: -0.0 ==
 * +0.0, +-inf allowed; NaN candidates are counted and must be rejected by the caller.  1 <= k <= n (n - 1) / 2.
 * Stages, in order 0 .. 7, each on every rank that holds a band:
 *   0, 2, 4  histogram of level 0, 1, 2 (2^11, 2^11, 2^10 bins of key bits 31..21, 20..10, 9..0, over the candidates that
 *            match the prefix selected so far): int64 hist[2049] at byte MCGRA_TOPK_HIST_OFFSET, the bins followed by
 *            the number of NaN candidates (stage 0 only).  With row bands the caller sums hist over ranks (all-reduce)
 *            before the next stage.
 *   1, 3, 5  select the bin of the remaining-th largest key from hist; after stage 5, int64 at byte 0 = tau (the key of
 *            the k-th largest candidate) and at byte 8 = t (candidates == tau still to take).  int64 at byte 32 is set to
 *            1 when hist holds fewer than k candidates.
 *   6        per-band counts: int64 at byte 16 = candidates > tau, at byte 24 = candidates == tau.
 *   7        write the band's candidates > tau and the first tie_quota candidates == tau (in index order) to
 *            out_idx / out_val [out_offset ...), as global indices i * n + j and raw scores.  One GPU: out_offset 0,
 *            tie_quota = t.  Row bands in row order: rank r uses out_offset = sum over q < r of (gt_q + quota_q) and
 *            quota_r = clamp(t - sum over q < r of eq_q, 0, eq_r).  Slots at or beyond k are never written.
 * Workspace: O(rows * ceil(n / 8192) + 2049) int64, never O(n^2).                                                 */
#define MCGRA_TOPK_HIST_OFFSET 256
int64_t mcgra_topk_workspace_bytes(int64_t rows, int64_t n, int64_t k);
int mcgra_topk_stage(int stage, const float* scores, int64_t row0, int64_t rows, int64_t n, int64_t k, void* ws,
                     int64_t out_offset, int64_t tie_quota, int64_t* out_idx, float* out_val, void* stream);

#ifdef __cplusplus
}
#endif
#endif
