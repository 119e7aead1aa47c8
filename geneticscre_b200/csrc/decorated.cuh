// Decorated p-values on the device (SURVEY section 8 row f4; reference: computeDecoratedPvalue, R/DecoratedPvalue.R:198-304),
// in the exact limit of the reference's Monte-Carlo estimate.
//
// For a split of a reported path into a sub-path (pos1 / neg1 carrier vectors) and the gene it is extended by (pos2 / neg2),
// the reference redraws the carriers the gene ADDS uniformly among the patients the sub-path does not cover and counts how
// often the re-scored path reaches the real score.  Only the number of redrawn carriers that land on cases matters, and that
// number is hypergeometric, so the estimate converges to
//     p = sum over (cp, cn) of P_pos(cp) * P_neg(cn) * [score_of(cp, cn) >= score]
// which is what decorated_exact_kernel evaluates: the same AND / popcount / value-table look-up shape as the join, one CTA per
// split.  Splits either come packed from the host (gcre_exec_decorated_exact) or are formed here from the gene rows of a path
// set (decorated_form_kernel: prefix / suffix ORs of whole paths, gcre_exec_decorated_paths).
//
// Stratified resampling (the reference's strataF, R/DecoratedPvalue.R:236-268) redraws the added carriers inside their own
// stratum, positives first, negatives from what is left of the stratum's pool; the exact limit is the 2-D convolution of the
// per-stratum joint distributions (geneticscre_b200/decorated.py, _stratified_joint_pmf, defines it).  On the device: a count
// pass (decorated_strata_count_kernel) sizes every split's joint distribution, the host cuts chunks that fit a scratch budget,
// and decorated_strata_joint_kernel convolves and sums the tail, one CTA per split, as a gather over output cells with
// fixed-order sums (repeated calls give identical bits).  The seeded Monte-Carlo mode stays a host utility.
#pragma once
#include <climits>

#include "common.cuh"

namespace gcre {

constexpr int DEC_THREADS = 256;

struct DecoratedOut {
  double pvalue;
  double score;
  int32_t cases1, ctrls1, cases2, ctrls2;
};

__device__ __forceinline__ double dec_block_sum(double v, double* s_red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < DEC_THREADS / 32; w++) t += s_red[w];  // fixed order: every thread gets the same bits
  return t;
}

// value table read with the engine's convention for entries outside the supplied table (-1.0, src/join_base.cpp:72)
__device__ __forceinline__ double dec_vt(const double* __restrict__ vt, int rows, int cols, long long r, long long c) {
  return (r >= 0 && c >= 0 && r < rows && c < cols) ? vt[(size_t)r * cols + c] : -1.0;
}

// The eight counts of R/DecoratedPvalue.R:206-225 (the gene's carriers already in the sub-path do not count) over the words
// load(k, pos1, neg1, pos2, neg2), k < W64, into s_cnt[8] (shared, zeroed and synchronised by the caller).
template <class Load>
__device__ __forceinline__ void dec_count8(Load load, int W64, int n_cases, int n, int* s_cnt) {
  int c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int k = threadIdx.x; k < W64; k += DEC_THREADS) {
    const uint64_t cm = case_mask_word(k, n_cases);
    const uint64_t valid = (k == W64 - 1 && (n & 63)) ? ((1ull << (n & 63)) - 1ull) : ~0ull;
    uint64_t w1, w2, w3, w4;
    load(k, w1, w2, w3, w4);
    const uint64_t p1 = w1 & valid, n1 = w2 & valid;
    const uint64_t p2 = w3 & valid & ~p1, n2 = w4 & valid & ~n1;
    c[0] += __popcll(p1 & cm);   // case_pos1
    c[1] += __popcll(p1 & ~cm);  // control_pos1
    c[2] += __popcll(n1 & ~cm);  // case_neg1 (the negative part counts controls as its "cases")
    c[3] += __popcll(n1 & cm);   // control_neg1
    c[4] += __popcll(p2 & cm);   // case_pos2
    c[5] += __popcll(p2 & ~cm);  // control_pos2
    c[6] += __popcll(n2 & ~cm);  // case_neg2
    c[7] += __popcll(n2 & cm);   // control_neg2
  }
#pragma unroll
  for (int q = 0; q < 8; q++) {
    const int v = __reduce_add_sync(0xffffffffu, c[q]);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&s_cnt[q], v);
  }
}

// The path's score when cp of tp redrawn positive carriers are cases and cn of tn redrawn negative carriers are controls;
// c = the eight counts of dec_count8
template <int M>
__device__ __forceinline__ double dec_score_of(const double* __restrict__ vt, int vt_rows, int vt_cols, const int* c, int cp, int tp, int cn, int tn) {
  if (M == 1)  // R/DecoratedPvalue.R:226-227, 285-286
    return dec_vt(vt, vt_rows, vt_cols, (long long)c[0] + cp + c[2] + cn, (long long)c[1] + (tp - cp) + c[3] + (tn - cn));
  return dec_vt(vt, vt_rows, vt_cols, c[0] + cp, c[1] + (tp - cp)) + dec_vt(vt, vt_rows, vt_cols, c[2] + cn, c[3] + (tn - cn));  // :228-229, :287-288
}

// Unnormalised hypergeometric probabilities w[x - lo], x = lo .. hi, of the number of "good" items among k drawn from good + bad,
// by the exact ratio recurrence P(x+1) / P(x) = (good - x)(k - x) / ((x + 1)(bad - k + x + 1)), started at the mode and run
// outwards (one thread: <= hi - lo steps of two multiplications).  Relative error ~1e-16 per step; log-gamma differences would
// lose ~n ln n * 1e-16 to cancellation.
__device__ __forceinline__ void dec_hyp_weights(long long good, long long bad, long long k, long long lo, long long hi, double* w) {
  long long mode = (k + 1) * (good + 1) / (good + bad + 2);
  mode = mode < lo ? lo : (mode > hi ? hi : mode);
  w[mode - lo] = 1.0;
  for (long long x = mode; x < hi; x++) w[x + 1 - lo] = w[x - lo] * ((double)((good - x) * (k - x)) / (double)((x + 1) * (bad - k + x + 1)));
  for (long long x = mode; x > lo; x--) w[x - 1 - lo] = w[x - lo] * ((double)(x * (bad - k + x)) / (double)((good - x + 1) * (k - x + 1)));
}

// rows: [n_items][4][W64] packed pos1, neg1, pos2, neg2; scratch: [n_items][2][n + 1] doubles
template <int M>
__global__ void __launch_bounds__(DEC_THREADS) decorated_exact_kernel(const uint64_t* __restrict__ rows, uint32_t n_items, int W64, int n_cases, int n_ctrls,
                                                                     const double* __restrict__ vt, int vt_rows, int vt_cols,
                                                                     double* __restrict__ scratch, DecoratedOut* __restrict__ out) {
  __shared__ double s_red[DEC_THREADS / 32];
  __shared__ int s_cnt[8];
  const uint32_t item = blockIdx.x;
  if (item >= n_items) return;
  const int n = n_cases + n_ctrls;
  const uint64_t* pos1 = rows + (size_t)item * 4 * W64;
  if (threadIdx.x < 8) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  dec_count8([&](int k, uint64_t& p1, uint64_t& n1, uint64_t& p2, uint64_t& n2) {
    p1 = pos1[k];
    n1 = pos1[W64 + k];
    p2 = pos1[2 * W64 + k];
    n2 = pos1[3 * W64 + k];
  }, W64, n_cases, n, s_cnt);
  __syncthreads();
  int cnt[8];
#pragma unroll
  for (int q = 0; q < 8; q++) cnt[q] = s_cnt[q];
  const int case_pos1 = s_cnt[0], ctrl_pos1 = s_cnt[1], case_neg1 = s_cnt[2], ctrl_neg1 = s_cnt[3];
  const int case_pos2 = s_cnt[4], ctrl_pos2 = s_cnt[5], case_neg2 = s_cnt[6], ctrl_neg2 = s_cnt[7];
  const int k_pos = case_pos2 + ctrl_pos2, k_neg = case_neg2 + ctrl_neg2;
  // pools (R/DecoratedPvalue.R:232-233): everything outside the sub-path's part; "good" = a case (positive part) / a control (negative)
  const int good_pos = n_cases - case_pos1, bad_pos = n_ctrls - ctrl_pos1;
  const int good_neg = n_ctrls - case_neg1, bad_neg = n_cases - ctrl_neg1;
  const double score = dec_score_of<M>(vt, vt_rows, vt_cols, cnt, case_pos2, k_pos, case_neg2, k_neg);

  // hypergeometric probabilities of the two independent counts over their supports
  const int lo_p = max(0, k_pos - bad_pos), hi_p = min(k_pos, good_pos), m_p = hi_p - lo_p + 1;
  const int lo_n = max(0, k_neg - bad_neg), hi_n = min(k_neg, good_neg), m_n = hi_n - lo_n + 1;
  double* pp = scratch + (size_t)item * 2 * (n + 1);
  double* pn = pp + (n + 1);
  if (threadIdx.x == 0) dec_hyp_weights(good_pos, bad_pos, k_pos, lo_p, hi_p, pp);
  if (threadIdx.x == 32) dec_hyp_weights(good_neg, bad_neg, k_neg, lo_n, hi_n, pn);
  __syncthreads();
  double sp = 0.0, sn = 0.0;
  for (int k = threadIdx.x; k < m_p; k += DEC_THREADS) sp += pp[k];
  for (int k = threadIdx.x; k < m_n; k += DEC_THREADS) sn += pn[k];
  sp = dec_block_sum(sp, s_red);
  sn = dec_block_sum(sn, s_red);
  __syncthreads();  // pp / pn are read by other threads below
  double acc = 0.0;
  const long long terms = (long long)m_p * m_n;
  for (long long q = threadIdx.x; q < terms; q += DEC_THREADS) {
    const int kp = (int)(q / m_n), kn = (int)(q % m_n);
    if (dec_score_of<M>(vt, vt_rows, vt_cols, cnt, lo_p + kp, k_pos, lo_n + kn, k_neg) >= score) acc += pp[kp] * pn[kn];
  }
  acc = dec_block_sum(acc, s_red);
  if (threadIdx.x == 0) {
    DecoratedOut o;
    o.pvalue = acc / (sp * sn);
    o.score = score;
    o.cases1 = case_pos1 + case_neg1;
    o.ctrls1 = ctrl_pos1 + ctrl_neg1;
    o.cases2 = case_pos2 + case_neg2;
    o.ctrls2 = ctrl_pos2 + ctrl_neg2;
    out[item] = o;
  }
}

// ---- splits of whole paths, formed from the gene rows of a path set ----

// One split: genes gene[0 .. n_sub) are the sub-path, gene[n_sub] is the gene it is extended by; bit j of `neg` sends gene j to
// the negative part (method 2, sign -1).  Gene rows are `stride` words apart and only their first (positive) half is read.
struct DecSplit {
  int32_t gene[5];
  int32_t n_sub;
  int32_t neg;
};

__device__ __forceinline__ void dec_split_word(const uint64_t* __restrict__ genes, size_t stride, const DecSplit& s, int k, uint64_t& p1, uint64_t& n1,
                                               uint64_t& p2, uint64_t& n2) {
  p1 = n1 = p2 = n2 = 0;
  for (int j = 0; j < s.n_sub; j++) {
    const uint64_t w = __ldg(genes + (size_t)s.gene[j] * stride + k);
    if ((s.neg >> j) & 1) n1 |= w;
    else p1 |= w;
  }
  const uint64_t w = __ldg(genes + (size_t)s.gene[s.n_sub] * stride + k);
  if ((s.neg >> s.n_sub) & 1) n2 = w;
  else p2 = w;
}

// rows := [n_items][4][W64] pos1, neg1, pos2, neg2 of the splits (what decorated_exact_kernel reads); one CTA per split
__global__ void __launch_bounds__(DEC_THREADS) decorated_form_kernel(const uint64_t* __restrict__ genes, size_t stride, const DecSplit* __restrict__ splits,
                                                                    uint32_t n_items, int W64, uint64_t* __restrict__ rows) {
  const uint32_t item = blockIdx.x;
  if (item >= n_items) return;
  const DecSplit s = splits[item];
  uint64_t* r = rows + (size_t)item * 4 * W64;
  for (int k = threadIdx.x; k < W64; k += DEC_THREADS) {
    uint64_t p1, n1, p2, n2;
    dec_split_word(genes, stride, s, k, p1, n1, p2, n2);
    r[k] = p1;
    r[W64 + k] = n1;
    r[2 * W64 + k] = p2;
    r[3 * W64 + k] = n2;
  }
}

// ---- stratified exact mode ----

// s_h[4 g + 0 .. 3] := per stratum g the sub-path's case and control carriers, and kp_g = |pos2' & free & g|, kn_g =
// |neg2' & free & g| with free = ~(pos1 | neg1), pos2' = pos2 & ~pos1, neg2' = neg2 & ~neg1 (so pos2' & free = pos2 & free).
// strata: dense stratum per patient (nullptr: one stratum).  s_h zeroed and synchronised by the caller.
__device__ __forceinline__ void dec_strata_hist(const uint64_t* __restrict__ genes, size_t stride, const DecSplit& s, int W64, int n_cases, int n,
                                                const int32_t* __restrict__ strata, int* s_h) {
  for (int k = threadIdx.x; k < W64; k += DEC_THREADS) {
    const uint64_t valid = (k == W64 - 1 && (n & 63)) ? ((1ull << (n & 63)) - 1ull) : ~0ull;
    uint64_t p1, n1, p2, n2;
    dec_split_word(genes, stride, s, k, p1, n1, p2, n2);
    const uint64_t cover = (p1 | n1) & valid;
    const uint64_t w[3] = {cover, p2 & ~cover & valid, n2 & ~cover & valid};
#pragma unroll
    for (int q = 0; q < 3; q++)
      for (uint64_t b = w[q]; b; b &= b - 1) {
        const int i = k * 64 + __ffsll((long long)b) - 1;
        const int g = strata ? strata[i] : 0;
        atomicAdd(&s_h[4 * g + (q == 0 ? (i < n_cases ? 0 : 1) : q + 1)], 1);
      }
  }
}

// Per-stratum pools of one split from its histogram: free cases c, free controls d, kp, kn.  tot: [S][2] cases / controls per stratum.
__device__ __forceinline__ int4 dec_stratum(const int* s_h, const int* __restrict__ tot, int g) {
  return make_int4(tot[2 * g] - s_h[4 * g], tot[2 * g + 1] - s_h[4 * g + 1], s_h[4 * g + 2], s_h[4 * g + 3]);
}

// Per split: sizes = {sum kp_g, sum kn_g, strata with kp_g + kn_g > 0, first stratum with fewer free patients than carriers to
// redraw (-1: none)}.  Dynamic shared memory: 4 * S ints.
__global__ void __launch_bounds__(DEC_THREADS) decorated_strata_count_kernel(const uint64_t* __restrict__ genes, size_t stride, const DecSplit* __restrict__ splits,
                                                                            uint32_t n_items, int W64, int n_cases, int n, const int32_t* __restrict__ strata, int S,
                                                                            const int* __restrict__ tot, int4* __restrict__ sizes) {
  extern __shared__ int s_h[];
  __shared__ int s_sum[4];
  const uint32_t item = blockIdx.x;
  if (item >= n_items) return;
  const DecSplit s = splits[item];
  for (int i = threadIdx.x; i < 4 * S; i += DEC_THREADS) s_h[i] = 0;
  if (threadIdx.x < 3) s_sum[threadIdx.x] = 0;
  if (threadIdx.x == 3) s_sum[3] = INT_MAX;
  __syncthreads();
  dec_strata_hist(genes, stride, s, W64, n_cases, n, strata, s_h);
  __syncthreads();
  int kp = 0, kn = 0, kept = 0, bad = INT_MAX;
  for (int g = threadIdx.x; g < S; g += DEC_THREADS) {
    const int4 p = dec_stratum(s_h, tot, g);
    kp += p.z;
    kn += p.w;
    kept += (p.z + p.w) > 0;
    if (p.z + p.w > p.x + p.y && g < bad) bad = g;  // R's sample(): "cannot take a sample larger than the population"
  }
  kp = __reduce_add_sync(0xffffffffu, kp);
  kn = __reduce_add_sync(0xffffffffu, kn);
  kept = __reduce_add_sync(0xffffffffu, kept);
  bad = (int)__reduce_min_sync(0xffffffffu, (unsigned)bad);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&s_sum[0], kp);
    atomicAdd(&s_sum[1], kn);
    atomicAdd(&s_sum[2], kept);
    atomicMin(&s_sum[3], bad);
  }
  __syncthreads();
  if (threadIdx.x == 0) sizes[item] = make_int4(s_sum[0], s_sum[1], s_sum[2], s_sum[3] == INT_MAX ? -1 : s_sum[3]);
}

// Scratch doubles of one split of the joint kernel: J and its next state, one stratum's joint, one stratum's positive pmf
__host__ __device__ inline size_t dec_joint_scratch(int sum_kp, int sum_kn) {
  return 3 * ((size_t)sum_kp + 1) * ((size_t)sum_kn + 1) + (size_t)sum_kp + 1;
}

// The stratified exact p-value of each split (decorated.py, compute_decorated_pvalue(strata=...), exact mode):
//   joint_g[x][y] = Hyp(c_g, d_g, kp_g)(x) * Hyp(d_g - (kp_g - x), c_g - x, kn_g)(y),  J = joint_0 * joint_1 * ... (2-D convolution
//   in dense-stratum order),  p = sum over (cp, cn) of J[cp][cn] * [score_of(cp, sum kp, cn, sum kn) >= score].
// One CTA per split; scratch + off[item]: dec_joint_scratch doubles.  Dynamic shared memory: 5 * S ints (histogram, kept strata).
template <int M>
__global__ void __launch_bounds__(DEC_THREADS) decorated_strata_joint_kernel(const uint64_t* __restrict__ genes, size_t stride, const DecSplit* __restrict__ splits,
                                                                            uint32_t n_items, int W64, int n_cases, int n_ctrls, const int32_t* __restrict__ strata,
                                                                            int S, const int* __restrict__ tot, const double* __restrict__ vt, int vt_rows,
                                                                            int vt_cols, const unsigned long long* __restrict__ off, double* __restrict__ scratch,
                                                                            DecoratedOut* __restrict__ out) {
  extern __shared__ int s_h[];
  int* s_kept = s_h + 4 * S;
  __shared__ double s_red[DEC_THREADS / 32];
  __shared__ double s_norm;
  __shared__ int s_cnt[8];
  __shared__ int s_nk, s_kp, s_kn;
  __shared__ DecSplit s;  // in shared memory: its gene list is indexed at run time
  const uint32_t item = blockIdx.x;
  if (item >= n_items) return;
  const int n = n_cases + n_ctrls;
  if (threadIdx.x == 0) s = splits[item];
  for (int i = threadIdx.x; i < 4 * S; i += DEC_THREADS) s_h[i] = 0;
  if (threadIdx.x < 8) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  dec_count8([&](int k, uint64_t& p1, uint64_t& n1, uint64_t& p2, uint64_t& n2) { dec_split_word(genes, stride, s, k, p1, n1, p2, n2); }, W64, n_cases, n, s_cnt);
  dec_strata_hist(genes, stride, s, W64, n_cases, n, strata, s_h);
  __syncthreads();
  // the strata that redraw anything, in dense order (warp 0, ballot compaction)
  if (threadIdx.x < 32) {
    int nk = 0, kp = 0, kn = 0;
    for (int g0 = 0; g0 < S; g0 += 32) {
      const int g = g0 + threadIdx.x;
      const bool keep = g < S && s_h[4 * g + 2] + s_h[4 * g + 3] > 0;
      const unsigned b = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        s_kept[nk + __popc(b & ((1u << threadIdx.x) - 1u))] = g;
        kp += s_h[4 * g + 2];
        kn += s_h[4 * g + 3];
      }
      nk += __popc(b);
    }
    kp = __reduce_add_sync(0xffffffffu, kp);
    kn = __reduce_add_sync(0xffffffffu, kn);
    if (threadIdx.x == 0) {
      s_nk = nk;
      s_kp = kp;
      s_kn = kn;
    }
  }
  __syncthreads();
  const int nk = s_nk, sum_kp = s_kp, sum_kn = s_kn, width = sum_kn + 1;
  const size_t cells = ((size_t)sum_kp + 1) * width;
  double* cur = scratch + off[item];
  double* nxt = cur + cells;
  double* joint = nxt + cells;
  double* pmf = joint + cells;
  if (threadIdx.x == 0) cur[0] = 1.0;
  int A = 0, B = 0;  // J covers [0, A] x [0, B] (row stride `width`)
  for (int t = 0; t < nk; t++) {
    const int4 p = dec_stratum(s_h, tot, s_kept[t]);
    const long long c = p.x, d = p.y, kp = p.z, kn = p.w;
    const long long lo1 = max(0ll, kp - d), hi1 = min(kp, c);
    if (threadIdx.x == 0) {
      dec_hyp_weights(c, d, kp, lo1, hi1, pmf);
      double sum = 0.0;
      for (long long x = lo1; x <= hi1; x++) sum += pmf[x - lo1];
      s_norm = sum;
    }
    __syncthreads();
    const int gw = (int)kn + 1;
    for (long long x = threadIdx.x; x <= kp; x += DEC_THREADS) {  // row x of joint_g: the negatives drawn from what the positives left
      double* row = joint + x * gw;
      for (int y = 0; y < gw; y++) row[y] = 0.0;
      if (x < lo1 || x > hi1) continue;
      const long long good = d - (kp - x), bad = c - x;
      const long long lo2 = max(0ll, kn - bad), hi2 = min(kn, good);
      dec_hyp_weights(good, bad, kn, lo2, hi2, row + lo2);
      double sum = 0.0;
      for (long long y = lo2; y <= hi2; y++) sum += row[y];
      const double px = pmf[x - lo1] / s_norm;
      for (long long y = lo2; y <= hi2; y++) row[y] = px * (row[y] / sum);
    }
    __syncthreads();
    // gather: nxt[a][b] = sum over (x, y) of joint_g[x][y] * J[a - x][b - y], in a fixed order
    const int A2 = A + (int)kp, B2 = B + (int)kn;
    const long long out_cells = (long long)(A2 + 1) * (B2 + 1);
    for (long long q = threadIdx.x; q < out_cells; q += DEC_THREADS) {
      const int a = (int)(q / (B2 + 1)), b = (int)(q % (B2 + 1));
      double acc = 0.0;
      for (int x = max(0, a - A); x <= min((int)kp, a); x++)
        for (int y = max(0, b - B); y <= min((int)kn, b); y++) acc += joint[(size_t)x * gw + y] * cur[(size_t)(a - x) * width + (b - y)];
      nxt[(size_t)a * width + b] = acc;
    }
    __syncthreads();
    double* t2 = cur;
    cur = nxt;
    nxt = t2;
    A = A2;
    B = B2;
  }
  int cnt[8];
#pragma unroll
  for (int q = 0; q < 8; q++) cnt[q] = s_cnt[q];
  const int k_pos = cnt[4] + cnt[5], k_neg = cnt[6] + cnt[7];
  const double score = dec_score_of<M>(vt, vt_rows, vt_cols, cnt, cnt[4], k_pos, cnt[6], k_neg);
  double acc = 0.0;
  for (long long q = threadIdx.x; q < (long long)cells; q += DEC_THREADS) {
    const int a = (int)(q / width), b = (int)(q % width);
    if (dec_score_of<M>(vt, vt_rows, vt_cols, cnt, a, sum_kp, b, sum_kn) >= score) acc += cur[q];
  }
  acc = dec_block_sum(acc, s_red);
  if (threadIdx.x == 0) {
    DecoratedOut o;
    o.pvalue = acc;
    o.score = score;
    o.cases1 = cnt[0] + cnt[2];
    o.ctrls1 = cnt[1] + cnt[3];
    o.cases2 = cnt[4] + cnt[6];
    o.ctrls2 = cnt[5] + cnt[7];
    out[item] = o;
  }
}

// per-stratum case / control totals: tot[2 g + (patient is a control)] (tot zeroed by the caller)
__global__ void strata_totals_kernel(const int32_t* __restrict__ strata, int n, int n_cases, int* __restrict__ tot) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicAdd(&tot[2 * strata[i] + (i < n_cases ? 0 : 1)], 1);
}

}  // namespace gcre
