// Seeded permutation masks generated on the device (gcre_exec_generate_permuted_masks).  geneticscre_b200/synth.py
// (make_perm_masks_philox) restates the definition in numpy; the two agree bit for bit.
//
// Permutation r of seed s: patient i draws u_i from Philox4x32-10 with key (lo32(s), hi32(s)) and counter
// (i >> 1, lo32(r), hi32(r), 0), u_i = x0 | x1 << 32 (i even) or x2 | x3 << 32 (i odd).  Patients are visited in index order;
// i is a case iff mulhi64(u_i, m_i) < k_g, with m_i the not-yet-visited patients of i's stratum g (i included) and k_g the
// cases still to place in g (initially g's patients with index < num_cases): sequential selection sampling per stratum.
//
// One warp per permutation, 64 patients (one output word) per step: lane l draws for patients 2l and 2l + 1 (one Philox call)
// and forms v_i = mulhi64(u_i, m_i) < 2^31.  Within the word the decisions depend on each other only through the number of
// cases among earlier patients of the same stratum, c_i, as d_i = [v_i < k_g - c_i] with k_g taken at the start of the word.
// The warp iterates d <- F(d) from d = [v < k_g]: after t rounds the first t patients are final (patient q depends on patients
// before q only), and a round that changes nothing has reached the unique solution of the sequential definition.  A draw is
// rarely within a few counts of k (probability ~ 64 / m), so a word is expected to settle in two or three rounds of two ballots
// and two popcounts; the serial compare-and-decrement chain is never walked patient by patient.
//
// Stratified masks read three per-patient arrays built once per strata setting (gcre_exec_set_permutation_strata): the dense
// stratum index, m_i with bit 31 set on the last patient of its stratum within its word (that lane writes k_g back), and the
// word's earlier same-stratum patients as a mask in ballot order (bit l = patient 2l, bit 32 + l = patient 2l + 1).  The k_g
// of a warp live in shared memory.  Without strata m_i = n - i and the earlier patients are a lane mask.
#pragma once
#include "common.cuh"

namespace gcre {

constexpr int PG_WARPS = 4;              // permutations per CTA
constexpr int PG_MAX_STRATA = 1024;      // k_g of one warp: 4 KB of shared memory

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// rows [0, iters) of masks (perm-major uint64[iters][W64]) := permutations first_perm + row
template <bool STRATA>
__global__ void __launch_bounds__(PG_WARPS * 32) perm_gen_kernel(uint64_t* __restrict__ masks, int iters, int W64, int n, int n_cases,
                                                                 uint64_t seed, uint64_t first_perm, const int2* __restrict__ sidx,
                                                                 const uint2* __restrict__ mlast, const ulonglong2* __restrict__ peer,
                                                                 const int32_t* __restrict__ k_init, int n_strata) {
  extern __shared__ int pg_k[];
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int row = blockIdx.x * PG_WARPS + wib;
  if (row >= iters) return;  // whole warps only; no block-wide barrier below
  int* ks = pg_k + wib * n_strata;
  if (STRATA) {
    for (int g = lane; g < n_strata; g += 32) ks[g] = k_init[g];
    __syncwarp();
  }
  const uint64_t r = first_perm + (uint64_t)row;
  const uint32_t key0 = (uint32_t)seed, key1 = (uint32_t)(seed >> 32);
  const unsigned lt = (1u << lane) - 1u, le = lt | (1u << lane);
  int K = n_cases;  // cases still to place (one stratum)
  uint64_t held = 0ull;
  uint64_t* out = masks + (size_t)row * W64;
  for (int w = 0; w < W64; w++) {
    const int j = w * 32 + lane;  // patient pair
    const int i0 = 2 * j, i1 = i0 + 1;
    const uint4 x = philox4x32_10(make_uint4((uint32_t)j, (uint32_t)r, (uint32_t)(r >> 32), 0u), key0, key1);
    const uint64_t u0 = (uint64_t)x.x | ((uint64_t)x.y << 32), u1 = (uint64_t)x.z | ((uint64_t)x.w << 32);
    unsigned m0, m1;
    int k0, k1, g0 = 0, g1 = 0;
    uint64_t p0, p1;
    bool last0 = false, last1 = false;
    if (STRATA) {
      const int2 g = sidx[j];
      const uint2 ml = mlast[j];
      const ulonglong2 pp = peer[j];
      g0 = g.x;
      g1 = g.y;
      m0 = ml.x & 0x7fffffffu;
      m1 = ml.y & 0x7fffffffu;
      last0 = ml.x >> 31;
      last1 = ml.y >> 31;
      p0 = pp.x;
      p1 = pp.y;
      k0 = ks[g0];
      k1 = ks[g1];
    } else {
      m0 = (unsigned)max(n - i0, 0);
      m1 = (unsigned)max(n - i1, 0);
      k0 = k1 = K;
      p0 = (uint64_t)lt | ((uint64_t)lt << 32);  // earlier patients of 2l: 2l' and 2l' + 1 for l' < l
      p1 = (uint64_t)le | ((uint64_t)lt << 32);  // of 2l + 1: also 2l
    }
    // v < m <= n < 2^31; patients >= n (m = 0 there) are never cases
    const int v0 = i0 < n ? (int)__umul64hi(u0, (uint64_t)m0) : 0x7fffffff;
    const int v1 = i1 < n ? (int)__umul64hi(u1, (uint64_t)m1) : 0x7fffffff;
    bool d0 = v0 < k0, d1 = v1 < k1;
    int c0, c1;
    uint64_t D;
    for (;;) {
      D = (uint64_t)__ballot_sync(FULL, d0) | ((uint64_t)__ballot_sync(FULL, d1) << 32);
      c0 = __popcll(D & p0);
      c1 = __popcll(D & p1);
      const bool e0 = v0 < k0 - c0, e1 = v1 < k1 - c1;
      if (!__any_sync(FULL, (e0 != d0) || (e1 != d1))) break;
      d0 = e0;
      d1 = e1;
    }
    if (STRATA) {
      __syncwarp();  // every lane has read its k_g of this word
      if (last0) ks[g0] = k0 - c0 - (int)d0;
      if (last1) ks[g1] = k1 - c1 - (int)d1;
      __syncwarp();
    } else {
      K -= __popcll(D);
    }
    // ballot order -> patient order: bit 2l + h of the word is (d0, d1)[h] of lane l
    const unsigned both = (unsigned)d0 | ((unsigned)d1 << 1);
    const unsigned a = __shfl_sync(FULL, both, lane >> 1), b = __shfl_sync(FULL, both, 16 + (lane >> 1));
    const uint64_t word = (uint64_t)__ballot_sync(FULL, (a >> (lane & 1)) & 1u) | ((uint64_t)__ballot_sync(FULL, (b >> (lane & 1)) & 1u) << 32);
    if (lane == (w & 31)) held = word;
    if ((w & 31) == 31 || w == W64 - 1) {  // 32 words at a time, one coalesced store
      const int w0 = w & ~31;
      if (w0 + lane <= w) out[w0 + lane] = held;
    }
  }
}

}  // namespace gcre
