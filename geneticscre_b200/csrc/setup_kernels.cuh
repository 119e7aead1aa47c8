// One-off input preparation kernels: bit packing, mask layouts, value-table re-layout, row gather.
#pragma once
#include "common.cuh"

namespace gcre {

// PathSet::load (src/gcre_paths.h:56-78): int32 matrix [rows][cols] -> bit c%64 of word c/64 of the pos half.
// One warp packs 64 consecutive patients of one row with two ballots (coalesced 128 B reads).
__global__ void pack_rows_i32_kernel(const int32_t* __restrict__ data, uint32_t rows, int cols, uint64_t* __restrict__ out,
                                     int row_words, int W64) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_items = (long long)rows * W64;
  if (warp >= n_items) return;
  const uint32_t r = (uint32_t)(warp / W64);
  const int k = (int)(warp % W64);
  const int c0 = k * 64 + lane, c1 = c0 + 32;
  const int32_t* row = data + (size_t)r * cols;
  const int v0 = (c0 < cols) ? row[c0] : 0;
  const int v1 = (c1 < cols) ? row[c1] : 0;
  const unsigned lo = __ballot_sync(0xffffffffu, v0 != 0);
  const unsigned hi = __ballot_sync(0xffffffffu, v1 != 0);
  if (lane == 0) out[(size_t)r * row_words + k] = ((uint64_t)hi << 32) | lo;
}

// packed rows uint64[rows][wsrc] -> pos half of device rows (row stride row_words), rest of the row untouched (zero)
__global__ void place_rows_kernel(const uint64_t* __restrict__ src, uint32_t rows, int wsrc, int wcopy, uint64_t* __restrict__ out, int row_words) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)rows * wcopy) return;
  const uint32_t r = (uint32_t)(i / wcopy);
  const int k = (int)(i % wcopy);
  out[(size_t)r * row_words + k] = src[(size_t)r * wsrc + k];
}

// Bits at patient indices >= n cannot mean anything (there are n = num_cases + num_ctrls patients); packed inputs and raw
// row writes may carry them.  Cleared on entry: the sparse kernels index the patient-major masks by patient, and the padding
// word of a half-row (Wp is W64 rounded up to 2) must stay zero.
__global__ void mask_tail_kernel(uint64_t* __restrict__ rows_io, long long n_halves, int Wp, int W64, int n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_halves) return;
  uint64_t* p = rows_io + (size_t)i * Wp;
  const int rem = n & 63;
  if (rem && W64 > 0) p[W64 - 1] &= (1ull << rem) - 1ull;
  for (int k = W64; k < Wp; k++) p[k] = 0ull;
}

// device rows -> unpadded host layout uint64[rows][W64*M]
template <int M>
__global__ void unpad_rows_kernel(const uint64_t* __restrict__ rows_in, uint32_t rows, int Wp, int W64, uint64_t* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int wout = W64 * M;
  if (i >= (long long)rows * wout) return;
  const uint32_t r = (uint32_t)(i / wout);
  const int k = (int)(i % wout);
  const int h = k / W64, kk = k % W64;
  out[i] = rows_in[(size_t)r * (Wp * M) + h * Wp + kk];
}

// PathSet::select (src/gcre_paths.h:82-92): out row k = in row idx[k]; 16-byte copies
__global__ void select_rows_kernel(const ulonglong2* __restrict__ in, const int32_t* __restrict__ idx, uint32_t n, int row_vec,
                                   ulonglong2* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * row_vec) return;
  const uint32_t r = (uint32_t)(i / row_vec);
  const int k = (int)(i % row_vec);
  out[(size_t)r * row_vec + k] = in[(size_t)idx[r] * row_vec + k];
}

// max over rows of the per-half carrier count (bounds the anti-diagonal range a join can touch)
template <int M>
__global__ void row_maxpop_kernel(const uint64_t* __restrict__ rows_in, uint32_t rows, int Wp, unsigned* __restrict__ out_max) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= (long long)rows * M) return;
  const uint64_t* p = rows_in + (size_t)warp * Wp;  // halves are contiguous: row r half h starts at (r*M + h) * Wp
  unsigned c = 0;
  for (int k = lane; k < Wp; k += 32) c += __popcll(p[k]);
  c = __reduce_add_sync(0xffffffffu, c);
  if (lane == 0 && c) atomicMax(out_max, c);
}

// setPermutedCases (src/join_base.cpp:85-125): int32 [rows][cols] (1 = kept) -> packed case masks, perm-major
// out[r][k] = case_mask[k] ^ flip_r[k].  One warp per (perm, word).
__global__ void pack_perm_i32_kernel(const int32_t* __restrict__ perm, int rows, int cols, int n_cases, int W64,
                                     uint64_t* __restrict__ out, int row0) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= (long long)rows * W64) return;
  const int r = (int)(warp / W64);
  const int k = (int)(warp % W64);
  const int c0 = k * 64 + lane, c1 = c0 + 32;
  const int32_t* row = perm + (size_t)r * cols;
  const bool f0 = (c0 < cols) && (row[c0] != 1);
  const bool f1 = (c1 < cols) && (row[c1] != 1);
  const unsigned lo = __ballot_sync(0xffffffffu, f0);
  const unsigned hi = __ballot_sync(0xffffffffu, f1);
  if (lane == 0) out[(size_t)(row0 + r) * W64 + k] = ((((uint64_t)hi) << 32) | lo) ^ case_mask_word(k, n_cases);
}

// cyclic reuse of supplied rows when fewer than iters were given (src/join_base.cpp:116-123)
__global__ void cycle_perm_rows_kernel(uint64_t* __restrict__ masks, int have, int iters, int W64) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)(iters - have) * W64) return;
  const int r = have + (int)(i / W64);
  const int k = (int)(i % W64);
  masks[(size_t)r * W64 + k] = masks[(size_t)(r % have) * W64 + k];
}

// perm-major packed masks [I][W64] -> word-major tile layout [Wp][Ip] (zero padded) for the dense kernels
__global__ void masks_to_word_major_kernel(const uint64_t* __restrict__ masks, int iters, int W64, uint64_t* __restrict__ pm, int Wp, int Ip) {
  __shared__ uint64_t tile[32][33];
  const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int r = r0 + j, k = k0 + threadIdx.x;
    tile[j][threadIdx.x] = (r < iters && k < W64) ? masks[(size_t)r * W64 + k] : 0ull;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int k = k0 + j, r = r0 + threadIdx.x;
    if (k < Wp && r < Ip) pm[(size_t)k * Ip + r] = tile[threadIdx.x][j];
  }
}

// perm-major packed masks [I][W64] -> patient-major bit matrix pt[c][w] (bit r%32 of word r/32 = patient c is a case
// under permutation r).  One warp transposes a 32 (perms) x 32 (patients) bit block with ballots.
__global__ void masks_to_patient_major_kernel(const uint64_t* __restrict__ masks, int iters, int W64, int n, uint32_t* __restrict__ pt, int Iw) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_cblk = (n + 31) / 32;
  if (warp >= (long long)Iw * n_cblk) return;
  const int w = (int)(warp / n_cblk);   // perm word
  const int cb = (int)(warp % n_cblk);  // block of 32 patients
  // slots beyond the requested permutations hold copies of real ones (r mod iters): they score like real permutations, so a
  // lane's threshold (thresholded look-ups, join_sparse.cuh) is not pinned at zero by padding; their maxima are never read
  const int r = (iters > 0) ? (w * 32 + lane) % iters : 0;
  uint32_t mine = 0;  // 32 patient bits of perm r
  if (iters > 0) {
    const uint64_t word = masks[(size_t)r * W64 + (cb >> 1)];
    mine = (uint32_t)(word >> ((cb & 1) * 32));
  }
  // lane j ends up with the word of patient cb*32 + j: bit i = bit j of lane i's `mine`
  uint32_t outw = 0;
  for (int j = 0; j < 32; j++) {
    const unsigned b = __ballot_sync(0xffffffffu, (mine >> j) & 1u);
    if (lane == j) outw = b;
  }
  const int c = cb * 32 + lane;
  if (c < n) pt[(size_t)c * Iw + w] = outw;
}

// value table (row-major R layout [cases][ctrls], reads outside give -1.0 like the reference's padded square,
// src/join_base.cpp:62-80) -> anti-diagonal-major tables up to total t_cap:
//   D [t(t+1)/2 + c] = vt[c][t-c]
//   F [..]           = (float) vt[c][t-c]              (method 1 permutation look-ups; NaN -> -1 so it can never win)
//   DM[..]           = std::max(vt[c][t-c], vt[t-c][c]) (src/methods.h:110-118; std::max(a,b) = a<b ? b : a)
//   FM[..]           = DM rounded up to f32 (method 2: upper bound used before the exact f64 look-ups, join_sparse.cuh)
__global__ void build_diag_kernel(const double* __restrict__ vt, int rows, int cols, unsigned t_cap, double* __restrict__ D,
                                  float* __restrict__ F, double* __restrict__ DM, float* __restrict__ FM) {
  const unsigned t = blockIdx.x;
  if (t > t_cap) return;
  const size_t base = diag_base(t);
  for (unsigned c = threadIdx.x; c <= t; c += blockDim.x) {
    const unsigned q = t - c;
    const double a = (c < (unsigned)rows && q < (unsigned)cols) ? vt[(size_t)c * cols + q] : -1.0;
    D[base + c] = a;
    if (F) F[base + c] = (a != a) ? -1.0f : (float)a;
    if (DM) {
      const double b = (q < (unsigned)rows && c < (unsigned)cols) ? vt[(size_t)q * cols + c] : -1.0;
      const double mx = (a < b) ? b : a;
      DM[base + c] = mx;
      FM[base + c] = __double2float_ru(mx);  // (NaN stays NaN: it never passes a `>` test, like the exact sum it stands for)
    }
  }
}

// ---- join index (UidRelSet) preparation on the device ---------------------------------------------------------------
// uid_ref array-of-structs (src/gcre_types.h:50-56; 24 bytes each) -> the arrays the join kernels read, plus the inputs
// of the two prefix sums (pairs per row, work units per row) and the bounds the pre-checks need.
struct UidRefPOD {
  int32_t src, trg, count;
  uint32_t location;
  unsigned long long path_idx;
};

struct UidStats {
  unsigned long long max_loc_end;   // max(location + count) over rows with count > 0
  unsigned long long max_res_end;   // max(path_idx + count)
  unsigned int res_not_prefix;      // != 0 if some path_idx differs from the running sum of counts
};

__global__ void split_uids_kernel(const UidRefPOD* __restrict__ uids, uint32_t n, int partners_per_unit, int32_t* __restrict__ count,
                                  uint32_t* __restrict__ loc, unsigned long long* __restrict__ res, unsigned long long* __restrict__ pairs_in,
                                  unsigned long long* __restrict__ units_in, UidStats* __restrict__ stats) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long le = 0, re = 0;
  if (u < n) {
    const UidRefPOD r = uids[u];
    const int32_t c = r.count > 0 ? r.count : 0;
    count[u] = c;
    loc[u] = r.location;
    res[u] = r.path_idx;
    pairs_in[u] = (unsigned long long)c;
    units_in[u] = ((unsigned long long)c + partners_per_unit - 1) / partners_per_unit;
    if (c > 0) {
      le = (unsigned long long)r.location + c;
      re = r.path_idx + c;
    }
  } else if (u == n) {  // the scans run over n + 1 entries
    pairs_in[u] = 0;
    units_in[u] = 0;
  }
  // warp-level max, then one atomic per warp
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    le = max(le, __shfl_xor_sync(0xffffffffu, le, d));
    re = max(re, __shfl_xor_sync(0xffffffffu, re, d));
  }
  if ((threadIdx.x & 31) == 0) {
    if (le) atomicMax(&stats->max_loc_end, le);
    if (re) atomicMax(&stats->max_res_end, re);
  }
}

// after the scans: unit -> upstream row table, and the "result rows are the running sums" check
__global__ void finish_uids_kernel(uint32_t n, const int32_t* __restrict__ count, const unsigned long long* __restrict__ res,
                                   const unsigned long long* __restrict__ prefix, const unsigned long long* __restrict__ units,
                                   uint32_t* __restrict__ unit_idx, UidStats* __restrict__ stats) {
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n) return;
  if (count[u] > 0 && res[u] != prefix[u]) stats->res_not_prefix = 1;
  for (unsigned long long q = units[u]; q < units[u + 1]; q++) unit_idx[q] = u;
}

// ---- provenance of kept rows (the tail form of the pre-counted sparse kernel, join_sparse.cuh) -------------------------
// Entries name a row of a base path set and its orientation: base row << 1 | 1 when the row's halves are swapped (method 2:
// joined half h holds base half 1 - h).  A KEEP join whose partner set is a selection of the base set records, per result
// row it writes, the partner's base row (`tail`) and - when every upstream row is exactly one oriented base row - the
// upstream row's entry (`head`).  `sel`: the selection's own entries (below).
// Both passes below run one thread per work unit of the join index (<= partners_per_unit partners of one upstream row; units
// [unit_lo, unit_hi) are those of upstream rows [ub, ue)).  The networks are heavy-tailed: one row of the benchmark's network has
// 4,622 partners, and a thread per upstream row left each launch as long as that row's serial loop.  A warp per unit idled
// most lanes instead: the level-4 rows of the benchmark average 9 partners (BASELINE config 3, B200 at 1,000 W, eligibility pass
// of methods 1 / 2: 0.37 / 0.39 ms with a thread per row, 0.21 / 0.25 with a warp per unit, 0.05 / 0.06 with a thread per unit).
template <int M>
__global__ void record_rows_kernel(unsigned long long unit_lo, unsigned long long unit_hi, const uint32_t* __restrict__ unit_idx,
                                   const unsigned long long* __restrict__ unit_prefix, int partners_per_unit, const int32_t* __restrict__ count,
                                   const uint32_t* __restrict__ location, const unsigned long long* __restrict__ res_idx,
                                   const int32_t* __restrict__ signs, int path_length, const uint32_t* __restrict__ sel,
                                   const uint32_t* __restrict__ tail0, uint32_t* __restrict__ tail_res, uint32_t* __restrict__ head_res) {
  const unsigned long long q = unit_lo + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= unit_hi) return;
  const uint32_t idx = unit_idx[q];
  const uint32_t j0 = (uint32_t)(q - unit_prefix[idx]) * (uint32_t)partners_per_unit;
  const uint32_t j1 = min((uint32_t)count[idx], j0 + (uint32_t)partners_per_unit);
  const uint32_t loc0 = location[idx];
  const unsigned long long r0 = res_idx[idx];
  const uint32_t head = head_res ? tail0[idx] : 0u;
  for (uint32_t j = j0; j < j1; j++) {
    const uint32_t loc = loc0 + j;
    const bool swap = (M == 2) && !need_flip(path_length, signs, idx, loc);  // src/methods.h:137-145: partner half 1 - h joins half h
    tail_res[r0 + j] = sel[loc] | (swap ? 1u : 0u);
    if (head_res) head_res[r0 + j] = head;
  }
}

// The entries of a selection (gcre_pathset_select): row k is base row idx[k], halves as they are; with idx null row k is row k
// (the map of a pre-counted join whose partners are scored through their own rows)
__global__ void selection_entries_kernel(const int32_t* __restrict__ idx, uint32_t n, uint32_t* __restrict__ sel) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) sel[k] = (idx ? (uint32_t)idx[k] : k) << 1;
}

// Does every pair of units [unit_lo, unit_hi) meet the tail form's condition: the partner's head, oriented as the pair joins it,
// is the upstream row's tail (same base row, same orientation)?  Partner rows outside [head_lo, head_hi) have no record.
// Any pair that does not sets *bad.  One thread per unit, as record_rows_kernel.
template <int M>
__global__ void tail_eligible_kernel(unsigned long long unit_lo, unsigned long long unit_hi, const uint32_t* __restrict__ unit_idx,
                                     const unsigned long long* __restrict__ unit_prefix, int partners_per_unit, const int32_t* __restrict__ count,
                                     const uint32_t* __restrict__ location, const int32_t* __restrict__ signs, int path_length,
                                     const uint32_t* __restrict__ tail0, const uint32_t* __restrict__ head1, unsigned long long head_lo,
                                     unsigned long long head_hi, unsigned* __restrict__ bad) {
  const unsigned long long q = unit_lo + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool ok = true;
  if (q < unit_hi) {
    const uint32_t idx = unit_idx[q];
    const uint32_t j0 = (uint32_t)(q - unit_prefix[idx]) * (uint32_t)partners_per_unit;
    const uint32_t j1 = min((uint32_t)count[idx], j0 + (uint32_t)partners_per_unit);
    const uint32_t loc0 = location[idx];
    const uint32_t t = tail0[idx];
    for (uint32_t j = j0; j < j1 && ok; j++) {
      const uint32_t loc = loc0 + j;
      if (loc < head_lo || loc >= head_hi) {
        ok = false;
        break;
      }
      uint32_t h = head1[loc];
      if (M == 2 && !need_flip(path_length, signs, idx, loc)) h ^= 1u;  // the pair swaps the partner's halves
      ok = (M == 2) ? h == t : (h >> 1) == (t >> 1);
    }
  }
  if (__any_sync(0xffffffffu, !ok) && (threadIdx.x & 31) == 0) atomicOr(bad, 1u);
}

}  // namespace gcre
