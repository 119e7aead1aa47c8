// Sparse join + permutation scoring (sm_100a): carrier-list walk over patient-major permutation masks.
//
// Rare-variant rows are sparse (R keeps genes with carriers <= 5 % of patients, R/Utils.R:185-188), so instead of
// AND+POPC over all W words per permutation (src/methods.h:73-88) the count |joined & mask_r| is formed as
//        sum over carriers c of the joined row of  PT[c][r]          (PT = permutation masks, patient-major bits)
// with 32 permutations per 32-bit word held in bit-sliced (vertical) counters: one LOP3 pair (carry-save adder) adds
// one carrier to 32 permutations at once.  The counts are exact integers, so every result is bit-identical to the
// dense formulation and to the reference.
//
// Work decomposition (one warp = one "unit" at a time, lanes = 32 permutation words = 1,024 permutations):
//   unit  = (upstream row idx, a block of <= PB of its partners, a block of 1,024 permutations)
//   base  : the upstream row's own carriers are accumulated once per unit        -> base counts (u16, shared memory)
//   pair  : only the partner's carriers NOT already in the upstream row (bit test against the dense upstream row) are
//           accumulated on top of the base (ballot-compacted into a shared-memory queue of row offsets, drained eight at a
//           time); partners that add no carrier reuse the base evaluation
//   score : counts -> anti-diagonal value-table look-ups (src/methods.h:96-103, 220-230) -> running per-permutation
//           max kept in registers across all units of the warp, merged at the end with an atomicMax per permutation it raises
//   true scores / top-K candidates / kept rows exactly as in the dense kernel.
//
// Kept rows carry their counts forward.  A KEEP join has the per-permutation counts of every row it writes in registers
// anyway; it stores them (2 KB per row, half and 1,024-permutation block, in the register image of this kernel) together
// with the rows' carrier totals.  The next level, whose upstream operand those rows are, loads its base counts from that
// table instead of walking the upstream carrier list per unit (a quarter of the level-4 gathers of BASELINE config 3) and
// needs no carrier lists of the upstream set at all.
//
// Pre-counted partners (template flag PC).  When every partner row is joined with several upstream rows, its own
// per-permutation counts P[row][half][perm] are formed once (build_precount_kernel) and a pair needs only
//        count(up | partner) = count(up) + count(partner) - count(up & partner)
// where up & partner - the partner's carriers that ARE already in the upstream row - is a handful of patients for
// rare-variant rows (|up|*|partner|/n) instead of the ~|partner| carriers the delta formulation walks.  A pair then costs
// one 2 KB read of P (coalesced, 4 x LDG.128 per lane), the filter pass over the partner's list and the look-ups.
//
// A pre-counted partner is always read through a row map: s.map1[loc] names the row of the pre-counted set whose carrier list
// and P stand for partner row loc, and its orientation (row << 1 | halves swapped); off1 / len1 / car1 / ncase1 / pcnt1 describe
// that set.  Three maps exist:
//  * the partner set itself: entries k << 1 (the exec's identity map);
//  * a selection of a base set (gcre_pathset_select: level 3's partners are copies of data1's gene rows): the selection's own
//    entries (base row << 1, halves as they are) - no lists of the copy, and one table shared with level 4;
//  * the tail form.  In the level schedule of the reference a level-4 partner row is a path g3 -> t whose first gene g3 is the
//    last gene of the upstream path (a paths2 row against a paths3 row).  When the engine knows where the rows came from
//    (gcre_capi.cu: provenance) and every pair of the join has that shape - the partner's first gene, oriented by the pair, is
//    exactly the upstream row's last gene - then  up | partner == up | gene row of t  and the partner is scored through the
//    base-set GENE row of t:
//        count(up | partner) = count(up) + P[t] - count(up & t)
//    up & t is a fraction of a carrier for rare-variant rows, P over the few thousand gene rows fits in L2, and the gene's list
//    is half as long as the partner's.  The map is the partner set's provenance: per row the base row of its last gene and
//    whether the pair orientation swaps its halves.
// A KEEP join in this form emits the final base + P - overlap counts in the same register image the delta form emits, so the
// next level cannot tell which form made them.
#pragma once
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace gcre {

namespace sparse {
constexpr int THREADS = 128;
constexpr int WARPS = THREADS / 32;
constexpr int PB = 64;          // partners per unit
constexpr int FLUSH_AT = 240;   // carrier slots accumulated in the 8 bit planes before they are flushed into u16 counters
constexpr int QCAP = 96;        // per-warp queue of filtered partner carriers (drained at 64)
// Resident CTAs per SM asked of ptxas (= register budget).  Measured on B200 with the level-4 join of BASELINE config 3:
//   running maxima in registers (THR = false): method 1 best at 8 CTAs (64 registers, a few hundred bytes spilled), method 2 at 5
//   (96 registers, no spills; 6 CTAs spill);
//   thresholded look-ups (THR = true): both methods compile to 64 registers without spills -> 8 CTAs = 32 warps per SM
//   (method 2 at 6 / 7 / 8 CTAs: 17.2 / 16.5 / 16.4 ms; method 1 at 8 / 10 / 12: 12.9 / 12.7 / 12.7 ms, profiles/r2_occupancy_variants.txt).
#ifndef GCRE_SPARSE_MB2
#define GCRE_SPARSE_MB2 5
#endif
#ifndef GCRE_SPARSE_MB1
#define GCRE_SPARSE_MB1 8
#endif
#ifndef GCRE_SPARSE_MB_THR
#define GCRE_SPARSE_MB_THR 8
#endif
constexpr int min_blocks(int m, bool thr) { return thr ? GCRE_SPARSE_MB_THR : (m == 1 ? GCRE_SPARSE_MB1 : GCRE_SPARSE_MB2); }
}  // namespace sparse

// Carrier-list (CSR) view of a path set: per (row, half) the ascending patient indices of its set bits.
// Every list starts on an 8-entry (16-byte) boundary and is padded to a multiple of 8 entries with the sentinel
// patient index n, whose row of the patient-major mask matrix is all zero - so lists can be consumed eight carriers
// at a time with one 16-byte load and no tail handling.
struct SparseView {
  unsigned long long* off = nullptr;  // [size*M + 1]  padded prefix (entries), multiples of 8; 64-bit: a kept level-3 set at 100,000
                                      // patients holds ~1e9 carriers and larger cohorts pass 2^32
  uint32_t* len = nullptr;    // [size*M]      true carrier counts
  void* car = nullptr;        // [off[size*M]] patient indices: u16 when n <= 65,535, else u32
  uint32_t* ncase = nullptr;  // [size*M] carriers < n_cases (a prefix of the ascending list)
  size_t total = 0;           // padded entries
  bool valid = false;         // lists (off, car) and stats (len, ncase) are built
  bool stats_valid = false;   // len / ncase alone are filled (by the join that produced the rows): enough for an upstream operand with pcnt
  // per-permutation counts of every (row, half), in the register image of the join kernel:
  // [item][perm block][q = 0..3][lane][4] u32 = packed u16 pairs (registers 4q..4q+3 of GCRE_C16_REG) - 2 KB per block
  uint32_t* pcnt = nullptr;
  unsigned long long pcnt_gen = 0;  // exec->mask_gen the table was built for
  int pcnt_layout = 0;              // 0: the image above; 4 / 8 / 16: the split-carrier kernels' (join_sparse_sc.cuh: [item][lane][NW / 2] u32)
  // rows whose counts / ranges / len / ncase were emitted: a KEEP join over a shard of its upstream rows (multi-GPU: each
  // rank builds only the rows its shard of the next level consumes) fills [emit_lo, emit_hi) only
  unsigned long long emit_lo = 0, emit_hi = 0;
  // per row, a 64-bit hash of its words (row_fingerprint), emitted with the counts over the same [emit_lo, emit_hi): what the
  // grouping of equal upstream rows (gcre_capi.cu: group_upstream_rows) sorts by.  Null for rows no join wrote.
  unsigned long long* fp = nullptr;
};

struct SparseParams {
  const unsigned long long* off0; const uint32_t* len0; const void* car0; const uint32_t* ncase0;   // car: CT[] (u16 or u32)
  const unsigned long long* off1; const uint32_t* len1; const void* car1; const uint32_t* ncase1;
  int n;                                  // patients; also the sentinel carrier index (zero row of pt)
  const unsigned long long* unit_prefix;  // [U+1] running sum of ceil(count/PB)
  const uint32_t* unit_idx;               // [n_units_total] upstream row of every unit (replaces a binary search per unit)
  unsigned long long unit_begin, n_units;  // units of this launch
  unsigned long long* work_counter;
  int n_perm_blocks;                      // ceil(Iw / 32)
  const uint32_t* pcnt1;                  // pre-counted partners (PC kernels), else null
  const uint32_t* pcnt0;                  // per-permutation counts of the upstream rows (emitted by the join that made them), else null
  uint32_t* pcnt_res;                     // KEEP: where to emit the counts / carrier totals of the kept rows, else null
  uint32_t* len_res;
  uint32_t* ncase_res;
  unsigned long long* exact_pairs;        // diagnostic (thresholded look-ups): pairs whose exact permutation scores had to be looked up
  const uint32_t* map1;                   // PC kernels: per partner row, the row of the pre-counted set it is scored through << 1 | halves swapped
  const uint32_t* unit_list;              // grouped upstream rows: the representatives' units; launch item k is unit unit_list[k], else unit k
  unsigned long long* fp_res;             // KEEP: where to emit the kept rows' fingerprints, else null
};

// ---- view construction ----------------------------------------------------------------------------------------------
// per (row, half): true carrier count and the padded count (multiple of 8) that is prefix-summed into offsets
__global__ void half_popcount_kernel(const uint64_t* __restrict__ rows, long long n_items, int Wp, uint32_t* __restrict__ len,
                                     unsigned long long* __restrict__ padded) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= n_items) return;
  const uint64_t* p = rows + (size_t)warp * Wp;
  unsigned c = 0;
  for (int k = lane; k < Wp; k += 32) c += __popcll(p[k]);
  c = __reduce_add_sync(0xffffffffu, c);
  if (lane == 0) {
    len[warp] = c;
    padded[warp] = (c + 7u) & ~7u;
  }
}

template <typename CT>
__global__ void build_lists_kernel(const uint64_t* __restrict__ rows, long long n_items, int Wp, int n_cases, int sentinel,
                                   const unsigned long long* __restrict__ off, CT* __restrict__ car, uint32_t* __restrict__ ncase) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= n_items) return;
  const uint64_t* p = rows + (size_t)warp * Wp;
  unsigned long long pos = off[warp];
  unsigned nc = 0;
  for (int k0 = 0; k0 < Wp; k0 += 32) {
    const int k = k0 + lane;
    uint64_t w = (k < Wp) ? p[k] : 0ull;
    const unsigned c = __popcll(w);
    // exclusive prefix over lanes keeps the list ascending
    unsigned incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    unsigned long long o = pos + incl - c;
    while (w) {
      const int b = __ffsll((long long)w) - 1;
      w &= w - 1;
      const int patient = k * 64 + b;
      car[o++] = (CT)patient;
      nc += patient < n_cases;
    }
    pos += __shfl_sync(0xffffffffu, incl, 31);
  }
  // pad with the sentinel up to the next list start
  const unsigned long long end = off[warp + 1];
  for (unsigned long long o = pos + lane; o < end; o += 32) car[o] = (CT)sentinel;
  nc = __reduce_add_sync(0xffffffffu, nc);
  if (lane == 0) ncase[warp] = nc;
}

// ---- bit-sliced counters -----------------------------------------------------------------------------------------------
__device__ __forceinline__ void csa(uint32_t& hi, uint32_t& lo, uint32_t a, uint32_t b, uint32_t c) {
  const uint32_t u = a ^ b;
  hi = (a & b) | (u & c);
  lo = u ^ c;
}

// add eight 1-bit-per-permutation words into the 8 bit planes (Harley-Seal carry-save tree: 3 LOP3 per carrier)
__device__ __forceinline__ void hs8(uint32_t (&pl)[8], const uint32_t (&x)[8]) {
  uint32_t ta, tb, fa, fb, e;
  csa(ta, pl[0], pl[0], x[0], x[1]);
  csa(tb, pl[0], pl[0], x[2], x[3]);
  csa(fa, pl[1], pl[1], ta, tb);
  csa(ta, pl[0], pl[0], x[4], x[5]);
  csa(tb, pl[0], pl[0], x[6], x[7]);
  csa(fb, pl[1], pl[1], ta, tb);
  csa(e, pl[2], pl[2], fa, fb);
#pragma unroll
  for (int j = 3; j < 8; j++) {
    const uint32_t t = pl[j] & e;
    pl[j] ^= e;
    e = t;
  }
}

// planes -> per-permutation counts, added into 16 registers of packed u16 pairs.
// bit b of the lane's word (permutation b of the lane's 32): s = b & 7, q = b >> 3 -> register 2s + (q >> 1), half q & 1.
__device__ __forceinline__ void flush_planes(uint32_t (&c16)[16], uint32_t (&pl)[8], int nbits) {
  uint32_t r8[8];
#pragma unroll
  for (int s = 0; s < 8; s++) r8[s] = 0;
  // plane-major with a warp-uniform early exit: only the planes a batch of `nbits` bits can populate cost instructions
  // (as predicated code every plane was paid for: 11 % of the kernel's issue slots, profiles/r1_sparse_m1_level4_hotlines.txt)
#pragma unroll
  for (int j = 0; j < 8; j++) {
    if (j >= nbits) break;
#pragma unroll
    for (int s = 0; s < 8; s++) {
      const uint32_t v = (s >= j) ? (pl[j] >> (s - j)) : (pl[j] << (j - s));
      r8[s] |= v & (0x01010101u << j);
    }
  }
#pragma unroll
  for (int s = 0; s < 8; s++) {
    c16[2 * s] += __byte_perm(r8[s], 0u, 0x4140);
    c16[2 * s + 1] += __byte_perm(r8[s], 0u, 0x4342);
  }
#pragma unroll
  for (int j = 0; j < 8; j++) pl[j] = 0;
}

__device__ __forceinline__ int bits_for(int count) { return 32 - __clz(count); }  // count in [1, 255] -> 1..8

// register index / half of permutation bit b inside the packed u16 counters
#define GCRE_C16_REG(b) (2 * ((b) & 7) + ((b) >> 4))
#define GCRE_C16_HI(b) (((b) >> 3) & 1)

// host: the count of permutation r in one (row, half) entry of a count table in this register image (SparseView::pcnt,
// layout 0: [perm block][q][lane][4] u32, register 4q + k in component k).  Tests read tables back through it
// (gcre_pathset_debug_counts) and so depend on neither image.
static inline uint32_t c16_table_count(const uint32_t* entry, int r) {
  const int b = r & 31, lane = (r >> 5) & 31, pb = r >> 10, reg = GCRE_C16_REG(b);
  const uint32_t v = entry[(((size_t)pb * 4 + (reg >> 2)) * 32 + lane) * 4 + (reg & 3)];
  return GCRE_C16_HI(b) ? v >> 16 : v & 0xffffu;
}

// eight consecutive carriers of a (16-byte aligned, padded) list -> eight patient indices
__device__ __forceinline__ void load8(const uint16_t* p, uint32_t (&c)[8]) {
  const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
  c[0] = v.x & 0xffffu; c[1] = v.x >> 16; c[2] = v.y & 0xffffu; c[3] = v.y >> 16;
  c[4] = v.z & 0xffffu; c[5] = v.z >> 16; c[6] = v.w & 0xffffu; c[7] = v.w >> 16;
}
__device__ __forceinline__ void load8(const uint32_t* p, uint32_t (&c)[8]) {
  const uint4 lo = __ldg(reinterpret_cast<const uint4*>(p)), hi = __ldg(reinterpret_cast<const uint4*>(p) + 1);
  c[0] = lo.x; c[1] = lo.y; c[2] = lo.z; c[3] = lo.w; c[4] = hi.x; c[5] = hi.y; c[6] = hi.z; c[7] = hi.w;
}

// base + 4 * word_offset with the base held as a 64-bit register pair: LEA + LEA.HI.X (ptxas strength-reduces the mad.wide).  Left
// to the compiler, `pt_lane + off` costs IADD3 + IMAD.X + LEA + LEA.HI.X per gather - four ALU-pipe instructions, and the ALU pipe
// is the busiest one in these kernels.
__device__ __forceinline__ const uint32_t* word_ptr(const uint32_t* base, uint32_t word_offset) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(r) : "r"(word_offset), "l"(base));
  return reinterpret_cast<const uint32_t*>(r);
}
// the same for the look-up tables: element `index` of a row held as a 64-bit register pair (the compiler otherwise keeps the table
// base and the row offset in uniform registers and spends IADD3 + IMAD.X + LEA + LEA.HI.X on every look-up)
__device__ __forceinline__ float lookup_f32(const float* row, uint32_t index) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(r) : "r"(index), "l"(row));
  return __ldg(reinterpret_cast<const float*>(r));
}
__device__ __forceinline__ double lookup_f64(const double* row, uint32_t index) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, 8, %2;" : "=l"(r) : "r"(index), "l"(row));
  return __ldg(reinterpret_cast<const double*>(r));
}

// Pre-count table of a path set (see the header): one warp per (item, permutation block).
template <typename CT>
__global__ void __launch_bounds__(128) build_precount_kernel(const unsigned long long* __restrict__ off, const CT* __restrict__ car, long long n_items, int n_perm_blocks,
                                                             const uint32_t* __restrict__ pt, int Iw, uint32_t* __restrict__ pcnt) {
  const int lane = threadIdx.x & 31;
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= n_items * n_perm_blocks) return;
  const long long item = w / n_perm_blocks;
  const int pb = (int)(w % n_perm_blocks);
  const uint32_t* pt_lane = pt + pb * 32 + lane;
  const unsigned long long o = off[item];
  const uint32_t plen = (uint32_t)(off[item + 1] - o);
  uint32_t pl[8], c16[16];
#pragma unroll
  for (int j = 0; j < 8; j++) pl[j] = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) c16[i] = 0;
  int inbatch = 0;
#pragma unroll 1
  for (uint32_t i = 0; i < plen; i += 8) {
    uint32_t c[8], x[8];
    load8(car + o + i, c);
#pragma unroll
    for (int q = 0; q < 8; q++) x[q] = __ldg(word_ptr(pt_lane, c[q] * (uint32_t)Iw));
    hs8(pl, x);
    inbatch += 8;
    if (inbatch > sparse::FLUSH_AT || i + 8 >= plen) {
      flush_planes(c16, pl, bits_for(inbatch));
      inbatch = 0;
    }
  }
  uint4* out = reinterpret_cast<uint4*>(pcnt) + (size_t)w * 128 + lane;
#pragma unroll
  for (int q = 0; q < 4; q++) out[q * 32] = make_uint4(c16[4 * q], c16[4 * q + 1], c16[4 * q + 2], c16[4 * q + 3]);
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// ---- per pair, shared with join_sparse_sc.cuh ----
// 64-bit hash of 16 bytes of a row at 16-byte position pos (SparseView::fp sums it over the row)
__device__ __forceinline__ unsigned long long row_fp_part(unsigned long long w0, unsigned long long w1, unsigned pos) {
  unsigned long long h = (w0 ^ (((w1 << 31) | (w1 >> 33)) * 0x9E3779B97F4A7C15ull)) + (pos + 1ull) * 0xD6E8FEB86659FD93ull;
  h ^= h >> 33;
  h *= 0xFF51AFD7ED558CCDull;
  h ^= h >> 33;
  h *= 0xC4CEB9FE1A85EC53ull;
  return h ^ (h >> 33);
}

// the kept joined row (src/join_base.cpp:246-249) = upstream row | partner row, written to result row r.  16-byte accesses (Wp is
// even, rows are 16-byte aligned), streaming stores: the row is next read by the following level's join.  At 100,000 patients a
// row is 12.5 KB per half and this copy is most of a KEEP join.  Wp: the caller's copy of a.Wp (re-read from the parameters here,
// it changes the register allocation of the whole kernel).
template <int M>
__device__ __forceinline__ void store_kept_row(const JoinParams& a, int Wp, const uint64_t* p0row, uint32_t loc, size_t r, bool flip, int lane) {
  const int row_words = Wp * M;
  const ulonglong2* u = reinterpret_cast<const ulonglong2*>(p0row);
  const ulonglong2* v = reinterpret_cast<const ulonglong2*>(a.p1 + (size_t)loc * row_words);
  ulonglong2* out = reinterpret_cast<ulonglong2*>(a.pres + r * row_words);
  const int Wv = Wp >> 1;
  const int vpos = (M == 2 && !flip) ? Wv : 0, vneg = (M == 2 && !flip) ? 0 : Wv;  // partner half joined into pos / neg
#pragma unroll 4
  for (int k = lane; k < Wv; k += 32) {
    const ulonglong2 x = u[k], y = __ldg(v + vpos + k);
    __stcs(out + k, make_ulonglong2(x.x | y.x, x.y | y.y));
    if (M == 2) {
      const ulonglong2 xn = u[Wv + k], yn = __ldg(v + vneg + k);
      __stcs(out + Wv + k, make_ulonglong2(xn.x | yn.x, xn.y | yn.y));
    }
  }
}

// The fingerprint of kept row r (SparseView::fp): a function of the row's words alone, whichever kernel wrote it - read back
// from L2 right behind store_kept_row.  Out of line: formed in the store loop it cost every KEEP instance registers and spills.
// Warp-uniform call.
__device__ __noinline__ void store_kept_fp(const SparseParams& s, const JoinParams& a, int row_words, size_t r, int lane) {
  __syncwarp();
  const ulonglong2* row = reinterpret_cast<const ulonglong2*>(a.pres + r * row_words);
  unsigned long long fp = 0;
  for (int k = lane; k < row_words / 2; k += 32) {
    const ulonglong2 x = __ldcg(row + k);
    fp += row_fp_part(x.x, x.y, (unsigned)k);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) fp += __shfl_xor_sync(0xffffffffu, fp, d);
  if (lane == 0) s.fp_res[r] = fp;
}

// the carrier totals of half h of kept row r, beside its emitted counts (t0 / nc0: the upstream half's, nd / ncn: what the
// partner adds)
template <int M>
__device__ __forceinline__ void store_kept_totals(const SparseParams& s, size_t r, int h, const uint32_t (&t0)[M], const uint32_t (&nd)[M],
                                                  const uint32_t (&nc0)[M], const uint32_t (&ncn)[M]) {
  s.len_res[r * M + h] = t0[h] + nd[h];
  s.ncase_res[r * M + h] = nc0[h] + ncn[h];
}

// True score -> top-K candidate (src/methods.h:90-94, 253-264): lane 0 parks the pair's totals in its slot of the warp's s_park
// rows (method 1: (carriers, case carriers); method 2: (tp, case_pos, tn, ctrl_pos)) ...
template <int M>
__device__ __forceinline__ void park_totals(uint32_t (&slot)[2 * M], const uint32_t (&t0)[M], const uint32_t (&nd)[M], const uint32_t (&nc0)[M],
                                            const uint32_t (&ncn)[M]) {
  if (M == 1) *reinterpret_cast<uint2*>(slot) = make_uint2(t0[0] + nd[0], nc0[0] + ncn[0]);
  else *reinterpret_cast<uint4*>(slot) = make_uint4(t0[0] + nd[0], nc0[0] + ncn[0], t0[M - 1] + nd[M - 1], nc0[M - 1] + ncn[M - 1]);
}

// ... and behind every 32nd pair and the unit's last one the scores of the parked pairs (slots 0..park, `loc`: the partner of slot
// `park`) are worked off by 32 lanes at once instead of by lane 0 behind every pair.  Candidates that beat the launch's threshold
// and the self-tightening one (JoinParams::slots) are appended; KEEP joins raise max_total.
template <int M, bool KEEP>
__device__ __forceinline__ void score_parked(const JoinParams& a, const uint32_t (*park_rows)[2 * M], uint32_t park, uint32_t idx, uint32_t loc, int lane) {
  __syncwarp();
  const bool mine = (uint32_t)lane <= park;
  const uint32_t locm = loc - park + (uint32_t)lane;
  uint32_t pk[2 * M];
  if (M == 1) {
    const uint2 t = *reinterpret_cast<const uint2*>(park_rows[lane]);
    pk[0] = t.x; pk[1] = t.y;
  } else {
    const uint4 t = *reinterpret_cast<const uint4*>(park_rows[lane]);
    pk[0] = t.x; pk[1] = t.y; pk[2 * M - 2] = t.z; pk[2 * M - 1] = t.w;
  }
  double score = 0.0;
  int cases = 0, ctrls = 0;
  unsigned tmax = 0;
  if (mine) {
    if (M == 1) {
      cases = (int)pk[1];
      tmax = pk[0];
      ctrls = (int)tmax - cases;
      score = a.diagD[diag_base(tmax) + cases];
    } else {
      const unsigned tp = pk[0], tn = pk[2 * M - 2];
      const unsigned case_pos = pk[1], ctrl_neg = tp - case_pos;
      const unsigned ctrl_pos = pk[2 * M - 1], case_neg = tn - ctrl_pos;
      score = a.diagD[diag_base(tp) + case_pos] + a.diagD[diag_base(tn) + case_neg];
      cases = (int)(case_pos + case_neg);
      ctrls = (int)(ctrl_pos + ctrl_neg);
      tmax = max(tp, tn);
    }
  }
  if (KEEP) {
    const unsigned m = __reduce_max_sync(0xffffffffu, tmax);
    if (lane == 0) atomicMax(a.max_total, m);
  }
  if (mine && score == score) {
    const unsigned long long key = score_key(score);
    const unsigned long long dyn = a.n_slots ? __ldcg(a.dyn_thr) : 0ull;
    if (key > a.thr_key && key >= dyn) {
      const unsigned slot = atomicAdd(a.cand_count, 1u);
      if (slot < a.cand_cap) {
        Cand cd;
        cd.key = key; cd.idx = idx; cd.loc = locm; cd.cases = cases; cd.ctrls = ctrls;
        a.cand[slot] = cd;
      }
      if (a.n_slots) {
        const unsigned bucket = ((idx * 0x9E3779B1u) ^ (locm * 0x85EBCA6Bu)) >> 8;
        if (atomicMax(a.slots + bucket % (unsigned)a.n_slots, key) < key) {
          unsigned long long m = ~0ull;
          for (int t = 0; t < a.n_slots; t++) m = min(m, __ldcg(a.slots + t));
          if (m > dyn) atomicMax(a.dyn_thr, m);
        }
      }
    }
  }
  __syncwarp();
}

// CT = carrier index type of the list views: uint16_t (n <= 65,535) or uint32_t
// PC: pre-counted partners, each scored through the row of the pre-counted set s.map1 names (see the header)
// THR: thresholded look-ups (below) instead of 32 running maxima per lane in registers
template <int M, bool KEEP, typename CT, bool PC, bool THR>
__global__ void __launch_bounds__(sparse::THREADS, sparse::min_blocks(M, THR)) join_sparse_kernel(const JoinParams a, const SparseParams s) {
  using namespace sparse;
  const CT* car0 = static_cast<const CT*>(s.car0);
  const CT* car1 = static_cast<const CT*>(s.car1);
  // per-thread slots indexed [half][register][threadIdx.x]: the address is a constant plus 4 * threadIdx.x, which costs two
  // instructions to rematerialise under register pressure (indexed [warp][..][lane] it cost ten, 5 % of method 2's issue slots)
  __shared__ uint32_t s_base[M][16][THREADS];              // base counts per half / packed register / thread
  __shared__ __align__(16) uint32_t s_queue[WARPS][QCAP];  // row offsets (carrier * Iw) of the partner's carriers that survive the filter
  // method 2: the two halves go through ONE instance of the filter / accumulate / flush code (a rolled loop), their counts
  // parked here for the look-up stage: unrolled per half the kernel was 62 KB of SASS and lost more issue slots to
  // instruction fetch than to memory latency (profiles/r1_sparse_final_full.txt, no_instruction 4.1 vs long_scoreboard 4.0)
  // method 2: counts parked for the look-up stage.  THR: half 0 only (the last half stays in registers); else both halves
  __shared__ uint32_t s_cnt[(M == 2 && !THR) ? 2 : 1][M == 2 ? 16 : 1][THREADS];
  __shared__ __align__(16) uint32_t s_park[WARPS][32][2 * M];  // totals of the last <= 32 pairs of the warp's unit (true scores)

  const int tid = threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Wp = a.Wp, Iw = a.Iw;  // Iw: words per patient row of pt (a multiple of 32: every lane owns a valid word)
  const int row_words = Wp * M;
  const unsigned long long n_work = s.n_units * (unsigned long long)s.n_perm_blocks;
  const unsigned lt_mask = (1u << lane) - 1u;
  uint32_t* queue = s_queue[warp];

  // THR = false: 32 running maxima per lane in registers, merged into a.perm_max with one atomicMax per permutation when the
  // warp changes permutation block or runs out of work.
  float best[THR ? 1 : 32];
#pragma unroll
  for (int b = 0; b < (THR ? 1 : 32); b++) best[b] = 0.0f;
  // Only records go out: the lane reads its 32 current maxima (one 128-byte line) and raises those its own beat.  Every warp of
  // the persistent grid flushes at the end of the launch, all at once and on the same lines of a.perm_max; issued
  // unconditionally, those atomics serialised the tail of every small join.  Skipping one is safe: maxima only grow.
  auto flush_best = [&](int pb) {
    const int r0 = (pb * 32 + lane) * 32;
    if constexpr (!THR) {
      if (r0 >= a.Ip) return;
      const int4* p = reinterpret_cast<const int4*>(a.perm_max + r0);
#pragma unroll
      for (int q = 0; q < 8; q++) {
        const int4 v = __ldcg(p + q);
        const int cur[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; k++)
          if (best[4 * q + k] > __int_as_float(cur[k])) atomicMax(a.perm_max + r0 + 4 * q + k, __float_as_int(best[4 * q + k]));
      }
    }
  };
  // THR = true: thresholded look-ups.  The per-permutation maxima live in global memory only (a.perm_max, float bit patterns
  // >= +0, raised with atomicMax).  A lane keeps ONE float, thr: a lower bound of the current maxima of its 32 permutations (their
  // minimum when last read - maxima only grow).  A pair's look-ups first only ask "does any permutation score above thr?" (one
  // compare per look-up, no running-maximum registers); only then - about one pair in a hundred on BASELINE config 3 - the pair's
  // exact scores are pushed with atomicMax and thr is re-read.  Method 2 asks the question with round-up f32 copies of its f64
  // table and a round-up add, an upper bound of the exactly rounded f64 sum, and computes the f64 sums only in the rare path.
  // This frees 31 registers: method 2 runs at 64 registers / 8 CTAs per SM instead of 96 / 5 (level-4 join of BASELINE config 3
  // 19.3 -> 15.0 ms, 2.4 % of the pairs take the exact path).  Method 1 - already at 8 CTAs - does not gain (10.8 ms with running
  // maxima, 11.1 thresholded), nor do small joins (every warp's first pairs take the exact path: the maxima start at zero).
  float thr = 0.0f;
  unsigned since_refresh = 0;
  auto load_thr = [&](int pb) -> float {
    const int r0 = (pb * 32 + lane) * 32;
    if (r0 >= a.Ip) return INFINITY;  // no result slots: the lane's permutations are padding copies of real ones
    const int4* p = reinterpret_cast<const int4*>(a.perm_max + r0);
    float m = INFINITY;
#pragma unroll
    for (int q = 0; q < 8; q++) {
      const int4 v = __ldcg(p + q);
      m = fminf(fminf(m, __int_as_float(v.x)), fminf(__int_as_float(v.y), fminf(__int_as_float(v.z), __int_as_float(v.w))));
    }
    return m;
  };
  int pb_cur = -1;

  while (true) {
    unsigned long long g = 0;
    if (lane == 0) g = atomicAdd(s.work_counter, 1ull);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g >= n_work) break;
    const int pb = (int)(g / s.n_units);
    const unsigned long long unit = s.unit_list ? s.unit_list[s.unit_begin + (g % s.n_units)] : s.unit_begin + (g % s.n_units);
    if (THR) {
      if (pb != pb_cur || (++since_refresh & 7u) == 0u) {  // other warps keep raising the maxima: re-read every 8th unit
        thr = load_thr(pb);
        pb_cur = pb;
      }
    } else if (pb != pb_cur) {
      if (pb_cur >= 0) flush_best(pb_cur);
#pragma unroll
      for (int b = 0; b < (THR ? 1 : 32); b++) best[b] = 0.0f;
      pb_cur = pb;
    }
    const bool first_pb = (pb == 0);
    const uint32_t idx = s.unit_idx[unit];
    const uint32_t sub = (uint32_t)(unit - s.unit_prefix[idx]);
    const uint32_t cnt_idx = (uint32_t)a.count[idx];
    const uint32_t j0 = sub * PB, j1 = min(cnt_idx, j0 + PB);
    const uint32_t* pt_lane = a.pt + pb * 32 + lane;
    const uint64_t* p0row = a.p0 + (size_t)idx * row_words;
    const uint32_t loc0 = a.location[idx];
    // PC: pull the pre-counted rows of a partner (2 KB per half and permutation block = 16 lines, one per lane) towards
    // the SM ahead of their use - the table is far larger than L2 and each row is read once per pair
    auto prefetch_partner = [&](uint32_t loc) {
      const uint32_t row = __ldg(s.map1 + loc) >> 1;
      if (lane < 16 * M)
        prefetch_l2(reinterpret_cast<const char*>(s.pcnt1) + (((size_t)row * M + (lane >> 4)) * s.n_perm_blocks + pb) * 2048 + (lane & 15) * 128);
    };
    if (PC && j0 < j1) prefetch_partner(loc0 + j0);

    uint32_t pl[8];
#pragma unroll
    for (int j = 0; j < 8; j++) pl[j] = 0;
    int inbatch = 0;  // carrier slots (sentinels included) in the planes
    int inreal = 0;   // upper bound of the count any permutation can have reached in the planes: sets how many planes a flush reads

    // add eight carriers of a list (sentinel entries hit the zero row) to the bit planes
    // `last`: nothing more will be added to these counters - flush what the planes hold.  The overflow flush (planes
    // nearly full) and the final flush are the same code on purpose: flush_planes is ~170 instructions and was inlined
    // five times before.
    auto add8 = [&](uint32_t (&c16)[16], const CT* lst8, bool last) {
      uint32_t c[8], x[8];
      load8(lst8, c);
#pragma unroll
      for (int q = 0; q < 8; q++) x[q] = __ldg(word_ptr(pt_lane, c[q] * (uint32_t)Iw));
      hs8(pl, x);
      inbatch += 8;
      inreal += 8;
      if (inbatch > FLUSH_AT || last) {
        flush_planes(c16, pl, bits_for(inreal));
        inbatch = inreal = 0;
      }
    };

    // the same for eight pre-multiplied row offsets (filtered partner carriers, multiplied once per lane in the filter)
    // (keeping a second group of gathers in flight while the first is added - method 2 has the registers - gained < 1 %)
    auto gather8 = [&](uint32_t (&x)[8], const uint32_t* q8) {
      const uint4 lo = *reinterpret_cast<const uint4*>(q8), hi = *reinterpret_cast<const uint4*>(q8 + 4);
      x[0] = __ldg(word_ptr(pt_lane, lo.x));
      x[1] = __ldg(word_ptr(pt_lane, lo.y));
      x[2] = __ldg(word_ptr(pt_lane, lo.z));
      x[3] = __ldg(word_ptr(pt_lane, lo.w));
      x[4] = __ldg(word_ptr(pt_lane, hi.x));
      x[5] = __ldg(word_ptr(pt_lane, hi.y));
      x[6] = __ldg(word_ptr(pt_lane, hi.z));
      x[7] = __ldg(word_ptr(pt_lane, hi.w));
    };
    auto acc8 = [&](uint32_t (&c16)[16], const uint32_t (&x)[8], int real, bool last) {
      hs8(pl, x);
      inbatch += 8;
      inreal += real;
      if (inbatch > FLUSH_AT || last) {
        flush_planes(c16, pl, bits_for(inreal));
        inbatch = inreal = 0;
      }
    };

    // ---- base: the upstream row's own carriers ----
    uint32_t t0[M], nc0[M];
#pragma unroll
    for (int h = 0; h < M; h++) t0[h] = nc0[h] = 0;
#pragma unroll 1
    for (int h = 0; h < M; h++) {
      const size_t item = (size_t)idx * M + h;
      const uint32_t t0h = s.len0[item], nc0h = s.ncase0[item];
      if (M == 1 || h == 0) { t0[0] = t0h; nc0[0] = nc0h; } else { t0[M - 1] = t0h; nc0[M - 1] = nc0h; }
      if (s.pcnt0) {  // counts emitted by the join that produced the upstream rows
        const uint4* B = reinterpret_cast<const uint4*>(s.pcnt0) + ((item * s.n_perm_blocks + pb) * 4) * 32 + lane;
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const uint4 v = __ldcs(B + q * 32);  // read once per unit: keep it from displacing the mask rows in L1
          s_base[h][4 * q][tid] = v.x;
          s_base[h][4 * q + 1][tid] = v.y;
          s_base[h][4 * q + 2][tid] = v.z;
          s_base[h][4 * q + 3][tid] = v.w;
        }
      } else {
        uint32_t acc[16];
#pragma unroll
        for (int i = 0; i < 16; i++) acc[i] = 0;
        const CT* lst = car0 + s.off0[item];
        const uint32_t plen = (uint32_t)(s.off0[item + 1] - s.off0[item]);
#pragma unroll 1
        for (uint32_t i = 0; i < plen; i += 8) add8(acc, lst + i, i + 8 >= plen);
#pragma unroll
        for (int i = 0; i < 16; i++) s_base[h][i][tid] = acc[i];
      }
    }
    __syncwarp();

    bool base_done = false;
    // ---- partners ----
    for (uint32_t j = j0; j < j1; j++) {
      const uint32_t loc = loc0 + j;
      if (PC && j + 1 < j1) prefetch_partner(loc + 1);
      bool flip = true;
      if (M == 2) flip = need_flip(a.path_length, a.signs, idx, loc);
      const uint32_t mapped = PC ? __ldg(s.map1 + loc) : 0u;
      uint32_t c16[16];          // counts of the half being accumulated (PC: of up & partner only)
      uint32_t nd[M], ncn[M];    // carriers / case carriers the partner adds to the upstream half
      size_t pitem[M];           // PC: the partner item joined into half h
#pragma unroll
      for (int h = 0; h < M; h++) { nd[h] = ncn[h] = 0; pitem[h] = 0; }
#pragma unroll 1
      for (int h = 0; h < M; h++) {
#pragma unroll
        for (int i = 0; i < 16; i++) c16[i] = PC ? 0u : s_base[h][i][tid];
        // joined half h = upstream half h | partner half hh   (src/methods.h:137-145)
        const int hh = (M == 1) ? 0 : (flip ? h : 1 - h);
        // PC: half hh of the partner row is half hh ^ swapped of the row it is scored through
        const size_t item = PC ? (size_t)(mapped >> 1) * M + (M == 1 ? 0 : (hh ^ (int)(mapped & 1u))) : (size_t)loc * M + hh;
        const CT* lst1 = car1 + s.off1[item];
        const uint32_t len = s.len1[item];
        const uint64_t* p0h = p0row + h * Wp;
        uint32_t ndh = 0, ncnh = 0;
        uint32_t qn = 0;  // carriers waiting in the queue (warp-uniform)
#pragma unroll 1
        for (uint32_t i0 = 0; i0 < len; i0 += 32) {
          const uint32_t i = i0 + lane;
          const bool valid = i < len;
          const uint32_t c = valid ? (uint32_t)lst1[i] : 0u;
          const uint32_t w0 = valid ? __ldg(reinterpret_cast<const uint32_t*>(p0h) + (c >> 5)) : 0u;
          // delta: carriers not yet in the upstream row are added to the base; PC: carriers already in it are subtracted
          const bool keep = valid && (((w0 >> (c & 31)) & 1u) != 0u) == PC;
          const unsigned km = __ballot_sync(0xffffffffu, keep);
          ncnh += __popc(__ballot_sync(0xffffffffu, keep && (int)c < a.n_cases));
          if (keep) queue[qn + __popc(km & lt_mask)] = c * (uint32_t)Iw;
          qn += __popc(km);
          const bool last_chunk = i0 + 32 >= len;
          if (qn >= 64 || (last_chunk && (qn > 0 || inbatch > 0))) {
            // drain: everything (padded to a multiple of 8 with the zero row) after the last chunk, else eight groups with
            // the remainder (< 32 entries) moved to the front
            // (after the last chunk at least one group runs, if only of zero rows, so that counts an earlier drain left in
            // the planes are flushed)
            const uint32_t take = last_chunk ? max((qn + 7u) & ~7u, 8u) : 64u;
            if (last_chunk && lane < take - qn) queue[qn + lane] = (uint32_t)s.n * (uint32_t)Iw;
            __syncwarp();
#pragma unroll 1
            for (uint32_t q0 = 0; q0 < take; q0 += 8) {
              uint32_t x[8];
              gather8(x, queue + q0);
              acc8(c16, x, (int)min(8u, qn > q0 ? qn - q0 : 0u), last_chunk && q0 + 8 >= take);
            }
            const uint32_t rem = last_chunk ? 0u : qn - 64u;
            const uint32_t keepv = (lane < rem) ? queue[64 + lane] : 0u;
            __syncwarp();
            if (lane < rem) queue[lane] = keepv;
            ndh += qn - rem;
            qn = rem;
          }
        }
        if (PC) {  // what the filter kept is the overlap: added = partner - overlap
          ndh = len - ndh;
          ncnh = s.ncase1[item] - ncnh;
        }
        if (M == 2) {
          if (h == 0 || !THR) {
#pragma unroll
            for (int i = 0; i < 16; i++) s_cnt[THR ? 0 : h][M == 2 ? i : 0][tid] = c16[i];
          }
          if (h == 0) { nd[0] = ndh; ncn[0] = ncnh; pitem[0] = item; } else { nd[M - 1] = ndh; ncn[M - 1] = ncnh; pitem[M - 1] = item; }
        } else {
          nd[0] = ndh;
          ncn[0] = ncnh;
          pitem[0] = item;
        }
      }

      bool empty = nd[0] == 0;
      if (M == 2) empty = empty && nd[M - 1] == 0;
      // KEEP + PC: the final counts formed below are the kept row's emitted counts (a partner skipped as empty has the base's);
      // with running maxima they are stored where they are formed, at emit_at
      const bool scored = !empty || !base_done;
      uint4* emit_at = nullptr;
      if (KEEP && PC && !THR && s.pcnt_res) emit_at = reinterpret_cast<uint4*>(s.pcnt_res) + ((((size_t)(a.res_idx[idx] + j) * M) * s.n_perm_blocks + pb) * 4) * 32 + lane;
      if (scored) {
        if (empty) base_done = true;
        if constexpr (THR) {
          if (PC) {
            // counts = base + P[partner] - overlap, packed u16 pairs (whole-register arithmetic is exact: every final half is a
            // count in [0, 65535]); finalised in place: half 0 of method 2 in its shared-memory slots, the last half in c16
            const uint4* P0 = reinterpret_cast<const uint4*>(s.pcnt1) + ((pitem[0] * s.n_perm_blocks + pb) * 4) * 32 + lane;
            const uint4* P1 = reinterpret_cast<const uint4*>(s.pcnt1) + ((pitem[M - 1] * s.n_perm_blocks + pb) * 4) * 32 + lane;
#pragma unroll
            for (int q = 0; q < 4; q++) {
              const uint4 pv = __ldg(P1 + q * 32);
              const uint32_t pr[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
              for (int k = 0; k < 4; k++) c16[4 * q + k] = s_base[M - 1][4 * q + k][tid] + pr[k] - c16[4 * q + k];
              if (M == 2) {
                const uint4 pw = __ldg(P0 + q * 32);
                const uint32_t pr0[4] = {pw.x, pw.y, pw.z, pw.w};
#pragma unroll
                for (int k = 0; k < 4; k++)
                  s_cnt[0][M == 2 ? 4 * q + k : 0][tid] = s_base[0][4 * q + k][tid] + pr0[k] - s_cnt[0][M == 2 ? 4 * q + k : 0][tid];
              }
            }
          }
          // final counts of permutation bit b: register GCRE_C16_REG(b), half GCRE_C16_HI(b); the last half (method 1: the only
          // one) is in c16, half 0 of method 2 in shared memory
          bool hit = false;
          if (M == 1) {
            const float* row = a.diagF + diag_base(t0[0] + nd[0]);
#pragma unroll
            for (int b = 0; b < 32; b++) {
              const uint32_t v = c16[GCRE_C16_REG(b)];
              const uint32_t c = GCRE_C16_HI(b) ? (v >> 16) : (v & 0xffffu);
              hit |= lookup_f32(row, c) > thr;
            }
          } else {
            // src/methods.h:223-227: vtmax[pcp][total_pos - pcp] + vtmax[total_neg - pnp][pnp]
            const unsigned tn = t0[M - 1] + nd[M - 1];
            const float* frp = a.diagFM + diag_base(t0[0] + nd[0]);
            const float* frn = a.diagFM + diag_base(tn);  // indexed by tn - cn
#pragma unroll
            for (int b = 0; b < 32; b++) {
              const uint32_t vp = s_cnt[0][M == 2 ? GCRE_C16_REG(b) : 0][tid], vn = c16[GCRE_C16_REG(b)];
              const uint32_t cp = GCRE_C16_HI(b) ? (vp >> 16) : (vp & 0xffffu);
              const uint32_t cn = GCRE_C16_HI(b) ? (vn >> 16) : (vn & 0xffffu);
              hit |= __fadd_ru(lookup_f32(frp, cp), lookup_f32(frn, tn - cn)) > thr;  // >= the exactly rounded f64 sum
            }
          }
          if (__any_sync(0xffffffffu, hit)) {
            // rare: exact scores of the pair -> global maxima.  A rolled loop (small code, no register pressure on the common path):
            // the last half's counts are copied to a dynamically indexed local array (thread-private memory, touched only here)
            uint32_t lc[16];
#pragma unroll
            for (int i = 0; i < 16; i++) lc[i] = c16[i];
            if (lane == 0) atomicAdd(s.exact_pairs, 1ull);  // diagnostic
            const int r0 = (pb * 32 + lane) * 32;
            const unsigned tp = t0[0] + nd[0], tn = t0[M - 1] + nd[M - 1];
#pragma unroll 1
            for (int b = 0; b < 32; b++) {
              const int reg = GCRE_C16_REG(b), sh = GCRE_C16_HI(b) * 16;
              float p;
              if (M == 1) {
                p = __ldg(a.diagF + diag_base(tp) + ((lc[reg] >> sh) & 0xffffu));
              } else {
                const uint32_t cp = (s_cnt[0][M == 2 ? reg : 0][tid] >> sh) & 0xffffu, cn = (lc[reg] >> sh) & 0xffffu;
                p = __double2float_rn(__ldg(a.diagDM + diag_base(tp) + cp) + __ldg(a.diagDM + diag_base(tn) + tn - cn));
              }
              // candidates only (p above the lane's bound) are compared with the permutation's CURRENT maximum, read past L1: an
              // atomic only for a genuine record (at a cold start every p beats the zero bound - 1,024 atomics per warp otherwise)
              if (p > thr && p > __int_as_float(__ldcg(a.perm_max + r0 + b))) atomicMax(a.perm_max + r0 + b, __float_as_int(p));
            }
            thr = load_thr(pb);
          }
        } else {
          if (PC) {
            // counts = base + P[partner] - overlap, packed u16 pairs (whole-register arithmetic is exact: every final half
            // is a count in [0, 65535]); register i holds permutation bits b = ((i & 1) * 2 + hf) * 8 + (i >> 1), hf = 0, 1
            const uint4* P0 = reinterpret_cast<const uint4*>(s.pcnt1) + ((pitem[0] * s.n_perm_blocks + pb) * 4) * 32 + lane;
            if (M == 1) {
              const unsigned total = t0[0] + nd[0];
              const float* row = a.diagF + diag_base(total);
#pragma unroll
              for (int q = 0; q < 4; q++) {
                const uint4 pv = __ldg(P0 + q * 32);
                const uint32_t pr[4] = {pv.x, pv.y, pv.z, pv.w};
                uint32_t v[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  const int i = 4 * q + k;
                  v[k] = s_base[0][i][tid] + pr[k] - c16[i];
                  best[((i & 1) * 2) * 8 + (i >> 1)] = fmaxf(best[((i & 1) * 2) * 8 + (i >> 1)], lookup_f32(row, v[k] & 0xffffu));
                  best[((i & 1) * 2 + 1) * 8 + (i >> 1)] = fmaxf(best[((i & 1) * 2 + 1) * 8 + (i >> 1)], lookup_f32(row, v[k] >> 16));
                }
                if (KEEP && emit_at) __stcs(emit_at + q * 32, make_uint4(v[0], v[1], v[2], v[3]));
              }
            } else {
              const uint4* P1 = reinterpret_cast<const uint4*>(s.pcnt1) + ((pitem[M - 1] * s.n_perm_blocks + pb) * 4) * 32 + lane;
              const unsigned tp = t0[0] + nd[0], tn = t0[M - 1] + nd[M - 1];
              const double* rowp = a.diagDM + diag_base(tp);
              const double* rown = a.diagDM + diag_base(tn);  // indexed by tn - cn
#pragma unroll
              for (int q = 0; q < 4; q++) {
                const uint4 pvp = __ldg(P0 + q * 32), pvn = __ldg(P1 + q * 32);
                const uint32_t prp[4] = {pvp.x, pvp.y, pvp.z, pvp.w}, prn[4] = {pvn.x, pvn.y, pvn.z, pvn.w};
                uint32_t vp[4], vn[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  const int i = 4 * q + k;
                  vp[k] = s_base[0][i][tid] + prp[k] - s_cnt[0][M == 2 ? i : 0][tid];
                  vn[k] = s_base[M - 1][i][tid] + prn[k] - s_cnt[M == 2 ? 1 : 0][M == 2 ? i : 0][tid];
                  // src/methods.h:223-227: vtmax[pcp][total_pos - pcp] + vtmax[total_neg - pnp][pnp]
                  const double vlo = lookup_f64(rowp, vp[k] & 0xffffu) + lookup_f64(rown, tn - (vn[k] & 0xffffu));
                  const double vhi = lookup_f64(rowp, vp[k] >> 16) + lookup_f64(rown, tn - (vn[k] >> 16));
                  best[((i & 1) * 2) * 8 + (i >> 1)] = fmaxf(best[((i & 1) * 2) * 8 + (i >> 1)], __double2float_rn(vlo));
                  best[((i & 1) * 2 + 1) * 8 + (i >> 1)] = fmaxf(best[((i & 1) * 2 + 1) * 8 + (i >> 1)], __double2float_rn(vhi));
                }
                if (KEEP && emit_at) {  // halves 0 and 1 of the kept row, n_perm_blocks * 128 uint4 apart
                  __stcs(emit_at + q * 32, make_uint4(vp[0], vp[1], vp[2], vp[3]));
                  __stcs(emit_at + (size_t)s.n_perm_blocks * 128 + q * 32, make_uint4(vn[0], vn[1], vn[2], vn[3]));
                }
              }
            }
          } else if (M == 1) {
            const unsigned total = t0[0] + nd[0];
            const float* row = a.diagF + diag_base(total);
#pragma unroll
            for (int b = 0; b < 32; b++) {
              const uint32_t v = c16[GCRE_C16_REG(b)];
              const uint32_t c = GCRE_C16_HI(b) ? (v >> 16) : (v & 0xffffu);
              best[b] = fmaxf(best[b], lookup_f32(row, c));
            }
          } else {
            const unsigned tp = t0[0] + nd[0], tn = t0[M - 1] + nd[M - 1];
            const double* rowp = a.diagDM + diag_base(tp);
            const double* rown = a.diagDM + diag_base(tn);  // indexed by tn - cn
#pragma unroll
            for (int b = 0; b < 32; b++) {
              const uint32_t vp = s_cnt[0][M == 2 ? GCRE_C16_REG(b) : 0][tid], vn = s_cnt[M == 2 ? 1 : 0][M == 2 ? GCRE_C16_REG(b) : 0][tid];
              const uint32_t cp = GCRE_C16_HI(b) ? (vp >> 16) : (vp & 0xffffu);
              const uint32_t cn = GCRE_C16_HI(b) ? (vn >> 16) : (vn & 0xffffu);
              // src/methods.h:223-227: vtmax[pcp][total_pos - pcp] + vtmax[total_neg - pnp][pnp]
              const double v = lookup_f64(rowp, cp) + lookup_f64(rown, tn - cn);
              best[b] = fmaxf(best[b], __double2float_rn(v));
            }
          }
        }
      }

      if (KEEP && s.pcnt_res) {
        // ---- the kept row's counts and carrier totals travel with it (base of the next level) ----
        // (PC with running maxima stored its final counts beside the look-ups already)
        const size_t r = (size_t)(a.res_idx[idx] + j);
#pragma unroll
        for (int h = 0; h < M; h++) {
          if (!(PC && !THR && scored)) {
            uint4* out = reinterpret_cast<uint4*>(s.pcnt_res) + (((r * M + h) * s.n_perm_blocks + pb) * 4) * 32 + lane;
            uint32_t v16[16];  // method 1 / THR: the last half is in registers; method 2: parked halves in shared memory
#pragma unroll
            for (int i = 0; i < 16; i++)
              v16[i] = (PC && !scored) ? s_base[h][i][tid]
                                       : (M == 1 || (THR && h == M - 1)) ? c16[i] : s_cnt[(M == 2 && !THR) ? h : 0][M == 2 ? i : 0][tid];
#pragma unroll
            for (int q = 0; q < 4; q++) __stcs(out + q * 32, make_uint4(v16[4 * q], v16[4 * q + 1], v16[4 * q + 2], v16[4 * q + 3]));
          }
          if (first_pb && lane == 0) store_kept_totals<M>(s, r, h, t0, nd, nc0, ncn);
        }
      }

      // on the first permutation block only: the kept row, the true score and the candidate
      if (first_pb) {
        if (KEEP) {
          const size_t r = (size_t)(a.res_idx[idx] + j);
          store_kept_row<M>(a, Wp, p0row, loc, r, flip, lane);
          if (s.fp_res) store_kept_fp(s, a, row_words, r, lane);
        }
        const uint32_t park = (j - j0) & 31u;
        if (lane == 0) park_totals<M>(s_park[warp][park], t0, nd, nc0, ncn);
        if (park == 31u || j + 1 == j1) score_parked<M, KEEP>(a, s_park[warp], park, idx, loc, lane);
      }
    }
    __syncwarp();
  }
  if (!THR && pb_cur >= 0) flush_best(pb_cur);
}

// can the sparse kernel run this shape at all: packed u16 counters, 32-bit row offsets into the patient-major masks
static inline bool sparse_supported(int n, long long t_needed, int Iw) {
  return t_needed <= 65535 && ((unsigned long long)n + 1) * (unsigned long long)Iw < 0xffffffffull;
}

// AUTO choice: a cost model in nanoseconds per pair, calibrated on B200 (profiles/r2_density_sweep.json).
//   dense : every pair pays W64 * Ip * M word-ops (Ip = permutations padded to the 128-wide tile) at the measured 2.1e12 word-ops/s
//           of the POPC pipe, whatever the rows hold;
//   sparse: a fixed part per pair and 1,024-permutation block (filter pass, flush, look-ups) plus a part proportional to the
//           carriers the partner ADDS to the upstream row (gathers + carry-save adds).
// The sparse walk wins for rare-variant rows at any cohort size; the dense kernel wins for very short rows (the vignette:
// W64 = 4) and when partner rows add thousands of carriers (common variants: GWASPA(threshold = 0.5)).  The carriers added per
// pair are bounded by the densest partner half-row; when that bound does not decide, a 2,048-pair sample (sample_overlap_kernel)
// measures them.
static inline double dense_pair_ns(int W64, int Ip_dense, int M) { return (double)W64 * Ip_dense * M / 2100.0; }
// (density sweep at n = 10,000, 425 k pairs, 1,000 permutations: dense 77 ns per pair whatever the rows hold; sparse 3.5 / 7.3 / 20 /
// 41 ns at ~22 / 80 / 260 / 570 carriers added per pair - method 2 about a third more)
static inline double sparse_pair_ns(int n_perm_blocks, int M, double new_carriers_per_pair) {
  return n_perm_blocks * ((M == 1 ? 1.5 : 2.0) + (M == 1 ? 0.075 : 0.1) * new_carriers_per_pair);
}

// Thresholded look-ups pay on large method-2 joins only (see the kernel); forced = 0 / 1 (GCRE_THR) turns them off / on for
// every join, -1 applies that rule
static inline bool sparse_thr(int M, unsigned long long n_pairs, int forced) {
  return forced >= 0 ? forced == 1 : M == 2 && n_pairs >= (1ull << 20);
}

template <int M, bool KEEP, bool PC, bool THR>
static inline void launch_sparse_ct(unsigned grid, cudaStream_t stream, const JoinParams& jp, const SparseParams& sp, bool wide) {
  if (wide) join_sparse_kernel<M, KEEP, uint32_t, PC, THR><<<grid, sparse::THREADS, 0, stream>>>(jp, sp);
  else join_sparse_kernel<M, KEEP, uint16_t, PC, THR><<<grid, sparse::THREADS, 0, stream>>>(jp, sp);
}

template <int M, bool THR>
static inline void launch_sparse_form(unsigned grid, cudaStream_t stream, const JoinParams& jp, const SparseParams& sp, bool keep, bool pc, bool wide) {
  if (keep && pc) launch_sparse_ct<M, true, true, THR>(grid, stream, jp, sp, wide);
  else if (keep) launch_sparse_ct<M, true, false, THR>(grid, stream, jp, sp, wide);
  else if (pc) launch_sparse_ct<M, false, true, THR>(grid, stream, jp, sp, wide);
  else launch_sparse_ct<M, false, false, THR>(grid, stream, jp, sp, wide);
}

// `pc`: the pre-counted-partner kernels (sp.pcnt1 and sp.map1 set); `thr`: the thresholded look-ups; `wide`: u32 carrier indices
static inline cudaError_t launch_join_sparse(cudaStream_t stream, const JoinParams& jp, const SparseParams& sp, int M, bool keep, int sm_count, bool pc,
                                             bool thr, bool wide) {
  const unsigned long long n_work = sp.n_units * (unsigned long long)sp.n_perm_blocks;
  if (n_work == 0) return cudaSuccess;
  const unsigned long long want = (n_work + sparse::WARPS - 1) / sparse::WARPS;
  const unsigned grid = (unsigned)std::min<unsigned long long>(want, (unsigned long long)sm_count * sparse::min_blocks(M, thr));
  if (M == 1) {
    if (thr) launch_sparse_form<1, true>(grid, stream, jp, sp, keep, pc, wide);
    else launch_sparse_form<1, false>(grid, stream, jp, sp, keep, pc, wide);
  } else {
    if (thr) launch_sparse_form<2, true>(grid, stream, jp, sp, keep, pc, wide);
    else launch_sparse_form<2, false>(grid, stream, jp, sp, keep, pc, wide);
  }
  return cudaGetLastError();
}

// Pre-counted partners replace the walk over the partner's new carriers by a 2 KB read plus a walk over the carriers
// the two rows SHARE.  In the level schedule of the reference a partner path always starts at the gene the upstream path
// ends in, so at level 4 the shared part is as long as the new part and the form loses (BASELINE config 3, ms per launch,
// delta / pre-counted: level 4 method 1 13.1 / 15.0, method 2 22.4 / 27.0), while at level 5 (two new genes per shared one)
// and level 3 (single-gene partners, nothing shared) method 1 gains: 147 / 123 and 2.7 / 2.4; method 2, whose look-ups
// dominate, does not (244 / 242, 5.8 / 5.8).  So: method 1, large score-only joins, and only when a sample of the pairs
// (sample_overlap_kernel) shows the shared part below 0.6 of the new part.
// KEEP joins whose partners are a selection (levels 2 and 3: single gene rows) are scored through the base set's rows and table
// and emit their counts (see the header).  Measured on B200 (BASELINE config 3, delta -> this form, ms per join, methods 1 / 2):
// level 2 (150 k pairs) 0.72 -> 0.64 / 0.90 -> 0.85, level 3 (1.35 M pairs) 2.24 -> 2.11 / 3.91 -> 4.06 (thresholded look-ups);
// the step also loses the carrier lists of the two partner copies (~0.3 / 0.5 ms of list builds per method): 31.0 -> 30.2 ms
// per step (profiles/r5_selection_ab.txt).  So: such joins of >= 128 K pairs, either method, when the sample agrees.
// `forced` (GCRE_PRECOUNT=1 / 0, GCRE_TEST_PRECOUNT in the tests; -1: not set) forces it on / off for every join (KEEP joins
// included), or with PRECOUNT_SAMPLE lets the sample decide whatever the method and the size.
enum { PRECOUNT_NO = 0, PRECOUNT_YES = 1, PRECOUNT_SAMPLE = 2 };
// `table_rows`: rows of the set the table is built over (the partner set, or the base set of a selection partner)
// `kept_selection`: a KEEP join whose partners are a selection, scored through the base set (SELECTION_MIN_PAIRS below)
static inline int precount_mode(unsigned long long pairs, unsigned long long table_rows, int M, int n_perm_blocks, size_t budget_bytes, int forced,
                                bool kept_selection) {
  if (table_rows == 0 || pairs == 0) return PRECOUNT_NO;
  if (table_rows >= (1ull << 31)) return PRECOUNT_NO;  // partners are read through a map of row << 1 (SparseParams::map1)
  if ((size_t)table_rows * M * n_perm_blocks * 2048 > budget_bytes) return PRECOUNT_NO;
  if (forced >= 0) return forced;
  if (kept_selection) return pairs >= (1ull << 17) ? PRECOUNT_SAMPLE : PRECOUNT_NO;
  return (M == 1 && pairs >= (1ull << 20)) ? PRECOUNT_SAMPLE : PRECOUNT_NO;
}

// One warp per sampled pair (evenly spaced over the pairs of the join): out[0] += |partner & upstream|,
// out[1] += |partner & ~upstream| over the halves that are joined (method 2: routed by need_flip).
template <int M>
__global__ void sample_overlap_kernel(const JoinParams a, unsigned long long pair_lo, unsigned long long pair_hi, int n_samples,
                                      unsigned long long* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (w >= n_samples) return;
  const unsigned long long p = pair_lo + (pair_hi - pair_lo) * (unsigned long long)w / (unsigned long long)n_samples;
  const uint32_t idx = find_uid(a.prefix, a.n_uids, p);
  const uint32_t loc = a.location[idx] + (uint32_t)(p - a.prefix[idx]);
  const bool flip = (M == 2) ? need_flip(a.path_length, a.signs, idx, loc) : true;
  const uint64_t* u = a.p0 + (size_t)idx * a.Wp * M;
  const uint64_t* v = a.p1 + (size_t)loc * a.Wp * M;
  unsigned ov = 0, dl = 0;
  for (int h = 0; h < M; h++) {
    const int hh = (M == 1) ? 0 : (flip ? h : 1 - h);
    for (int k = lane; k < a.Wp; k += 32) {
      const uint64_t x = u[h * a.Wp + k], y = v[hh * a.Wp + k];
      ov += __popcll(x & y);
      dl += __popcll(y & ~x);
    }
  }
  ov = __reduce_add_sync(0xffffffffu, ov);
  dl = __reduce_add_sync(0xffffffffu, dl);
  if (lane == 0) {
    atomicAdd(out, (unsigned long long)ov);
    atomicAdd(out + 1, (unsigned long long)dl);
  }
}

}  // namespace gcre
