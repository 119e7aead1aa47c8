// Sparse join for FEW permutations (<= 512, e.g. GWASPA's default of 100): the carriers of one pair are split across the
// lanes of the warp.
//
// join_sparse_kernel gives every lane one 32-permutation word of the patient-major masks; with <= 128 permutations only 4
// of the 32 lanes have a word and 28 idle through the gathers, the flush and the look-ups (8 of 32 busy up to 256, 16 up to
// 512).  Here the warp is G = 32 / NW sub-groups x NW words (NW = 4, 8, 16; w = lane % NW, s = lane / NW): sub-group s walks
// every G-th group of eight carriers of the SAME pair, so a batch of 8 G carriers costs each lane eight gathers; the G partial
// count vectors of a word are then combined with a reduce-scatter over shuffles (log2 G rounds), which leaves lane (w, s)
// with 16 / G of the 16 packed count registers - for NW = 4 the counts of the four permutations w*32 + {s, s+8, s+16, s+24} -
// the only ones it looks up and keeps a running maximum for.  Same integers as every other
// kernel, so results are bit-identical.  (Splitting the warp over different PARTNERS instead was tried first and lost to
// the heavy-tailed list lengths; splitting one pair's carriers has no such imbalance.)
//
// Everything else - units, filter against the dense upstream row, true scores, candidates with the self-tightening
// threshold, kept rows - is as in join_sparse.cuh.
//
// Per-pair cost is what matters here (a pair of the bench cohort brings ~32 new carriers of 4 words on average, most pairs far
// fewer), so:
//  * a half whose new carriers fit HALF a batch (<= 4 per sub-group: the common case) takes a short path - 1 or 4 gathers per
//    lane, a 3-plane carry-save sum, BYTE counts and a 7-shuffle reduce-scatter over bytes instead of the 8-gather / 8-plane /
//    16-register form (about 90 fewer warp instructions per half);
//  * the totals behind the true score of a pair are parked in shared memory (16 bytes) and the scores of 32 pairs (two 64-bit
//    triangle offsets, f64 loads, candidate test each) are worked off by 32 lanes at once instead of by lane 0 behind every pair;
//  * the offsets / lengths of the next partner's lists are loaded one pair ahead;
//  * KEEP joins emit the counts of the kept rows (R registers per lane and half: 256 B per row and half at <= 128
//    permutations) with their carrier totals, and the next level takes them as the base of its units: it then needs neither
//    the carrier lists of its upstream rows (two passes over the kept rows to build) nor the walk over them.
#pragma once
#include "join_sparse.cuh"

namespace gcre {

namespace sparse_sc {
constexpr int THREADS = 128;
constexpr int WARPS = THREADS / 32;
// PTS form (<= 128 permutations, small cohorts): ONE CTA of 32 warps per SM with the whole patient-major mask matrix
// ((n + 1) x 16 B) staged in its shared memory by a bulk async copy - the gathers of the hot loop become LDS, and L1 is left
// to the carrier lists, the upstream rows and the score tables.  Measured gain 4 % (config 3, 100 permutations): the kernel is
// bound by its instruction count and the filter's dependent loads, not by these gathers (profiles/r2_sc_full.txt).
#ifndef GCRE_SC_PTS_THREADS
#define GCRE_SC_PTS_THREADS 1024  // measured: 768 threads (80 registers, no spills) +15 % time, 512 threads +50 % - resident warps matter more
#endif
constexpr int PTS_THREADS = GCRE_SC_PTS_THREADS;
constexpr size_t PTS_SMEM_MAX = 232448;  // 227 KB opt-in limit of a CTA on sm_100
constexpr int QCAP = 128;       // the batch being drained (<= 64 slots) + the < 32 entries that can wait behind it, in whole batches
constexpr int MAX_PERMS = 512;  // 16 words of 32
#ifndef GCRE_SC_MB4
#define GCRE_SC_MB4 8  // resident CTAs per SM the <= 128-permutation kernels are compiled for (64 registers)
#endif
constexpr int min_blocks(int nw) { return nw == 16 ? 6 : nw == 8 ? 8 : GCRE_SC_MB4; }
}  // namespace sparse_sc

// position of the t-th queued carrier: inside its batch of B = 8 G the entries of sub-group s = t % G are contiguous (two
// 16-byte shared loads per lane and batch)
template <int G>
__device__ __forceinline__ uint32_t sc_slot(uint32_t t) {
  constexpr uint32_t B = 8 * G;
  return (t / B) * B + ((t % G) << 3) + ((t % B) / G);
}

// 16 packed count registers per lane (partial sums over the lane's share of the carriers) -> the R = NW / 2 registers
// R*s .. R*s + R-1 summed over the G sub-groups of the lane's word (s = lane / NW)
template <int NW>
__device__ __forceinline__ void sc_reduce_scatter(const uint32_t (&c16)[16], int lane, uint32_t (&out)[NW / 2]) {
  const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
  uint32_t r8[8];
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const uint32_t send = b4 ? c16[k] : c16[k + 8], keep = b4 ? c16[k + 8] : c16[k];
    r8[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  if constexpr (NW == 16) {
#pragma unroll
    for (int k = 0; k < 8; k++) out[k] = r8[k];
  } else {
    uint32_t r4[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const uint32_t send = b3 ? r8[k] : r8[k + 4], keep = b3 ? r8[k + 4] : r8[k];
      r4[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    if constexpr (NW == 8) {
#pragma unroll
      for (int k = 0; k < 4; k++) out[k] = r4[k];
    } else {
#pragma unroll
      for (int k = 0; k < 2; k++) {
        const uint32_t send = b2 ? r4[k] : r4[k + 2], keep = b2 ? r4[k + 2] : r4[k];
        out[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
    }
  }
}

// the same over BYTE counts (every sum <= 255): r8[s] holds the four counts of bits s, s+8, s+16, s+24 -> the NW / 4
// registers NW/4 * sub .. of the lane's sub-group, 7 / 6 / 4 shuffles
template <int NW>
__device__ __forceinline__ void sc_reduce_scatter_bytes(const uint32_t (&r8)[8], int lane, uint32_t (&ob)[NW / 4]) {
  const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
  uint32_t r4[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint32_t send = b4 ? r8[k] : r8[k + 4], keep = b4 ? r8[k + 4] : r8[k];
    r4[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  if constexpr (NW == 16) {
#pragma unroll
    for (int k = 0; k < 4; k++) ob[k] = r4[k];
  } else {
    uint32_t r2[2];
#pragma unroll
    for (int k = 0; k < 2; k++) {
      const uint32_t send = b3 ? r4[k] : r4[k + 2], keep = b3 ? r4[k + 2] : r4[k];
      r2[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    if constexpr (NW == 8) {
      ob[0] = r2[0];
      ob[1] = r2[1];
    } else {
      const uint32_t send = b2 ? r2[0] : r2[1], keep = b2 ? r2[1] : r2[0];
      ob[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
  }
}

// R packed-u16 registers of one lane and half in a count table (emitted by a KEEP join, base of the next level's units)
template <int R>
__device__ __forceinline__ void sc_table_load(const uint32_t* p, uint32_t (&v)[R]) {
  if constexpr (R == 2) {
    const uint2 t = __ldcs(reinterpret_cast<const uint2*>(p));
    v[0] = t.x; v[1] = t.y;
  } else {
#pragma unroll
    for (int k = 0; k < R; k += 4) {
      const uint4 t = __ldcs(reinterpret_cast<const uint4*>(p + k));
      v[k] = t.x; v[k + 1] = t.y; v[k + 2] = t.z; v[k + 3] = t.w;
    }
  }
}
template <int R>
__device__ __forceinline__ void sc_table_store(uint32_t* p, const uint32_t (&v)[R]) {
  if constexpr (R == 2) {
    __stcs(reinterpret_cast<uint2*>(p), make_uint2(v[0], v[1]));
  } else {
#pragma unroll
    for (int k = 0; k < R; k += 4) __stcs(reinterpret_cast<uint4*>(p + k), make_uint4(v[k], v[k + 1], v[k + 2], v[k + 3]));
  }
}

// one 1-D bulk copy global -> shared (TMA engine, SASS UBLKCP), completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar_smem) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar_smem)
               : "memory");
}

template <int M, bool KEEP, typename CT, int NW, bool PTS>
__global__ void __launch_bounds__(PTS ? sparse_sc::PTS_THREADS : sparse_sc::THREADS, PTS ? 1 : sparse_sc::min_blocks(NW))
    join_sparse_sc_kernel(const JoinParams a, const SparseParams s) {
  using namespace sparse_sc;
  constexpr int WARPS = (PTS ? PTS_THREADS : THREADS) / 32;
  constexpr int PB = sparse::PB, FLUSH_AT = sparse::FLUSH_AT;
  constexpr int G = 32 / NW;          // sub-groups sharing one pair's carriers
  constexpr uint32_t B = 8 * G;       // carriers per batch
  constexpr uint32_t SHORT = B / 2;   // new carriers of a half the short path takes (<= 4 per sub-group)
  constexpr int R = NW / 2;           // packed count registers (2 permutations each) a lane keeps after the reduce-scatter
  constexpr int NCOPY = (B == 64) ? 2 : 1;  // 32-slot pieces that can hold the < 32 entries left behind a drained batch
  const CT* car0 = static_cast<const CT*>(s.car0);
  const CT* car1 = static_cast<const CT*>(s.car1);
  __shared__ __align__(16) uint32_t s_queue[WARPS][QCAP];
  __shared__ __align__(16) uint32_t s_park[WARPS][32][2 * M];  // totals of the last <= 32 pairs of the warp's unit

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int w = lane % NW, sub = lane / NW;
  const int Wp = a.Wp, Iw = a.Iw;
  const int row_words = Wp * M;
  const unsigned lt_mask = (1u << lane) - 1u;
  uint32_t* queue = s_queue[warp];
  const uint32_t* pt_lane = a.pt + w;
  const uint32_t zero_row = (uint32_t)s.n * (uint32_t)Iw;
  extern __shared__ __align__(128) uint32_t s_pt[];  // PTS: [(n + 1) * Iw] copy of a.pt
  if constexpr (PTS) {
    __shared__ __align__(8) unsigned long long s_bar;
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
    const uint32_t total = ((uint32_t)s.n + 1u) * (uint32_t)Iw * 4u;  // multiple of 16: Iw == 4
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_pt);
      constexpr uint32_t PIECE = 32768;
      for (uint32_t o = 0; o < total; o += PIECE) bulk_copy_g2s(dst + o, reinterpret_cast<const char*>(a.pt) + o, min(PIECE, total - o), bar);
    }
    uint32_t done = 0;
    while (!done) {
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(done) : "r"(bar) : "memory");
    }
  }
  // word w of mask row `off` (a word offset c * Iw): shared memory (PTS) or the read-only path
  auto pt_word = [&](uint32_t off) -> uint32_t {
    if constexpr (PTS) return s_pt[off + (uint32_t)w];
    else return __ldg(word_ptr(pt_lane, off));
  };

  // permutations of this lane: (register i = R*sub + k, half hf)  <->  bit ((i & 1)*2 + hf)*8 + (i >> 1) of word w
  float best[2 * R];
#pragma unroll
  for (int j = 0; j < 2 * R; j++) best[j] = 0.0f;

  while (true) {
    unsigned long long g = 0;
    if (lane == 0) g = atomicAdd(s.work_counter, 1ull);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g >= s.n_units) break;
    const unsigned long long unit = s.unit_begin + g;
    const uint32_t idx = s.unit_idx[unit];
    const uint32_t subu = (uint32_t)(unit - s.unit_prefix[idx]);
    const uint32_t cnt_idx = (uint32_t)a.count[idx];
    const uint32_t j0 = subu * PB, j1 = min(cnt_idx, j0 + PB);
    const uint64_t* p0row = a.p0 + (size_t)idx * row_words;
    const uint32_t loc0 = a.location[idx];

    // eight words into the bit planes of a walk; flushed into the packed counters when nearly full and behind the last batch
    // (planes and batch counters belong to one walk and are zero again after its last flush)
    auto acc8 = [&](uint32_t (&c16)[16], uint32_t (&pl)[8], int& inbatch, int& inreal, const uint32_t (&x)[8], int real, bool last) {
      hs8(pl, x);
      inbatch += 8;
      inreal += real;
      if (inbatch > FLUSH_AT || last) {
        flush_planes(c16, pl, bits_for(inreal));
        inbatch = inreal = 0;
      }
    };

    // ---- base: counts of the upstream row's own carriers for this lane's permutations ----
    uint32_t t0[M], nc0[M], base[M][R];
    if (s.pcnt0) {  // emitted by the join that made the upstream rows
#pragma unroll
      for (int h = 0; h < M; h++) {
        const size_t item = (size_t)idx * M + h;
        t0[h] = s.len0[item];
        nc0[h] = s.ncase0[item];
        sc_table_load<R>(s.pcnt0 + (item * 32 + lane) * R, base[h]);
      }
    } else {  // walk the row's carrier list, 8 G per step, sub-group `sub` takes the sub-th group of eight
#pragma unroll
      for (int h = 0; h < M; h++) {
        t0[h] = nc0[h] = 0;
#pragma unroll
        for (int k = 0; k < R; k++) base[h][k] = 0;
      }
#pragma unroll 1
      for (int h = 0; h < M; h++) {
        uint32_t acc[16], pl[8];
#pragma unroll
        for (int i = 0; i < 16; i++) acc[i] = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) pl[i] = 0;
        int inbatch = 0, inreal = 0;
        const size_t item = (size_t)idx * M + h;
        const CT* lst0 = car0 + s.off0[item];
        const uint32_t plen = (uint32_t)(s.off0[item + 1] - s.off0[item]);
        const uint32_t t0h = s.len0[item], nc0h = s.ncase0[item];
#pragma unroll 1
        for (uint32_t i = 0; i < plen; i += B) {
          uint32_t x[8];
          if (i + sub * 8 < plen) {
            uint32_t c[8];
            load8(lst0 + i + sub * 8, c);
#pragma unroll
            for (int q = 0; q < 8; q++) x[q] = pt_word(c[q] * (uint32_t)Iw);
          } else {
#pragma unroll
            for (int q = 0; q < 8; q++) x[q] = 0u;
          }
          acc8(acc, pl, inbatch, inreal, x, 8, i + B >= plen);
        }
        uint32_t rr[R];
        sc_reduce_scatter<NW>(acc, lane, rr);
        if (M == 1 || h == 0) {
          t0[0] = t0h; nc0[0] = nc0h;
#pragma unroll
          for (int k = 0; k < R; k++) base[0][k] = rr[k];
        } else {
          t0[M - 1] = t0h; nc0[M - 1] = nc0h;
#pragma unroll
          for (int k = 0; k < R; k++) base[M - 1][k] = rr[k];
        }
      }
    }

    // list offsets / lengths of a partner's halves (in the order they are joined into the upstream halves): loaded one pair ahead
    bool flip_n = true;
    unsigned long long off_n[M];
    uint32_t len_n[M];
    auto load_meta = [&](uint32_t loc) {
      if (M == 2) flip_n = need_flip(a.path_length, a.signs, idx, loc);
#pragma unroll
      for (int h = 0; h < M; h++) {
        const int hh = (M == 1) ? 0 : (flip_n ? h : 1 - h);
        const size_t item = (size_t)loc * M + hh;
        off_n[h] = s.off1[item];
        len_n[h] = s.len1[item];
      }
    };
    load_meta(loc0 + j0);

    bool base_done = false;
    // ---- partners ----
    for (uint32_t j = j0; j < j1; j++) {
      const uint32_t loc = loc0 + j;
      const uint32_t park = (j - j0) & 31u;  // slot of this pair in s_park
      const bool flip = flip_n;
      unsigned long long off[M];
      uint32_t lenh[M];
#pragma unroll
      for (int h = 0; h < M; h++) {
        off[h] = off_n[h];
        lenh[h] = len_n[h];
      }
      load_meta(loc0 + min(j + 1, j1 - 1));
      uint32_t nd[M], ncn[M], cnt[M][R];
#pragma unroll
      for (int h = 0; h < M; h++) {
        nd[h] = ncn[h] = 0;
#pragma unroll
        for (int k = 0; k < R; k++) cnt[h][k] = 0;
      }
#pragma unroll 1
      for (int h = 0; h < M; h++) {
        const CT* lst1 = car1 + ((M == 1 || h == 0) ? off[0] : off[M - 1]);
        const uint32_t len = (M == 1 || h == 0) ? lenh[0] : lenh[M - 1];
        const uint64_t* p0h = p0row + h * Wp;
        uint32_t c16[16], pl[8];  // general path only: zeroed by its first drain
        int inbatch = 0, inreal = 0;
        uint32_t rr[R];    // counts of the half's new carriers for this lane's permutations
#pragma unroll
        for (int k = 0; k < R; k++) rr[k] = 0;
        bool counted = len == 0;
        uint32_t ndh = 0, ncnh = 0;
        uint32_t qn = 0;
#pragma unroll 1
        for (uint32_t i0 = 0; i0 < len; i0 += 32) {
          const uint32_t i = i0 + lane;
          const bool valid = i < len;
          const uint32_t c = valid ? (uint32_t)lst1[i] : 0u;
          const uint32_t w0 = valid ? __ldg(reinterpret_cast<const uint32_t*>(p0h) + (c >> 5)) : 0u;
          const bool keep = valid && !((w0 >> (c & 31)) & 1u);
          const unsigned km = __ballot_sync(0xffffffffu, keep);
          ncnh += __popc(__ballot_sync(0xffffffffu, keep && (int)c < a.n_cases));
          if (keep) queue[sc_slot<G>(qn + __popc(km & lt_mask))] = c * (uint32_t)Iw;
          qn += __popc(km);
          const bool last_chunk = i0 + 32 >= len;
          if (last_chunk && ndh == 0 && qn <= SHORT) {
            // ---- short path: everything new fits half a batch; entry t sits at position t / G (< 4) of sub-group t % G ----
            if (qn > 0) {
              if ((uint32_t)lane >= qn && (uint32_t)lane < SHORT) queue[sc_slot<G>((uint32_t)lane)] = zero_row;
              __syncwarp();
              const uint4 lo = *reinterpret_cast<const uint4*>(queue + sub * 8);
              __syncwarp();
              uint32_t r8[8];  // byte counts: byte q of r8[t] <-> bit q*8 + t of the lane's word
              if (qn <= (uint32_t)G) {  // at most one carrier per sub-group
                const uint32_t x0 = pt_word(lo.x);
#pragma unroll
                for (int t = 0; t < 8; t++) r8[t] = (x0 >> t) & 0x01010101u;
              } else {
                const uint32_t x0 = pt_word(lo.x), x1 = pt_word(lo.y);
                const uint32_t x2 = pt_word(lo.z), x3 = pt_word(lo.w);
                uint32_t c1, s1;
                csa(c1, s1, x0, x1, x2);
                const uint32_t q0 = s1 ^ x3, c2 = s1 & x3;
                const uint32_t q1 = c1 ^ c2, q2 = c1 & c2;
#pragma unroll
                for (int t = 0; t < 8; t++) r8[t] = ((q0 >> t) & 0x01010101u) | ((t >= 1 ? (q1 >> (t - 1)) : (q1 << 1)) & 0x02020202u);
                if (qn > 3u * G) {  // some sub-group holds four
#pragma unroll
                  for (int t = 0; t < 8; t++) r8[t] |= (t >= 2 ? (q2 >> (t - 2)) : (q2 << (2 - t))) & 0x04040404u;
                }
              }
              uint32_t ob[NW / 4];
              sc_reduce_scatter_bytes<NW>(r8, lane, ob);
#pragma unroll
              for (int k = 0; k < NW / 4; k++) {
                rr[2 * k] = __byte_perm(ob[k], 0u, 0x4140);
                rr[2 * k + 1] = __byte_perm(ob[k], 0u, 0x4342);
              }
              ndh = qn;
              qn = 0;
            }
            counted = true;
            break;
          }
          // drain whole batches of B; after the last chunk also the remainder (padded with the zero row), and at least once
          // when counts of an earlier batch are still in the planes
#pragma unroll 1
          while (qn >= B || (last_chunk && (qn > 0 || inbatch > 0))) {
            if (ndh == 0) {
#pragma unroll
              for (int t = 0; t < 16; t++) c16[t] = 0;
#pragma unroll
              for (int t = 0; t < 8; t++) pl[t] = 0;
            }
            const uint32_t real = min(qn, B);
            if (real < B) {
              for (uint32_t t = real + lane; t < B; t += 32) queue[sc_slot<G>(t)] = zero_row;
            }
            __syncwarp();
            uint32_t x[8];
            const uint4 lo = *reinterpret_cast<const uint4*>(queue + sub * 8), hi = *reinterpret_cast<const uint4*>(queue + sub * 8 + 4);
            x[0] = pt_word(lo.x);
            x[1] = pt_word(lo.y);
            x[2] = pt_word(lo.z);
            x[3] = pt_word(lo.w);
            x[4] = pt_word(hi.x);
            x[5] = pt_word(hi.y);
            x[6] = pt_word(hi.z);
            x[7] = pt_word(hi.w);
            const uint32_t rem = qn - real;                      // < 32 entries waiting behind the drained batch
            acc8(c16, pl, inbatch, inreal, x, (int)((real + G - 1) / G), last_chunk && rem == 0);
            // they move to the front: the slot layout is per batch, so whole batches are copied as they are
            uint32_t mv[NCOPY];
#pragma unroll
            for (int k = 0; k < NCOPY; k++) mv[k] = queue[B + 32 * k + lane];
            __syncwarp();
            if (rem) {
#pragma unroll
              for (int k = 0; k < NCOPY; k++) queue[32 * k + lane] = mv[k];
            }
            __syncwarp();
            ndh += real;
            qn = rem;
          }
        }
        if (!counted) sc_reduce_scatter<NW>(c16, lane, rr);
        if (M == 1 || h == 0) {
          nd[0] = ndh; ncn[0] = ncnh;
#pragma unroll
          for (int k = 0; k < R; k++) cnt[0][k] = base[0][k] + rr[k];
        } else {
          nd[M - 1] = ndh; ncn[M - 1] = ncnh;
#pragma unroll
          for (int k = 0; k < R; k++) cnt[M - 1][k] = base[M - 1][k] + rr[k];
        }
      }

      bool empty = nd[0] == 0;
      if (M == 2) empty = empty && nd[M - 1] == 0;
      if (!empty || !base_done) {
        if (empty) base_done = true;
        if (M == 1) {
          const unsigned total = t0[0] + nd[0];
          const float* row = a.diagF + diag_base(total);
#pragma unroll
          for (int q = 0; q < 2 * R; q++) {
            const uint32_t v = cnt[0][q >> 1];
            const uint32_t c = (q & 1) ? (v >> 16) : (v & 0xffffu);
            best[q] = fmaxf(best[q], lookup_f32(row, c));
          }
        } else {
          const unsigned tp = t0[0] + nd[0], tn = t0[M - 1] + nd[M - 1];
          const double* rowp = a.diagDM + diag_base(tp);
          const double* rown = a.diagDM + diag_base(tn);  // indexed by tn - cn
#pragma unroll
          for (int q = 0; q < 2 * R; q++) {
            const uint32_t vp = cnt[0][q >> 1], vn = cnt[M - 1][q >> 1];
            const uint32_t cp = (q & 1) ? (vp >> 16) : (vp & 0xffffu);
            const uint32_t cn = (q & 1) ? (vn >> 16) : (vn & 0xffffu);
            // src/methods.h:223-227: vtmax[pcp][total_pos - pcp] + vtmax[total_neg - pnp][pnp]
            const double v = lookup_f64(rowp, cp) + lookup_f64(rown, tn - cn);
            best[q] = fmaxf(best[q], __double2float_rn(v));
          }
        }
      }

      if (KEEP) {
        const size_t r = (size_t)(a.res_idx[idx] + j);
        // ---- the kept row's counts and carrier totals travel with it (base of the next level's units) ----
        if (s.pcnt_res) {
#pragma unroll
          for (int h = 0; h < M; h++) {
            sc_table_store<R>(s.pcnt_res + ((r * M + h) * 32 + lane) * R, cnt[h]);
            if (lane == 0) store_kept_totals<M>(s, r, h, t0, nd, nc0, ncn);
          }
        }
        store_kept_row<M>(a, Wp, p0row, loc, r, flip, lane);
      }
      if (lane == 0) park_totals<M>(s_park[warp][park], t0, nd, nc0, ncn);
      if (park == 31u || j + 1 == j1) score_parked<M, KEEP>(a, s_park[warp], park, idx, loc, lane);
    }
    __syncwarp();
  }
  // best[q]: register i = R*sub + (q >> 1), half q & 1  ->  permutation w*32 + ((i & 1)*2 + (q & 1))*8 + (i >> 1)
#pragma unroll
  for (int q = 0; q < 2 * R; q++) {
    const int i = R * sub + (q >> 1);
    const int r = w * 32 + ((i & 1) * 2 + (q & 1)) * 8 + (i >> 1);
    if (r < a.Ip && best[q] > 0.0f) atomicMax(a.perm_max + r, __float_as_int(best[q]));
  }
}

// words per lane group (4, 8, 16): also the tag of the count-table layout these kernels emit and consume; pcnt0 / pcnt_res,
// when set, must be in that layout (gcre_capi.cu tags every table with the layout it was emitted in)
static inline int sparse_sc_words(int Ip) { return Ip <= 128 ? 4 : Ip <= 256 ? 8 : 16; }
// bytes of one (row, half) entry of that table: 32 lanes x NW / 2 registers
static inline size_t sparse_sc_table_bytes(int Ip) { return (size_t)32 * (sparse_sc_words(Ip) / 2) * 4; }
// host: the count of permutation r in one (row, half) entry of a table in that layout (nw words per lane group): lane
// sub * nw + w holds registers R * sub .. R * sub + R - 1 of word w, R = nw / 2 (sc_reduce_scatter)
static inline uint32_t sc_table_count(const uint32_t* entry, int nw, int r) {
  const int b = r & 31, reg = GCRE_C16_REG(b), R = nw / 2;
  const uint32_t v = entry[((reg / R) * nw + (r >> 5)) * R + reg % R];
  return GCRE_C16_HI(b) ? v >> 16 : v & 0xffffu;
}

// PTS applies to <= 128 permutations when the matrix fits beside the CTA's static shared memory (queues, parked totals:
// n <= ~12,400) and the launch has enough units to pay for staging it (160 KB per SM, ~10 us); pts_forced = 0 / 1 (GCRE_SC_PTS,
// a test hook; -1: not set) turns it off / on where it fits
static inline bool sparse_sc_pts_wanted(const JoinParams& jp, const SparseParams& sp, int sm_count, bool wide, int pts_forced) {
  if (jp.Iw != 4 || wide) return false;
  if (pts_forced >= 0) return pts_forced == 1;
  return sp.n_units >= (unsigned long long)sm_count * (sparse_sc::PTS_THREADS / 32) * 4;
}

template <int M, bool KEEP, int NW>
static inline cudaError_t launch_sparse_sc_ct(cudaStream_t stream, const JoinParams& jp, const SparseParams& sp, int sm_count, bool wide, int pts_forced,
                                              bool* pts) {
  if constexpr (NW == 4) {
    if (sparse_sc_pts_wanted(jp, sp, sm_count, wide, pts_forced)) {
      constexpr int warps = sparse_sc::PTS_THREADS / 32;
      auto kern = join_sparse_sc_kernel<M, KEEP, uint16_t, 4, true>;
      static int static_smem[64];  // per instantiation and device: static shared memory of the kernel, 0 = not asked yet
      int dev = 0;
      cudaGetDevice(&dev);
      if (dev >= 0 && dev < 64) {
        if (static_smem[dev] == 0) {
          cudaFuncAttributes fa;
          cudaError_t e = cudaFuncGetAttributes(&fa, kern);
          if (e != cudaSuccess) return e;
          e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sparse_sc::PTS_SMEM_MAX - fa.sharedSizeBytes));
          if (e != cudaSuccess) return e;
          static_smem[dev] = (int)fa.sharedSizeBytes;
        }
        const size_t dyn = ((size_t)sp.n + 1) * jp.Iw * 4;
        if (dyn + (size_t)static_smem[dev] <= sparse_sc::PTS_SMEM_MAX) {
          const unsigned long long want = (sp.n_units + warps - 1) / warps;
          const unsigned grid = (unsigned)std::min<unsigned long long>(want, (unsigned long long)sm_count);
          kern<<<grid, sparse_sc::PTS_THREADS, dyn, stream>>>(jp, sp);
          *pts = true;
          return cudaGetLastError();
        }
      }
    }
  }
  const unsigned long long want = (sp.n_units + sparse_sc::WARPS - 1) / sparse_sc::WARPS;
  const unsigned grid = (unsigned)std::min<unsigned long long>(want, (unsigned long long)sm_count * sparse_sc::min_blocks(NW));
  if (wide) join_sparse_sc_kernel<M, KEEP, uint32_t, NW, false><<<grid, sparse_sc::THREADS, 0, stream>>>(jp, sp);
  else join_sparse_sc_kernel<M, KEEP, uint16_t, NW, false><<<grid, sparse_sc::THREADS, 0, stream>>>(jp, sp);
  return cudaGetLastError();
}

template <int M, bool KEEP>
static inline cudaError_t launch_sparse_sc_nw(cudaStream_t stream, const JoinParams& jp, const SparseParams& sp, int sm_count, bool wide, int pts_forced,
                                              bool* pts) {
  const int nw = sparse_sc_words(jp.Ip);
  if (nw == 4) return launch_sparse_sc_ct<M, KEEP, 4>(stream, jp, sp, sm_count, wide, pts_forced, pts);
  if (nw == 8) return launch_sparse_sc_ct<M, KEEP, 8>(stream, jp, sp, sm_count, wide, pts_forced, pts);
  return launch_sparse_sc_ct<M, KEEP, 16>(stream, jp, sp, sm_count, wide, pts_forced, pts);
}

// `wide`: u32 carrier indices; *pts is set when the shared-memory form was launched
static inline cudaError_t launch_join_sparse_sc(cudaStream_t stream, const JoinParams& jp, const SparseParams& sp, int M, bool keep, int sm_count, bool wide,
                                                int pts_forced, bool* pts) {
  if (sp.n_units == 0) return cudaSuccess;
  if (M == 1)
    return keep ? launch_sparse_sc_nw<1, true>(stream, jp, sp, sm_count, wide, pts_forced, pts)
                : launch_sparse_sc_nw<1, false>(stream, jp, sp, sm_count, wide, pts_forced, pts);
  return keep ? launch_sparse_sc_nw<2, true>(stream, jp, sp, sm_count, wide, pts_forced, pts)
              : launch_sparse_sc_nw<2, false>(stream, jp, sp, sm_count, wide, pts_forced, pts);
}

}  // namespace gcre
