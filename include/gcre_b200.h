/*
 * gcre_b200.h -- C ABI of the B200-native path-join + permutation-scoring engine.
 *
 * This is the drop-in boundary for geneticsCRE's C++ join loop: every entry point below stands in for one member
 * of the reference's JoinExec / PathSet / UidRelSet class surface (citations are paths in the reference checkout).
 * Plain pointers and sizes only; all buffers passed in are HOST memory unless the name says "device".  Inputs are
 * copied, never aliased (the reference copies too: src/wrapper.cpp:71-96).
 *
 * All functions return GCRE_OK (0) or a negative gcre_status; gcre_last_error() gives the message of the last
 * failure on the calling thread.  There is no CPU fallback: without a CUDA device every compute entry point fails
 * with GCRE_ERR_CUDA.
 *
 * The C++ class layer in include/gcre/ (JoinExec, PathSet, UidRelSet, Score, joined_res, uid_ref, Timer -- same
 * names and members as src/gcre.h, src/gcre_paths.h, src/gcre_types.h, src/util.h) is a thin wrapper over this ABI
 * and rethrows failures as the reference's exception types (src/gcre_types.h:58-76).
 */
#ifndef GCRE_B200_H
#define GCRE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  GCRE_OK = 0,
  GCRE_ERR_ASSERT = -1, /* reference: check_true / check_equal -> std::logic_error("assertion")  (src/gcre_types.h:58-66) */
  GCRE_ERR_RANGE = -2,  /* reference: check_index / check_range -> std::out_of_range("assertion") (src/gcre_types.h:68-76) */
  GCRE_ERR_ARG = -3,    /* null pointer / bad enum: reference: std::logic_error("bad method") (src/join_base.cpp:135) */
  GCRE_ERR_CUDA = -4,   /* CUDA runtime failure or no device */
  GCRE_ERR_NOMEM = -5   /* host or device allocation failed (reference prints and crashes: src/gcre_paths.h:25-36) */
} gcre_status;

/* Score (src/gcre_types.h:32-43): src = row in uids/paths0, trg = row in paths1 (NOT gene uids). */
typedef struct {
  double score;
  int32_t src;
  int32_t trg;
  int32_t cases;
  int32_t ctrls;
} gcre_score;

/* uid_ref (src/gcre_types.h:50-56). location may be 0xFFFFFFFF (R's -1) when count == 0. */
typedef struct {
  int32_t src;
  int32_t trg;
  int32_t count;
  uint32_t location;
  uint64_t path_idx;
} gcre_uid_ref;

typedef struct gcre_exec gcre_exec;       /* JoinExec  (src/gcre.h:103-180) */
typedef struct gcre_pathset gcre_pathset; /* PathSet   (src/gcre_paths.h:10-98), rows live in HBM */

/* Sizes the reference exposes as public JoinExec fields (src/gcre.h:113-123). */
typedef struct {
  int32_t method;          /* 1 or 2 */
  int32_t num_cases;
  int32_t num_ctrls;
  int32_t width_ul;        /* 64-bit words per half-row as stored on the device (W64 rounded up to 2) */
  int32_t iterations;      /* padded permutation count used on the device */
  int32_t iters_requested;
  int32_t device;
  int32_t sm_count;
} gcre_exec_info;

/* which kernel family a join may use */
typedef enum {
  GCRE_KERNEL_AUTO = 0,   /* pick by row length, permutation count and operand density (cost model in join_sparse.cuh; the carriers a
                             partner adds per pair are bounded by the densest row or, when that does not decide, sampled) */
  GCRE_KERNEL_DENSE = 1,  /* AND + POPC against word-major permutation mask tiles */
  GCRE_KERNEL_SPARSE = 2  /* carrier-list walk over patient-major permutation masks (bit-sliced counters) */
} gcre_kernel;

/* Optional controls of one join (zero-initialise for defaults). */
typedef struct {
  uint32_t uid_begin;       /* shard of upstream rows [uid_begin, uid_end); uid_end == 0 means "all" */
  uint32_t uid_end;
  int32_t kernel;           /* gcre_kernel */
  int32_t skip_host_perm;   /* 1: leave permutation maxima on the device only (caller reads gcre_exec_device_perm_max) */
  uint64_t pairs_scored;    /* out: pairs this call scored */
  double kernel_ms;         /* out: device time of the join kernels of this call (CUDA events) */
  int32_t kernel_used;      /* out: gcre_kernel actually run */
  int32_t launches;         /* out: kernel launches made by this call */
  int32_t precounted;       /* out: 1 when the sparse kernel ran in its pre-counted-partner form (join_sparse.cuh) */
  int32_t split_carrier;    /* out: 1 when the <= 512-permutation form of the sparse kernel ran (join_sparse_sc.cuh) */
  int32_t thresholded;      /* out: 1 when the sparse kernel ran with thresholded look-ups (join_sparse.cuh: large method-2 joins) */
  int32_t shared_masks;     /* out: 1 when that form ran with the permutation masks staged in shared memory (<= 128 permutations, small cohorts) */
  uint64_t exact_pairs;     /* out: with thresholded look-ups, the pairs (per 1,024-permutation block) whose exact permutation scores
                               had to be looked up; every other pair was ruled out by one compare per look-up */
  int32_t tail_form;        /* out: 1 when the pre-counted form ran against the gene rows of the base set the partner rows were
                               selected from (join_sparse.cuh, tail form: every partner adds one gene to its upstream path) */
  uint32_t dedup_rows;      /* out: upstream rows not scored because they equal a smaller row of the join in every word and index
                               entry (score-only sparse joins): that row's candidates were appended for them too */
} gcre_join_opts;

/* One split of a reported path for the decorated p-value (R/DecoratedPvalue.R:198-304). */
typedef struct {
  double pvalue;            /* exact limit of the reference's Monte-Carlo estimate: P(re-scored path >= score) */
  double score;             /* score of the real path from the value table */
  int32_t cases1, ctrls1;   /* lst$cases1 / lst$controls1: the sub-path */
  int32_t cases2, ctrls2;   /* lst$cases2 / lst$controls2: what the added gene contributes */
} gcre_decorated;

const char* gcre_last_error(void);
const char* gcre_version(void);
int gcre_device_count(int* count);
/* Number of CUDA kernels this library has launched in this process so far (all execs, all streams). */
int gcre_kernel_launch_count(uint64_t* count);
/* Device memory freed by execs / path sets is kept in a per-device cache for reuse; this returns it to the driver. */
int gcre_release_cached_memory(void);

/* JoinExec::JoinExec(method_name, num_cases, num_ctrls, iters)  (src/join_base.cpp:37-59).
 * method: 1 = "method1", 2 = anything else (JoinExec::to_method, src/gcre.h:125-133).  device: CUDA ordinal. */
int gcre_exec_create(int method, int num_cases, int num_ctrls, int iters, int device, gcre_exec** out);
int gcre_exec_destroy(gcre_exec* ex);
int gcre_exec_get_info(const gcre_exec* ex, gcre_exec_info* out);
/* computeDecoratedPvalue (R/DecoratedPvalue.R:198-304), non-stratified, in the exact limit of its Monte-Carlo estimate, for
 * n_items splits at once against this exec's value table and method.  rows: uint64[n_items][4][ceil(n/64)] packed carrier
 * vectors pos1, neg1 (sub-path), pos2, neg2 (added gene), patient c -> word c/64 bit c%64, cases first. */
int gcre_exec_decorated_exact(gcre_exec* ex, const uint64_t* rows, uint32_t n_items, gcre_decorated* out);
/* Decorated p-values of n_paths whole paths whose genes are rows of `genes` (a path set of this exec; only the first, positive
 * half of each row is read), every split formed on the device.  gene_idx / signs: int32[n_paths][5], lengths[i] in 1..5 (slots
 * past a path's length are not read); signs +1 / -1 (method 2; ignored, and may be NULL, for method 1).
 * out: gcre_decorated[n_paths][8]: path i's 2(L-1) splits in the order of decorated_pvalues_for_path (forward j = 1 .. L-1:
 * genes 0 .. j-1 + gene j; then backward j = L-1 .. 1: genes L-1 .. j + gene j-1), the remaining slots zeroed.
 * stratified = 0: exactly gcre_exec_decorated_exact on those splits.  stratified = 1: the exact limit of stratified resampling
 * (the reference's strataF, R/DecoratedPvalue.R:236-268) under the strata set by gcre_exec_set_permutation_strata (none set: one
 * stratum), so one setting serves the permutations and the decorated p-values.  Per stratum g, with free = ~(pos1 | neg1):
 * c_g / d_g the free cases / controls, kp_g = |pos2 & ~pos1 & free & g|, kn_g = |neg2 & ~neg1 & free & g|,
 *   joint_g[x][y] = Hyp(c_g, d_g, kp_g)(x) * Hyp(d_g - (kp_g - x), c_g - x, kn_g)(y),
 * J = the 2-D convolution of the joint_g in dense-stratum order, p = sum J[cp][cn] * [score_of(cp, sum kp, cn, sum kn) >= score]
 * (score and the counts as in the non-stratified mode).
 * Errors: `genes` of another exec, a method-2 sign not +-1: GCRE_ERR_ARG; a gene index outside [0, size of genes) or a length
 * outside 1..5: GCRE_ERR_RANGE; no value table: GCRE_ERR_ASSERT; a stratum with fewer free patients than carriers to redraw:
 * GCRE_ERR_RANGE naming the path and split (R's sample() stops there).  n_paths = 0: GCRE_OK. */
int gcre_exec_decorated_paths(gcre_exec* ex, const gcre_pathset* genes, const int32_t* gene_idx, const int32_t* signs,
                              const int32_t* lengths, uint32_t n_paths, int stratified, gcre_decorated* out);
/* Run this exec's work on a caller-owned CUDA stream (cudaStream_t passed as void*); NULL restores the internal one. */
int gcre_exec_set_stream(gcre_exec* ex, void* cuda_stream);

/* JoinExec::setValueTable(const vec2d_d&)  (src/join_base.cpp:62-80).  Row-major rows x cols doubles, [cases][ctrls].
 * Entries outside the supplied table read as -1.0, as in the reference's (n+1)x(n+1) padding. */
int gcre_exec_set_value_table(gcre_exec* ex, const double* table, int rows, int cols);
/* The same from a buffer in this exec's device memory (see gcre_pathset_load_bits_device for the ordering rule). */
int gcre_exec_set_value_table_device(gcre_exec* ex, const double* d_table, int rows, int cols);

/* getValuesTable(nCases, nControls) (R/Utils.R:137-159) computed on the device for this exec's own case/control counts:
 * vt[x][y] = -log(two-sided hypergeometric p of x cases among x + y carriers), infinities -> max finite + 1.  The R version
 * is O(n * range^2) and infeasible for n >= 50,000.  gcre_exec_get_value_table copies the table in use to the host. */
int gcre_exec_generate_value_table(gcre_exec* ex);
/* log(k!) for k = 0..n (n + 1 doubles, host only): the table the generator starts from (lets a host-side check make the
 * same decisions at exactly tied probabilities). */
int gcre_log_factorial_table(int n, double* out);
int gcre_exec_get_value_table(const gcre_exec* ex, double* out, int rows, int cols);

/* JoinExec::setPermutedCases(const vec2d_i&)  (src/join_base.cpp:85-125).  Row-major rows x cols int32,
 * 1 = label kept, anything else = flipped; rows reused cyclically if rows < iters, surplus rows ignored. */
int gcre_exec_set_permuted_cases_i32(gcre_exec* ex, const int32_t* perm, int rows, int cols);
/* Same masks already packed: uint64[n_perms][ceil(n/64)], bit c of row r set iff patient c is a case under
 * permutation r (what setPermutedCases computes, without the 32x larger int matrix). */
int gcre_exec_set_permuted_masks_u64(gcre_exec* ex, const uint64_t* masks, int n_perms);
/* The same from a buffer in this exec's device memory (e.g. one batch of a resident set of permutations); ordered on the
 * exec's stream, returns without waiting. */
int gcre_exec_set_permuted_masks_device(gcre_exec* ex, const uint64_t* d_masks, int n_perms);

/* Seeded permutation masks made on the device (extension; no host matrix).  Permutation r (a global 64-bit index) of seed s:
 *   draws    patient i takes u_i = x0 | x1 << 32 (i even) or x2 | x3 << 32 (i odd) of Philox4x32-10 (Salmon et al. 2011; M0 =
 *            0xD2511F53, M1 = 0xCD9E8D57, W0 = 0x9E3779B9, W1 = 0xBB67AE85) with key (lo32(s), hi32(s)) and counter
 *            (i >> 1, lo32(r), hi32(r), 0);
 *   choice   patients are visited in index order i = 0 .. n-1; with g the stratum of i, m_g the patients of g not yet visited
 *            (i included) and k_g the cases still to place in g (initially g's patients with index < num_cases), i is a case
 *            iff mulhi64(u_i, m_g) < k_g (the high 64 bits of the 128-bit product); then m_g -= 1 and, if i was picked, k_g -= 1.
 * So every row keeps each stratum's true case count, each decision's probability is within 2^-64 of k_g / m_g and, with one
 * stratum, every case set of num_cases patients is equally likely: the null of R's permutation matrix, not R's sample() stream.
 * Permutation r is the same whatever batch or GPU makes it.  geneticscre_b200/synth.py (make_perm_masks_philox) restates this
 * in numpy bit for bit.
 *
 * gcre_exec_set_permutation_strata: labels = one arbitrary int32 per patient (n must be num_cases + num_ctrls, GCRE_ERR_ASSERT
 * otherwise); only the partition matters, so relabelling gives identical masks.  At most 1,024 distinct labels
 * (GCRE_ERR_RANGE beyond, the setting is left as it was).  labels = NULL with n = 0 goes back to one stratum.  The host buffer
 * has been read on return; the per-patient tables stay on the device.  The current masks are not changed. */
int gcre_exec_set_permutation_strata(gcre_exec* ex, const int32_t* labels, int n);
/* Rows 0 .. iters_requested-1 := permutations first_perm, first_perm + 1, ... of seed (bit i % 64 of word i / 64 set iff
 * patient i is a case; bits at i >= n zero: what gcre_exec_set_permuted_masks_* accepts).  Ordered on the exec's stream,
 * returns without waiting; nothing to do with 0 iterations.  A batched or sharded job gives batch b of rank r
 * first_perm = (r * n_batches + b) * iters_requested. */
int gcre_exec_generate_permuted_masks(gcre_exec* ex, uint64_t seed, uint64_t first_perm);
/* Copy the first n_perms (<= iters_requested, GCRE_ERR_RANGE otherwise) of the current masks to the host as
 * uint64[n_perms][ceil(n/64)], whichever setter made them (setPermutedCases' int matrix included); waits for the exec's stream. */
int gcre_exec_get_permuted_masks(const gcre_exec* ex, uint64_t* out, int n_perms);

/* JoinExec::createPathSet(size)  (src/join_base.cpp:156-161): size rows of width_ul*method words, zero-filled. */
int gcre_pathset_create(const gcre_exec* ex, uint32_t size, gcre_pathset** out);
int gcre_pathset_destroy(gcre_pathset* ps);
int gcre_pathset_size(const gcre_pathset* ps, uint32_t* size);

/* PathSet::load(const vec2d_i&)  (src/gcre_paths.h:56-78): rows x cols int32, non-zero = carrier, fills the first
 * (pos) half of each row.  rows must equal the set's size; cols must be < 64*ceil64(n) + 1 (any cols <= n works). */
int gcre_pathset_load_i32(gcre_pathset* ps, const int32_t* data, uint32_t rows, int cols);
/* The same rows already packed: uint64[rows][words_per_row], patient c -> word c/64 bit c%64. */
int gcre_pathset_load_bits(gcre_pathset* ps, const uint64_t* bits, uint32_t rows, int words_per_row);
/* The same from a buffer in this exec's device memory (e.g. the target of an NCCL broadcast): ordered on the exec's stream,
 * no host synchronisation; d_bits must stay valid until that stream has passed the copy (any later join synchronises). */
int gcre_pathset_load_bits_device(gcre_pathset* ps, const uint64_t* d_bits, uint32_t rows, int words_per_row);
/* Host utility (no GPU involved): packs rows x cols int32 (non-zero = carrier, src/gcre_paths.h:65-67) into
 * uint64[rows][ceil(cols/64)] for gcre_pathset_load_bits, on `threads` host threads (<= 0: all hardware threads, at most 16).
 * gcre_pathset_load_i32 uses it by itself for large inputs when the host has >= 8 threads to spare. */
int gcre_host_pack_i32(const int32_t* data, uint32_t rows, int cols, uint64_t* bits, int threads);

/* PathSet::select(const vector<int>&)  (src/gcre_paths.h:82-92): new set, row k = row indices[k] of ps. */
int gcre_pathset_select(const gcre_pathset* ps, const int32_t* indices, uint32_t n, gcre_pathset** out);

/* PathSet::set(idx, data) / PathSet::operator[](idx)  (src/gcre_paths.h:44-52).  Rows are exchanged UNPADDED:
 * ceil(n/64)*method words, method-2 rows as [pos | neg]. */
int gcre_pathset_set_row(gcre_pathset* ps, uint32_t idx, const uint64_t* words);
int gcre_pathset_get_row(const gcre_pathset* ps, uint32_t idx, uint64_t* words);
/* all rows, unpadded, uint64[size][ceil(n/64)*method] */
int gcre_pathset_download(const gcre_pathset* ps, uint64_t* out);

/*
 * JoinExec::join(uids, paths0, paths1, paths_res)  (src/join_base.cpp:189-264) with UidRelSet(path_length, uids,
 * signs) (src/gcre.h:49-90) flattened into arrays.
 *
 *   paths_res   NULL or a set of size 0: score only.  Otherwise its size must equal sum(count) and joined rows are
 *               written at uid.path_idx + j (src/join_base.cpp:239,246-249).
 *   top_k       JoinExec::top_k (src/gcre.h:120).
 *   out_scores  capacity top_k + 1; ascending score; holds the -inf sentinel {src=trg=-1} first when fewer than top_k
 *               pairs were pushed (src/join_base.cpp:192-194, 138-154).  Among equal scores the smaller (src, trg)
 *               wins a place (the reference's choice among ties is heap- and thread-dependent).
 *   out_perm    iters_requested doubles holding float-rounded maxima: (float) max(+0, max over pairs p_score)
 *               (src/methods.h:96-103, 220-230; src/join_base.cpp:142-146).
 *   opts        NULL for defaults.
 * Pre-checks as src/join_base.cpp:196-200: n_uids == paths0.size (GCRE_ERR_ASSERT), paths_res size (GCRE_ERR_ASSERT),
 * location + count - 1 < paths1.size (GCRE_ERR_RANGE).
 */
int gcre_join(gcre_exec* ex, int path_length, const gcre_uid_ref* uids, uint32_t n_uids, const int32_t* signs,
              uint32_t n_signs, const gcre_pathset* paths0, const gcre_pathset* paths1, gcre_pathset* paths_res,
              int top_k, gcre_score* out_scores, int* n_scores, double* out_perm, gcre_join_opts* opts);

/* UidRelSet kept on the device: build the join index once, join with it many times (the level schedule of a run reuses
 * nothing, but a resident service / benchmark does).  gcre_join(...) == create + gcre_join_uidset + destroy. */
typedef struct gcre_uidset gcre_uidset;
int gcre_uidset_create(gcre_exec* ex, int path_length, const gcre_uid_ref* uids, uint32_t n_uids, const int32_t* signs,
                       uint32_t n_signs, gcre_uidset** out);
int gcre_uidset_destroy(gcre_uidset* uidset);
int gcre_join_uidset(gcre_exec* ex, const gcre_uidset* uidset, const gcre_pathset* paths0, const gcre_pathset* paths1,
                     gcre_pathset* paths_res, int top_k, gcre_score* out_scores, int* n_scores, double* out_perm,
                     gcre_join_opts* opts);

/* Device pointer (float[iterations]) to the permutation maxima of the last join on this exec -- lets a multi-GPU
 * driver merge shards with one allreduce(max) (NCCL) without a host round trip.  Valid until the next join. */
int gcre_exec_device_perm_max(const gcre_exec* ex, void** device_ptr, int* n_floats);
/* Device-to-device copy of those maxima into / out of a caller-owned device buffer (e.g. a torch tensor that
 * torch.distributed all-reduces); count floats, on this exec's stream. */
int gcre_exec_export_perm_max(const gcre_exec* ex, void* device_dst, int count);
int gcre_exec_import_perm_max(gcre_exec* ex, const void* device_src, int count);
/* After an external allreduce: read the maxima back (float-rounded, widened to double). */
int gcre_exec_read_perm_max(const gcre_exec* ex, double* out_perm);

/* Merge shard-local top-K lists (each ascending, sentinel allowed) into the global list under the same rule. */
int gcre_merge_topk(const gcre_score* lists, const int* list_sizes, int n_lists, int top_k, gcre_score* out_scores,
                    int* n_scores);

/*
 * ---- Test and diagnostics only ----
 * Read-backs of the state the sparse kernels keep per path set, so that tests can check it directly and not only through
 * the join results it feeds.  Each copies on the exec's stream and waits for it.  Not part of the reference's surface.
 *
 * gcre_pathset_debug_view_info: out = int64[8]: [0] carrier lists built, [1] their padded entries, [2] len / ncase filled,
 *   [3] a count table present, [4] its layout (0: the 1,024-permutation register image of join_sparse.cuh; 4 / 8 / 16: the
 *   split-carrier layout of join_sparse_sc.cuh), [5] it was built for the exec's current permutation masks, [6] / [7] the rows
 *   [lo, hi) it holds (a KEEP join's emitted rows, or every row of a pre-count table).
 * gcre_pathset_debug_counts: the table decoded: counts = uint16[hi - lo][method][iters_requested], the count of permutation r
 *   in half h of row lo + i; len / ncase = uint32[hi - lo][method] carriers and carriers < num_cases per half (NULL: not
 *   copied).  GCRE_ERR_ASSERT when the set holds no table.
 * gcre_pathset_debug_lists: the carrier lists: off = uint64[size * method + 1] (list starts, in entries), len / ncase =
 *   uint32[size * method], car = uint32[off[size * method]] (patient indices, sentinel num_cases + num_ctrls as padding).
 *   GCRE_ERR_ASSERT when the lists are not built.
 * gcre_pathset_debug_bounds: out = int64[2]: [0] the largest carrier count of any half-row as the set records it (not
 *   recomputed; -1 = unknown, computed by the next join that reads the set), which sizes its carrier lists and the exec's
 *   anti-diagonal tables and must never be below the true one; [1] the carrier-list entries allocated (0: no lists built).
 * gcre_exec_debug_diag_cap: out = the largest joined half-row total the exec's anti-diagonal value tables cover (-1: none
 *   built since the value table last changed).
 */
int gcre_pathset_debug_view_info(const gcre_pathset* ps, int64_t* out);
int gcre_pathset_debug_counts(const gcre_pathset* ps, uint16_t* counts, uint32_t* len, uint32_t* ncase);
int gcre_pathset_debug_lists(const gcre_pathset* ps, uint64_t* off, uint32_t* len, uint32_t* ncase, uint32_t* car);
int gcre_pathset_debug_bounds(const gcre_pathset* ps, int64_t* out);
int gcre_exec_debug_diag_cap(const gcre_exec* ex, int64_t* out);

#ifdef __cplusplus
}
#endif
#endif /* GCRE_B200_H */
