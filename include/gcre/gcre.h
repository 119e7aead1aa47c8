// Drop-in replacement for the reference's src/gcre.h: UidRelSet, JoinMethod (interface kept for source compatibility)
// and JoinExec with the same public surface, implemented over the C ABI of the B200 engine (include/gcre_b200.h).
// With this directory first on the include path and -lgcre_b200 on the link line, the reference's own
// src/wrapper.cpp / src/RcppExports.cpp (R entry points) and test/harness.cpp compile and run unchanged; the
// reference's src/join_base.cpp and src/methods.h are no longer compiled.  Reference: src/gcre.h:49-180,
// src/join_base.cpp:37-264.
#ifndef GCRE_H
#define GCRE_H

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <memory>
#include <queue>
#include <string>
#include <vector>

#include <atomic>
#include <mutex>
#include <thread>

// the reference picks a SIMD width at compile time and pads to it (src/gcre.h:19-39); here the "vector unit" is a B200
const int gs_vec_width = 64;
const std::string gs_instr_label = "B200 sm_100a";
#define gs_align_size 16
#define ALIGNED __attribute__((aligned(gs_align_size)))

#include "gcre_types.h"
#include "gcre_paths.h"

using namespace std;  // the reference header exports this and src/wrapper.cpp relies on it (src/gcre.h:47)

// Join index: for upstream row idx the partners are rows [location, location + count) of the downstream set
// (src/gcre.h:49-90).
class UidRelSet {
 public:
  const int path_length;
  const vector<uid_ref> uids;
  const vector<int> signs;

  UidRelSet(int path_length_, vector<uid_ref> uids_, vector<int> signs_) : path_length(path_length_), uids(uids_), signs(signs_) {}

  size_t size() const { return uids.size(); }

  const uid_ref& operator[](int idx) const {
    check_index(idx, uids.size());
    return uids[idx];
  }

  // which half of a method-2 downstream row joins the positive half (src/gcre.h:71-81); evaluated on the device in
  // the join kernels, kept here for callers that ask
  bool need_flip(int idx, int loc) const {
    int sign;
    if (path_length > 3) sign = signs[idx];
    else if (path_length < 3) sign = signs[loc];
    else sign = (signs[idx] + signs[loc] == 0) ? -1 : 1;
    return sign == 1;
  }

  st_path_count count_total_paths() const {
    st_path_count total = 0;
    for (const auto& uid : uids) total += uid.count;
    return total;
  }
};

// Kept so code that names the type still compiles (src/gcre.h:92-101); the scoring methods are CUDA kernels now.
class JoinMethod {
 public:
  virtual ~JoinMethod() {}
  virtual void score_permute(int idx, int loc, const uint64_t* path0, const uint64_t* path1, uint64_t* path_res, bool keep_paths) = 0;
  virtual void merge_scores() = 0;
};
using TJoinMethod = unique_ptr<JoinMethod>;

class JoinExec {
 public:
  const Method method;
  const int num_cases;
  const int num_ctrls;
  const int width_ul;         // host-visible words per half-row: ceil(n / 64)
  const int iterations;       // permutations as padded on the device
  const int iters_requested;

  int top_k = 12;    // src/gcre.h:120
  int nthreads = 0;  // accepted for compatibility; the join runs on the GPU(s)
  int width_vec = 0;

  static Method to_method(string name) { return name == "method1" ? Method::method1 : Method::method2; }  // src/gcre.h:125-133

  // src/join_base.cpp:37-59.  GPUs: GCRE_DEVICES="0,2,3" (explicit ordinals) or GCRE_GPUS=N (ordinals 0..N-1) or
  // GCRE_DEVICE=k (one GPU, default 0).  With several GPUs every path set is replicated, joins that keep their rows run
  // on every GPU, and score-only joins (levels 4 and 5 - where the pairs are) are sharded over the GPUs by upstream row.
  JoinExec(string method_name, int num_cases_, int num_ctrls_, int iters)
      : method(to_method(method_name)),
        num_cases(num_cases_),
        num_ctrls(num_ctrls_),
        width_ul((num_cases_ + num_ctrls_ + 63) / 64),
        iterations(padded_iterations(iters)),
        iters_requested(iters) {
    check_true(num_cases > 0 && num_ctrls > 0 && iters >= 0);
    const std::vector<int> devices = devices_from_env();
    handles_.assign(devices.size(), nullptr);
    try {
      gcre_for_each_device(devices.size(), [&](size_t d) {
        return gcre_exec_create((int)method, num_cases, num_ctrls, iters, devices[d], &handles_[d]);
      });
    } catch (...) {
      for (gcre_exec* h : handles_) gcre_exec_destroy(h);
      throw;
    }
  }
  JoinExec(const JoinExec&) = delete;
  JoinExec& operator=(const JoinExec&) = delete;
  ~JoinExec() {
    for (gcre_exec* h : handles_) gcre_exec_destroy(h);
  }

  void print_vector_info() {}  // src/gcre.h:144-152: all output is commented out upstream

  // src/join_base.cpp:62-80
  void setValueTable(const vec2d_d& table) {
    const size_t rows = table.size(), cols = rows ? table.front().size() : 0;
    std::vector<double> flat(rows * cols, -1.0);  // ragged rows read as the reference's -1.0 padding
    for (size_t r = 0; r < rows; r++)
      for (size_t c = 0; c < std::min(cols, table[r].size()); c++) flat[r * cols + c] = table[r][c];
    gcre_for_each_device(handles_.size(), [&](size_t d) { return gcre_exec_set_value_table(handles_[d], flat.data(), (int)rows, (int)cols); });
  }

  // src/join_base.cpp:85-125 (same WARN lines)
  void setPermutedCases(const vec2d_i& data) {
    if ((size_t)iters_requested < data.size()) printf("  ** WARN more permuted cases than iterations, input will be truncated\n");
    const size_t rows = std::min(data.size(), (size_t)iters_requested), cols = (size_t)num_cases + num_ctrls;
    std::vector<int32_t> flat(rows * cols);
    for (size_t r = 0; r < rows; r++) {
      check_equal(cols, data[r].size());
      for (size_t c = 0; c < cols; c++) flat[r * cols + c] = data[r][c];
    }
    if ((size_t)iters_requested > data.size())
      printf("  ** WARN not enough permuted cases, some will be reused to match iterations - hope this is for testing!\n");
    gcre_for_each_device(handles_.size(),
                         [&](size_t d) { return gcre_exec_set_permuted_cases_i32(handles_[d], flat.data(), (int)rows, (int)cols); });
  }

  // Extensions (include/gcre_b200.h): strata of the seeded generator (one label per patient; empty = one stratum) and
  // permutations first_perm .. first_perm + iters_requested - 1 of seed made on every GPU - identical seeds give identical
  // masks everywhere, so the sharded joins see the same permutations on each device.
  void setPermutationStrata(const vector<int>& labels) {
    if (!labels.empty()) check_equal(labels.size(), (size_t)num_cases + num_ctrls);
    std::vector<int32_t> lab(labels.begin(), labels.end());
    gcre_for_each_device(handles_.size(), [&](size_t d) {
      return gcre_exec_set_permutation_strata(handles_[d], lab.empty() ? nullptr : lab.data(), (int)lab.size());
    });
  }
  void generatePermutedMasks(uint64_t seed, uint64_t first_perm = 0) {
    gcre_for_each_device(handles_.size(), [&](size_t d) { return gcre_exec_generate_permuted_masks(handles_[d], seed, first_perm); });
  }

  // src/join_base.cpp:156-161
  TPathSet createPathSet(st_pathset_size size) const {
    std::vector<gcre_pathset*> ps(handles_.size(), nullptr);
    gcre_for_each_device(handles_.size(), [&](size_t d) { return gcre_pathset_create(handles_[d], size, &ps[d]); });
    return TPathSet(new PathSet(ps, size, width_ul, (uint16_t)(width_ul * (int)method)));
  }

  // src/join_base.cpp:189-264 (+ result formatting :138-154)
  joined_res join(const UidRelSet& uids, const PathSet& paths0, const PathSet& paths1, PathSet& paths_res) const {
    static_assert(sizeof(uid_ref) == sizeof(gcre_uid_ref), "uid_ref layout must match the C ABI");
    printf("progress:");
    const int k = top_k > 0 ? top_k : 1;
    const size_t nd = handles_.size();
    const bool keep = paths_res.size != 0;
    const gcre_uid_ref* u = reinterpret_cast<const gcre_uid_ref*>(uids.uids.data());
    const uint32_t n_uids = (uint32_t)uids.uids.size();

    // shards of upstream rows balanced by pair count (score-only joins on several GPUs); one shard otherwise
    std::vector<uint32_t> cut(nd + 1, n_uids);
    cut[0] = 0;
    if (nd > 1 && !keep) {
      st_path_count total = uids.count_total_paths(), run = 0;
      size_t next = 1;
      for (uint32_t i = 0; i < n_uids && next < nd; i++) {
        run += uids.uids[i].count > 0 ? uids.uids[i].count : 0;
        while (next < nd && run * nd >= total * next) cut[next++] = i + 1;
      }
    }

    std::vector<std::vector<gcre_score>> sc(nd, std::vector<gcre_score>((size_t)k + 1));
    std::vector<int> n_sc(nd, 0);
    std::vector<std::vector<double>> perm(nd, std::vector<double>((size_t)std::max(iters_requested, 1), 0.0));
    gcre_for_each_device(nd, [&](size_t d) {
      gcre_join_opts opts;
      std::memset(&opts, 0, sizeof opts);
      if (nd > 1 && !keep) {
        if (cut[d] == cut[d + 1]) return (int)GCRE_OK;  // empty shard
        opts.uid_begin = cut[d];
        opts.uid_end = cut[d + 1];
      }
      return gcre_join(handles_[d], uids.path_length, u, n_uids, uids.signs.data(), (uint32_t)uids.signs.size(), paths0.handle(d),
                       paths1.handle(d), paths_res.handle(d), k, sc[d].data(), &n_sc[d], perm[d].data(), &opts);
    });

    joined_res res;
    res.permuted_scores.assign((size_t)iters_requested, 0.0);
    std::vector<gcre_score> merged((size_t)k + 1);
    int n_merged = 0;
    if (nd > 1 && !keep) {
      // merge_scores of the reference (src/methods.h:25-39): element-wise max of the maxima, union of the top-K lists
      for (size_t d = 0; d < nd; d++)
        for (int r = 0; r < iters_requested; r++) res.permuted_scores[r] = std::max(res.permuted_scores[r], perm[d][r]);
      std::vector<gcre_score> all;
      std::vector<int> sizes;
      for (size_t d = 0; d < nd; d++) {
        all.insert(all.end(), sc[d].begin(), sc[d].begin() + n_sc[d]);
        sizes.push_back(n_sc[d]);
      }
      gcre_detail::raise(gcre_merge_topk(all.data(), sizes.data(), (int)nd, k, merged.data(), &n_merged));
    } else {
      for (int r = 0; r < iters_requested; r++) res.permuted_scores[r] = perm[0][r];
      merged = sc[0];
      n_merged = n_sc[0];
    }
    res.scores.reserve((size_t)n_merged);
    for (int i = 0; i < n_merged; i++) res.scores.push_back(Score(merged[i].score, merged[i].src, merged[i].trg, merged[i].cases, merged[i].ctrls));
    printf(" - done!\n\n");
    return res;
  }

  gcre_exec* handle(size_t device_slot = 0) const { return handles_[device_slot]; }
  size_t device_count() const { return handles_.size(); }

 protected:
  static int padded_iterations(int iters) { return ((std::max(iters, 1) + 127) / 128) * 128; }

  static std::vector<int> devices_from_env() {
    std::vector<int> out;
    if (const char* list = std::getenv("GCRE_DEVICES")) {
      const char* p = list;
      while (*p) {
        char* e = nullptr;
        const long v = std::strtol(p, &e, 10);
        if (e == p) break;
        out.push_back((int)v);
        p = (*e == ',') ? e + 1 : e;
      }
    } else if (const char* n = std::getenv("GCRE_GPUS")) {
      for (int d = 0; d < std::atoi(n); d++) out.push_back(d);
    }
    if (out.empty()) {
      const char* dev = std::getenv("GCRE_DEVICE");
      out.push_back(dev ? std::atoi(dev) : 0);
    }
    return out;
  }

  std::vector<gcre_exec*> handles_;
};

#endif
