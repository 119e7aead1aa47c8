// Known-answer test of the seeded permutation masks through the C++ class layer (include/gcre/gcre.h extensions
// setPermutationStrata / generatePermutedMasks): the masks every GPU of the JoinExec holds must be the words below (from
// geneticscre_b200/synth.py make_perm_masks_philox), and a score-only join against them must equal the same join after
// setPermutedCases with the int matrix those words stand for.  Prints the join result on a "join:" line so that runs under
// GCRE_GPUS=1 and GCRE_GPUS=2 (rows sharded over the GPUs) can be compared.
// Built and run by tests/test_perm_gen_gpu.py:  g++ -std=c++11 -Iinclude/gcre ... -lgcre_b200
#include <cmath>
#include <cstdio>
#include <stdexcept>

#include "gcre.h"

static int failures = 0;
#define EXPECT(cond)                                                    \
  do {                                                                  \
    if (!(cond)) {                                                      \
      std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond);     \
      failures++;                                                       \
    }                                                                   \
  } while (0)

static const int kCases = 50, kCtrls = 50, kIters = 4;
static const uint64_t kSeed = 0x0123456789ABCDEFull, kFirst = 0xFFFFFFFEull;  // permutations 2^32 - 2 .. 2^32 + 1
static const uint64_t kPlain[kIters * 2] = {0xb1aa3fc4827a104full, 0x0000000e21f9d533ull, 0x3d8c375505da153cull, 0x0000000a827cdf8aull,
                                            0xf4408ce92de5101bull, 0x000000035debb5d8ull, 0x07be9041e18d8fd9ull, 0x0000000bb0759d68ull};
// strata: patient i in stratum i % 3
static const uint64_t kStrata[kIters * 2] = {0xb1aa3fc4827a104full, 0x0000000e03f9d533ull, 0x348c371501da153cull, 0x0000000ba07cdfafull,
                                             0xf4008ce92de5101bull, 0x000000057dafb5d8ull, 0x07be9041e18d8fd1ull, 0x00000007a4f59d68ull};

static bool masks_are(const JoinExec& ex, const uint64_t* want) {
  bool ok = true;
  for (size_t d = 0; d < ex.device_count(); d++) {
    uint64_t got[kIters * 2] = {0};
    gcre_detail::raise(gcre_exec_get_permuted_masks(ex.handle(d), got, kIters));
    for (int i = 0; i < kIters * 2; i++) ok = ok && got[i] == want[i];
  }
  return ok;
}

static uint32_t lcg(uint32_t& s) { return s = s * 1664525u + 1013904223u; }

static joined_res score_join(JoinExec& ex) {
  const int n = kCases + kCtrls;
  uint32_t s = 12345;
  vec2d_i r0(6, vec_i(n)), r1(6, vec_i(n));
  for (auto* m : {&r0, &r1})
    for (auto& row : *m)
      for (auto& c : row) c = (lcg(s) >> 24) < 40;  // ~16 % carriers
  TPathSet p0 = ex.createPathSet(6), p1 = ex.createPathSet(6), none = ex.createPathSet(0);
  p0->load(r0);
  p1->load(r1);
  vector<uid_ref> uids(6);
  for (int i = 0; i < 6; i++) {
    uids[i].src = i;
    uids[i].trg = i;
    uids[i].count = 3;
    uids[i].location = (uint32_t)(i % 4);
    uids[i].path_idx = 3 * (uint64_t)i;
  }
  return ex.join(UidRelSet(2, uids, vector<int>{1, -1, 1, 1, -1, 1}), *p0, *p1, *none);
}

static void setup(JoinExec& ex) {
  ex.top_k = 5;
  vec2d_d table(kCases + 1, vec_d(kCtrls + 1));
  for (int i = 0; i <= kCases; i++)
    for (int j = 0; j <= kCtrls; j++) table[i][j] = std::fmod(7.3 * i + 1.1 * j + 0.01 * i * j, 13.0);
  ex.setValueTable(table);
}

static bool same(const joined_res& a, const joined_res& b) {
  if (a.scores.size() != b.scores.size() || a.permuted_scores != b.permuted_scores) return false;
  for (size_t i = 0; i < a.scores.size(); i++)
    if (a.scores[i].score != b.scores[i].score || a.scores[i].src != b.scores[i].src || a.scores[i].trg != b.scores[i].trg) return false;
  return true;
}

int main() {
  for (const char* method : {"method1", "method2"}) {
    JoinExec gen(method, kCases, kCtrls, kIters);
    setup(gen);
    gen.generatePermutedMasks(kSeed, kFirst);
    EXPECT(masks_are(gen, kPlain));
    vector<int> labels(kCases + kCtrls);
    for (size_t i = 0; i < labels.size(); i++) labels[i] = (int)(i % 3);
    gen.setPermutationStrata(labels);
    EXPECT(masks_are(gen, kPlain));  // setting strata leaves the current masks alone
    gen.generatePermutedMasks(kSeed, kFirst);
    EXPECT(masks_are(gen, kStrata));
    gen.setPermutationStrata(vector<int>());
    gen.generatePermutedMasks(kSeed, kFirst);
    EXPECT(masks_are(gen, kPlain));
    const joined_res a = score_join(gen);

    // the same permutations as R's CaseORControl int matrix: 1 = label kept
    JoinExec mat(method, kCases, kCtrls, kIters);
    setup(mat);
    vec2d_i perm(kIters, vec_i(kCases + kCtrls));
    for (int r = 0; r < kIters; r++)
      for (int c = 0; c < kCases + kCtrls; c++) perm[r][c] = (int)(((kPlain[r * 2 + c / 64] >> (c % 64)) & 1) == (c < kCases ? 1u : 0u));
    mat.setPermutedCases(perm);
    EXPECT(masks_are(mat, kPlain));
    const joined_res b = score_join(mat);
    EXPECT(same(a, b));
    EXPECT(a.scores.size() == 5 && a.permuted_scores.size() == (size_t)kIters);

    std::printf("join: %s", method);
    for (const Score& sc : a.scores) std::printf(" (%.17g %d %d %d %d)", sc.score, sc.src, sc.trg, sc.cases, sc.ctrls);
    for (double p : a.permuted_scores) std::printf(" %.17g", p);
    std::printf("\n");

    bool threw = false;
    try {  // one label per patient
      gen.setPermutationStrata(vector<int>(7, 1));
    } catch (const std::logic_error& e) {
      threw = std::string(e.what()) == "assertion";
    }
    EXPECT(threw);
  }
  std::printf(failures ? "perm gen: %d FAILURES\n" : "perm gen: OK\n", failures);
  return failures ? 1 : 0;
}
