"""Generates the golden fixtures in this directory by running the UNMODIFIED reference (oracle/_ref, built by
oracle/build_ref.sh from the reference checkout named by $GCRE_REF) on seeded inputs:

    python tests/golden/make_golden.py

Fixtures (npz, inputs + the reference's outputs for every level of the schedule):
  vignette_m1_len2_p100.npz   BASELINE config 1: bundled inst/extdata/random.phenotype.data (3000 genes x 200 patients,
                              100 cases) on a seeded synthetic edge list (Rels.dat is absent from the checkout),
                              method 1, path length 2, 100 permutations
  vignette_m2_len3_p1000.npz  BASELINE config 2: same data, method 2, path length 3, 1,000 permutations
  synth_m{1,2}_len5.npz       small synthetic cohort (n = 333, irregular table) through all six joins

    python tests/golden/make_golden.py bench

  bench_level4_p1000.npz      the level-4 join of bench.py's default workload (BASELINE config 3), methods 1 and 2: pair
                              count, top-K and the 1,000 permutation maxima.  Computed by the scalar C restatement
                              (oracle/gcre_oracle.c, pinned to the reference by the fixtures above) over upstream-row shards
                              on all host cores, about 10 minutes on 8 cores; the inputs are regenerated from bench.py's seed.
"""
import argparse
import multiprocessing
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from geneticscre_b200 import schedule, synth  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

REF = os.environ.get("GCRE_REF", "/root/reference")


def vignette_workload(n_perms, seed, n_edges=4000, max_len=3):
    """Bundled phenotype data restricted to genes known to Ents.dat, with a seeded synthetic signed edge list."""
    ents = {}
    with open(os.path.join(REF, "inst/extdata/Ents.dat")) as f:
        next(f)
        for line in f:
            parts = line.split()
            uid, sym = int(parts[1]), parts[3].strip('"')
            if sym != "-1" and sym not in ents:
                ents[sym] = uid
    syms, rows = [], []
    with open(os.path.join(REF, "inst/extdata/random.phenotype.data")) as f:
        next(f)
        for line in f:
            parts = line.split()
            syms.append(parts[1].strip('"'))  # parts[0] is the R row name
            rows.append(np.array(parts[2:], dtype=np.int32))
    data = np.stack(rows)
    data[data == 2] = 1  # R/Utils.R:174
    n = data.shape[1]
    n_cases = n // 2
    freqs = data.sum(axis=1)
    keep = [i for i, s in enumerate(syms) if s in ents and freqs[i] <= 0.05 * (n + 1)]  # R/Utils.R:185-188
    keep.sort(key=lambda i: ents[syms[i]])  # Ents order (by uid)
    data = data[keep]
    g = data.shape[0]
    rng = np.random.default_rng(seed)
    pairs = set()
    while len(pairs) < n_edges:
        s, t = rng.integers(0, g, 2)
        if s != t:
            pairs.add((int(s), int(t)))
    pairs = np.array(sorted(pairs))
    used = np.unique(pairs)
    remap = -np.ones(g, dtype=np.int64)
    remap[used] = np.arange(used.size)
    pairs = remap[pairs]
    order = np.lexsort((pairs[:, 1], pairs[:, 0]))
    pairs = pairs[order]
    sign = np.where(rng.random(pairs.shape[0]) < 0.7, 1, -1).astype(np.int32)
    net = synth.network_from_edges(used.size, pairs[:, 0], pairs[:, 1], sign, max_path_length=max_len)
    bits = synth.pack_bits(data[used])
    masks = synth.make_perm_masks(n_cases, n - n_cases, n_perms, seed + 3)
    table = synth.make_value_table(n_cases, n - n_cases)
    return synth.Workload(n_cases, n - n_cases, n_perms, bits, np.ascontiguousarray(bits[net.ents2]), masks, table, net)


def run_reference(w, method, path_length, top_k):
    ex = po.RefExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.nthreads = 0  # deterministic top-K ties (SURVEY section 8c)
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    res, kept = schedule.replay_levels(ex, po.UidRelSet, w, path_length, use_int_matrices=True)
    return res, {k: v.to_numpy() for k, v in kept.items()}


def save(name, w, method, path_length, top_k):
    res, kept = run_reference(w, method, path_length, top_k)
    out = {
        "method": method, "path_length": path_length, "top_k": top_k, "n_cases": w.n_cases, "n_ctrls": w.n_ctrls, "n_perms": w.n_perms,
        "gene_bits": w.gene_bits, "gene_bits2": w.gene_bits2, "perm_masks": w.perm_masks, "value_table": w.value_table,
        "n_genes": w.net.n_genes, "edges_src": w.net.edges_src, "edges_trg": w.net.edges_trg, "edges_sign": w.net.edges_sign,
        "ents2": w.net.ents2, "levels": np.array(sorted(res.keys())),
    }
    for lvl, r in res.items():
        out[f"scores_{lvl}"] = np.array([[s.score, s.src, s.trg, s.cases, s.ctrls] for s in r.scores], dtype=np.float64).reshape(-1, 5)
        out[f"perm_{lvl}"] = r.permuted_scores
    for k, v in kept.items():
        out[f"kept_{k}"] = v
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **out)
    print(name, os.path.getsize(path), "bytes", {l: len(r.scores) for l, r in res.items()})


_SHARD = {}


def _join_shard(bounds):
    """Level-4 join of upstream rows [a, b) on the oracle prepared in _SHARD (inherited by fork); src made absolute."""
    a, b = bounds
    ex, kept, lv = _SHARD["ex"], _SHARD["kept"], _SHARD["lv"]
    uids = po.UidRelSet(4, lv.src[a:b], lv.trg[a:b], lv.count[a:b], lv.location[a:b], lv.signs[a:b])
    r = ex.join(uids, kept["paths3"].select(np.arange(a, b, dtype=np.int32)), kept["paths2"], ex.createPathSet(0))
    return [(s.score, s.src + a, s.trg, s.cases, s.ctrls) for s in r.scores if s.src >= 0], r.permuted_scores


def bench_level4(method, workers):
    import bench
    from geneticscre_b200 import dist

    a = argparse.Namespace(table="host", **bench.WORKLOAD)
    w, _ = bench.make_workload(a)
    ex = po.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = a.top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    _, kept = schedule.replay_levels(ex, po.UidRelSet, w, 3, only=())
    lv = w.net.levels["4"]
    _SHARD.update(ex=ex, kept=kept, lv=lv)
    shards = [b for b in dist.shard_bounds(lv.count, 4 * workers) if b[1] > b[0]]
    with multiprocessing.get_context("fork").Pool(workers) as pool:
        parts = pool.map(_join_shard, shards, chunksize=1)
    perm = np.max(np.stack([p for _, p in parts]), axis=0)
    # the oracle's deterministic rule: the K largest scores, ties to the smaller (upstream row, downstream row)
    best = sorted((e for s, _ in parts for e in s), key=lambda e: (-e[0], e[1], e[2]))[: a.top_k]
    scores = sorted(best, key=lambda e: (e[0], -e[1], -e[2]))  # the oracle's output order: ascending, later pairs first among ties
    if len(scores) < a.top_k:
        scores.insert(0, (-np.inf, -1, -1, 0, 0))
    return int(lv.n_pairs), np.array(scores, dtype=np.float64).reshape(-1, 5), perm


def save_bench(workers):
    out = {}
    for method in ("method1", "method2"):
        pairs, scores, perm = bench_level4(method, workers)
        out.update({f"pairs_{method}": pairs, f"scores_{method}": scores, f"perm_{method}": perm})
        print(method, pairs, "pairs, max permutation maximum", perm.max(), flush=True)
    path = os.path.join(HERE, "bench_level4_p1000.npz")
    np.savez_compressed(path, **out)
    print("bench_level4_p1000.npz", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    po.build()
    if sys.argv[1:] == ["bench"]:
        save_bench(os.cpu_count() or 1)
        sys.exit(0)
    save("vignette_m1_len2_p100.npz", vignette_workload(100, 101, max_len=2), "method1", 2, 10)
    save("vignette_m2_len3_p1000.npz", vignette_workload(1000, 102, max_len=3), "method2", 3, 10)
    w = synth.make_workload(150, 183, 400, 1100, 77, seed=7, max_path_length=5, real_table=False, max_freq=0.08, zero_frac=0.3)
    save("synth_m1_len5.npz", w, "method1", 5, 12)
    save("synth_m2_len5.npz", w, "method2", 5, 12)
