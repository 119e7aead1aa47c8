"""Parity on WHAT IS BENCHMARKED: the level-4 join of bench.py's default workload (BASELINE config 3: 10,000 patients,
150,000 edges => 1.35 M three-gene paths, 12 M level-4 pairs, 1,000 permutations) on the GPU, both methods, against
tests/golden/bench_level4_p1000.npz: pair count, top-K and permutation maxima of the whole join computed on the host by the
scalar C restatement (tests/golden/make_golden.py bench), which the other fixtures pin to the reference.  Where oracle/_ref
is built, the reference's own join_base.cpp is run live as well (all host threads: permutation maxima and - under the A.7
rule - the top-K do not depend on the thread count, SURVEY section 8c), in the worker subprocesses of bench.py's
cpu_baseline leg (it never frees its per-thread copies of the value table).
"""
import argparse
import os

import numpy as np
import pytest

from geneticscre_b200 import _lib, schedule

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bench_mod():
    import bench

    return bench


@pytest.fixture(scope="module")
def workload(bench_mod):
    a = argparse.Namespace(table="host", impl="ours", shard="perms", **bench_mod.WORKLOAD)
    w, _ = bench_mod.make_workload(a)
    return a, w


def test_level4_of_the_bench_workload_matches_the_reference(engine, oracles, bench_mod, workload):
    a, w = workload
    lv = w.net.levels["4"]
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bench_level4_p1000.npz"))
    expected = {"stored": {m: {"pairs": int(z[f"pairs_{m}"]), "scores": z[f"scores_{m}"], "perm": z[f"perm_{m}"]} for m in ("method1", "method2")}}
    if oracles.ref_available():
        arm = bench_mod.ReferenceArm(w, a)
        try:
            for method in arm.methods:
                arm.plan[method] = (lv.n_uids, 0.0)  # the whole join
            _, expected["live reference"] = arm.sample(60.0, results=True)
        finally:
            arm.close()
    for method in ("method1", "method2"):
        ex = engine.JoinExec(method, w.n_cases, w.n_ctrls, w.n_perms)
        ex.top_k = a.top_k
        ex.setValueTable(w.value_table)
        ex.setPermutedMasks(w.perm_masks)
        got, _ = schedule.replay_levels(ex, engine.UidRelSet, w, 4, only=("4",))
        for source, out in expected.items():
            r = out[method]
            assert r["pairs"] == lv.n_pairs == got["4"].info["pairs"]
            want = oracles.JoinedRes([oracles.Score(float(s[0]), int(s[1]), int(s[2]), int(s[3]), int(s[4])) for s in r["scores"]],
                                     np.asarray(r["perm"], dtype=np.float64))
            oracles.compare_results(got["4"], want, what=f"bench workload level 4 {method} vs {source}")
            assert float(want.permuted_scores.max()) > 0.0
        assert got["4"].info["kernel"] == _lib.KERNEL_SPARSE
        ex.close()
