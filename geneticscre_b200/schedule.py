"""Host-side replay of the level schedule that calls ``join`` (the caller of the hot path).

Mirrors ``ProcessPaths`` (src/wrapper.cpp:176-281) and the standalone harness (test/harness.cpp:109-181): six joins
1a, 1b, 2, 3, 4, 5 in that order, with the kept path sets of levels 1a/2/3 feeding the next level.  It is written
against the reference class surface (JoinExec / PathSet / UidRelSet) so any implementation of that surface can run it.
"""
from __future__ import annotations

import numpy as np


def replay_levels(ex, uidrelset_cls, workload, path_length: int, use_int_matrices: bool = False, only=None,
                  on_level=None):
    """Run levels 1..path_length through ``ex``; returns ``{level: joined_res}`` and the kept path sets.

    ``ex`` must already hold the value table and permutation masks.  ``use_int_matrices`` feeds ``PathSet.load`` with
    the 0/1 IntegerMatrix exactly as R does (src/wrapper.cpp:216-217) instead of packed bits (our extension).
    ``only`` (iterable of level names) restricts which joins are *scored*; kept levels needed as inputs always run.
    """
    from . import synth

    net = workload.net
    lv = net.levels
    n = workload.n_patients

    def uids(level):
        return uidrelset_cls(level.path_length, level.src, level.trg, level.count, level.location, level.signs)

    def loaded(bits):
        ps = ex.createPathSet(bits.shape[0])
        if use_int_matrices:
            ps.load(synth.unpack_bits(bits, n))
        else:
            ps.load_bits(bits)
        return ps

    results, kept = {}, {}

    def run(name, p0, p1, res):
        r = ex.join(uids(lv[name]), p0, p1, res)
        results[name] = r
        if on_level is not None:
            on_level(name, r)
        return r

    data1 = loaded(workload.gene_bits)
    zero_set = ex.createPathSet(0)
    # level 1 (src/wrapper.cpp:225-244)
    paths1 = ex.createPathSet(lv["1a"].n_pairs)
    run("1a", ex.createPathSet(lv["1a"].n_uids), data1.select(net.data_idx["1a"]), paths1)
    kept["paths1"] = paths1
    if only is None or "1b" in only:
        data2 = loaded(workload.gene_bits2)
        run("1b", ex.createPathSet(lv["1b"].n_uids), data2.select(net.data_idx["1b"]), zero_set)
    if path_length >= 2:  # src/wrapper.cpp:246-253
        paths2 = ex.createPathSet(lv["2"].n_pairs)
        run("2", paths1, data1.select(net.data_idx["2"]), paths2)
        kept["paths2"] = paths2
    if path_length >= 3:  # src/wrapper.cpp:255-262
        paths3 = ex.createPathSet(lv["3"].n_pairs)
        run("3", paths2, data1.select(net.data_idx["3"]), paths3)
        kept["paths3"] = paths3
    if path_length >= 4 and (only is None or "4" in only):  # src/wrapper.cpp:264-269
        run("4", paths3, paths2, zero_set)
    if path_length >= 5 and (only is None or "5" in only):  # src/wrapper.cpp:271-276
        run("5", paths3, paths3, zero_set)
    return results, kept


def replay_permutation_batches(ex, uidrelset_cls, workload, path_length: int, n_perms: int, seed: int, first_perm: int = 0):
    """Score the levels against permutations ``first_perm .. first_perm + n_perms - 1`` of ``seed`` in batches of
    ``ex.iters_requested``, the masks made on the device (``generatePermutedMasks``): no host mask at any permutation count.

    Batch b holds permutations ``first_perm + b * I ...`` (I = ``ex.iters_requested``).  Returns ``{level: joined_res}`` with the
    batches' maxima concatenated and cut to ``n_perms``, and the top-K, which does not depend on the permutations (checked:
    every batch must give the same).  ``ex`` must already hold the value table (and any strata).
    """
    per = int(ex.iters_requested)
    if per <= 0:
        raise ValueError("the exec scores no permutations")
    out, perms = {}, {}
    for b in range(-(-int(n_perms) // per)):
        ex.generatePermutedMasks(seed, first_perm + b * per)
        results, _ = replay_levels(ex, uidrelset_cls, workload, path_length)
        for name, r in results.items():
            top = [(s.score, s.src, s.trg, s.cases, s.ctrls) for s in r.scores]
            if name in out:
                if top != out[name]:
                    raise RuntimeError(f"level {name}: the top-K of permutation batch {b} differs from batch 0's")
            else:
                out[name] = top
                perms[name] = (r, [])
            perms[name][1].append(np.asarray(r.permuted_scores, dtype=np.float64))
    return {name: type(r)(r.scores, np.concatenate(ps)[: int(n_perms)]) for name, (r, ps) in perms.items()}
