"""synth.path_genes: a level's top-K scores mapped back to the genes and cumulative signs of their paths (the inverse of the row
layouts of synth._derive_levels), checked against the scores the CPU oracle's joins report for those paths."""
import numpy as np
import pytest

from geneticscre_b200 import decorated, schedule, synth


def oracle_replay(oracles, w, method, top_k):
    ex = oracles.OracleExec(method, w.n_cases, w.n_ctrls, w.n_perms)
    ex.top_k = top_k
    ex.setValueTable(w.value_table)
    ex.setPermutedMasks(w.perm_masks)
    res, _ = schedule.replay_levels(ex, oracles.UidRelSet, w, 5)
    return res


@pytest.fixture(scope="module")
def workload():
    return synth.make_workload(60, 70, 40, 160, 8, seed=3, max_path_length=5, real_table=True, max_freq=0.15, zero_frac=0.2)


@pytest.mark.parametrize("method", ["method1", "method2"])
def test_last_forward_split_reproduces_the_join_score(oracles, workload, method):
    """For every top-K path of levels 2-5, the last forward split (the whole path) scores what the join scored, and its counts
    add up to the join's cases / controls."""
    w = workload
    n = w.n_patients
    m = 1 if method == "method1" else 2
    rows = synth.unpack_bits(w.gene_bits, n).astype(bool)
    res = oracle_replay(oracles, w, method, 40)
    checked = mismatches = 0
    for lv in ("2", "3", "4", "5"):
        sc = [s for s in res[lv].scores if s.src >= 0]
        assert sc, lv
        genes, signs, lengths = synth.path_genes(w.net, lv, [s.src for s in sc], [s.trg for s in sc])
        assert (lengths == int(lv)).all()
        for s, g, sg, L in zip(sc, genes, signs, lengths):
            d = decorated.decorated_pvalues_for_path(rows[g[:L]], sg[:L], w.n_cases, w.n_ctrls, m, w.value_table)
            last = [x for x in d if x["direction"] == "Forward"][-1]
            checked += 1
            mismatches += not (last["score"] == s.score and last["cases1"] + last["cases2"] == s.cases
                               and last["controls1"] + last["controls2"] == s.ctrls)
    assert checked >= 100
    assert mismatches == 0


def test_paths_follow_network_edges_with_cumulative_signs(oracles, workload):
    w = workload
    net = w.net
    edge_sign = {(int(a), int(b)): int(c) for a, b, c in zip(net.edges_src, net.edges_trg, net.edges_sign)}
    res = oracle_replay(oracles, w, "method2", 40)
    for lv in ("2", "3", "4", "5"):
        sc = [s for s in res[lv].scores if s.src >= 0]
        genes, signs, lengths = synth.path_genes(net, lv, [s.src for s in sc], [s.trg for s in sc])
        for g, sg, L in zip(genes, signs, lengths):
            assert sg[0] == 1
            for j in range(1, L):
                e = (int(g[j - 1]), int(g[j]))
                assert e in edge_sign, (lv, g, j)
                assert sg[j] == sg[j - 1] * edge_sign[e]
            assert (g[L:] == 0).all() and (sg[L:] == 0).all()


def test_level_one_paths_have_one_gene(workload):
    net = workload.net
    g, s, L = synth.path_genes(net, "1a", [3, 5], [3, 5])
    assert (L == 1).all() and list(g[:, 0]) == [3, 5] and (s[:, 0] == 1).all() and (g[:, 1:] == 0).all()
    k = np.arange(min(4, net.ents2.shape[0]))
    g, s, L = synth.path_genes(net, "1b", k, k)
    assert (L == 1).all() and list(g[:, 0]) == list(net.ents2[k]) and (s[:, 0] == 1).all()


def test_a_sentinel_entry_names_no_path(workload):
    with pytest.raises(ValueError):
        synth.path_genes(workload.net, "3", [0, -1], [0, -1])
    with pytest.raises(ValueError):
        synth.path_genes(workload.net, "6", [0], [0])
