"""The identity the tail form of the pre-counted sparse kernel relies on (join_sparse.cuh), checked in numpy on the bench network.

A level-4 pair joins a paths3 row u (g1 -> g2 -> g3) with a paths2 row p (g3 -> t).  The engine records, per kept row, the
data1 row of its last gene and its orientation (tail), and per paths2 row the entry of its first gene (head); a pair may be
scored through gene t alone when the partner's head, oriented by the pair, is u's tail.  Then u | flip(p) == u | orient(t).
This replays that bookkeeping with the formulas of setup_kernels.cuh (record_rows_kernel, tail_eligible_kernel) and checks,
bit for bit and for every level-4 pair of both methods, that every pair is eligible and that the identity holds.
"""
import numpy as np
import pytest

from geneticscre_b200 import synth

# bench.py's default network (WORKLOAD: 15,000 genes, 150,000 edges, seed 20261021) on a small cohort
N_GENES, N_EDGES, SEED, N_CASES, N_CTRLS = 15000, 150000, 20261021, 70, 60


def pairs(level):
    """flattened pairs of a level in join order: (upstream row, partner row)"""
    c = np.maximum(level.count.astype(np.int64), 0)
    idx = np.repeat(np.arange(c.shape[0], dtype=np.int64), c)
    within = np.arange(int(c.sum()), dtype=np.int64) - np.repeat(np.cumsum(c) - c, c)
    loc = np.repeat(level.location.astype(np.int64), c) + within
    return idx, loc


def swapped(level, idx, loc):
    """UidRelSet::need_flip (src/gcre.h:71-81) is false: the partner's halves are swapped"""
    s = level.signs.astype(np.int64)
    if level.path_length > 3:
        sign = s[idx]
    elif level.path_length < 3:
        sign = s[loc]
    else:
        sign = np.where(s[idx] + s[loc] == 0, -1, 1)
    return sign != 1


def orient(rows, swap, m):
    """[k][W] rows -> [k][m*W] with the row in half `swap` (method 2) or as is (method 1)"""
    if m == 1:
        return rows
    w = rows.shape[1]
    out = np.zeros((rows.shape[0], 2 * w), dtype=np.uint64)
    out[~swap, :w] = rows[~swap]
    out[swap, w:] = rows[swap]
    return out


def swap_halves(rows, swap, m):
    if m == 1:
        return rows
    w = rows.shape[1] // 2
    out = rows.copy()
    out[swap] = np.concatenate([rows[swap, w:], rows[swap, :w]], axis=1)
    return out


@pytest.fixture(scope="module")
def workload():
    return synth.make_workload(N_CASES, N_CTRLS, N_GENES, N_EDGES, 1, SEED, max_path_length=4, host_table=False)


@pytest.mark.parametrize("m", [1, 2])
def test_level4_partner_adds_one_gene(workload, m):
    w = workload
    lv, didx, gene = w.net.levels, w.net.data_idx, w.gene_bits

    def keep(level, up_rows, sel_idx, up_tail):
        """a KEEP join whose partner set is data1.select(sel_idx): rows, tails (row, swap) and heads of the result"""
        idx, loc = pairs(lv[level])
        sw = swapped(lv[level], idx, loc) if m == 2 else np.zeros(idx.shape[0], dtype=bool)
        rows = up_rows[idx] | orient(gene[sel_idx[loc]], sw, m)
        tail = (sel_idx[loc].astype(np.int64), sw)
        head = None if up_tail is None else (up_tail[0][idx], up_tail[1][idx])
        return rows, tail, head

    zero = np.zeros((lv["1a"].n_uids, m * gene.shape[1]), dtype=np.uint64)
    paths1, tail1, _ = keep("1a", zero, didx["1a"], None)
    assert np.array_equal(paths1, orient(gene[tail1[0]], tail1[1], m)), "level-1a rows are single genes"
    paths2, tail2, head2 = keep("2", paths1, didx["2"], tail1)
    paths3, tail3, _ = keep("3", paths2, didx["3"], None)

    idx, loc = pairs(lv["4"])
    assert idx.shape[0] > 10_000_000, "the bench's level-4 join"
    for b in range(0, idx.shape[0], 1 << 21):
        i, l = idx[b: b + (1 << 21)], loc[b: b + (1 << 21)]
        sw = swapped(lv["4"], i, l) if m == 2 else np.zeros(i.shape[0], dtype=bool)
        # eligibility (tail_eligible_kernel): the head, oriented by the pair, is the upstream row's tail
        assert np.array_equal(head2[0][l], tail3[0][i])
        if m == 2:
            assert np.array_equal(head2[1][l] ^ sw, tail3[1][i])
        u = paths3[i]
        joined = u | swap_halves(paths2[l], sw, m)
        via_gene = u | orient(gene[tail2[0][l]], tail2[1][l] ^ sw, m)
        assert np.array_equal(joined, via_gene)
