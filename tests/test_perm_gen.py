"""CPU tests of the seeded permutation-mask generator's definition (synth.make_perm_masks_philox, the numpy restatement the
device generator is held to bit for bit): Philox known answers, exact per-stratum case counts, relabelling and batch
invariance, and the null distribution (uniform case sets, within strata too, uniform marginals, independent rows)."""
import itertools
import math

import numpy as np
import pytest
from scipy import stats

from geneticscre_b200 import synth

P_FLOOR = 1e-4  # fixed seeds: each statistical check passes deterministically; the floor says how far off a failure would be


def unpack(masks, n):
    return np.unpackbits(masks.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(bool)


def set_index(masks, n, k):
    """row -> index of its case set among all C(n, k) sets (n <= 64)"""
    sets = np.array(sorted(sum(1 << i for i in c) for c in itertools.combinations(range(n), k)), dtype=np.uint64)
    idx = np.searchsorted(sets, masks[:, 0])
    assert (sets[idx] == masks[:, 0]).all(), "a row has the wrong number of cases"
    return idx, sets.shape[0]


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    """Random123's known-answer vectors of Philox4x32-10."""
    got = synth.philox4x32_10(*ctr, *key)
    assert tuple(int(x) for x in got) == want


@pytest.mark.parametrize("nc,nt,strata", [(1, 1, None), (5, 58, None), (64, 1, None), (33, 32, None), (70, 130, None),
                                          (70, 130, "3"), (37, 63, "37"), (500, 501, "stairs")])
def test_exact_counts_per_stratum_and_no_tail_bits(nc, nt, strata):
    n = nc + nt
    rng = np.random.default_rng(n)
    lab = None
    if strata == "stairs":
        lab = np.arange(n) // 7  # strata of 7 consecutive patients, some all cases, some all controls, one mixed
    elif strata is not None:
        lab = rng.integers(-1000, 1000, size=int(strata))[rng.integers(0, int(strata), size=n)]
    masks = synth.make_perm_masks_philox(nc, nt, 300, seed=0xC0FFEE, first_perm=11, strata=lab)
    assert masks.shape == (300, synth.words_for(n)) and masks.dtype == np.uint64
    if n % 64:
        assert not (masks[:, -1] >> np.uint64(n % 64)).any(), "bits at patient indices >= n"
    case = unpack(masks, n)
    lab = np.zeros(n, int) if lab is None else lab
    for g in np.unique(lab):
        sel = lab == g
        assert (case[:, sel].sum(1) == sel[:nc].sum()).all(), f"stratum {g} lost its case count"
    assert len({r.tobytes() for r in masks}) > 1 or n <= 2


def test_relabelled_strata_give_identical_masks():
    rng = np.random.default_rng(3)
    lab = rng.integers(0, 9, size=300)
    perm_labels = rng.permutation(9) * 1000 - 4000  # a bijection onto other, negative and sparse, label values
    a = synth.make_perm_masks_philox(120, 180, 64, seed=5, strata=lab)
    b = synth.make_perm_masks_philox(120, 180, 64, seed=5, strata=perm_labels[lab])
    assert np.array_equal(a, b)
    c = synth.make_perm_masks_philox(120, 180, 64, seed=5, strata=np.zeros(300, np.int32) + 7)
    assert np.array_equal(c, synth.make_perm_masks_philox(120, 180, 64, seed=5)), "one stratum is no strata"
    assert not np.array_equal(a, c)


@pytest.mark.parametrize("seed", [0, 12345, 0xDEADBEEF00000001, 2**64 - 1])
@pytest.mark.parametrize("a,p,q", [(0, 7, 13), (2**32 - 5, 3, 9), (2**32 - 1, 1, 1), (2**40 + 17, 10, 30), (2**64 - 4, 3, 1)])
def test_batches_concatenate(seed, a, p, q):
    """Permutation r is a function of (seed, r) alone: (a, p + q) == (a, p) ++ (a + p, q), across r = 2^32 and with the
    seed's high word set."""
    whole = synth.make_perm_masks_philox(40, 37, p + q, seed, first_perm=a)
    parts = np.concatenate([synth.make_perm_masks_philox(40, 37, p, seed, first_perm=a),
                            synth.make_perm_masks_philox(40, 37, q, seed, first_perm=(a + p) % 2**64)])
    assert np.array_equal(whole, parts)
    one = synth.make_perm_masks_philox(40, 37, 1, seed, first_perm=(a + p) % 2**64)
    assert np.array_equal(whole[p], one[0])


def test_seed_words_and_counter_words_matter():
    base = synth.make_perm_masks_philox(50, 50, 4, 1)
    for other in (synth.make_perm_masks_philox(50, 50, 4, 1 + 2**32), synth.make_perm_masks_philox(50, 50, 4, 1, first_perm=2**32),
                  synth.make_perm_masks_philox(50, 50, 4, 2)):
        assert not (base == other).all(axis=1).any()


def test_uniform_over_all_case_sets():
    """n = 12, 5 cases: 200,000 rows against the 792 equally likely case sets."""
    masks = synth.make_perm_masks_philox(5, 7, 200_000, seed=20261020)
    idx, cells = set_index(masks, 12, 5)
    assert cells == math.comb(12, 5)
    p = stats.chisquare(np.bincount(idx, minlength=cells)).pvalue
    assert p > P_FLOOR, p


def test_uniform_within_strata():
    """Two strata of 6 patients, 3 and 2 true cases: the joint case sets (20 x 15 = 300 cells) are uniform - uniform within
    each stratum and independent across them."""
    lab = np.array([0, 0, 0, 1, 1, 1, 0, 0, 0, 1, 1, 1])
    masks = synth.make_perm_masks_philox(5, 7, 200_000, seed=99, strata=lab)
    case = unpack(masks, 12)
    assert (case[:, lab == 0].sum(1) == 3).all() and (case[:, lab == 1].sum(1) == 2).all()
    ids = []
    for g, k in ((0, 3), (1, 2)):
        sub = synth.pack_bits(case[:, lab == g].astype(np.int32))
        ids.append(set_index(sub, 6, k)[0])
    joint = ids[0] * 15 + ids[1]
    p = stats.chisquare(np.bincount(joint, minlength=300)).pvalue
    assert p > P_FLOOR, p


@pytest.mark.parametrize("strata", [None, "two"])
def test_per_patient_marginals(strata):
    """Every patient is a case with probability k_g / |g| (Bonferroni over the patients)."""
    n, nc, rows = 101, 40, 50_000
    lab = None if strata is None else (np.arange(n) % 3 == 0).astype(int)
    case = unpack(synth.make_perm_masks_philox(nc, n - nc, rows, seed=4242, first_perm=2**33, strata=lab), n)
    lab = np.zeros(n, int) if lab is None else lab
    prob = np.array([(lab[:nc] == lab[i]).sum() / (lab == lab[i]).sum() for i in range(n)])
    z = (case.sum(0) - rows * prob) / np.sqrt(rows * prob * (1 - prob))
    p = min(1.0, n * 2 * stats.norm.sf(np.abs(z).max()))
    assert p > P_FLOOR, (p, np.abs(z).max())


@pytest.mark.parametrize("offset", [0, 1])
def test_consecutive_rows_independent(offset):
    """n = 6, 3 cases: the case sets of rows r and r + 1 (disjoint pairs) fill the 20 x 20 joint table uniformly."""
    masks = synth.make_perm_masks_philox(3, 3, 200_001, seed=77, first_perm=2**32 - 100_000)
    idx, cells = set_index(masks, 6, 3)
    a, b = idx[offset:-1:2], idx[offset + 1::2]
    m = min(a.shape[0], b.shape[0])
    p = stats.chisquare(np.bincount(a[:m] * cells + b[:m], minlength=cells * cells)).pvalue
    assert p > P_FLOOR, p
