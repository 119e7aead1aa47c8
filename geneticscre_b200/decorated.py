"""Decorated p-values of the reported top-K paths (SURVEY section 8 row f4; reference: R/DecoratedPvalue.R:49-304).

For every top-K path of length L and every split point, the path is cut into a sub-path (the first j genes, or the last
ones for the backward direction) and the next gene; the carriers that gene ADDS to the sub-path are re-drawn uniformly
without replacement among the patients the sub-path does not cover, the path is re-scored from the value table, and the
decorated p-value is the share of redraws scoring at least as high as the real path (computeDecoratedPvalue,
R/DecoratedPvalue.R:198-304).

The exact limit also runs on the GPU (csrc/decorated.cuh: one CTA per split, AND + popcount for the eight counts,
hypergeometric weights by the ratio recurrence, value-table look-ups over the support): `decorated_exact_device` for splits
packed on the host, and `decorated_pvalues_device` for whole top-K lists whose splits are formed on the device from the gene
rows already there (`synth.path_genes` maps a level's scores to genes and signs), non-stratified or stratified under the
exec's permutation strata.  The Monte-Carlo mode is a host utility.  Only
the number of redrawn carriers that fall among the cases matters, and that number is hypergeometric, so besides the
reference's Monte-Carlo estimate (`n_permutations` redraws; R's `sample()` stream cannot be reproduced, a seeded numpy
generator is used) the exact limit of that estimate is available (`n_permutations=None`): the tail probability is summed
over the support of the (independent) positive and negative hypergeometric counts.

Stratified resampling (`strata=`, R/DecoratedPvalue.R:236-268): the added carriers are redrawn inside their own stratum.
Per stratum the pool is the stratum minus every carrier of the sub-path (positive or negative part); as many patients as
the gene adds positive carriers in that pool are drawn, then - from what is left of the pool - as many as it adds negative
carriers.  So per stratum the case count of the positive draw is hypergeometric and that of the negative draw is
hypergeometric given the first; the strata are independent and their counts add up.  The Monte-Carlo mode samples exactly
that; the exact mode convolves the per-stratum joint distributions.  (Added carriers that sit in the other part of the
sub-path belong to no pool and are not redrawn, as in the reference.)
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np


def _hypergeom_pmf(n_good: int, n_bad: int, n_draw: int) -> tuple[np.ndarray, np.ndarray]:
    """Support and probabilities of the number of 'good' items among n_draw drawn without replacement."""
    from scipy.special import gammaln

    lo, hi = max(0, n_draw - n_bad), min(n_draw, n_good)
    x = np.arange(lo, hi + 1)

    def lch(a, b):
        return gammaln(a + 1.0) - gammaln(b + 1.0) - gammaln(a - b + 1.0)

    logp = lch(n_good, x) + lch(n_bad, n_draw - x) - lch(n_good + n_bad, n_draw)
    p = np.exp(logp)
    return x, p / p.sum()


@dataclass
class DecoratedResult:
    decorated_pvalue: float
    cases1: int
    controls1: int
    cases2: int
    controls2: int
    score: float


def _stratified_counts(pool_case, pool_ctrl, k_pos, k_neg, n_permutations, rng):
    """Monte-Carlo (cp, cn) totals over strata: per stratum cp_g ~ Hyp(cases, ctrls, k_pos_g); the negatives are drawn from
    what is left and count CONTROLS: cn_g ~ Hyp(ctrls - (k_pos_g - cp_g), cases - cp_g, k_neg_g)."""
    cp = np.zeros(n_permutations, dtype=np.int64)
    cn = np.zeros(n_permutations, dtype=np.int64)
    for c, d, kp, kn in zip(pool_case, pool_ctrl, k_pos, k_neg):
        cpg = rng.hypergeometric(c, d, kp, size=n_permutations) if kp else np.zeros(n_permutations, dtype=np.int64)
        cp += cpg
        if kn:
            good, bad = d - (kp - cpg), c - cpg
            cn += rng.hypergeometric(good, bad, kn)
    return cp, cn


def _stratified_joint_pmf(pool_case, pool_ctrl, k_pos, k_neg):
    """Exact joint distribution P[cp, cn] of the totals (2-D convolution of the per-stratum joints)."""
    joint = np.ones((1, 1))
    for c, d, kp, kn in zip(pool_case, pool_ctrl, k_pos, k_neg):
        g = np.zeros((kp + 1, kn + 1))
        xp, pp = _hypergeom_pmf(c, d, kp)
        for x, px in zip(xp, pp):
            xn, pn = _hypergeom_pmf(d - (kp - x), c - x, kn)
            g[x, xn] += px * pn
        out = np.zeros((joint.shape[0] + kp, joint.shape[1] + kn))
        for i in range(kp + 1):  # strata are few and their draws small: a direct convolution is plenty
            for j in range(kn + 1):
                if g[i, j]:
                    out[i:i + joint.shape[0], j:j + joint.shape[1]] += g[i, j] * joint
        joint = out
    return joint


def compute_decorated_pvalue(pos1, neg1, pos2, neg2, n_cases: int, n_ctrls: int, method: int, value_table: np.ndarray,
                             n_permutations: int | None = None, rng: np.random.Generator | None = None, strata=None) -> DecoratedResult:
    """computeDecoratedPvalue (R/DecoratedPvalue.R:198-304) for boolean patient vectors (cases first).

    pos1/neg1: carriers of the sub-path (positive / negative part); pos2/neg2: carriers of the gene being added.
    strata: optional stratum label per patient (the `stratum` column of the reference's strata file, in patient order).
    """
    pos1, neg1, pos2, neg2 = (np.asarray(v, dtype=bool) for v in (pos1, neg1, pos2, neg2))
    n = n_cases + n_ctrls
    is_case = np.arange(n) < n_cases
    pos2 = pos2 & ~pos1  # only what the gene adds (R/DecoratedPvalue.R:206-209)
    neg2 = neg2 & ~neg1
    # counts as in R/DecoratedPvalue.R:218-225: the negative part counts controls as "cases"
    case_pos1, case_neg1 = int((pos1 & is_case).sum()), int((neg1 & ~is_case).sum())
    ctrl_pos1, ctrl_neg1 = int((pos1 & ~is_case).sum()), int((neg1 & is_case).sum())
    case_pos2, case_neg2 = int((pos2 & is_case).sum()), int((neg2 & ~is_case).sum())
    ctrl_pos2, ctrl_neg2 = int((pos2 & ~is_case).sum()), int((neg2 & is_case).sum())
    vt = np.asarray(value_table)

    def score_of(cp, tp, cn, tn):
        """cp of tp redrawn positive carriers are cases; cn of tn redrawn negative carriers are controls."""
        if method == 1:  # R/DecoratedPvalue.R:226-227, 285-286
            return vt[case_pos1 + cp + case_neg1 + cn, ctrl_pos1 + (tp - cp) + ctrl_neg1 + (tn - cn)]
        return vt[case_pos1 + cp, ctrl_pos1 + (tp - cp)] + vt[case_neg1 + cn, ctrl_neg1 + (tn - cn)]  # :228-229, :287-288

    k_pos, k_neg = int(pos2.sum()), int(neg2.sum())
    score = float(score_of(case_pos2, k_pos, case_neg2, k_neg))
    # pools the carriers are redrawn from (R/DecoratedPvalue.R:232-233): everything outside the sub-path
    good_pos, bad_pos = int((~pos1 & is_case).sum()), int((~pos1 & ~is_case).sum())    # "good" = a case
    good_neg, bad_neg = int((~neg1 & ~is_case).sum()), int((~neg1 & is_case).sum())    # "good" = a control
    if strata is not None:
        strata = np.asarray(strata)
        if strata.shape[0] != n:
            raise ValueError("one stratum label per patient is required")
        free = ~(pos1 | neg1)  # R/DecoratedPvalue.R:240-242: the stratum minus every carrier of the sub-path
        groups = list(dict.fromkeys(strata.tolist()))  # unique(), in order of appearance (R/DecoratedPvalue.R:80)
        pool_case = [int((free & (strata == g) & is_case).sum()) for g in groups]
        pool_ctrl = [int((free & (strata == g) & ~is_case).sum()) for g in groups]
        kp = [int((pos2 & free & (strata == g)).sum()) for g in groups]
        kn = [int((neg2 & free & (strata == g)).sum()) for g in groups]
        for c, d, a_, b_ in zip(pool_case, pool_ctrl, kp, kn):
            if a_ + b_ > c + d:  # R's sample() stops with "cannot take a sample larger than the population"
                raise ValueError("a stratum has fewer free patients than carriers to redraw")
        tp, tn = sum(kp), sum(kn)  # (carriers outside every pool are not redrawn)
        if n_permutations is None:
            joint = _stratified_joint_pmf(pool_case, pool_ctrl, kp, kn)
            cp_ax, cn_ax = np.arange(joint.shape[0]), np.arange(joint.shape[1])
            sc = score_of(cp_ax[:, None], tp, cn_ax[None, :], tn)
            pvalue = float(joint[(sc >= score) & (joint > 0)].sum())
        else:
            rng = rng or np.random.default_rng(0)
            cp, cn = _stratified_counts(pool_case, pool_ctrl, kp, kn, n_permutations, rng)
            pvalue = float((score_of(cp, tp, cn, tn) >= score).mean())
    elif n_permutations is None:
        xp, pp = _hypergeom_pmf(good_pos, bad_pos, k_pos)
        xn, pn = _hypergeom_pmf(good_neg, bad_neg, k_neg)
        s = score_of(xp[:, None], k_pos, xn[None, :], k_neg)
        pvalue = float((pp[:, None] * pn[None, :])[s >= score].sum())
    else:
        rng = rng or np.random.default_rng(0)
        cp = rng.hypergeometric(good_pos, bad_pos, k_pos, size=n_permutations) if k_pos else np.zeros(n_permutations, dtype=np.int64)
        cn = rng.hypergeometric(good_neg, bad_neg, k_neg, size=n_permutations) if k_neg else np.zeros(n_permutations, dtype=np.int64)
        pvalue = float((score_of(cp, k_pos, cn, k_neg) >= score).mean())  # R/DecoratedPvalue.R:293
    return DecoratedResult(pvalue, case_pos1 + case_neg1, ctrl_pos1 + ctrl_neg1, case_pos2 + case_neg2, ctrl_pos2 + ctrl_neg2, score)


def decorated_exact_device(ex, splits) -> list[DecoratedResult]:
    """Exact-limit decorated p-values of many splits in one call on the GPU (gcre_exec_decorated_exact, csrc/decorated.cuh).

    ex: a JoinExec holding the value table (its method and cohort sizes are used); splits: iterable of
    (pos1, neg1, pos2, neg2) boolean patient vectors as for :func:`compute_decorated_pvalue`."""
    import ctypes as C

    from . import _lib, synth

    splits = list(splits)
    n = ex.num_cases + ex.num_ctrls
    if not splits:
        return []
    flat = np.stack([np.asarray(v, dtype=bool) for sp in splits for v in sp])
    if flat.shape[1] != n:
        raise ValueError("carrier vectors must have one entry per patient")
    bits = np.ascontiguousarray(synth.pack_bits(flat))  # [4 * items][W64]
    out = (_lib.DecoratedC * len(splits))()
    _lib.check(ex._lib.gcre_exec_decorated_exact(ex._h, bits.ctypes.data_as(C.POINTER(C.c_uint64)), len(splits), out))
    return [DecoratedResult(o.pvalue, o.cases1, o.ctrls1, o.cases2, o.ctrls2, o.score) for o in out]


def _split_labels(L: int) -> list[dict]:
    """direction / subpath1 / subpath2 of a path's splits (R/DecoratedPvalue.R:123-180): forward, then backward."""
    labels = [{"direction": "Forward", "subpath1": list(range(j)), "subpath2": j} for j in range(1, L)]
    labels += [{"direction": "Backward", "subpath1": list(range(L - 1, j - 1, -1)), "subpath2": j - 1} for j in range(L - 1, 0, -1)]
    return labels


def decorated_pvalues_device(ex, gene_set, genes, signs, lengths, stratified: bool = False) -> list[list[dict]]:
    """Exact decorated p-values of many paths in one device call (gcre_exec_decorated_paths, csrc/decorated.cuh).

    ex: a JoinExec holding the value table; gene_set: a PathSet of ``ex`` whose rows are the genes (data1);
    genes / signs: int [k][<= 5] per path (gene rows in path order, +1 / -1 cumulative signs as :func:`synth.path_genes` gives);
    lengths: int [k].  stratified: redraw inside the strata set by ``ex.setPermutationStrata`` (one stratum when none is set).
    Returns per path what :func:`decorated_pvalues_for_path` returns for it (same labels, order and fields)."""
    import ctypes as C

    from . import _lib

    lengths = np.ascontiguousarray(np.atleast_1d(lengths), dtype=np.int32)
    k = lengths.shape[0]
    g = np.zeros((k, 5), dtype=np.int32)
    sg = np.zeros((k, 5), dtype=np.int32)
    gin, sin = (np.asarray(v, dtype=np.int32).reshape(k, -1) if k else np.zeros((0, 5), np.int32) for v in (genes, signs))
    if gin.shape[1] > 5 or sin.shape[1] > 5:
        raise ValueError("paths have at most 5 genes")
    g[:, :gin.shape[1]] = gin
    sg[:, :sin.shape[1]] = sin
    out = (_lib.DecoratedC * (8 * max(k, 1)))()
    i32 = C.POINTER(C.c_int32)
    _lib.check(ex._lib.gcre_exec_decorated_paths(ex._h, gene_set._h, g.ctypes.data_as(i32), sg.ctypes.data_as(i32), lengths.ctypes.data_as(i32),
                                                 k, 1 if stratified else 0, out))
    res = []
    for i in range(k):
        labels = _split_labels(int(lengths[i]))
        res.append([{**lab, **DecoratedResult(o.pvalue, o.cases1, o.ctrls1, o.cases2, o.ctrls2, o.score).__dict__}
                    for lab, o in zip(labels, out[8 * i:8 * i + len(labels)])])
    return res


def decorated_pvalues_for_path(gene_rows: np.ndarray, signs, n_cases: int, n_ctrls: int, method: int, value_table: np.ndarray,
                               n_permutations: int | None = None, rng: np.random.Generator | None = None, strata=None,
                               device_exec=None) -> list[dict]:
    """All forward and backward splits of one path (R/DecoratedPvalue.R:123-180).

    gene_rows: bool/0-1 array [L][n] of the path's genes in order; signs: +1/-1 per gene (method 2 moves the genes with a
    negative sign to the negative part, R/DecoratedPvalue.R:129-132).
    """
    rows = np.asarray(gene_rows) != 0
    L = rows.shape[0]
    signs = np.asarray(signs)
    pos = rows.copy()
    neg = np.zeros_like(rows)
    if method == 2:
        neg[signs == -1] = rows[signs == -1]
        pos[signs == -1] = False
    splits = [(pos[:j].any(0), neg[:j].any(0), pos[j], neg[j]) for j in range(1, L)]  # forward: genes 1..j, then gene j+1
    splits += [(pos[j:].any(0), neg[j:].any(0), pos[j - 1], neg[j - 1]) for j in range(L - 1, 0, -1)]  # backward: genes L..j+1, then gene j
    labels = _split_labels(L)
    if device_exec is not None:  # all splits of the path in one kernel launch (exact mode, no strata)
        if n_permutations is not None or strata is not None:
            raise ValueError("the device path computes the exact, non-stratified limit")
        results = decorated_exact_device(device_exec, splits)
    else:
        results = [compute_decorated_pvalue(*sp, n_cases, n_ctrls, method, value_table, n_permutations, rng, strata) for sp in splits]
    return [{**lab, **r.__dict__} for lab, r in zip(labels, results)]
