"""Seeded synthetic inputs for the path-join hot path (SURVEY.md section 8d).

Everything the reference's R layer prepares before calling ``ProcessPaths`` is produced here with numpy from a
seed: the cohort (gene x patient carrier bits, cases first), the signed directed gene network, the per-level join
indices, the permutation label masks and the hypergeometric value table.  The index derivation mirrors
R/ProcessPaths.R:206-256 and getRels3 (src/wrapper.cpp:18-48); the permutation matrix mirrors
R/Utils.R:22-46,246-262 (``CaseORControl``: 1 = label kept); the value table mirrors R/Utils.R:137-159.

This module is host-side input preparation only; it performs no scoring.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

NO_LOCATION = np.uint32(0xFFFFFFFF)  # R passes location -1 with count 0 (R/PathMethods.R:147) -> stored in a uint32


def words_for(n_patients: int) -> int:
    """64-bit words per patient bit-vector, unpadded (SURVEY section 8: W64 = ceil(n/64))."""
    return (int(n_patients) + 63) // 64


# ----------------------------------------------------------------------------------------------------------------
# cohort
# ----------------------------------------------------------------------------------------------------------------
def make_cohort_bits(n_patients: int, n_genes: int, seed: int, max_freq: float = 0.05, zero_frac: float = 0.6) -> np.ndarray:
    """Packed carrier bits ``uint64[n_genes][W64]`` (patient c -> word c//64, bit c%64, LSB first).

    Gene carrier frequency is log-uniform in [1/n, max_freq]; ``zero_frac`` of the genes carry nothing (the bundled
    vignette data has 1,831 of 3,000 all-zero genes); carriers are capped at ``max_freq * (n + 1)`` like
    PreprocessTable (R/Utils.R:185-188).
    """
    rng = np.random.default_rng(seed)
    n, w = int(n_patients), words_for(n_patients)
    bits = np.zeros((n_genes, w), dtype=np.uint64)
    cap = int(np.floor(max_freq * (n + 1)))
    freq = np.exp(rng.uniform(np.log(min(1.0 / n, max_freq)), np.log(max_freq), size=n_genes))
    k = np.minimum(rng.binomial(n, freq), cap)
    k[rng.random(n_genes) < zero_frac] = 0
    for g in np.nonzero(k)[0]:
        cols = rng.choice(n, size=int(k[g]), replace=False)
        np.bitwise_or.at(bits[g], cols >> 6, np.uint64(1) << (cols & 63).astype(np.uint64))
    return bits


def unpack_bits(bits: np.ndarray, n_patients: int) -> np.ndarray:
    """``uint64[rows][W]`` -> ``int32[rows][n]`` 0/1 matrix (the IntegerMatrix the R layer passes, SURVEY App. A.1)."""
    b = np.unpackbits(bits.view(np.uint8), axis=1, bitorder="little")
    return b[:, :n_patients].astype(np.int32)


def pack_bits(mat: np.ndarray) -> np.ndarray:
    """``[rows][n]`` (any non-zero = carrier) -> ``uint64[rows][W64]``."""
    rows, n = mat.shape
    w = words_for(n)
    padded = np.zeros((rows, w * 64), dtype=np.uint8)
    padded[:, :n] = mat != 0
    return np.packbits(padded, axis=1, bitorder="little").view(np.uint64).reshape(rows, w)


# ----------------------------------------------------------------------------------------------------------------
# permutations and value table
# ----------------------------------------------------------------------------------------------------------------
def make_perm_matrix(n_cases: int, n_ctrls: int, n_perms: int, seed: int) -> np.ndarray:
    """``CaseORControl`` int32[n_perms][n]: 1 where the permuted column keeps its label (R/Utils.R:246-262)."""
    rng = np.random.default_rng(seed)
    n = n_cases + n_ctrls
    out = np.empty((n_perms, n), dtype=np.int32)
    for r in range(n_perms):
        p = rng.permutation(n)
        out[r, :n_cases] = p[:n_cases] < n_cases
        out[r, n_cases:] = p[n_cases:] >= n_cases
    return out


def make_perm_masks(n_cases: int, n_ctrls: int, n_perms: int, seed: int) -> np.ndarray:
    """Packed permuted case masks ``uint64[n_perms][W64]`` - the same masks ``setPermutedCases`` derives from
    :func:`make_perm_matrix` with the same seed (src/join_base.cpp:85-125), built without the 32x larger int matrix."""
    rng = np.random.default_rng(seed)
    n = n_cases + n_ctrls
    w = words_for(n)
    out = np.zeros((n_perms, w), dtype=np.uint64)
    for r in range(n_perms):
        p = rng.permutation(n)
        case = np.empty(n, dtype=bool)
        case[:n_cases] = p[:n_cases] < n_cases  # kept case stays case; flipped case becomes control
        case[n_cases:] = ~(p[n_cases:] >= n_cases)  # flipped control becomes case
        cols = np.nonzero(case)[0]
        np.bitwise_or.at(out[r], cols >> 6, np.uint64(1) << (cols & 63).astype(np.uint64))
    return out


PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57  # Philox4x32-10 (Salmon et al. 2011): round multipliers
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85  # ... and key increments


def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    """Philox4x32-10 on numpy arrays (any broadcastable shapes) of 32-bit counter words; returns the four output words as uint64
    arrays holding 32-bit values."""
    u32 = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, dtype=np.uint64) & u32 for x in (c0, c1, c2, c3)]
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    m0, m1, s = np.uint64(PHILOX_M0), np.uint64(PHILOX_M1), np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c[0], m1 * c[2]  # exact: 32 x 32 -> 64 bits
        c = [(p1 >> s) ^ c[1] ^ np.uint64(k0), p1 & u32, (p0 >> s) ^ c[3] ^ np.uint64(k1), p0 & u32]
        k0, k1 = (k0 + PHILOX_W0) & 0xFFFFFFFF, (k1 + PHILOX_W1) & 0xFFFFFFFF
    return c


def _perm_strata_plan(n_cases: int, n_ctrls: int, strata=None):
    """(stratum index int64[n], m int64[n], k0 int64[S]) of the seeded generator: patient i's dense stratum, the number of its
    stratum's patients with index >= i, and each stratum's true case count.  Only the partition ``strata`` induces matters."""
    n = n_cases + n_ctrls
    if strata is None:
        g = np.zeros(n, dtype=np.int64)
    else:
        lab = np.asarray(strata)
        if lab.shape != (n,):
            raise ValueError("strata must hold one label per patient")
        g = np.unique(lab, return_inverse=True)[1].reshape(n).astype(np.int64)
    s = int(g.max()) + 1 if n else 0
    seen_after = np.zeros(s, dtype=np.int64)
    m = np.empty(n, dtype=np.int64)
    for i in range(n - 1, -1, -1):  # O(n) once per strata setting
        seen_after[g[i]] += 1
        m[i] = seen_after[g[i]]
    return g, m, np.bincount(g[:n_cases], minlength=s).astype(np.int64)


def make_perm_masks_philox(n_cases: int, n_ctrls: int, n_perms: int, seed: int, first_perm: int = 0, strata=None) -> np.ndarray:
    """Packed case masks ``uint64[n_perms][W64]`` of permutations ``first_perm .. first_perm + n_perms - 1`` of ``seed``: the
    numpy restatement of the device generator (``gcre_exec_generate_permuted_masks``, csrc/perm_gen.cuh), bit for bit.

    Patient i of permutation r draws ``u_i`` from Philox4x32-10 with key (lo32(seed), hi32(seed)) and counter
    (i >> 1, lo32(r), hi32(r), 0): ``x0 | x1 << 32`` for even i, ``x2 | x3 << 32`` for odd i.  Patients are visited in index
    order (sequential selection sampling per stratum); i is a case iff ``mulhi64(u_i, m_i) < k_g``, where m_i counts the
    not-yet-visited patients of i's stratum g (i included) and k_g the cases still to place in g (initially g's patients with
    index < n_cases).  Every row keeps each stratum's true case count; with one stratum every case set is equally likely up to
    < 2^-64 per decision.  Pure numpy, no CUDA library: a CPU-only caller can feed the reference the same masks.
    """
    n = n_cases + n_ctrls
    w = words_for(n)
    out = np.zeros((n_perms, w), dtype=np.uint64)
    if n_perms <= 0 or n == 0:
        return out
    g, m, k0 = _perm_strata_plan(n_cases, n_ctrls, strata)
    seed, first_perm = int(seed) & (2**64 - 1), int(first_perm) & (2**64 - 1)
    pairs = (n + 1) // 2
    j = np.arange(pairs, dtype=np.uint64)[None, :]
    u32, s32 = np.uint64(0xFFFFFFFF), np.uint64(32)
    m_lo = m.astype(np.uint64)[None, :]
    block = max(1, min(n_perms, (1 << 23) // max(pairs, 1)))  # bounds the temporaries to ~ 8 M pairs at a time
    for b0 in range(0, n_perms, block):
        nb = min(block, n_perms - b0)
        r = ((np.arange(nb, dtype=object) + first_perm + b0) % (2**64)).astype(np.uint64)[:, None]
        x0, x1, x2, x3 = philox4x32_10(j, r & u32, r >> s32, np.uint64(0), seed, seed >> 32)
        u = np.empty((nb, 2 * pairs), dtype=np.uint64)
        u[:, 0::2] = x0 | (x1 << s32)
        u[:, 1::2] = x2 | (x3 << s32)
        u = u[:, :n]
        # mulhi64(u, m) for m < 2^32, exactly: (hi32(u) * m + ((lo32(u) * m) >> 32)) >> 32
        v = (((u >> s32) * m_lo + (((u & u32) * m_lo) >> s32)) >> s32).astype(np.int64).T.copy()  # [n][nb]
        k = np.repeat(k0[:, None], nb, axis=1)  # [S][nb]
        case = np.empty((n, nb), dtype=bool)
        for i in range(n):
            kg = k[g[i]]
            sel = v[i] < kg
            case[i] = sel
            kg -= sel
        out[b0 : b0 + nb] = pack_bits(case.T)
    return out


def log_factorials(n: int) -> np.ndarray:
    """log(k!) for k = 0..n from libm's lgamma (math.lgamma) - the same routine the engine's host code calls
    (gcre_log_factorial_table: std::lgamma), so the device generator and this restatement start from identical doubles.
    Pure Python on purpose: input preparation must not need the CUDA library (the CPU reference arm of bench.py uses it)."""
    import math

    return np.array([math.lgamma(k + 1.0) for k in range(n + 1)], dtype=np.float64)


VT_TIE_TOL = 1e-7  # as csrc/value_table.cuh: outcomes whose probabilities agree to 1e-7 relative are ties (R's fisher.test relErr)


def make_value_table(n_cases: int, n_ctrls: int) -> np.ndarray:
    """float64[(n_cases+1)][(n_ctrls+1)]: -log(two-sided hypergeometric p) (R/Utils.R:137-159).

    For every total i the number of cases among i carriers is hypergeometric; the two-sided p of an outcome is the sum of
    all probabilities <= its own; infinities are replaced by (max finite + 1).  Log-probabilities come from a
    log-factorial table (math.lgamma) and the "<= own" selection is made on the log-probabilities with the tie tolerance
    VT_TIE_TOL: exact ties between outcomes are common and belong to the sum when the reference's expression is evaluated
    exactly (its own float comparison keeps or drops them by dhyper's last-bit rounding).  tests/test_value_table.py pins this
    function and the device generator (csrc/value_table.cuh) to an exact big-integer evaluation and to scipy.stats.hypergeom.
    """
    n = n_cases + n_ctrls
    lf = log_factorials(n)
    table = np.full((n_cases + 1, n_ctrls + 1), np.nan)
    for i in range(n + 1):
        lo, hi = max(0, i - n_ctrls), min(i, n_cases)
        x = np.arange(lo, hi + 1)
        a = (lf[n_cases] - lf[x]) - lf[n_cases - x]
        b = (lf[n_ctrls] - lf[i - x]) - lf[n_ctrls - (i - x)]
        c = (lf[n] - lf[i]) - lf[n - i]
        logp = (a + b) - c
        order = np.argsort(logp, kind="stable")
        ls = logp[order]
        csum = np.cumsum(np.exp(ls))
        last = np.searchsorted(ls, ls + VT_TIE_TOL, side="right") - 1  # last sorted position with a probability <= own (ties included)
        two = np.empty_like(logp)
        two[order] = csum[last]
        with np.errstate(divide="ignore"):
            table[x, i - x] = -np.log(two)
    fin = np.isfinite(table)
    table[~fin] = table[fin].max() + 1.0
    table[table == 0] = 0.0  # -0.0 (= -log 1) kept as a zero; both signs behave identically downstream (App. A.6)
    return table


def make_test_table(n_cases: int, n_ctrls: int, seed: int) -> np.ndarray:
    """An arbitrary deterministic table with irregular doubles (stresses float rounding / max logic in parity tests)."""
    rng = np.random.default_rng(seed)
    t = rng.gamma(2.0, 3.0, size=(n_cases + 1, n_ctrls + 1))
    t[rng.random(t.shape) < 0.02] = 0.0
    t[rng.random(t.shape) < 0.01] *= -1.0
    return t


# ----------------------------------------------------------------------------------------------------------------
# network and per-level join indices
# ----------------------------------------------------------------------------------------------------------------
@dataclass
class Level:
    """One ``join`` call of the level schedule (src/wrapper.cpp:225-276): the UidRelSet fields plus operand roles."""

    name: str
    path_length: int
    src: np.ndarray  # int32[U]  (gene uids; carried through, unused by the arithmetic)
    trg: np.ndarray  # int32[U]
    count: np.ndarray  # int32[U]
    location: np.ndarray  # uint32[U]
    signs: np.ndarray  # int32[...]
    keep: bool

    @property
    def n_uids(self) -> int:
        return int(self.count.shape[0])

    @property
    def n_pairs(self) -> int:
        return int(self.count.sum(dtype=np.int64))


@dataclass
class Network:
    n_genes: int  # genes in `Ents` order == rows of data1
    edges_src: np.ndarray  # int32[E] indices into Ents, sorted by (src, trg)
    edges_trg: np.ndarray
    edges_sign: np.ndarray  # +1 / -1
    ents2: np.ndarray  # int32[n1'] rows of data2 == source genes of Rels2
    levels: dict = field(default_factory=dict)
    data_idx: dict = field(default_factory=dict)  # '1a','1b','2','3' -> int32 row selectors
    rels3: dict = field(default_factory=dict)


def make_network(n_genes: int, n_edges: int, seed: int, tail: float = 1.2, max_path_length: int = 5) -> Network:
    """Random signed directed network with heavy-tailed degrees, plus the index vectors of all six joins.

    Edges are unique (src, trg), no self loops, sorted by (src, trg) (R/ProcessPaths.R:145-149, 210).  Genes that
    touch no edge are dropped from `Ents` like the R filtering does (R/ProcessPaths.R:160-164), so ``n_genes`` of the
    result can be below the request.
    """
    rng = np.random.default_rng(seed)
    w_out = rng.pareto(tail, n_genes) + 1.0
    w_in = rng.pareto(tail, n_genes) + 1.0
    w_out /= w_out.sum()
    w_in /= w_in.sum()
    want = int(n_edges)
    pairs = np.empty((0, 2), dtype=np.int64)
    while pairs.shape[0] < want:
        m = int((want - pairs.shape[0]) * 1.3) + 16
        s = rng.choice(n_genes, size=m, p=w_out)
        t = rng.choice(n_genes, size=m, p=w_in)
        ok = s != t
        pairs = np.unique(np.concatenate([pairs, np.stack([s[ok], t[ok]], axis=1)]), axis=0)
    if pairs.shape[0] > want:
        pairs = pairs[np.sort(rng.choice(pairs.shape[0], size=want, replace=False))]
    # drop isolated genes and renumber (Ents <- Ents[uid %in% leftuids])
    used = np.unique(pairs)
    remap = -np.ones(n_genes, dtype=np.int64)
    remap[used] = np.arange(used.shape[0])
    pairs = remap[pairs]
    order = np.lexsort((pairs[:, 1], pairs[:, 0]))
    pairs = pairs[order]
    sign = np.where(rng.random(pairs.shape[0]) < 0.7, 1, -1).astype(np.int32)
    net = network_from_edges(int(used.shape[0]), pairs[:, 0], pairs[:, 1], sign, max_path_length=max_path_length)
    net.used_genes = used.astype(np.int64)  # rows of the original cohort that became Ents rows
    return net


def network_from_edges(n_genes: int, src, trg, sign, ents2=None, max_path_length: int = 5) -> Network:
    """Build the join indices for a given edge list (already unique, self-loop free, sorted by (src, trg))."""
    src = np.ascontiguousarray(src, dtype=np.int32)
    trg = np.ascontiguousarray(trg, dtype=np.int32)
    sign = np.ascontiguousarray(sign, dtype=np.int32)
    if ents2 is None:
        ents2 = np.unique(src)
    net = Network(n_genes=int(n_genes), edges_src=src, edges_trg=trg, edges_sign=sign, ents2=np.ascontiguousarray(ents2, dtype=np.int32))
    net.used_genes = np.arange(n_genes, dtype=np.int64)
    _derive_levels(net, max_path_length)
    return net


def _derive_levels(net: Network, max_path_length: int) -> None:
    g, src, trg, sign = net.n_genes, net.edges_src, net.edges_trg, net.edges_sign
    e = src.shape[0]
    outdeg = np.bincount(src, minlength=g).astype(np.int32)
    first = np.zeros(g, dtype=np.int64)
    first[1:] = np.cumsum(outdeg)[:-1]
    loc_of_gene = np.where(outdeg > 0, first, -1).astype(np.int64).astype(np.uint32)  # -1 -> 0xFFFFFFFF

    genes = np.arange(g, dtype=np.int32)
    ones = np.ones(g, dtype=np.int32)
    # level 1a: one uid per gene of Ents, partner = its own row (R/ProcessPaths.R:212-218)
    net.levels["1a"] = Level("1a", 1, genes, genes, ones.copy(), genes.astype(np.uint32), ones.copy(), keep=True)
    net.data_idx["1a"] = genes.copy()
    # level 1b: source genes of Rels2 against data2 (R/ProcessPaths.R:220-224)
    n2 = net.ents2.shape[0]
    k2 = np.arange(n2, dtype=np.int32)
    net.levels["1b"] = Level("1b", 1, net.ents2.copy(), net.ents2.copy(), np.ones(n2, np.int32), k2.astype(np.uint32),
                             np.ones(n2, np.int32), keep=False)
    net.data_idx["1b"] = k2.copy()
    # level 2: per gene, its out-edges; operand rows = target gene of each edge (R/ProcessPaths.R:226-230)
    net.levels["2"] = Level("2", 2, genes, genes, outdeg.copy(), loc_of_gene.copy(), sign.copy(), keep=True)
    net.data_idx["2"] = trg.copy()
    # level 3: per edge, the out-edges of its target (R/ProcessPaths.R:232-236)
    net.levels["3"] = Level("3", 3, src.copy(), trg.copy(), outdeg[trg].copy(), loc_of_gene[trg].copy(), sign.copy(), keep=True)
    net.data_idx["3"] = trg.copy()
    if max_path_length < 4:
        return
    # Rels3 in getRels3 order (src/wrapper.cpp:32-45): for edge i, for j in [loc, loc+count)
    cnt3 = outdeg[trg].astype(np.int64)
    p3 = int(cnt3.sum())
    e_i = np.repeat(np.arange(e, dtype=np.int64), cnt3)
    start = np.repeat(first[trg], cnt3)
    within = np.arange(p3, dtype=np.int64) - np.repeat(np.cumsum(cnt3) - cnt3, cnt3)
    e_j = start + within
    g1, g2, g3 = src[e_i], trg[e_i], trg[e_j]
    third_sign = (sign[e_i] * sign[e_j]).astype(np.int32)  # R/ProcessPaths.R:243-245
    net.rels3 = {"g1": g1, "g2": g2, "g3": g3, "sign": third_sign, "e_i": e_i, "e_j": e_j}
    # level 4: per 3-path, out-edges of its third gene; operand = paths2 (R/ProcessPaths.R:247-250)
    net.levels["4"] = Level("4", 4, g1.copy(), g3.copy(), outdeg[g3].copy(), loc_of_gene[g3].copy(), third_sign.copy(), keep=False)
    if max_path_length < 5:
        return
    # level 5: per 3-path, the 3-paths that start at its third gene; operand = paths3 (R/ProcessPaths.R:253-256)
    p3_from = np.bincount(g1, minlength=g).astype(np.int32)
    first3 = np.zeros(g, dtype=np.int64)
    first3[1:] = np.cumsum(p3_from)[:-1]
    loc3 = np.where(p3_from > 0, first3, -1).astype(np.int64).astype(np.uint32)
    net.levels["5"] = Level("5", 5, g1.copy(), g3.copy(), p3_from[g3].copy(), loc3[g3].copy(), third_sign.copy(), keep=False)


@dataclass
class Workload:
    """Everything one GWASPA run hands to the join path."""

    n_cases: int
    n_ctrls: int
    n_perms: int
    gene_bits: np.ndarray  # uint64[n_genes][W64] rows in Ents order (data1)
    gene_bits2: np.ndarray  # uint64[n1'][W64] rows of data2
    perm_masks: np.ndarray  # uint64[n_perms][W64]
    value_table: np.ndarray  # float64[(n_cases+1)][(n_ctrls+1)]
    net: Network

    @property
    def n_patients(self) -> int:
        return self.n_cases + self.n_ctrls


def make_workload(n_cases: int, n_ctrls: int, n_genes: int, n_edges: int, n_perms: int, seed: int,
                  max_path_length: int = 5, real_table: bool = True, max_freq: float = 0.05, zero_frac: float = 0.6,
                  host_table: bool = True) -> Workload:
    """``host_table=False`` leaves ``value_table`` as None: the caller generates it on the device
    (``JoinExec.generateValueTable``), which is the only practical way for n >= 50,000."""
    n = n_cases + n_ctrls
    net = make_network(n_genes, n_edges, seed + 1, max_path_length=max_path_length)
    bits_all = make_cohort_bits(n, n_genes, seed + 2, max_freq=max_freq, zero_frac=zero_frac)
    bits = np.ascontiguousarray(bits_all[net.used_genes])
    bits2 = np.ascontiguousarray(bits[net.ents2])
    masks = make_perm_masks(n_cases, n_ctrls, n_perms, seed + 3)
    table = None if not host_table else (make_value_table(n_cases, n_ctrls) if real_table else make_test_table(n_cases, n_ctrls, seed + 4))
    return Workload(n_cases, n_ctrls, n_perms, bits, bits2, masks, table, net)
