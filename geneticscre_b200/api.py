"""Python mirror of the reference's join class surface, backed by the CUDA engine through the C ABI.

Same names, argument meaning and error behaviour as the reference's C++ classes so that parity tests read like the
reference's own harness (test/harness.cpp:50-181):

    JoinExec(method_name, num_cases, num_ctrls, iters)   src/gcre.h:103-180, src/join_base.cpp:37-59
      .top_k .nthreads .setValueTable .setPermutedCases .createPathSet .join
    PathSet  .size .load .select                          src/gcre_paths.h:10-98
    UidRelSet(path_length, uids, signs)                   src/gcre.h:49-90
    Score, joined_res, uid_ref                            src/gcre_types.h:32-56

Extensions (not in the reference): packed inputs (``load_bits``, ``setPermutedMasks``), seeded permutation masks made on the
device (``setPermutationStrata``, ``generatePermutedMasks``, ``getPermutedMasks``), ``PathSet.to_numpy`` and the
sharding / kernel-selection options of ``join``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import check


@dataclass
class Score:
    score: float = float("-inf")
    src: int = -1
    trg: int = -1
    cases: int = 0
    ctrls: int = 0


@dataclass
class joined_res:
    scores: list
    permuted_scores: np.ndarray
    info: dict | None = None


def _as(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class UidRelSet:
    """UidRelSet(path_length, uids, signs) with the uid_ref fields given as parallel arrays."""

    def __init__(self, path_length, src, trg, count, location, signs, path_idx=None):
        self.path_length = int(path_length)
        self.src, self.trg, self.count = _as(src, np.int32), _as(trg, np.int32), _as(count, np.int32)
        self.location, self.signs = _as(location, np.uint32), _as(signs, np.int32)
        n = self.count.shape[0]
        if path_idx is None:  # running sum of counts, as assemble_uids does (src/wrapper.cpp:128-130)
            c = np.maximum(self.count.astype(np.int64), 0)
            path_idx = np.cumsum(c) - c
        self.path_idx = _as(path_idx, np.uint64)
        self._packed = np.zeros(n, dtype=np.dtype([("src", "<i4"), ("trg", "<i4"), ("count", "<i4"), ("location", "<u4"), ("path_idx", "<u8")]))
        self._packed["src"], self._packed["trg"], self._packed["count"] = self.src, self.trg, self.count
        self._packed["location"], self._packed["path_idx"] = self.location, self.path_idx

        self._resident = None  # (exec, device handle) once make_resident() was called

    def size(self):
        return int(self.count.shape[0])

    def count_total_paths(self):  # src/gcre.h:83-88
        return int(self.count.sum(dtype=np.int64))

    def make_resident(self, ex):
        """Upload the join index to ``ex``'s device once; later joins with this object reuse it (extension)."""
        self.release()
        h = C.c_void_p()
        check(ex._lib.gcre_uidset_create(ex._h, self.path_length, self._packed.ctypes.data_as(C.POINTER(_lib.UidRefC)), self.size(),
                                         _ptr(self.signs, C.c_int32), self.signs.shape[0], C.byref(h)))
        self._resident = (ex, h)
        return self

    def release(self):
        r, self._resident = getattr(self, "_resident", None), None
        if r is not None:  # legal after the exec is gone: gcre_exec_destroy orphans its children
            r[0]._lib.gcre_uidset_destroy(r[1])

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class PathSet:
    def __init__(self, ex, handle):
        self.ex, self._h = ex, handle
        sz = C.c_uint32(0)
        check(ex._lib.gcre_pathset_size(handle, C.byref(sz)))
        self.size = sz.value
        self.width_ul = ex.width_ul
        self.vlen = ex.width_ul * ex.m

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:  # legal after the exec is gone: gcre_exec_destroy orphans its children
            self.ex._lib.gcre_pathset_destroy(h)

    def load(self, data):
        """PathSet::load - int matrix rows x patients, non-zero = carrier (src/gcre_paths.h:56-78)."""
        d = _as(data, np.int32)
        rows = d.shape[0]
        cols = d.shape[1] if d.ndim == 2 else 0
        check(self.ex._lib.gcre_pathset_load_i32(self._h, _ptr(d, C.c_int32), rows, cols))

    def load_bits(self, bits):
        b = _as(bits, np.uint64)
        check(self.ex._lib.gcre_pathset_load_bits(self._h, _ptr(b, C.c_uint64), b.shape[0], b.shape[1] if b.ndim == 2 else 0))

    def load_bits_device(self, device_ptr, rows, words_per_row):
        """Packed rows already in this GPU's memory (e.g. after an NCCL broadcast); ordered on the exec's stream."""
        check(self.ex._lib.gcre_pathset_load_bits_device(self._h, C.c_void_p(int(device_ptr)), int(rows), int(words_per_row)))

    def select(self, indices):
        """PathSet::select (src/gcre_paths.h:82-92)."""
        i = _as(indices, np.int32)
        out = C.c_void_p()
        check(self.ex._lib.gcre_pathset_select(self._h, _ptr(i, C.c_int32), i.shape[0], C.byref(out)))
        return PathSet(self.ex, out)

    def set(self, idx, words):
        w = _as(words, np.uint64)
        if w.shape[0] != self.ex.w64 * self.ex.m:
            raise ValueError("row must hold ceil(n/64)*method words")
        check(self.ex._lib.gcre_pathset_set_row(self._h, int(idx), _ptr(w, C.c_uint64)))

    def __getitem__(self, idx):
        out = np.zeros(self.ex.w64 * self.ex.m, dtype=np.uint64)
        if idx < 0:
            raise _lib.GcreOutOfRange(_lib.GCRE_ERR_RANGE, "assertion")
        check(self.ex._lib.gcre_pathset_get_row(self._h, int(idx), _ptr(out, C.c_uint64)))
        return out

    def to_numpy(self):
        out = np.zeros((self.size, self.ex.w64 * self.ex.m), dtype=np.uint64)
        check(self.ex._lib.gcre_pathset_download(self._h, _ptr(out, C.c_uint64)))
        return out

    def debug_view(self):
        """The sparse kernels' state of this set, read back for tests and diagnostics (include/gcre_b200.h, gcre_pathset_debug_*):
        ``{"lists": {off, len, ncase, car} or None, "table": {counts [rows][method][iters_requested] uint16, len, ncase
        [rows][method], lo, hi, layout, current} or None, "stats_valid": bool}``."""
        lib, m = self.ex._lib, self.ex.m
        info = np.zeros(8, dtype=np.int64)
        check(lib.gcre_pathset_debug_view_info(self._h, _ptr(info, C.c_int64)))
        lists = table = None
        if info[0]:
            items = self.size * m
            off = np.zeros(items + 1, dtype=np.uint64)
            ln, nc = np.zeros(max(items, 1), dtype=np.uint32), np.zeros(max(items, 1), dtype=np.uint32)
            car = np.zeros(max(int(info[1]), 1), dtype=np.uint32)
            check(lib.gcre_pathset_debug_lists(self._h, _ptr(off, C.c_uint64), _ptr(ln, C.c_uint32), _ptr(nc, C.c_uint32), _ptr(car, C.c_uint32)))
            lists = {"off": off, "len": ln[:items].reshape(self.size, m), "ncase": nc[:items].reshape(self.size, m), "car": car[: int(info[1])]}
        if info[3]:
            lo, hi = int(info[6]), int(info[7])
            counts = np.zeros((max(hi - lo, 1), m, max(self.ex.iters_requested, 1)), dtype=np.uint16)
            ln, nc = np.zeros((max(hi - lo, 1), m), dtype=np.uint32), np.zeros((max(hi - lo, 1), m), dtype=np.uint32)
            check(lib.gcre_pathset_debug_counts(self._h, _ptr(counts, C.c_uint16), _ptr(ln, C.c_uint32), _ptr(nc, C.c_uint32)))
            table = {"counts": counts[: hi - lo, :, : self.ex.iters_requested], "len": ln[: hi - lo], "ncase": nc[: hi - lo], "lo": lo, "hi": hi,
                     "layout": int(info[4]), "current": bool(info[5])}
        return {"lists": lists, "table": table, "stats_valid": bool(info[2])}


class JoinExec:
    """JoinExec (src/gcre.h:103-180).  ``nthreads`` is accepted and ignored (the join runs on the GPU)."""

    def __init__(self, method_name, num_cases, num_ctrls, iters, device=0):
        self._h = None
        self._lib = _lib.load()
        self.method = method_name
        self.m = 1 if method_name == "method1" else 2  # JoinExec::to_method (src/gcre.h:125-133)
        h = C.c_void_p()
        check(self._lib.gcre_exec_create(self.m, int(num_cases), int(num_ctrls), int(iters), int(device), C.byref(h)))
        self._h = h
        info = _lib.ExecInfoC()
        check(self._lib.gcre_exec_get_info(h, C.byref(info)))
        self.num_cases, self.num_ctrls = info.num_cases, info.num_ctrls
        self.width_ul, self.iterations, self.iters_requested = info.width_ul, info.iterations, info.iters_requested
        self.device, self.sm_count = info.device, info.sm_count
        self.w64 = (self.num_cases + self.num_ctrls + 63) // 64
        self.top_k = 12  # src/gcre.h:120
        self.nthreads = 0
        self.kernel = _lib.KERNEL_AUTO

    def close(self):
        h, self._h = self._h, None
        if h:
            self._lib.gcre_exec_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def print_vector_info(self):  # src/gcre.h:144-152 (all output commented out in the reference)
        pass

    def set_stream(self, cuda_stream_ptr):
        check(self._lib.gcre_exec_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def setValueTable(self, table):
        t = _as(table, np.float64)
        if t.ndim != 2:
            t = t.reshape(0, 0)
        check(self._lib.gcre_exec_set_value_table(self._h, _ptr(t, C.c_double), t.shape[0], t.shape[1]))

    def setValueTableDevice(self, device_ptr, rows, cols):
        """The value table from a buffer in this GPU's memory (multi-GPU fan-out); ordered on the exec's stream."""
        check(self._lib.gcre_exec_set_value_table_device(self._h, C.c_void_p(int(device_ptr)), int(rows), int(cols)))

    def generateValueTable(self):
        """getValuesTable (R/Utils.R:137-159) on the device for this exec's (num_cases, num_ctrls) (extension)."""
        check(self._lib.gcre_exec_generate_value_table(self._h))

    def getValueTable(self):
        out = np.zeros((self.num_cases + 1, self.num_ctrls + 1), dtype=np.float64)
        check(self._lib.gcre_exec_get_value_table(self._h, _ptr(out, C.c_double), out.shape[0], out.shape[1]))
        return out

    def setPermutedCases(self, perm_cases):
        p = _as(perm_cases, np.int32)
        rows = p.shape[0]
        cols = p.shape[1] if p.ndim == 2 else 0
        check(self._lib.gcre_exec_set_permuted_cases_i32(self._h, _ptr(p, C.c_int32), rows, cols))

    def setPermutedMasks(self, masks):
        m = _as(masks, np.uint64)
        if m.ndim != 2 or (m.shape[0] and m.shape[1] != self.w64):
            raise ValueError("masks must be uint64[n_perms][ceil(n/64)]")
        check(self._lib.gcre_exec_set_permuted_masks_u64(self._h, _ptr(m, C.c_uint64), m.shape[0]))

    def setPermutedMasksDevice(self, device_ptr, n_perms):
        """Packed masks uint64[n_perms][ceil(n/64)] already in this GPU's memory; ordered on the exec's stream (extension)."""
        check(self._lib.gcre_exec_set_permuted_masks_device(self._h, C.c_void_p(int(device_ptr)), int(n_perms)))

    def setPermutationStrata(self, labels):
        """One int32 label per patient for generatePermutedMasks (cases keep their count within every stratum); None or an
        empty sequence goes back to one stratum (extension)."""
        if labels is None or len(labels) == 0:
            check(self._lib.gcre_exec_set_permutation_strata(self._h, None, 0))
            return
        lab = _as(labels, np.int32)
        check(self._lib.gcre_exec_set_permutation_strata(self._h, _ptr(lab, C.c_int32), int(lab.shape[0])))

    def generatePermutedMasks(self, seed, first_perm=0):
        """Permutations first_perm .. first_perm + iters_requested - 1 of ``seed``, made on the device (include/gcre_b200.h,
        synth.make_perm_masks_philox); ordered on the exec's stream (extension)."""
        check(self._lib.gcre_exec_generate_permuted_masks(self._h, int(seed) & (2**64 - 1), int(first_perm) & (2**64 - 1)))

    def getPermutedMasks(self, n_perms=None):
        """The current masks as uint64[n_perms][ceil(n/64)] (default: all iters_requested rows), whichever setter made them."""
        n_perms = self.iters_requested if n_perms is None else int(n_perms)
        out = np.zeros((max(n_perms, 0), self.w64), dtype=np.uint64)
        check(self._lib.gcre_exec_get_permuted_masks(self._h, _ptr(out, C.c_uint64), n_perms))
        return out

    def createPathSet(self, size):
        out = C.c_void_p()
        check(self._lib.gcre_pathset_create(self._h, int(size), C.byref(out)))
        return PathSet(self, out)

    def join(self, uids, paths0, paths1, paths_res, uid_range=None, skip_host_perm=False):
        """JoinExec::join (src/join_base.cpp:189-264) -> joined_res."""
        cap = max(int(self.top_k), 1) + 1
        sc = (_lib.ScoreC * cap)()
        n_sc = C.c_int(0)
        perm = np.zeros(max(self.iters_requested, 1), dtype=np.float64)
        opts = _lib.JoinOptsC()
        opts.kernel = int(self.kernel)
        opts.skip_host_perm = 1 if skip_host_perm else 0
        if uid_range is not None:
            opts.uid_begin, opts.uid_end = int(uid_range[0]), int(uid_range[1])
            if opts.uid_end == 0:  # empty shard at the front: nothing to do, still go through the call for the checks
                opts.uid_begin, opts.uid_end = uids.size(), uids.size()
        res_h = paths_res._h if paths_res is not None else None
        if uids._resident is not None and uids._resident[0] is self:
            check(self._lib.gcre_join_uidset(self._h, uids._resident[1], paths0._h, paths1._h, res_h, int(self.top_k), sc, C.byref(n_sc),
                                             _ptr(perm, C.c_double), C.byref(opts)))
        else:
            check(self._lib.gcre_join(self._h, uids.path_length, uids._packed.ctypes.data_as(C.POINTER(_lib.UidRefC)), uids.size(),
                                      _ptr(uids.signs, C.c_int32), uids.signs.shape[0], paths0._h, paths1._h, res_h, int(self.top_k), sc,
                                      C.byref(n_sc), _ptr(perm, C.c_double), C.byref(opts)))
        scores = [Score(s.score, s.src, s.trg, s.cases, s.ctrls) for s in sc[: n_sc.value]]
        info = {"pairs": int(opts.pairs_scored), "kernel_ms": float(opts.kernel_ms), "kernel": int(opts.kernel_used), "launches": int(opts.launches),
                "precounted": bool(opts.precounted), "tail_form": bool(opts.tail_form), "split_carrier": bool(opts.split_carrier), "thresholded": bool(opts.thresholded), "shared_masks": bool(opts.shared_masks),
                "exact_pairs": int(opts.exact_pairs)}
        return joined_res(scores, perm[: self.iters_requested].copy(), info)

    def device_perm_max(self):
        """(device pointer, n_floats) of the last join's permutation maxima (float32) - for an NCCL allreduce(max)."""
        p, n = C.c_void_p(), C.c_int(0)
        check(self._lib.gcre_exec_device_perm_max(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def read_perm_max(self):
        out = np.zeros(max(self.iters_requested, 1), dtype=np.float64)
        check(self._lib.gcre_exec_read_perm_max(self._h, _ptr(out, C.c_double)))
        return out[: self.iters_requested].copy()


def host_pack(data, threads=0, out=None):
    """int matrix (any non-zero = carrier) -> uint64[rows][ceil(cols/64)] on host threads (gcre_host_pack_i32)."""
    d = _as(data, np.int32)
    rows, cols = d.shape
    w = (cols + 63) // 64
    if out is None:
        out = np.zeros((rows, w), dtype=np.uint64)
    check(_lib.load().gcre_host_pack_i32(_ptr(d, C.c_int32), rows, cols, _ptr(out, C.c_uint64), int(threads)))
    return out


def merge_topk(score_lists, top_k):
    """Merge shard-local top-K lists under the engine's rule (K largest, ties -> smaller (src, trg))."""
    lib = _lib.load()
    flat = [s for lst in score_lists for s in lst]
    arr = (_lib.ScoreC * max(len(flat), 1))()
    for i, s in enumerate(flat):
        arr[i].score, arr[i].src, arr[i].trg, arr[i].cases, arr[i].ctrls = s.score, s.src, s.trg, s.cases, s.ctrls
    sizes = (C.c_int * max(len(score_lists), 1))(*[len(l) for l in score_lists])
    out = (_lib.ScoreC * (top_k + 1))()
    n = C.c_int(0)
    check(lib.gcre_merge_topk(arr, sizes, len(score_lists), int(top_k), out, C.byref(n)))
    return [Score(s.score, s.src, s.trg, s.cases, s.ctrls) for s in out[: n.value]]
