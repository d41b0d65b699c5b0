"""ctypes binding of the C-ABI in include/phylocsf_b200.h (lib/libphylocsf_b200.so).

This is the only door from Python into the product.  There is no CPU fallback: if the CUDA library has
not been built, or no CUDA device is present, every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libphylocsf_b200.so")
if os.environ.get("PCSF_LIB_VARIANT"):          # kernel experiments (tools/build_variant.sh): lib/libphylocsf_b200_<variant>.so
    LIB_PATH = os.path.join(_HERE, "lib", f"libphylocsf_b200_{os.environ['PCSF_LIB_VARIANT']}.so")

PCSF_OK = 0
PCSF_ERR_INVALID = 1
PCSF_ERR_CUDA = 2
PCSF_ERR_NUMERIC = 3
PCSF_ERR_UNSUPPORTED = 4
PCSF_ERR_BAD_CHAR = 37

TRACKS_SCORES = 0x1
TRACKS_BLS = 0x2
TRACKS_NO_DEDUP = 0x4
TRACKS_TC5 = 0x10

STRATEGY_MLE = 0
STRATEGY_FIXED = 1
STRATEGY_OMEGA = 2

ORF_ASIS = 0
ORF_STOPSTOP = 1
ORF_ATGSTOP = 2

# pcsf_region (include/phylocsf_b200.h), 48 bytes
REGION_DTYPE = np.dtype([("aln", np.int32), ("strand", np.int8), ("frame", np.int8), ("pad", np.int16), ("col_begin", np.int64),
                         ("col_end", np.int64), ("codons", np.int64), ("phylo", np.float32), ("anc", np.float32),
                         ("bls", np.float32)], align=True)

EXPORTS = [
    "pcsf_model_create", "pcsf_model_destroy", "pcsf_last_error", "pcsf_abi_version", "pcsf_tracks",
    "pcsf_tracks_device", "pcsf_tracks_device_finish", "pcsf_set_chunk_columns", "pcsf_set_timing",
    "pcsf_score_msa", "pcsf_model_get", "pcsf_alloc_pinned", "pcsf_free_pinned", "pcsf_device_count", "pcsf_score_msa_stats", "pcsf_register_host", "pcsf_unregister_host",
    "pcsf_score_regions", "pcsf_score_regions_get", "pcsf_score_given_regions",
]


class PcsfError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"pcsf status {status}: {msg}")
        self.status = status


class ModelDesc(C.Structure):
    _fields_ = [("nl", C.c_int32), ("child1", C.c_void_p), ("child2", C.c_void_p), ("branch_len", C.c_void_p),
                ("branch_len_f64", C.c_void_p), ("ecm_c", C.c_void_p), ("freq_c", C.c_void_p),
                ("ecm_nc", C.c_void_p), ("freq_nc", C.c_void_p)]


class TracksStats(C.Structure):
    _fields_ = [("n_windows", C.c_int64), ("n_unique", C.c_int64), ("n_chunks", C.c_int32), ("n_launches", C.c_int32),
                ("ms_pack", C.c_float), ("ms_hash", C.c_float), ("ms_dedup", C.c_float), ("ms_prune", C.c_float),
                ("ms_scatter", C.c_float), ("ms_bls", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class MsaStats(C.Structure):
    _fields_ = [("alignments", C.c_int64), ("evaluations", C.c_int64), ("rounds", C.c_int32), ("slots", C.c_int32),
                ("ms_step", C.c_float), ("ms_plan", C.c_float), ("ms_expm", C.c_float), ("ms_prune", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load():
    """Loads the CUDA library.  Raises (loudly) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          f"(nvcc, sm_100a).  phylocsfpp_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.pcsf_last_error.restype = C.c_char_p
    L.pcsf_abi_version.restype = C.c_int
    L.pcsf_alloc_pinned.restype = C.c_void_p
    L.pcsf_alloc_pinned.argtypes = [C.c_size_t]
    L.pcsf_free_pinned.restype = None
    L.pcsf_free_pinned.argtypes = [C.c_void_p]
    L.pcsf_model_create.argtypes = [C.POINTER(ModelDesc), C.c_int, C.POINTER(C.c_void_p)]
    L.pcsf_model_destroy.argtypes = [C.c_void_p]
    L.pcsf_model_destroy.restype = None
    L.pcsf_tracks.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_uint32, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.POINTER(TracksStats)]
    L.pcsf_tracks_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_uint32, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pcsf_tracks_device_finish.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(TracksStats)]
    L.pcsf_set_chunk_columns.argtypes = [C.c_void_p, C.c_int64]
    L.pcsf_set_timing.argtypes = [C.c_void_p, C.c_int]
    L.pcsf_score_msa.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]
    L.pcsf_model_get.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.pcsf_score_msa_stats.argtypes = [C.c_void_p, C.POINTER(MsaStats)]
    L.pcsf_device_count.restype = C.c_int
    L.pcsf_score_regions.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                     C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]
    L.pcsf_score_regions_get.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    L.pcsf_score_given_regions.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = L
    return L


def _check(status: int):
    if status != PCSF_OK:
        raise PcsfError(status, load().pcsf_last_error().decode(errors="replace"))


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


class DeviceModel:
    """pcsf_model: the device-resident model blob (what the reference rebuilds on every run_tracks call)."""

    def __init__(self, model, device: int = 0):
        """model: phylocsfpp_b200.models.Model (or anything with .tree, .S_c, .f_c, .S_nc, .f_nc)."""
        L = load()
        t = model.tree
        self.nl, self.n = t.nl, t.n
        self._keep = [np.ascontiguousarray(t.child1, np.int16), np.ascontiguousarray(t.child2, np.int16),
                      np.ascontiguousarray(t.branch_len, np.float32), np.ascontiguousarray(t.branch_len_f64, np.float64),
                      np.ascontiguousarray(model.S_c, np.float64), np.ascontiguousarray(model.f_c, np.float64),
                      np.ascontiguousarray(model.S_nc, np.float64), np.ascontiguousarray(model.f_nc, np.float64)]
        d = ModelDesc(t.nl, *[a.ctypes.data for a in self._keep])
        h = C.c_void_p()
        _check(L.pcsf_model_create(C.byref(d), device, C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            load().pcsf_model_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_chunk_columns(self, columns: int):
        _check(load().pcsf_set_chunk_columns(self.h, columns))

    def set_timing(self, enabled: bool):
        _check(load().pcsf_set_timing(self.h, int(enabled)))

    def get(self, which: int):
        lam, pi, P = np.zeros(64), np.zeros(64), np.zeros((self.n - 1, 64, 64))
        _check(load().pcsf_model_get(self.h, which, lam.ctypes.data, pi.ctypes.data, P.ctypes.data))
        return lam, pi, P

    def tracks(self, seqs: np.ndarray, scores: bool = True, bls: bool = True, dedup: bool = True,
               want_patterns: bool = False, tc5: bool = False):
        """Host-buffer call (H2D + kernels + D2H).  seqs: uint8 ASCII [nl, L].
        Returns dict(plus, minus, bls, pattern_index, stats)."""
        seqs = np.ascontiguousarray(seqs, np.uint8)
        nl, Lc = seqs.shape
        assert nl == self.nl
        W = max(Lc - 2, 0)
        flags = ((TRACKS_SCORES if scores else 0) | (TRACKS_BLS if bls else 0) | (0 if dedup else TRACKS_NO_DEDUP)
                 | (TRACKS_TC5 if tc5 else 0))
        plus = np.zeros(W, np.float64) if scores else None
        minus = np.zeros(W, np.float64) if scores else None
        b = np.zeros(Lc, np.float64) if bls else None
        pat = np.zeros(2 * W, np.uint32) if (want_patterns and scores) else None
        st = TracksStats()
        _check(load().pcsf_tracks(self.h, seqs.ctypes.data, Lc, Lc, flags, _ptr(plus), _ptr(minus), _ptr(b), _ptr(pat),
                                  C.byref(st)))
        return dict(plus=plus, minus=minus, bls=b, pattern_index=pat, stats=st.as_dict())

    def tracks_device(self, d_seqs: int, L: int, ld: int, flags: int, d_plus: int, d_minus: int, d_bls: int,
                      d_pattern: int, stream: int):
        """Device-pointer call: enqueues on `stream` without synchronising (see pcsf_tracks_device)."""
        _check(load().pcsf_tracks_device(self.h, d_seqs, L, ld, flags, d_plus, d_minus, d_bls, d_pattern, stream))

    def tracks_device_finish(self, stream: int):
        st = TracksStats()
        _check(load().pcsf_tracks_device_finish(self.h, stream, C.byref(st)))
        return st.as_dict()

    def score_msa_stats(self):
        st = MsaStats()
        _check(load().pcsf_score_msa_stats(self.h, C.byref(st)))
        return st.as_dict()

    def _batch(self, alignments):
        n = len(alignments)
        lens = np.array([a.shape[1] for a in alignments], np.int64)
        offs = np.zeros(n, np.int64)
        if n:
            offs[1:] = np.cumsum(lens[:-1] * self.nl)
        blob = np.concatenate([np.ascontiguousarray(a, np.uint8).reshape(-1) for a in alignments]) if n else np.zeros(1, np.uint8)
        if blob.size == 0:
            blob = np.zeros(1, np.uint8)
        return n, lens, offs, blob

    def score_msa(self, alignments, strategy: int = STRATEGY_FIXED, comp_phylo: bool = True, comp_anc: bool = True,
                  comp_bls: bool = True):
        """alignments: list of uint8 ASCII [nl, L_i] matrices.  Returns (phylo, anc, bls) float32 arrays, None for a score not
        asked for."""
        n, lens, offs, blob = self._batch(alignments)
        phylo = np.full(n, np.nan, np.float32) if comp_phylo else None
        anc = np.full(n, np.nan, np.float32) if comp_anc else None
        b = np.full(n, np.nan, np.float32) if comp_bls else None
        _check(load().pcsf_score_msa(self.h, strategy, n, blob.ctypes.data, offs.ctypes.data, lens.ctypes.data,
                                     _ptr(phylo), _ptr(anc), _ptr(b)))
        return phylo, anc, b

    def score_regions(self, alignments, ref_rows, strategy: int = STRATEGY_FIXED, frames: int = 6, orf: int = ORF_ATGSTOP,
                      min_codons: int = 25, best_only: bool = False, comp_anc: bool = True, comp_bls: bool = True) -> np.ndarray:
        """Reading frames / ORFs of every alignment, scored on the device (pcsf_score_regions).  ref_rows: model row of each
        alignment's reference species.  Returns a structured array of REGION_DTYPE records (phylocsfpp_b200.orf mirrors the
        enumeration and the best-only rule)."""
        n, lens, offs, blob = self._batch(alignments)
        refs = np.ascontiguousarray(np.asarray(ref_rows, np.int32).reshape(-1))
        if refs.size != n:
            raise ValueError("one reference row per alignment")
        if refs.size == 0:
            refs = np.zeros(1, np.int32)
        L = load()
        nreg = C.c_int64(0)
        _check(L.pcsf_score_regions(self.h, strategy, n, blob.ctypes.data, offs.ctypes.data, lens.ctypes.data, refs.ctypes.data,
                                    frames, orf, min_codons, int(best_only), int(comp_anc), int(comp_bls), C.byref(nreg)))
        out = np.zeros(nreg.value, REGION_DTYPE)
        _check(L.pcsf_score_regions_get(self.h, out.ctypes.data if out.size else None, nreg.value))
        return out

    def score_given_regions(self, alignments, region_aln, region_begin, region_end, strategy: int = STRATEGY_FIXED,
                            comp_anc: bool = True, comp_bls: bool = True):
        """Column ranges [region_begin[r], region_end[r]) of alignments[region_aln[r]], each scored in frame +1 from its begin
        (pcsf_score_given_regions).  Returns (phylo, anc, bls) float32 arrays, None for a score not asked for; bit for bit what
        score_msa returns for the ranges cut out on the host."""
        n, lens, offs, blob = self._batch(alignments)
        ra = np.ascontiguousarray(np.asarray(region_aln, np.int32).reshape(-1))
        rb = np.ascontiguousarray(np.asarray(region_begin, np.int64).reshape(-1))
        re_ = np.ascontiguousarray(np.asarray(region_end, np.int64).reshape(-1))
        if not (ra.size == rb.size == re_.size):
            raise ValueError("region_aln, region_begin and region_end differ in length")
        nr = ra.size
        phylo = np.full(nr, np.nan, np.float32)
        anc = np.full(nr, np.nan, np.float32) if comp_anc else None
        b = np.full(nr, np.nan, np.float32) if comp_bls else None
        _check(load().pcsf_score_given_regions(self.h, strategy, n, blob.ctypes.data, offs.ctypes.data, lens.ctypes.data, nr,
                                               _ptr(ra), _ptr(rb), _ptr(re_), _ptr(phylo), _ptr(anc), _ptr(b)))
        return phylo, anc, b
