"""Plain-Python mirror of the reading-frame / ORF regions of pcsf_score_regions (csrc/regions.cuh).

A frame phi = (strand, f) with offset f = 0, 1, 2 reads W = A ('+') or W = RC(A) ('-'); codon k is W columns f+3k .. f+3k+2 for
k < K = max(0, (L - f) // 3).  On the reference row (case-folded) TAA, TAG and TGA are stops and ATG is a start; a codon with any
other character is neither.  Regions of one frame:
  asis      one region: W columns [min(f, L), L), the trailing partial codon included (frame +1 is the whole alignment)
  stopstop  every stop-delimited segment (closing stop included) and the non-empty open tail after the last stop
  atgstop   per segment with an ATG before its stop: the first such ATG through the stop; the open tail never yields one
In the ORF modes a region is kept if it has at least min_codons codons (stop included).  Order: frame (+1 +2 +3 -1 -2 -3), then
codon index.  Region columns are reported in the input alignment: a '-' region over W columns [a, b) is [L - b, L - a).
"""
from __future__ import annotations

from typing import List, NamedTuple, Optional, Sequence

import numpy as np

ASIS, STOPSTOP, ATGSTOP = 0, 1, 2
MODES = {"asis": ASIS, "stopstop": STOPSTOP, "atgstop": ATGSTOP}
FRAMES = {1: [(1, 0)], 3: [(1, 0), (1, 1), (1, 2)], 6: [(1, 0), (1, 1), (1, 2), (-1, 0), (-1, 1), (-1, 2)]}

_COMP = {ord(a): ord(b) for a, b in zip("ACGTacgt", "TGCAtgca")}
STOPS = (b"TAA", b"TAG", b"TGA")


class Region(NamedTuple):
    strand: int       # +1 / -1 (0: none)
    frame: int        # 1..3 (0: none)
    k0: int           # first codon of the frame
    codons: int
    col_begin: int    # [col_begin, col_end) in the input alignment's columns
    col_end: int


def frame_codon(ref: bytes, strand: int, f: int, k: int) -> bytes:
    """Codon k of frame (strand, f) of one row, upper case; '-' codons read the complemented row backwards."""
    L = len(ref)
    if strand > 0:
        c = ref[f + 3 * k:f + 3 * k + 3]
    else:
        o = L - 3 - f - 3 * k
        c = bytes(_COMP.get(x, x) for x in reversed(ref[o:o + 3]))
    return c.upper()


def codon_class(c: bytes) -> str:
    if c in STOPS:
        return "stop"
    return "start" if c == b"ATG" else ""


def regions(ref, L: Optional[int] = None, frames: int = 6, orf: int = ATGSTOP, min_codons: int = 25) -> List[Region]:
    """All regions of one alignment whose reference row is `ref` (bytes or a uint8 array of ASCII)."""
    ref = bytes(np.asarray(ref, np.uint8).tobytes()) if not isinstance(ref, (bytes, bytearray)) else bytes(ref)
    L = len(ref) if L is None else L
    if frames not in FRAMES or orf not in (ASIS, STOPSTOP, ATGSTOP) or min_codons < 1:
        raise ValueError("bad frames / orf / min_codons")
    out: List[Region] = []
    for strand, f in FRAMES[frames]:
        K = max(0, (L - f) // 3)

        def region(k0: int, n: int, a: int, b: int) -> Region:
            return Region(strand, f + 1, k0, n, *((a, b) if strand > 0 else (L - b, L - a)))

        if orf == ASIS:
            a = min(f, L)
            out.append(region(0, K, a, L))
            continue
        seg, atg = 0, -1
        for k in range(K):
            cls = codon_class(frame_codon(ref, strand, f, k))
            if cls == "start" and atg < 0:
                atg = k
            elif cls == "stop":
                start = seg if orf == STOPSTOP else atg
                if start >= 0 and k - start + 1 >= min_codons:
                    out.append(region(start, k - start + 1, f + 3 * start, f + 3 * (k + 1)))
                seg, atg = k + 1, -1
        if orf == STOPSTOP and K - seg >= max(1, min_codons):
            out.append(region(seg, K - seg, f + 3 * seg, f + 3 * K))
    return out


def sub_alignment(seqs: np.ndarray, r: Region) -> np.ndarray:
    """S(r): the region's columns of W (reverse complement of the input's [col_begin, col_end) on the '-' strand)."""
    s = np.ascontiguousarray(seqs[:, r.col_begin:r.col_end], np.uint8)
    if r.strand < 0:
        lut = np.arange(256, dtype=np.uint8)
        for a, b in _COMP.items():
            lut[a] = b
        s = np.ascontiguousarray(lut[s[:, ::-1]])
    return s


def best_index(phylo: Sequence[float]) -> int:
    """The best-only rule over one alignment's regions in enumeration order: the largest phylo; NaN never wins; ties go to the
    earlier region; all NaN: the first region; no region: -1 (the "none" record)."""
    best = -1
    for i, v in enumerate(phylo):
        if v == v and (best < 0 or v > phylo[best]):
            best = i
    if best < 0 and len(phylo) > 0:
        best = 0
    return best
