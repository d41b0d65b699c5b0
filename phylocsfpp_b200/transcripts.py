"""Plain-Python mirror of the transcript alignments of annotate-with-maf (host/transcripts.hpp); the tests use it as the reference.

MAF chains are read with build-tracks' semantics (maf.MafReader, concatenate): chain column j is reference position start_pos + j.
A position no chain covers is N in every row; where two chains cover it (the +2 columns past a 1 Mb breakpoint), the chain that
starts last is used.  Chains whose reference row is on '-' are not used.

GFF/GTF records are the runs of lines from one `transcript` line up to the next (the first record also holds the lines before the
first transcript).  A record with CDS lines: the CDS intervals in genomic order, concatenated, reverse-complemented as a whole on '-'
(oracle.reverse_complement), the phase of the 5'-most CDS dropped from the front; regions: the whole alignment, then one per CDS line
in file order, its own columns from after its own phase.  A record without CDS (ORF search): its `exon` intervals, or its own span,
spliced the same way; ref_row is the reference row of the chains used (-1: none, -2: they disagree).
"""
from __future__ import annotations

import bisect
import re
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

from .maf import MafReader

_NUM = re.compile(rb"\s*\+?(\d+)")


def _num(tok: bytes) -> int:
    m = _NUM.match(tok)
    return int(m.group(1)) if m else 0


@dataclass
class GffLine:
    text: bytes
    feature: bytes
    chrom: str
    begin: int
    end: int
    strand: str
    phase: int          # 0..2 ('.' or anything else: 0)


@dataclass
class TxAlignment:
    coding: bool
    strand: str
    ref_row: int
    seqs: np.ndarray                                      # [nl, L] uint8 ASCII
    segs: List[Tuple[int, int]]                           # genomic [begin, end] (1-based) of the columns, in the alignment's order
    regions: List[Tuple[int, int]] = field(default_factory=list)   # coding: whole, then one per CDS line

    @property
    def L(self) -> int:
        return int(self.seqs.shape[1])

    def genomic(self, j: int) -> int:
        for b, e in self.segs:
            n = e - b + 1
            if j < n:
                return e - j if self.strand == "-" else b + j
            j -= n
        raise IndexError(j)


def read_gff(path: str) -> List[List[GffLine]]:
    text = open(path, "rb").read()
    lines = text.split(b"\n")
    if text.endswith(b"\n"):
        lines.pop()
    recs: List[List[GffLine]] = []
    cur: List[GffLine] = []
    for ln in lines:
        c = ln.split(b"\t")
        feat = c[2] if len(c) > 2 else b""
        if feat == b"transcript" and any(g.feature == b"transcript" for g in cur):
            recs.append(cur)
            cur = []
        ph = c[7][0] - 48 if len(c) > 7 and c[7] else 0
        cur.append(GffLine(ln, feat, c[0].decode(errors="replace"), _num(c[3]) if len(c) > 3 else 0, _num(c[4]) if len(c) > 4 else 0,
                           "-" if len(c) > 6 and c[6][:1] == b"-" else "+", ph if 0 <= ph <= 2 else 0))
    if cur:
        recs.append(cur)
    return recs


class ChainIndex:
    def __init__(self, maf_paths: List[str], model):
        self.nl = model.nl
        self.minus_chains = 0
        self.by_chrom: Dict[str, List[Tuple[int, int, int, np.ndarray]]] = {}
        for p in maf_paths:
            for a in MafReader(p, model.seqid_to_phyloid, model.nl, True, warn=False, minus_ref=True):
                if a.ref_row < 0:
                    continue
                if a.strand != "+":
                    self.minus_chains += 1
                    continue
                self.by_chrom.setdefault(a.chrom, []).append((a.start_pos, a.start_pos + a.L, a.ref_row, a.seqs))
        for v in self.by_chrom.values():
            v.sort(key=lambda e: e[0])          # stable
        self.starts = {k: [e[0] for e in v] for k, v in self.by_chrom.items()}

    def extract(self, chrom: str, b: int, e: int) -> Tuple[np.ndarray, List[int]]:
        """Positions [b, e] (1-based, inclusive): the [nl, e - b + 1] columns and the reference rows of the chains used."""
        out = np.full((self.nl, max(0, e - b + 1)), ord("N"), np.uint8)
        ent, st = self.by_chrom.get(chrom, []), self.starts.get(chrom, [])
        refs = []
        p = b
        while p <= e:
            i = bisect.bisect_right(st, p)
            q = min(e + 1, st[i] if i < len(st) else e + 1)
            if i > 0 and p < ent[i - 1][1]:
                s0, s1, ref, seqs = ent[i - 1]
                q = min(q, s1)
                out[:, p - b:q - b] = seqs[:, p - s0:q - s0]
                refs.append(ref)
            p = q
        return out, refs


def extract_transcript(idx: ChainIndex, rec: List[GffLine], find_orf: bool) -> Optional[TxAlignment]:
    from oracle.oracle import reverse_complement
    tx = [g for g in rec if g.feature == b"transcript"]
    cds = [g for g in rec if g.feature == b"CDS"]
    if not tx or (not cds and not find_orf):
        return None
    t = tx[0]
    strand = "-" if t.strand == "-" else "+"
    chrom = t.chrom
    if cds:
        order = sorted(range(len(cds)), key=lambda i: cds[i].begin)
        iv = [(cds[i].begin, cds[i].end) for i in order]
    else:
        exons = [g for g in rec if g.feature == b"exon"]
        iv = sorted([(g.begin, g.end) for g in exons] or [(t.begin, t.end)], key=lambda x: x[0])
    glen = [max(0, e - b + 1) for b, e in iv]
    goff = np.concatenate([[0], np.cumsum(glen)]).astype(int).tolist()
    parts, refs = [], []
    for (b, e), n in zip(iv, glen):
        if n:
            m, r = idx.extract(chrom, b, e)
            parts.append(m)
            refs += r
    raw = np.concatenate(parts, axis=1) if parts else np.zeros((idx.nl, 0), np.uint8)
    if strand == "-":
        raw = reverse_complement(raw)
    Lraw = raw.shape[1]
    ref_row = -1 if not refs else (refs[0] if all(r == refs[0] for r in refs) else -2)
    drop = min(cds[order[-1] if strand == "-" else order[0]].phase, Lraw) if cds else 0
    segs = [s for s, n in zip(iv, glen) if n]
    if strand == "-":
        segs = segs[::-1]
    x = TxAlignment(bool(cds), strand, ref_row, np.ascontiguousarray(raw[:, drop:]), segs)
    if cds:
        x.regions.append((0, x.L))
        for i, c in enumerate(cds):
            k = order.index(i)
            tpos = Lraw - goff[k + 1] if strand == "-" else goff[k]
            end = max(0, tpos + glen[k] - drop)
            x.regions.append((min(end, max(0, tpos - drop + c.phase)), end))
    return x


def region_hash(seqs: np.ndarray, b: int, e: int) -> str:
    """sum of byte_i * P^(i+1) mod 2^64 over columns [b, e) of every row, row after row (dump-transcripts' hash)."""
    v = np.ascontiguousarray(seqs[:, b:e]).reshape(-1).astype(np.uint64)
    if v.size == 0:
        return "%016x" % 0
    with np.errstate(over="ignore"):
        pw = np.cumprod(np.full(v.size, 1099511628211, np.uint64), dtype=np.uint64)
        return "%016x" % int((v * pw).sum(dtype=np.uint64))


def dump_lines(idx: ChainIndex, gff_paths: List[str]) -> List[str]:
    """What `phylocsf_b200 dump-transcripts` prints after its header line."""
    out = []
    for fi, path in enumerate(gff_paths):
        for ri, rec in enumerate(read_gff(path)):
            x = extract_transcript(idx, rec, True)
            if x is None:
                continue
            if not x.coding:
                out.append(f"{fi}\t{ri}\texons\t{x.L}\t0\t{x.L}\t{region_hash(x.seqs, 0, x.L)}\t{x.ref_row}")
                continue
            for r, (b, e) in enumerate(x.regions):
                out.append(f"{fi}\t{ri}\t{'transcript' if r == 0 else 'CDS'}\t{x.L}\t{b}\t{e}\t{region_hash(x.seqs, b, e)}\t.")
    return out
