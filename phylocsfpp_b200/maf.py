"""MAF alignment reader with the reference's block-concatenation semantics.

Host-side mirror of `parallel_maf_reader::get_next_alignment` (src/parallel_file_reader.hpp:430-700) and
`alignment_t` (:19-114).  Only the *semantics* are kept (SURVEY.md Appendix C): which blocks are
concatenated, where a chain is cut, how absent species and reference gaps are handled.  The reference's
page-range job splitting (:254-357, :396-425) only decides which thread reads which chain and is designed
so the output is independent of the job count; this reader walks the file once, which equals jobs = 1.

  * `s` lines: `s <species>.<chrom> <start0> <size> <strand> <srcSize> <text>`; species = text before the
    first '.', lower-cased (:489-507); species unknown to the model are skipped with a one-time warning.
  * first matched row of a chain's first block is the reference: start_pos = start0 + 1 (:528-554).
  * concatenate=True (build-tracks): the next block is appended iff same chrom and
    start0 == (start_pos - 1) + cumulative reference length (:494-505); absent species are padded with 'N'
    (:603-611); a chain that crosses a multiple of BREAKPOINT_POS keeps reading until >= 2 more reference
    bases are in, is truncated to exactly +2 and the cursor is rewound to the first block after the
    crossing block (:456-473, :547-569, :616-629, :671-679).
  * columns where the reference row has '-' are deleted from every row (:631-669).
  * concatenate=False (score-msa): one block = one alignment, any reference strand.
"""
from __future__ import annotations

import gzip
import sys
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

BREAKPOINT_POS = 1000000


@dataclass
class Alignment:
    """alignment_t (parallel_file_reader.hpp:19-44); seqs is a [nl, L] uint8 matrix of ASCII."""
    start_pos: int = 0
    chrom_len: int = 0
    strand: str = "+"
    chrom: str = ""
    seqs: np.ndarray = field(default_factory=lambda: np.zeros((0, 0), np.uint8))
    ref_row: int = -1   # model row of the reference species (the first matched species of the first block); -1: none

    @property
    def L(self) -> int:
        return int(self.seqs.shape[1])


def _atoi(tok: bytes) -> int:
    # the reference parses numbers with atoi (:213-225)
    return int(tok)


class MafReader:
    def __init__(self, path: str, seqid_to_phyloid: Dict[str, int], nl: int, concatenate: bool,
                 warn=True):
        opener = gzip.open if path.endswith(".gz") else open
        with opener(path, "rb") as fh:
            data = fh.read()
        self.lines: List[bytes] = data.split(b"\n")
        if self.lines and self.lines[-1] == b"":
            self.lines.pop()
        self.nlines = len(self.lines)
        self.map = seqid_to_phyloid
        self.nl = nl
        self.concatenate = concatenate
        self.unresolved = set()
        self.species_seen = np.zeros(nl, bool)
        self.warn = warn
        # constructor (:321-343): start at the first "a " line
        self.pos = 0
        while self.pos < self.nlines and not self.lines[self.pos].startswith(b"a "):
            self.pos += 1

    def __iter__(self):
        return self

    def __next__(self) -> Alignment:
        aln = self.get_next_alignment()
        if aln is None:
            raise StopIteration
        return aln

    def get_next_alignment(self, single_block_scoring: Optional[bool] = None) -> Optional[Alignment]:
        if single_block_scoring is None:
            single_block_scoring = not self.concatenate
        if self.pos >= self.nlines:
            return None
        lines, nlines = self.lines, self.nlines
        rows: List[List[bytes]] = [[] for _ in range(self.nl)]
        row_len = [0] * self.nl
        aln = Alignment()

        first_block = True
        abort_next = not self.concatenate
        reached_bp = False
        stop_saving = False
        saved_pos = self.pos
        ref_seq_id = -1
        prev_cum = 0
        cum_after_bp = 0

        while (not abort_next or first_block) and self.pos < nlines:
            if not stop_saving:
                if reached_bp:
                    stop_saving = True
                saved_pos = self.pos
            self.pos += 1  # skip "a score=..."
            ref_seq_id_sub = -1
            if reached_bp and prev_cum >= cum_after_bp + 2:
                abort_next = True

            while (not abort_next or first_block) and self.pos < nlines and not lines[self.pos].startswith(b"a"):
                line = lines[self.pos]
                if not line.startswith(b"s"):
                    self.pos += 1
                    continue
                self.pos += 1
                tok = line.split(b" ")
                tok = [t for t in tok if t]  # strtok_r collapses runs of spaces
                ident = tok[1].decode()
                start0 = _atoi(tok[2])
                size = _atoi(tok[3])
                strand = chr(tok[4][0])
                chrom_len = _atoi(tok[5])
                seq = tok[6]
                dot = ident.find(".")
                assert dot >= 0, "expect format species_name.chrom_name"
                species, chrom = ident[:dot], ident[dot + 1:]

                if not first_block:
                    if ref_seq_id_sub == -1 and not ((aln.start_pos - 1) + prev_cum == start0 and chrom == aln.chrom):
                        abort_next = True
                        break
                species = species.lower()
                alnid = self.map.get(species)
                if alnid is None:
                    if species not in self.unresolved:
                        self.unresolved.add(species)
                        if self.warn:
                            print(f"WARNING: Not able to match species {species} in alignment file to model "
                                  f"(Use `--mapping` to fix it)!", file=sys.stderr)
                    continue

                if ref_seq_id == -1 and first_block:
                    aln.start_pos = start0 + 1
                    aln.chrom = chrom
                    aln.chrom_len = chrom_len
                    aln.strand = strand
                    ref_seq_id = alnid
                    prev_cum = size
                    if strand != "+" and not single_block_scoring:
                        raise ValueError(f"Reference sequence is not on the + strand ({species}.{chrom} at position {start0})!")
                    prev_end = aln.start_pos
                    new_end = aln.start_pos + size
                    if not reached_bp and prev_end // BREAKPOINT_POS < new_end // BREAKPOINT_POS:
                        reached_bp = True
                        cum_after_bp = prev_cum
                elif ref_seq_id_sub == -1 and not first_block:
                    ref_seq_id_sub = alnid
                    prev_end = aln.start_pos + prev_cum
                    new_end = aln.start_pos + prev_cum + size
                    prev_cum += size
                    if not reached_bp and prev_end // BREAKPOINT_POS < new_end // BREAKPOINT_POS:
                        reached_bp = True
                        cum_after_bp = prev_cum
                    if ref_seq_id != ref_seq_id_sub:
                        raise ValueError(f"Encountered an alignment block that didn't start with the reference species: "
                                         f"{species}.{chrom} at position {start0}!")
                    if strand != "+" and not single_block_scoring:
                        raise ValueError(f"Reference sequence is not on the + strand ({species}.{chrom} at position {start0})!")

                rows[alnid].append(seq)
                row_len[alnid] += len(seq)
                self.species_seen[alnid] = True

            # absent species get N (:603-611)
            if ref_seq_id >= 0:
                new_len = row_len[ref_seq_id]
                for i in range(self.nl):
                    if row_len[i] != new_len:
                        rows[i].append(b"N" * (new_len - row_len[i]))
                        row_len[i] = new_len
            first_block = False

        if reached_bp and prev_cum >= cum_after_bp + 2:
            abort_next = True
        if abort_next and self.concatenate:
            self.pos = saved_pos

        if ref_seq_id < 0:
            # a block with no species known to the model: the reference would index seqs[-1]; treat as empty
            aln.seqs = np.zeros((self.nl, 0), np.uint8)
            return aln
        mat = np.frombuffer(b"".join(b"".join(r) for r in rows), np.uint8).reshape(self.nl, row_len[ref_seq_id])
        keep = mat[ref_seq_id] != ord("-")
        mat = mat[:, keep]
        if reached_bp and prev_cum > cum_after_bp + 2:
            mat = mat[:, :cum_after_bp + 2]
        aln.seqs = np.ascontiguousarray(mat)
        aln.ref_row = ref_seq_id
        return aln
