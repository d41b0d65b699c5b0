"""Reading-frame / ORF regions (score-msa --frames, --orf): the plain-Python mirror phylocsfpp_b200.orf against a brute-force
enumerator built on the oracle's translate / reverse_complement, the command line's option checks (they run before any device is
touched), and the register budget of the region kernels.  No GPU needed."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import orf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")

_IDS = {c: int(orc.translate(np.frombuffer(c, np.uint8)[None, :])[0, 0]) for c in (b"TAA", b"TAG", b"TGA", b"ATG")}
STOP_IDS = {_IDS[b"TAA"], _IDS[b"TAG"], _IDS[b"TGA"]}
ATG_ID = _IDS[b"ATG"]


def brute_force(ref: bytes, frames: int, mode: int, min_codons: int):
    """Translate every frame of the (upper-cased) row with the oracle, split on stops, and map W columns back to the input."""
    row = np.frombuffer(ref.upper(), np.uint8)[None, :] if ref else np.zeros((1, 0), np.uint8)
    L = row.shape[1]
    out = []
    for strand, f in orf.FRAMES[frames]:
        W = row if strand > 0 else orc.reverse_complement(row)
        ids = list(orc.translate(W, skip=f)[0]) if L > f else []
        K = len(ids)

        def emit(a, b, k0, n):
            out.append(orf.Region(strand, f + 1, k0, n, *((a, b) if strand > 0 else (L - b, L - a))))

        if mode == orf.ASIS:
            emit(min(f, L), L, 0, K)
            continue
        stops = [k for k in range(K) if ids[k] in STOP_IDS]
        prev = -1
        for s in stops:
            seg = list(range(prev + 1, s + 1))
            if mode == orf.STOPSTOP:
                start = seg[0]
            else:
                atgs = [k for k in seg[:-1] if ids[k] == ATG_ID]
                start = atgs[0] if atgs else None
            if start is not None and s - start + 1 >= min_codons:
                emit(f + 3 * start, f + 3 * (s + 1), start, s - start + 1)
            prev = s
        if mode == orf.STOPSTOP and K - (prev + 1) >= max(1, min_codons):
            emit(f + 3 * (prev + 1), f + 3 * K, prev + 1, K - prev - 1)
    return out


def _rc(s: bytes) -> bytes:
    return bytes(orc.reverse_complement(np.frombuffer(s, np.uint8)[None, :])[0]) if s else b""


# hand-built reference rows (forward strand; the reverse complement of a planted ORF plants it on the '-' strand)
ROWS = [
    b"TAAATGAAACCCTGA",                 # stop as the first codon, ORF ending in the last codon
    b"ATGCCCTAGTAATGAATG",              # adjacent stops, ATG in the open tail (never an ORF)
    b"CCCATGAAAGGG",                    # ATG in a segment without a stop
    b"ATGAAATAA" + b"ATGTAA",            # ORFs of exactly 3 and 3-1 codons (min_codons = 3)
    b"atgaaacccgggtaa",                 # lower case
    b"ATGNAATAGATG-CCTGAATGCCCTAA",     # N and - inside codons
    _rc(b"ATGAAACCCGGGTTTTAA") + b"C",  # ORF on the '-' strand, len = 1 mod 3
    b"TTAGGTAAAGCATCATTT",              # stops only visible in the reverse complement
    b"", b"A", b"AT", b"ATG", b"TAAT", b"ATGTA",  # len 0 ... 5
    b"ATGAAATGA" * 4 + b"GG",          # len = 2 mod 3
]


@pytest.mark.parametrize("mode", [orf.ASIS, orf.STOPSTOP, orf.ATGSTOP])
@pytest.mark.parametrize("frames", [1, 3, 6])
@pytest.mark.parametrize("min_codons", [1, 2, 3, 25])
def test_mirror_equals_brute_force_hand_rows(mode, frames, min_codons):
    for ref in ROWS:
        assert orf.regions(ref, frames=frames, orf=mode, min_codons=min_codons) == brute_force(ref, frames, mode, min_codons), ref


def test_min_codons_boundary():
    ref = b"ATGAAATAA" + b"ATGTAA"       # ORFs of 3 and 2 codons on +1
    assert [r.codons for r in orf.regions(ref, frames=1, orf=orf.ATGSTOP, min_codons=3)] == [3]
    assert [r.codons for r in orf.regions(ref, frames=1, orf=orf.ATGSTOP, min_codons=2)] == [3, 2]
    assert [r.codons for r in orf.regions(ref, frames=1, orf=orf.STOPSTOP, min_codons=2)] == [3, 2]
    exact = b"ATGCCCTAA"
    assert len(orf.regions(exact, frames=1, orf=orf.ATGSTOP, min_codons=3)) == 1
    assert len(orf.regions(exact, frames=1, orf=orf.ATGSTOP, min_codons=4)) == 0


def test_asis_frame_plus1_is_whole_alignment():
    for L in range(0, 8):
        ref = b"ACGTACGT"[:L]
        rs = orf.regions(ref, frames=6, orf=orf.ASIS)
        assert len(rs) == 6
        assert (rs[0].col_begin, rs[0].col_end, rs[0].codons) == (0, L, L // 3)
        for r in rs:
            f = r.frame - 1
            assert r.codons == max(0, (L - f) // 3)
            assert r.col_end - r.col_begin == L - min(f, L)


@pytest.mark.parametrize("seed", range(12))
@pytest.mark.parametrize("L", [0, 1, 2, 3, 4, 5, 29, 30, 31, 299, 300, 301])
def test_mirror_equals_brute_force_random(seed, L):
    rng = np.random.default_rng(1000 * seed + L)
    # a row rich in stops and starts: random codons drawn from a small set, plus noise
    pieces = [b"ATG", b"TAA", b"TAG", b"TGA", b"CCC", b"GGA", b"AAA", b"tga", b"aTg", b"NNN", b"T-A", b"C", b"G"]
    ref = b"".join(pieces[i] for i in rng.integers(0, len(pieces), size=L))[:L]
    for frames in (1, 3, 6):
        for mode in (orf.ASIS, orf.STOPSTOP, orf.ATGSTOP):
            for mc in (1, 2, 5):
                assert orf.regions(ref, frames=frames, orf=mode, min_codons=mc) == brute_force(ref, frames, mode, mc)


@pytest.mark.parametrize("L", [0, 1, 2, 3, 4, 5, 6, 7, 8, 30, 31, 32])
def test_minus_strand_columns_pick_rc_slice(L):
    """S(r) taken through the input columns equals RC(A) sliced at the region's W columns, and every codon of it is the device's
    codon_minus reading at original column L-3-f-3k."""
    rng = np.random.default_rng(L)
    A = np.frombuffer(b"ACGTacgtN-", np.uint8)[rng.integers(0, 10, size=(3, L))]
    RC = orc.reverse_complement(A)
    for r in orf.regions(A[0], frames=6, orf=orf.ASIS):
        f = r.frame - 1
        S = orf.sub_alignment(A, r)
        if r.strand < 0:
            a, b = L - r.col_end, L - r.col_begin
            assert np.array_equal(S, RC[:, a:b])
            for k in range(r.codons):
                o = L - 3 - f - 3 * k
                comp = bytes(orc.reverse_complement(A[:1, o:o + 3])[0]).upper()
                assert orf.frame_codon(bytes(A[0]), -1, f, k) == comp
                assert np.array_equal(S[:, 3 * k:3 * k + 3], orc.reverse_complement(A[:, o:o + 3]))
        else:
            assert np.array_equal(S, A[:, r.col_begin:r.col_end])


def test_best_index_rule():
    nan = float("nan")
    assert orf.best_index([]) == -1
    assert orf.best_index([nan, nan]) == 0
    assert orf.best_index([nan, 1.0, 3.0, 3.0, nan]) == 2
    assert orf.best_index([-5.0, nan, -4.0]) == 2
    assert orf.best_index([2.0]) == 0


def _cli(*args):
    if not os.path.exists(BIN):
        pytest.fail(f"{BIN} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    return subprocess.run([BIN, "score-msa", *args, "100vertebrates", "/nonexistent/input.maf"], capture_output=True, text=True)


@pytest.mark.parametrize("args,msg", [
    (["--frames", "2"], "--frames must be 1, 3 or 6"),
    (["--frames", "six"], "--frames must be 1, 3 or 6"),
    (["--orf", "foo"], "--orf must be"),
    (["--min-codons", "0"], "--min-codons must be"),
    (["--strategy", "fixed_mean", "--genome-length", "100", "--coding-exons", "x.gff", "--frames", "6"], "FIXED_MEAN cannot"),
    (["--frames", "6", "--comp-phylo", "0"], "--comp-phylo 0 needs --all-scores 1"),
])
def test_cli_rejects_before_touching_a_device(args, msg):
    r = _cli(*args)
    assert r.returncode == 255, (r.stdout, r.stderr)
    assert msg in r.stdout


def test_region_kernels_do_not_spill(tmp_path):
    """Every kernel of the region path (and the strand-aware window consumers) compiles for sm_100a without local-memory spills."""
    import __graft_entry__ as g
    out = subprocess.run([g.NVCC] + [f for f in g.NVCC_FLAGS if f != "-shared"] + ["-c", "-Xptxas", "-v", "-o", str(tmp_path / "capi.o"),
                          os.path.join(g.CSRC, "pcsf_capi.cu")], capture_output=True, text=True, check=True).stderr
    props = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       out)
    seen = set()
    for name, _, st, ld in props:
        for k in ("k_orf_count", "k_orf_emit", "k_unit_offsets", "k_region_windows", "k_region_sums", "k_region_records",
                  "k_best_region", "k_keys_list", "k_insert", "k_tc5_ids", "k_omega_counts"):
            if k in name:
                seen.add(k)
                assert int(st) == 0 and int(ld) == 0, (name, st, ld)
    assert len(seen) == 11, seen
