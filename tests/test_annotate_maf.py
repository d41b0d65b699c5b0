"""annotate-with-maf: transcript alignments cut from whole-genome MAF chains (host/transcripts.hpp against the Python mirror
phylocsfpp_b200/transcripts.py), pcsf_score_given_regions against pcsf_score_msa, and the annotated files."""
import ctypes
import gzip
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi, orf
from phylocsfpp_b200 import transcripts as T
from phylocsfpp_b200.models import load_model
from tests.util import random_alignment

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")
sys.path.insert(0, os.path.join(ROOT, "tools"))
from annotate_maf_bench import write_annotation  # noqa: E402
from make_synth_maf import write_synth_maf  # noqa: E402

SETS = ["ensGene", "ncbiRefSeq", "refGene"]
STRATEGIES = {"fixed": capi.STRATEGY_FIXED, "mle": capi.STRATEGY_MLE, "omega": capi.STRATEGY_OMEGA}


def _gunzip(src, dst_dir):
    dst = os.path.join(dst_dir, os.path.basename(src)[:-3])
    with gzip.open(src, "rb") as fi, open(dst, "wb") as fo:
        shutil.copyfileobj(fi, fo)
    return dst


def _dump(model_arg, mafs, gffs):
    out = subprocess.run([BIN, "dump-transcripts", "--threads", "3", model_arg, ",".join(mafs)] + gffs, check=True, capture_output=True,
                         text=True).stdout.splitlines()
    assert out[0].startswith("# minus_chains ")
    return int(out[0].split()[-1]), out[1:]


@pytest.fixture(scope="module")
def birds(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("birds"))
    G = os.path.join(ROOT, "tests", "golden")
    maf = _gunzip(os.path.join(G, "build-tracks", "galGal6_chr22_25_28_each_30k_bases.maf.gz"), d)
    gtfs = [_gunzip(os.path.join(G, "annotate-with-tracks", f"galGal6_chr22_25_28_subset_{n}.gtf.gz"), d) for n in SETS]
    return dict(dir=d, model_arg=os.path.join(G, "build-tracks", "53birds"), model=load_model(os.path.join(G, "build-tracks", "53birds")),
                mafs=[maf], gffs=gtfs)


@pytest.fixture(scope="module")
def synth(tmp_path_factory):
    """12flies, chr1 from 985,001 over the 1 Mb breakpoint with holes; chr2 the same columns in a second MAF, with one block with
    the reference on '-'; a GTF and a GFF3 with '-' transcripts, phases 0-2, CDS across a hole and across the breakpoint, transcripts on
    a chromosome absent from the MAF, and transcripts without CDS with and without exon lines."""
    d = str(tmp_path_factory.mktemp("synth"))
    model = load_model("12flies")
    rng = np.random.default_rng(3)
    n = 30000
    mat = rng.choice(np.frombuffer(b"ACGTACGTacgtN-", np.uint8), size=(model.nl, n)).astype(np.uint8)
    mat[0] = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=n)
    m1 = os.path.join(d, "chr1.maf")
    write_synth_maf(m1, model, n, seed=4, start0=985000, mean_block=150, hole_p=1 / 40.0, ref_gap=0.01, alien_p=0.02, mat=mat)
    text = open(m1).read()
    ref_name = text.split("\ns ")[1].split(".")[0]
    m2 = os.path.join(d, "chr2.maf")
    with open(m2, "w") as fh:
        fh.write(text.replace(".chr1 ", ".chr2 "))
        fh.write(f"a score=0\ns {ref_name}.chr2 5000000 30 - 6000000 {'ACGTAC' * 5}\n\n")
    idx = T.ChainIndex([m1, m2], model)
    ch = idx.by_chrom["chr1"]
    hole = next((a, b) for a, b in zip(ch, ch[1:]) if a[1] < b[0])
    bp = next((a, b) for a, b in zip(ch, ch[1:]) if a[1] > b[0])          # the +2 columns past the breakpoint
    extra = [("chr1", "+", [(hole[0][1] - 100, hole[1][0] + 100)], [(hole[0][1] - 90, hole[1][0] + 90, 1)], True),
             ("chr2", "-", [(hole[0][1] - 200, hole[0][1] - 50), (hole[1][0] + 10, hole[1][0] + 300)],
              [(hole[0][1] - 180, hole[0][1] - 50, 2), (hole[1][0] + 10, hole[1][0] + 200, 1)], True),
             ("chr1", "-", [(bp[1][0] - 300, bp[1][0] + 300)], [(bp[1][0] - 250, bp[1][0] + 250, 2)], True),
             ("chr2", "+", [(999000, 999400), (999800, 1000500)], [(999100, 999400, 0), (999800, 1000400, 2)], True),
             ("chrUn", "+", [(1000, 1300)], [(1010, 1290, 1)], True),
             ("chrUn", "-", [(1000, 1300)], None, True),
             ("chr1", "+", [(990000, 990800)], None, False)]
    gtf, gff = os.path.join(d, "synth.gtf"), os.path.join(d, "synth.gff3")
    chroms = [("chr1", 985001, 985000 + n), ("chr2", 985001, 985000 + n)]
    write_annotation(gtf, chroms, 150, seed=8, fmt="gtf", extra=extra)
    write_annotation(gff, chroms, 150, seed=9, fmt="gff3", extra=extra[:4])
    return dict(dir=d, model_arg="12flies", model=model, mafs=[m1, m2], gffs=[gtf, gff], idx=idx, bp=bp, hole=hole)


def _check_dump(case, idx):
    minus, got = _dump(case["model_arg"], case["mafs"], case["gffs"])
    want = T.dump_lines(idx, case["gffs"])
    assert minus == idx.minus_chains
    assert got == want
    return want


def test_dump_transcripts_matches_mirror_on_birds(birds):
    idx = T.ChainIndex(birds["mafs"], birds["model"])
    rows = _check_dump(birds, idx)
    kinds = [r.split("\t")[2] for r in rows]
    assert kinds.count("transcript") >= 50 and kinds.count("CDS") >= 500
    # the MAF covers only parts of the transcripts: some regions are all N, some partly covered, some fully
    cover = []
    for path in birds["gffs"]:
        for rec in T.read_gff(path):
            x = T.extract_transcript(idx, rec, False)
            if x is not None:
                cover.append(float((x.seqs[0] != ord("N")).mean()) if x.L else 0.0)
    assert min(cover) == 0.0 and any(0.0 < c < 1.0 for c in cover) and max(cover) > 0.5


def test_dump_transcripts_matches_mirror_on_synthetic(synth):
    idx = synth["idx"]
    rows = _check_dump(synth, idx)
    assert idx.minus_chains == 1
    # the two chains around the breakpoint hold the same bytes in the columns both cover
    a, b = synth["bp"]
    assert a[1] - b[0] == 2 and np.array_equal(a[3][:, b[0] - a[0]:], b[3][:, :2])
    assert synth["hole"][0][1] < synth["hole"][1][0]
    recs = T.read_gff(synth["gffs"][0])
    xs = [T.extract_transcript(idx, r, True) for r in recs]
    xs_rec = [(x, r) for x, r in zip(xs, recs) if x is not None]
    assert any(x.coding and x.strand == "-" for x, _ in xs_rec)
    phases = {g.phase for _, r in xs_rec for g in r if g.feature == b"CDS"}
    assert {1, 2} <= phases
    assert any(not x.coding and not any(g.feature == b"exon" for g in r) for x, r in xs_rec)
    assert any(not x.coding and any(g.feature == b"exon" for g in r) for x, r in xs_rec)
    chrun = [x for x, r in xs_rec if any(g.feature == b"transcript" and g.chrom == "chrUn" for g in r)]
    assert len(chrun) == 2 and all((x.seqs == ord("N")).all() and x.ref_row == -1 for x in chrun)
    # the first transcript's CDS crosses a hole: N columns inside, bases on both sides
    row = xs_rec[0][0].seqs[0]
    assert (row == ord("N")).any() and (row != ord("N")).any()
    assert len(rows) > 300


def test_given_regions_rejected_before_any_device_is_touched():
    """Argument and range checks run before the handle is used: an opaque zeroed buffer stands in for the model here."""
    lib = capi.load()
    fake = ctypes.create_string_buffer(4096)
    seqs = np.frombuffer(b"ACGTAC" * 2, np.uint8).copy()
    off, ln = np.array([0], np.int64), np.array([6], np.int64)

    def call(aln, b, e, n=1, strategy=capi.STRATEGY_FIXED):
        ra, rb, re_ = np.array([aln], np.int32), np.array([b], np.int64), np.array([e], np.int64)
        ph = np.zeros(1, np.float32)
        return lib.pcsf_score_given_regions(fake, strategy, 1, seqs.ctypes.data, off.ctypes.data, ln.ctypes.data, n, ra.ctypes.data,
                                            rb.ctypes.data, re_.ctypes.data, ph.ctypes.data, None, None)
    for args in ((0, 4, 3), (0, 0, 7), (0, -1, 3), (1, 0, 3), (-1, 0, 3)):
        assert call(*args) == capi.PCSF_ERR_INVALID, args
        assert b"region 0" in lib.pcsf_last_error()
    assert call(0, 0, 3, n=-1) == capi.PCSF_ERR_INVALID
    assert call(0, 0, 3, strategy=7) == capi.PCSF_ERR_INVALID


# ------------------------------------------------------------------------------------------------------------------------ GPU
def _annotate(case, out, *opts, gffs=None):
    r = subprocess.run([BIN, "annotate-with-maf", "--output", out] + list(opts) + [case["model_arg"], ",".join(case["mafs"])] +
                       (gffs or case["gffs"]), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r


def _out_path(out, gff):
    base, ext = os.path.splitext(os.path.basename(gff))
    return os.path.join(out, base + ".PhyloCSF++maf" + ext)


def _attributes(line):
    """(line without the appended attributes, {key: value}) for GFF3 (;k=v) and GTF ( k "v";) syntax."""
    if ";phylocsf_" in line:
        head, tail = line.split(";phylocsf_", 1)
        kv = dict(p.split("=", 1) for p in ("phylocsf_" + tail).split(";"))
        return head, kv
    if ' phylocsf_' in line:
        head, tail = line.split(" phylocsf_", 1)
        kv = {}
        for p in ("phylocsf_" + tail).split(";"):
            p = p.strip()
            if p:
                k, v = p.split(" ", 1)
                kv[k] = v.strip('"')
        return head, kv
    return line, {}


@pytest.mark.gpu
@pytest.mark.parametrize("strategy", ["fixed", "mle", "omega"])
def test_score_given_regions_equals_score_msa_on_extracted(strategy):
    model = load_model("29mammals", "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat")
    dm = capi.DeviceModel(model)
    rng = np.random.default_rng(21)
    alns = [random_alignment(model.nl, L, seed=300 + i, gap=0.2, conserve=0.8) for i, L in enumerate((0, 2, 3, 7, 40, 151, 302, 600))]
    ra, rb, re_ = [], [], []
    for i, a in enumerate(alns):
        L = a.shape[1]
        ra += [i, i]; rb += [0, L]; re_ += [L, L]          # the whole alignment and an empty range at its end
        if L >= 3:
            b = int(rng.integers(0, L - 2))
            ra.append(i); rb.append(b); re_.append(b + 3)          # one codon
        for _ in range(3):
            b = int(rng.integers(0, L + 1)); e = int(rng.integers(b, L + 1))
            ra.append(i); rb.append(b); re_.append(e)
    order = rng.permutation(len(ra))
    ra, rb, re_ = [ra[k] for k in order], [rb[k] for k in order], [re_[k] for k in order]
    subs = [np.ascontiguousarray(alns[a][:, b:e]) for a, b, e in zip(ra, rb, re_)]
    st = STRATEGIES[strategy]
    anc_ok = strategy != "omega"
    want = dm.score_msa(subs, st, comp_anc=anc_ok, comp_bls=True)
    for comp_anc, comp_bls in ((anc_ok, True), (False, False), (anc_ok, False)):
        got = dm.score_given_regions(alns, ra, rb, re_, st, comp_anc=comp_anc, comp_bls=comp_bls)
        assert np.array_equal(got[0], want[0], equal_nan=True)
        if comp_anc:
            assert np.array_equal(got[1], want[1], equal_nan=True)
        if comp_bls:
            assert np.array_equal(got[2], want[2], equal_nan=True)
    if strategy == "omega":
        got = dm.score_given_regions(alns, ra, rb, re_, st, comp_anc=True)
        assert np.isnan(got[1]).all()
    with pytest.raises(capi.PcsfError) as e:
        dm.score_given_regions(alns, [0], [0], [1])
    assert e.value.status == capi.PCSF_ERR_INVALID
    dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("strategy", ["fixed", "mle"])
def test_annotation_scores_equal_score_msa_and_oracle(birds, synth, tmp_path, strategy):
    st = STRATEGIES[strategy]
    for case in (birds, synth):
        out = os.path.join(str(tmp_path), strategy + os.path.basename(case["dir"]))
        opts = ["--strategy", strategy, "--comp-anc", "1", "--threads", "4"]
        _annotate(case, out, *opts)
        model = case["model"]
        idx = T.ChainIndex(case["mafs"], model)
        dm = capi.DeviceModel(model)
        mc, mnc = orc.OracleModel(model.tree, model.S_c, model.f_c), orc.OracleModel(model.tree, model.S_nc, model.f_nc)
        n_checked, tight, n_oracle = 0, 0, 0
        for gff in case["gffs"]:
            src = open(gff, "rb").read()
            got = open(_out_path(out, gff), "rb").read()
            stripped = "\n".join(_attributes(ln)[0] for ln in got.decode().split("\n")).encode()
            assert stripped == src          # every input line, unchanged, and nothing else
            lines = got.decode().split("\n")
            subs, keys = [], []
            li = 0
            for rec in T.read_gff(gff):
                x = T.extract_transcript(idx, rec, False)
                for k, g in enumerate(rec):
                    kv = _attributes(lines[li + k])[1]
                    if x is None or g.feature not in (b"transcript", b"CDS"):
                        assert not kv
                        continue
                    r = 0 if g.feature == b"transcript" else 1 + sum(1 for h in rec[:k] if h.feature == b"CDS")
                    b, e = x.regions[r]
                    subs.append(np.ascontiguousarray(x.seqs[:, b:e]))
                    keys.append(kv)
                li += len(rec)
            phylo, anc, bls = dm.score_msa(subs, st)
            for s, kv, p, a, bl in zip(subs, keys, phylo, anc, bls):
                assert kv["phylocsf_score"] == "%.6f" % p and kv["phylocsf_anc"] == "%.6f" % a and kv["phylocsf_bls"] == "%.6f" % bl
                assert int(kv["phylocsf_codons"]) == s.shape[1] // 3
                n_checked += 1
            # the oracle on a spread of the regions (MLE: the Brent-fork allowance of the score-msa tests)
            for s, p, a in list(zip(subs, phylo, anc))[::max(1, len(subs) // 40)]:
                n_oracle += 1
                if strategy == "fixed":
                    rp, ra_ = orc.run_fixed(mc, mnc, orc.translate(s), True)
                    assert abs(float(p) - float(rp)) <= 1e-3 and abs(float(a) - float(ra_)) <= 1e-3
                else:
                    rp, ra_, _info = orc.run_mle(mc, mnc, orc.translate(s), True)
                    assert (float(p) - float(rp)) ** 2 <= 0.001 and (float(a) - float(ra_)) ** 2 <= 0.001
                    tight += abs(float(p) - float(rp)) <= 1e-3 and abs(float(a) - float(ra_)) <= 1e-3
        assert n_checked > 100
        if strategy == "mle":
            assert tight >= n_oracle - max(1, n_oracle // 50)
        dm.close()


@pytest.mark.gpu
def test_find_orf_reports_the_mirror_best_orf(synth, tmp_path):
    out = str(tmp_path / "orf")
    _annotate(synth, out, "--strategy", "fixed", "--find-orf", "1", "--min-codons", "5", "--threads", "3")
    model, idx = synth["model"], synth["idx"]
    dm = capi.DeviceModel(model)
    n_found, n_none = 0, 0
    for gff in synth["gffs"]:
        lines = open(_out_path(out, gff)).read().split("\n")
        li = 0
        for rec in T.read_gff(gff):
            x = T.extract_transcript(idx, rec, True)
            kv = _attributes(lines[li + [g.feature for g in rec].index(b"transcript")])[1] if x is not None else {}
            li += len(rec)
            if x is None or x.coding:
                continue
            regs = orf.regions(x.seqs[x.ref_row], frames=3, orf=orf.ATGSTOP, min_codons=5) if x.ref_row >= 0 else []
            if not regs:
                assert kv["phylocsf_orf_start"] == "." and kv["phylocsf_orf_score"] == "nan"
                n_none += 1
                continue
            phylo, _, bls = dm.score_msa([orf.sub_alignment(x.seqs, r) for r in regs], capi.STRATEGY_FIXED)
            best = regs[orf.best_index(phylo)]
            g0, g1 = x.genomic(best.col_begin), x.genomic(best.col_end - 1)
            assert kv["phylocsf_orf_score"] == "%.6f" % phylo[orf.best_index(phylo)]
            assert (int(kv["phylocsf_orf_start"]), int(kv["phylocsf_orf_end"])) == (min(g0, g1), max(g0, g1))
            assert int(kv["phylocsf_orf_codons"]) == best.codons
            # the reported genomic interval, cut through the exons in transcript orientation, reads ATG ... stop on the reference row
            cols = [j for j in range(x.L) if min(g0, g1) <= x.genomic(j) <= max(g0, g1)]
            codons = bytes(x.seqs[x.ref_row, cols]).upper()
            assert codons[:3] == b"ATG" and codons[-3:] in (b"TAA", b"TAG", b"TGA")
            n_found += 1
    assert n_found >= 5 and n_none >= 1
    dm.close()


@pytest.mark.gpu
def test_output_independent_of_threads_and_gpus(synth, birds, tmp_path):
    import torch
    for case in (synth, birds):
        outs = {}
        for tag, opts in (("t1", ["--threads", "1", "--gpus", "1"]), ("t8", ["--threads", "8", "--gpus", "1"]), ("g2", ["--threads", "8", "--gpus", "2"])):
            if tag == "g2" and torch.cuda.device_count() < 2:
                continue
            out = os.path.join(str(tmp_path), tag + os.path.basename(case["dir"]))
            _annotate(case, out, "--strategy", "mle", "--find-orf", "1", *opts)
            outs[tag] = [open(_out_path(out, g), "rb").read() for g in case["gffs"]]
        assert outs["t1"] == outs["t8"]
        if "g2" in outs:
            assert outs["g2"] == outs["t1"]
    if torch.cuda.device_count() < 2:
        pytest.skip("one device: --gpus 2 against --gpus 1 not checked")


@pytest.mark.gpu
def test_command_line_errors(synth, tmp_path):
    out = str(tmp_path / "e")
    base = [BIN, "annotate-with-maf", "--output", out]
    tail = [synth["model_arg"], ",".join(synth["mafs"]), synth["gffs"][0]]
    r = subprocess.run(base + ["--strategy", "bogus"] + tail, capture_output=True, text=True)
    assert r.returncode != 0 and "valid strategy" in r.stdout
    r = subprocess.run(base + ["--strategy", "omega", "--comp-anc", "1"] + tail, capture_output=True, text=True)
    assert r.returncode != 0 and "Omega" in r.stdout
    bad = os.path.join(str(tmp_path), "bad.maf")
    open(bad, "w").write(open(synth["mafs"][0]).read().replace("ACGT", "ACJT", 50))
    r = subprocess.run(base + [synth["model_arg"], bad, synth["gffs"][0]], capture_output=True, text=True)
    assert r.returncode == 37
