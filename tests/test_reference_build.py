"""The reference itself as the checker.

oracle/_ref/phylocsf_ref is the reference's UNMODIFIED build-tracks / score-msa compiled where the sources lie in a PhyloCSF++
checkout with oracle/ref/gsl standing in for the absent GSL (oracle/ref/Makefile).  Three layers:

  1. (CPU, needs the binary) the shim-built reference reproduces the reference's own golden files -> the shim is sound;
  2. (CPU) the oracle restatement + the Python reader mirror reproduce what the reference wrote for the synthetic inputs of
     tests/golden/ref-generated/ (made by tests/golden/make_ref_fixtures.py): a chain crossing the 1 Mb breakpoint, holes,
     reference gaps, unknown species, --species reduction, single-block alignments;
  3. (GPU) the product (C++ host over the C-ABI over the CUDA kernels) reproduces the same files.

The differential runs (4.) feed fresh synthetic MAFs to the oracle and to the product and compare what they write with what the
reference binary writes for the same input, stored as sha256 digests in tests/golden/ref-generated/digests.json
(tests/golden/make_ref_digests.py), so that they need no binary outside the repository.
"""
import gzip
import hashlib
import json
import os
import shutil
import subprocess
from multiprocessing import get_context

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import tracks
from phylocsfpp_b200.maf import MafReader
from phylocsfpp_b200.models import load_model
from tests.util import read_lines

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "phylocsf_ref")
BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")
DIGESTS = os.path.join(ROOT, "tests", "golden", "ref-generated", "digests.json")
SPECIES29 = "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat"
WIGS = ["PhyloCSFpower.wig"] + [f"PhyloCSFRaw{s}{f}.wig" for s in "+-" for f in (1, 2, 3)]


def _gunzip(src, dst):
    with gzip.open(src, "rb") as fi, open(dst, "wb") as fo:
        shutil.copyfileobj(fi, fo)
    return dst


def _rows(path):
    return [ln.rstrip("\n").split("\t") for ln in open(path) if not ln.startswith("#") and not ln.startswith("seq\t")]


def _need_ref():
    if not os.path.exists(REF):
        pytest.skip("oracle/_ref/phylocsf_ref not built (needs the reference's sources: `make -C oracle/ref REF=<PhyloCSF++ checkout>`)")


def _sha(data: bytes) -> str:
    return hashlib.sha256(data).hexdigest()


def _ref_digest(group: str, key: str):
    """What the reference binary wrote for one input: sha256 per output (tests/golden/make_ref_digests.py)."""
    with open(DIGESTS) as fh:
        return json.load(fh)[group][key]


# ------------------------------------------------------------------------------------------------ 1. the shim is sound
def test_shim_built_reference_reproduces_reference_goldens(golden_dir, tmp_path):
    """test/tests.sh:15-19 (without the smoothing inputs the repository does not ship) and :35-37, run with the shim build:
    7 wig files byte-identical, FIXED .scores identical."""
    _need_ref()
    G = os.path.join(golden_dir, "build-tracks")
    maf = _gunzip(os.path.join(G, "galGal6_chr22_25_28_each_30k_bases.maf.gz"), os.path.join(str(tmp_path), "in.maf"))
    out = os.path.join(str(tmp_path), "bt")
    threads = str(min(8, os.cpu_count() or 1))
    subprocess.run([REF, "build-tracks", "--threads", threads, "--output", out, os.path.join(G, "53birds"), maf], check=True,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    for n in WIGS:
        assert open(os.path.join(out, n), "rb").read() == gzip.open(os.path.join(G, n + ".gz"), "rb").read(), n
    S = os.path.join(golden_dir, "score-msa")
    maf = shutil.copy(os.path.join(S, "chr22.50alignments.maf"), os.path.join(str(tmp_path), "small.maf"))
    subprocess.run([REF, "score-msa", "--threads", threads, "--strategy", "fixed", "--comp-phylo", "1", "--comp-anc", "1",
                    "100vertebrates", maf], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    assert _rows(maf + ".scores") == _rows(os.path.join(S, "chr22.50alignments.fixed.scores"))


# ------------------------------------------------------------------------------------------------ 2. oracle vs reference
_W = {}


def _init(name):
    m = load_model(name)
    _W["m"] = (orc.OracleModel(m.tree, m.S_c, m.f_c), orc.OracleModel(m.tree, m.S_nc, m.f_nc))


def _work(pep):
    return orc.run_tracks(_W["m"][0], _W["m"][1], pep)


def test_oracle_and_reader_mirror_vs_reference_tracks12(golden_dir):
    R = os.path.join(golden_dir, "ref-generated")
    m = load_model("12flies")
    alns = list(MafReader(os.path.join(R, "tracks12.maf.gz"), m.seqid_to_phyloid, m.nl, True, warn=False))
    assert len(alns) >= 3 and any(a.start_pos <= 1000000 < a.start_pos + a.L for a in alns)   # a chain that meets BREAKPOINT_POS
    out = {k: [] for k in tracks.FRAMES}
    power = []
    with get_context("fork").Pool(min(8, os.cpu_count() or 1), initializer=_init, initargs=("12flies",)) as pool:
        for a in alns:
            plus, minus = orc.window_codons(a.seqs)
            W = plus.shape[1]
            chunks = [np.ascontiguousarray(x[:, i:i + 500]) for x in (plus, minus) for i in range(0, W, 500)]
            res = pool.map(_work, chunks)
            half = len(res) // 2
            p, mi = np.concatenate(res[:half]), np.concatenate(res[half:])
            b = orc.bls(m.tree, a.seqs)[1]
            power += tracks.power_wig(a.chrom, a.start_pos, b)
            r = tracks.raw_wigs(a.chrom, a.start_pos, a.chrom_len, p, mi, b)
            for k in out:
                out[k] += r[k]
    assert power == read_lines(os.path.join(R, "tracks12.PhyloCSFpower.wig.gz"))
    for (s, f), lines in out.items():
        assert lines == read_lines(os.path.join(R, "tracks12." + tracks.wig_filename(s, f) + ".gz")), (s, f)


def test_oracle_vs_reference_msa29(golden_dir):
    R = os.path.join(golden_dir, "ref-generated")
    m = load_model("29mammals", SPECIES29)
    mc, mnc = orc.OracleModel(m.tree, m.S_c, m.f_c), orc.OracleModel(m.tree, m.S_nc, m.f_nc)
    alns = list(MafReader(os.path.join(R, "msa29.maf.gz"), m.seqid_to_phyloid, m.nl, False, warn=False))
    fixed, mle = _rows(os.path.join(R, "msa29.fixed.scores")), _rows(os.path.join(R, "msa29.mle.scores"))
    assert len(alns) == len(fixed) == len(mle)
    exact = 0
    for i, (a, g) in enumerate(zip(alns, fixed)):
        s, anc = orc.run_fixed(mc, mnc, orc.translate(a.seqs), True)
        b = orc.bls(m.tree, a.seqs, per_base=False)[0]
        assert [a.chrom, str(a.start_pos), str(a.start_pos + a.L - 1), a.strand] == g[:4]
        assert "%.6f" % np.float32(b) == g[6]
        assert abs(float(s) - float(g[4])) <= 1e-3 and abs(float(anc) - float(g[5])) <= 1e-3
        exact += ("%.6f" % s == g[4]) + ("%.6f" % anc == g[5])
    assert exact >= 2 * len(alns) - 2          # float32 print noise at most
    tight = 0
    picks = list(range(0, len(alns), 4))
    for i in picks:
        s, anc, info = orc.run_mle(mc, mnc, orc.translate(alns[i].seqs), True)
        gs, ga = float(mle[i][4]), float(mle[i][5])
        assert (float(s) - gs) ** 2 <= 0.001 and (float(anc) - ga) ** 2 <= 0.001, (i, s, anc, mle[i])   # test/tests.sh:41
        tight += abs(float(s) - gs) <= 1e-3 and abs(float(anc) - ga) <= 1e-3
    assert tight >= len(picks) - 1


def test_oracle_omega_vs_reference_msa29(golden_dir):
    """OMEGA restatement (orc_omega) against the reference's own output: the reference's CI tolerance for this strategy is
    a squared error of 0.1 (test/tests.sh:46) because the result is the LAST Brent evaluation of a 1 %-bracket search."""
    R = os.path.join(golden_dir, "ref-generated")
    m = load_model("29mammals", SPECIES29)
    alns = list(MafReader(os.path.join(R, "msa29.maf.gz"), m.seqid_to_phyloid, m.nl, False, warn=False))
    gold = _rows(os.path.join(R, "msa29.omega.scores"))
    assert len(alns) == len(gold)
    close = 0
    picks = [0, 2, 5, 7, 10, 12]
    for i in picks:
        s, info = orc.run_omega(m.tree, orc.translate(alns[i].seqs))
        assert info["status"] == 0 and 150 <= info["evals"] <= 12 * 260
        assert (float(s) - float(gold[i][4])) ** 2 <= 0.1, (i, s, gold[i])
        close += abs(float(s) - float(gold[i][4])) <= 0.01
    assert close >= 2


# ------------------------------------------------------------------------------------------------ 3. product vs reference
@pytest.mark.gpu
def test_cli_build_tracks_vs_reference_tracks12(golden_dir, tmp_path):
    R = os.path.join(golden_dir, "ref-generated")
    maf = _gunzip(os.path.join(R, "tracks12.maf.gz"), os.path.join(str(tmp_path), "tracks12.maf"))
    for prec, threads in (("f64", 1), ("f64", 4), ("tc5", 3)):
        out = os.path.join(str(tmp_path), f"o_{prec}_{threads}")
        subprocess.run([BIN, "build-tracks", "--threads", str(threads), "--precision", prec, "--output", out, "12flies", maf], check=True,
                       capture_output=True)
        for n in WIGS:
            ours = open(os.path.join(out, n)).read().split("\n")
            gold = gzip.open(os.path.join(R, "tracks12." + n + ".gz"), "rt").read().split("\n")
            if prec == "f64":
                assert ours == gold, n
            else:
                assert len(ours) == len(gold)
                for x, y in zip(ours, gold):
                    if x != y:
                        assert not x.startswith("fixedStep") and abs(float(x) - float(y)) <= 0.0011, (n, x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("strategy", ["fixed", "mle"])
def test_cli_score_msa_vs_reference_msa29(golden_dir, tmp_path, strategy):
    R = os.path.join(golden_dir, "ref-generated")
    maf = _gunzip(os.path.join(R, "msa29.maf.gz"), os.path.join(str(tmp_path), "msa29.maf"))
    out = os.path.join(str(tmp_path), "o")
    subprocess.run([BIN, "score-msa", "--strategy", strategy, "--comp-anc", "1", "--species", SPECIES29, "--output", out, "29mammals", maf],
                   check=True, capture_output=True)
    ours, gold = _rows(os.path.join(out, "msa29.maf.scores")), _rows(os.path.join(R, f"msa29.{strategy}.scores"))
    assert len(ours) == len(gold)
    loose = 0
    for o, g in zip(ours, gold):
        assert o[:4] == g[:4] and o[6] == g[6]
        d = max(abs(float(o[4]) - float(g[4])), abs(float(o[5]) - float(g[5])))
        if strategy == "fixed":
            assert d <= 1e-3
        else:
            assert d ** 2 <= 0.001          # the reference's own CI tolerance (test/tests.sh:41)
            loose += d > 1e-3               # a Brent trajectory that forks on ~1e-13 differences in P(t) (DESIGN.md section 7)
    assert loose <= max(1, len(gold) // 25)


@pytest.mark.gpu
def test_cli_score_msa_omega_vs_reference_msa29(golden_dir, tmp_path):
    """score-msa --strategy omega (batched Jacobi eigensolver + twelve Brent fits per alignment on the GPU) against the
    reference's own output, at the reference's CI tolerance for this strategy (squared error <= 0.1, test/tests.sh:46)."""
    R = os.path.join(golden_dir, "ref-generated")
    maf = _gunzip(os.path.join(R, "msa29.maf.gz"), os.path.join(str(tmp_path), "msa29.maf"))
    out = os.path.join(str(tmp_path), "o")
    subprocess.run([BIN, "score-msa", "--strategy", "omega", "--species", SPECIES29, "--output", out, "29mammals", maf], check=True, capture_output=True)
    ours, gold = _rows(os.path.join(out, "msa29.maf.scores")), _rows(os.path.join(R, "msa29.omega.scores"))
    assert len(ours) == len(gold)
    d = []
    for o, g in zip(ours, gold):
        assert o[:4] == g[:4] and o[5] == g[5] and len(o) == 6
        d.append(abs(float(o[4]) - float(g[4])))
    print("omega |d| vs reference: max %.3g, median %.3g, <=1e-2: %d of %d" % (max(d), sorted(d)[len(d) // 2], sum(x <= 1e-2 for x in d), len(d)))
    assert max(d) ** 2 <= 0.1
    r = subprocess.run([BIN, "score-msa", "--strategy", "omega", "--comp-anc", "1", "29mammals", maf], capture_output=True, text=True)
    assert r.returncode != 0 and "Omega mode" in r.stdout


@pytest.mark.gpu
def test_cli_score_msa_fixed_mean_vs_reference_msa29(golden_dir, tmp_path):
    """score-msa --strategy fixed_mean (score_msa.hpp:136-213): per-codon decibans from the CUDA tracks path through the host's
    PhyloCSF-HMM, mean posterior log-odds per alignment — against the reference's own output."""
    from tests.util import write_synthetic_exons
    R = os.path.join(golden_dir, "ref-generated")
    maf = _gunzip(os.path.join(R, "msa29.maf.gz"), os.path.join(str(tmp_path), "msa29.maf"))
    exons = os.path.join(str(tmp_path), "exons.txt")
    write_synthetic_exons(exons)
    out = os.path.join(str(tmp_path), "o")
    subprocess.run([BIN, "score-msa", "--strategy", "fixed_mean", "--species", SPECIES29, "--genome-length", "400000000", "--coding-exons", exons,
                    "--output", out, "29mammals", maf], check=True, capture_output=True)
    ours, gold = _rows(os.path.join(out, "msa29.maf.scores")), _rows(os.path.join(R, "msa29.fixed_mean.scores"))
    assert len(ours) == len(gold)
    exact = 0
    for o, g in zip(ours, gold):
        assert o[:4] == g[:4] and o[5] == g[5]
        assert abs(float(o[4]) - float(g[4])) <= 1e-4
        exact += o[4] == g[4]
    assert exact >= len(gold) - 2
    r = subprocess.run([BIN, "score-msa", "--strategy", "fixed_mean", "29mammals", maf], capture_output=True, text=True)
    assert r.returncode != 0 and "FIXED_MEAN" in r.stdout


# ------------------------------------------------------------------------------------------------ 4. differential runs
def _oracle_build_tracks(model_name, maf, threshold=0.1, species=""):
    """The oracle + reader-mirror pipeline of build-tracks: dict file name -> list of lines."""
    m = load_model(model_name, species) if species else load_model(model_name)
    mc, mnc = orc.OracleModel(m.tree, m.S_c, m.f_c), orc.OracleModel(m.tree, m.S_nc, m.f_nc)
    out = {tracks.wig_filename(s, f): [] for s, f in tracks.FRAMES}
    out["PhyloCSFpower.wig"] = []
    for a in MafReader(maf, m.seqid_to_phyloid, m.nl, True, warn=False):
        if a.L == 0:
            continue
        plus, minus = orc.window_codons(a.seqs)
        p, mi = orc.run_tracks(mc, mnc, plus), orc.run_tracks(mc, mnc, minus)
        b = orc.bls(m.tree, a.seqs)[1]
        out["PhyloCSFpower.wig"] += tracks.power_wig(a.chrom, a.start_pos, b)
        for (s, f), lines in tracks.raw_wigs(a.chrom, a.start_pos, a.chrom_len, p, mi, b, threshold=threshold).items():
            out[tracks.wig_filename(s, f)] += lines
    return out


def oracle_build_tracks_for(model_name, maf, extra):
    """_oracle_build_tracks with the options of a build-tracks command line: dict file name -> file contents (bytes)."""
    threshold = 0.1
    species = ""
    if "--power-threshold" in extra:
        threshold = 1.0 if extra[extra.index("--power-threshold") + 1] in ("1", "true", "one") else 0.0
    if "--species" in extra:
        species = extra[extra.index("--species") + 1]
    return {n: "".join(ln + "\n" for ln in lines).encode() for n, lines in _oracle_build_tracks(model_name, maf, threshold, species).items()}


def write_differential_maf(kind, path, model_name, cols, seed):
    """The synthetic MAF of one differential case (CPU generator: the same bytes on every machine)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    os.environ["PCSF_SYNTH_CPU"] = "1"
    from make_synth_maf import write_synth_maf
    kw = {"oracle": dict(mean_block=70, hole_p=1 / 15.0, ref_gap=0.03, alien_p=0.1),
          "cli": dict(mean_block=80, hole_p=1 / 20.0, ref_gap=0.03, alien_p=0.1),
          "acceptance": dict(mean_block=120, hole_p=1 / 40.0, ref_gap=0.02, alien_p=0.05, start0=1000000 - cols // 2)}[kind]
    write_synth_maf(path, load_model(model_name), cols, seed=seed, **kw)


ORACLE_CASES = [("7yeast", 2500, 21, []), ("20flies", 1800, 22, []), ("12flies", 2200, 23, ["--power-threshold", "1"]),
                ("12flies", 2200, 24, ["--power-threshold", "0.5"]), ("29mammals", 900, 25, ["--species", SPECIES29])]
CLI_CASES = [("20flies", 6000, 41, []), ("53birds", 4000, 42, ["--power-threshold", "1"]), ("29mammals", 5000, 43, ["--species", SPECIES29])]
ACCEPTANCE_CASES = [("58mammals", 60000, 51), ("100vertebrates", 50000, 52)]
MODEL_INFO_MODELS = ["100vertebrates", "53birds", "23flies", "7yeast"]


@pytest.mark.parametrize("model_name,cols,seed,extra", ORACLE_CASES)
def test_differential_build_tracks_oracle_vs_reference_binary(tmp_path, model_name, cols, seed, extra):
    """Fresh synthetic MAFs (holes, reference gaps, unknown species) through the oracle + reader mirror: byte for byte the wig files
    the reference binary writes for them.  Includes the --power-threshold quirk (read with get_bool, build_tracks.hpp:416-417: "1"
    gives 1.0, anything else 0.0) and a --species reduction."""
    maf = os.path.join(str(tmp_path), "d.maf")
    write_differential_maf("oracle", maf, model_name, cols, seed)
    ours = oracle_build_tracks_for(model_name, maf, extra)
    gold = _ref_digest("build_tracks", f"{model_name}-{seed}")
    for n in WIGS:
        assert _sha(ours[n]) == gold[n], n


@pytest.mark.parametrize("model_name,seed", [("7yeast", 31), ("12flies", 32)])
def test_differential_score_msa_oracle_vs_reference_binary(tmp_path, model_name, seed):
    """Single-block alignments through the reference binary (FIXED with the ancestral score, and MLE) and through the oracle."""
    _need_ref()
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    os.environ["PCSF_SYNTH_CPU"] = "1"
    from make_synth_maf import write_synth_maf
    m = load_model(model_name)
    maf = os.path.join(str(tmp_path), "b.maf")
    write_synth_maf(maf, m, 2500, seed=seed, loguniform_blocks=(20, 300), alien_p=0.1)
    alns = list(MafReader(maf, m.seqid_to_phyloid, m.nl, False, warn=False))
    mc, mnc = orc.OracleModel(m.tree, m.S_c, m.f_c), orc.OracleModel(m.tree, m.S_nc, m.f_nc)
    for strategy in ("fixed", "mle"):
        out = os.path.join(str(tmp_path), "o_" + strategy)
        subprocess.run([REF, "score-msa", "--threads", "4", "--strategy", strategy, "--comp-phylo", "1", "--comp-anc", "1", "--output", out, model_name, maf],
                       check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        gold = _rows(os.path.join(out, "b.maf.scores"))
        assert len(gold) == len(alns) >= 8
        forked = 0
        for a, g in zip(alns, gold):
            assert [a.chrom, str(a.start_pos), str(a.start_pos + a.L - 1), a.strand] == g[:4]
            assert "%.6f" % np.float32(orc.bls(m.tree, a.seqs, per_base=False)[0]) == g[6]
            pep = orc.translate(a.seqs)
            if strategy == "fixed":
                s, anc = orc.run_fixed(mc, mnc, pep, True)
                assert abs(float(s) - float(g[4])) <= 1e-3 and abs(float(anc) - float(g[5])) <= 1e-3
            else:
                s, anc, _ = orc.run_mle(mc, mnc, pep, True)
                d = max(abs(float(s) - float(g[4])), abs(float(anc) - float(g[5])))
                assert d ** 2 <= 0.001          # test/tests.sh:41
                forked += d > 1e-3
        assert forked <= 1


@pytest.mark.gpu
@pytest.mark.parametrize("model_name,cols,seed,extra", CLI_CASES)
def test_differential_cli_vs_reference_binary(tmp_path, model_name, cols, seed, extra):
    """The product's command line on a fresh synthetic MAF: on the FP64 path, byte for byte the seven wig files the reference binary
    writes for it."""
    maf = os.path.join(str(tmp_path), "d.maf")
    write_differential_maf("cli", maf, model_name, cols, seed)
    our_out = os.path.join(str(tmp_path), "ours")
    subprocess.run([BIN, "build-tracks", "--threads", "3", "--output", our_out] + extra + [model_name, maf], check=True, capture_output=True)
    gold = _ref_digest("build_tracks", f"{model_name}-{seed}")
    for n in WIGS:
        assert _sha(open(os.path.join(our_out, n), "rb").read()) == gold[n], n


def test_differential_omega_oracle_vs_reference_binary(tmp_path):
    """OMEGA on fresh single-block alignments (7yeast): the reference binary against orc_omega, at the reference's CI tolerance for this
    strategy (squared error <= 0.1, test/tests.sh:46); most rows agree far better."""
    _need_ref()
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    os.environ["PCSF_SYNTH_CPU"] = "1"
    from make_synth_maf import write_synth_maf
    m = load_model("7yeast")
    maf = os.path.join(str(tmp_path), "b.maf")
    write_synth_maf(maf, m, 1500, seed=51, loguniform_blocks=(30, 300), alien_p=0.0)
    alns = list(MafReader(maf, m.seqid_to_phyloid, m.nl, False, warn=False))
    out = os.path.join(str(tmp_path), "o")
    subprocess.run([REF, "score-msa", "--threads", "8", "--strategy", "omega", "--comp-phylo", "1", "--comp-anc", "0", "--output", out, "7yeast", maf],
                   check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    gold = _rows(os.path.join(out, "b.maf.scores"))
    assert len(gold) == len(alns) >= 6
    d = []
    for a, g in zip(alns, gold):
        s, info = orc.run_omega(m.tree, orc.translate(a.seqs))
        assert info["status"] == 0
        d.append(abs(float(s) - float(g[4])))
    assert max(d) ** 2 <= 0.1, d
    assert sorted(d)[len(d) // 2] <= 0.02, d


@pytest.mark.parametrize("model_name", MODEL_INFO_MODELS)
def test_model_info_matches_reference_binary(model_name):
    """--model-info (run.hpp:213-232): species and alternative names, the text the reference binary writes, from both sub-commands."""
    for tool in ("build-tracks", "score-msa"):
        ours = subprocess.run([BIN, tool, "--model-info", model_name], capture_output=True, text=True, check=True).stdout
        assert _sha(ours.encode()) == _ref_digest("model_info", f"{tool} {model_name}")
        assert model_name in ours and len(ours.splitlines()) > 5


def _wig_values(path):
    """(headers with their line numbers, values) of a wig file."""
    heads, vals = [], []
    with open(path) as fh:
        for i, ln in enumerate(fh):
            if ln.startswith("fixedStep"):
                heads.append((i, ln))
            else:
                vals.append(float(ln))
    return heads, np.array(vals)


@pytest.mark.gpu
@pytest.mark.parametrize("model_name,cols,seed", ACCEPTANCE_CASES)
def test_acceptance_baseline_models_vs_reference_binary(tmp_path, model_name, cols, seed):
    """North-star acceptance at BASELINE model size: build-tracks of the product against what the reference binary itself writes
    for the same synthetic MAF (58mammals = config 3's model, 100vertebrates = config 4's; holes, reference gaps, unknown species
    and a chain through the 1 Mb breakpoint).  FP64 path: seven wig files byte-identical.  tcgen05 path, against those same files:
    identical fixedStep headers at identical line numbers (gap / missing-species handling and wig positions are bit-exact), power
    track identical, every PhyloCSF value within 1e-3 decibans (one unit of the last printed digit)."""
    maf = os.path.join(str(tmp_path), "acc.maf")
    write_differential_maf("acceptance", maf, model_name, cols, seed)
    out64 = os.path.join(str(tmp_path), "f64")
    subprocess.run([BIN, "build-tracks", "--threads", "4", "--output", out64, model_name, maf], check=True, capture_output=True)
    gold = _ref_digest("build_tracks", f"{model_name}-{seed}")
    for n in WIGS:
        assert _sha(open(os.path.join(out64, n), "rb").read()) == gold[n], n
    ref_out = out64                 # byte for byte what the reference writes (checked just above)
    out5 = os.path.join(str(tmp_path), "tc5")
    subprocess.run([BIN, "build-tracks", "--threads", "4", "--precision", "tc5", "--output", out5, model_name, maf], check=True,
                   capture_output=True)
    assert open(os.path.join(out5, WIGS[0]), "rb").read() == open(os.path.join(ref_out, WIGS[0]), "rb").read()
    worst, nvals = 0.0, 0
    for n in WIGS[1:]:
        hr, vr = _wig_values(os.path.join(ref_out, n))
        h5, v5 = _wig_values(os.path.join(out5, n))
        assert h5 == hr, n
        assert v5.shape == vr.shape and vr.size > 0
        worst = max(worst, float(np.abs(v5 - vr).max()))
        nvals += vr.size
    print(f"{model_name}: tcgen05 path vs reference binary: max |delta| = {worst:.4f} decibans over {nvals} printed values")
    assert worst <= 1e-3 + 1e-9
