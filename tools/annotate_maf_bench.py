#!/usr/bin/env python3
"""annotate-with-maf end to end on one GPU: a seeded synthetic 58mammals MAF (one chromosome, holes every --chain columns) and a
generated GTF of coding and non-coding transcripts over it.  Runs the command under MLE and FIXED (with --find-orf 1) and reports
transcripts/s, the time split (MAF scan, GFF read, extraction, library calls, formatting, writing) and the card's name and power
limit, read in the same run.

    python tools/annotate_maf_bench.py [--columns 50000000] [--transcripts 100000] [--out profiles/annotate_maf_bench.json]

write_annotation() is also the annotation generator of tests/test_annotate_maf.py.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")


def _attrs(fmt, kind, tid, gid):
    if fmt == "gtf":
        return f'gene_id "{gid}"; transcript_id "{tid}";'
    return f"ID={tid};Parent={gid}" if kind == "transcript" else f"Parent={tid}"


def write_annotation(path, chroms, n, seed, fmt="gtf", coding=0.6, extra=()):
    """n random transcripts on chroms = [(name, lo, hi)] (1-based positions), plus the `extra` ones: (chrom, strand, exons [(b, e)],
    cds [(b, e, phase)] or None, with_exon_lines).  Coding transcripts get a CDS per exon (UTRs trimmed off the outer ones) with
    random phases; half of the non-coding ones have no exon lines."""
    rng = np.random.default_rng(seed)
    tx = []
    for _ in range(n):
        name, lo, hi = chroms[int(rng.integers(len(chroms)))]
        ne = int(rng.integers(1, 7))
        p = int(rng.integers(lo, max(lo + 1, hi - 12000)))
        exons = []
        for _k in range(ne):
            ln = int(rng.integers(60, 400))
            exons.append((p, p + ln - 1))
            p += ln + int(rng.integers(30, 1500))
        strand = "+-"[int(rng.integers(2))]
        if rng.random() < coding:
            cds = [(b, e, int(rng.integers(3))) for b, e in exons]
            b0, e0, ph0 = cds[0]
            cds[0] = (min(e0, b0 + int(rng.integers(0, 40))), e0, ph0)
            b1, e1, ph1 = cds[-1]
            cds[-1] = (b1, max(b1, e1 - int(rng.integers(0, 40))), ph1)
            tx.append((name, strand, exons, cds, True))
        else:
            tx.append((name, strand, exons, None, bool(rng.random() < 0.5)))
    tx = list(extra) + sorted(tx, key=lambda t: (t[0], t[2][0][0]))          # by chromosome and start, as annotations are distributed
    with open(path, "w") as fh:
        fh.write("##gff-version 3\n" if fmt == "gff3" else "#!genome-build synthetic\n")
        for i, (name, strand, exons, cds, with_exons) in enumerate(tx):
            tid, gid = f"t{i}", f"g{i}"
            order = (lambda v: v) if strand == "+" else (lambda v: v[::-1])
            fh.write(f"{name}\tsynth\ttranscript\t{exons[0][0]}\t{exons[-1][1]}\t.\t{strand}\t.\t{_attrs(fmt, 'transcript', tid, gid)}\n")
            if with_exons:
                for b, e in order(exons):
                    fh.write(f"{name}\tsynth\texon\t{b}\t{e}\t.\t{strand}\t.\t{_attrs(fmt, 'exon', tid, gid)}\n")
            for b, e, ph in order(cds or []):
                fh.write(f"{name}\tsynth\tCDS\t{b}\t{e}\t.\t{strand}\t{ph}\t{_attrs(fmt, 'CDS', tid, gid)}\n")
    return len(tx)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--columns", type=int, default=50_000_000)
    ap.add_argument("--transcripts", type=int, default=100_000)
    ap.add_argument("--chain", type=int, default=200_000)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "annotate_maf_bench.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("annotate_maf_bench: no CUDA device")
    from phylocsfpp_b200.models import load_model
    from phylocsfpp_b200.synth import synth_alignment
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "model": "58mammals", "columns": args.columns,
           "chain_columns": args.chain}
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 4 * 58 * args.columns else None
    with tempfile.TemporaryDirectory(dir=base) as d:
        t0 = time.time()
        model = load_model("58mammals")
        # [nl][columns] written piece by piece through a memmap (synth_alignment of the whole matrix at once needs far more memory)
        mbin = os.path.join(d, "mat.npy")
        mm = np.lib.format.open_memmap(mbin, mode="w+", dtype=np.uint8, shape=(model.nl, args.columns))
        piece = 1 << 23
        for c0 in range(0, args.columns, piece):
            n = min(piece, args.columns - c0)
            mm[:, c0:c0 + n] = synth_alignment(model, n, seed=11 + c0 // piece, device="cuda")[:, :n].cpu().numpy()
            print(f"synthetic columns: {c0 + n}", flush=True)
        off = mm.offset
        del mm
        maf = os.path.join(d, "chr1.maf")
        subprocess.run([BIN, "matrix-to-maf", "--chain", str(args.chain), "--start", "10000", "--chrom", "chr1", "--skip-bytes", str(off),
                        "58mammals", mbin, str(args.columns), maf], check=True, capture_output=True)
        os.unlink(mbin)
        print(f"MAF written: {os.path.getsize(maf)} bytes after {time.time() - t0:.1f} s", flush=True)
        gtf = os.path.join(d, "synth.gtf")
        res["transcripts"] = write_annotation(gtf, [("chr1", 10001, 10000 + args.columns)], args.transcripts, seed=5)
        print(f"annotation written: {res['transcripts']} transcripts", flush=True)
        res["generate_seconds"] = round(time.time() - t0, 1)
        res["maf_bytes"] = os.path.getsize(maf)
        res["runs"] = []
        for strat in ("fixed", "mle"):
            out = os.path.join(d, "o_" + strat)
            t1 = time.time()
            beat = threading.Event()
            threading.Thread(target=lambda: [print(f"{strat}: running", flush=True) for _ in iter(lambda: beat.wait(60), True)],
                             daemon=True).start()
            r = subprocess.run([BIN, "annotate-with-maf", "--strategy", strat, "--find-orf", "1", "--threads", str(args.threads), "--gpus", "1",
                                "--output", out, "58mammals", maf, gtf], capture_output=True, text=True, env=dict(os.environ, PCSF_HOST_STATS="1"))
            wall = time.time() - t1
            beat.set()
            if r.returncode != 0:
                sys.exit(f"annotate-with-maf failed ({r.returncode}): {r.stdout[-2000:]} {r.stderr[-2000:]}")
            stats = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
            stats.update(strategy=strat, process_seconds=round(wall, 3), transcripts_per_s=round(stats["transcripts"] / stats["seconds"], 1))
            res["runs"].append(stats)
            print(json.dumps(stats), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
