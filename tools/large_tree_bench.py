#!/usr/bin/env python3
"""Throughput on a large species tree (DESIGN.md section 12): a generated Yule tree of --nl leaves (default 470, the size of UCSC's
hg38 470-way alignment) with the 58mammals ECMs, written by tests/tree_shapes.py's generator.

Reports, as one JSON line, together with the card's name and power limit read in the same run:
  * FP64 pcsf_tracks columns/s on a synthetic config-3-style input (30 % missing cells), host buffers in and out;
  * the share of windows whose likelihood (either ECM) falls below 2^-512, the threshold under which k_prune_scaled rescales a
    partial (a lower bound of the windows that were rescaled), and the share below the double range (where the reference's
    unscaled product returns -inf / NaN), from the C oracle's per-codon log-likelihoods on a sample of windows;
  * MLE pcsf_score_msa alignments/s and the number of slots (alignments fitted at once) on short alignments.

usage: tools/large_tree_bench.py [--nl 470] [--columns 4194304] [--reps 3] [--alignments 512] [--sample 3000]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nl", type=int, default=470)
    ap.add_argument("--columns", type=int, default=1 << 22)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--alignments", type=int, default=512)
    ap.add_argument("--sample", type=int, default=3000)
    args = ap.parse_args()

    import torch
    from oracle import oracle as orc
    from phylocsfpp_b200 import capi
    from phylocsfpp_b200.models import load_model
    from phylocsfpp_b200.synth import synth_alignment
    from tests.tree_shapes import Shape, write_model
    from tests.util import random_alignment

    name, power = card()
    d = tempfile.mkdtemp()
    model = load_model(write_model(d, Shape("yule", args.nl)))
    dm = capi.DeviceModel(model)
    out = {"card": name, "power_limit": power, "nl": model.nl, "columns": args.columns}

    seqs = np.ascontiguousarray(synth_alignment(model, args.columns, seed=3, device="cuda").cpu().numpy()[:, :args.columns])
    dm.tracks(seqs)                                          # warm-up: buffers, module load
    times = []
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = dm.tracks(seqs)
        times.append(time.perf_counter() - t0)
    out["tracks_columns_per_s"] = args.columns / min(times)
    out["tracks_seconds"] = times
    out["unique_patterns"] = int(res["stats"]["n_unique"])

    rng = np.random.default_rng(1)
    cols = np.sort(rng.choice(args.columns - 2, size=min(args.sample, args.columns - 2), replace=False))
    plus, minus = orc.window_codons(seqs[:, np.concatenate([cols, cols + 1, cols + 2])].reshape(model.nl, 3, -1)
                                    .transpose(0, 2, 1).reshape(model.nl, -1))
    cod = np.concatenate([plus[:, 0::3], minus[:, 0::3]], axis=1)
    lz = [orc.OracleModel(model.tree, S, f).lpr_leaves(cod)[2] for S, f in ((model.S_c, model.f_c), (model.S_nc, model.f_nc))]
    low = np.minimum(lz[0], lz[1])
    out["windows_sampled"] = int(cod.shape[1])
    out["share_below_2^-512"] = float(np.mean(low < -512 * np.log(2.0)))
    out["share_below_double_range"] = float(np.mean(~np.isfinite(low) | (low < np.log(np.finfo(np.float64).tiny))))
    out["tracks_max_abs_decibans"] = float(np.nanmax(np.abs(res["plus"])))

    lens = rng.integers(30, 201, args.alignments)
    alns = [random_alignment(model.nl, 3 * int(k), seed=100 + i, gap=0.3, conserve=0.8) for i, k in enumerate(lens)]
    dm.score_msa(alns[:8], capi.STRATEGY_MLE)                # warm-up
    t0 = time.perf_counter()
    phylo, _, _ = dm.score_msa(alns, capi.STRATEGY_MLE)
    dt = time.perf_counter() - t0
    st = dm.score_msa_stats()
    out["mle_alignments"] = args.alignments
    out["mle_alignments_per_s"] = args.alignments / dt
    out["mle_slots"] = int(st["slots"])
    out["mle_finite"] = bool(np.isfinite(phylo).all())
    dm.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
