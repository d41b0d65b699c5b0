"""Six-frame and ORF scoring (pcsf_score_regions) against frame +1 scoring (pcsf_score_msa) on the config-5 alignment shape:
29mammals reduced to 12 species, synthetic single-block alignments of 30..600 columns (log-uniform), reference row 0.

Cases, for FIXED and MLE: score_msa (frame +1), regions --frames 6 --orf asis, regions --frames 6 --orf atgstop --min-codons 25.
Reports alignments/s, regions/s and (MLE) likelihood evaluations, with the GPU's name and power limit read in the same run.

    python tools/orf_bench.py [--fixed-alignments N] [--mle-alignments N] [--reps R] [--out profiles/orf_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SPECIES12 = "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat"


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def workload(model, n: int, seed: int):
    import torch
    from phylocsfpp_b200.synth import synth_alignment
    g = np.random.default_rng(seed)
    lens = np.exp(g.random(n) * (np.log(600.0) - np.log(30.0)) + np.log(30.0)).astype(np.int64)
    mat = synth_alignment(model, int(lens.sum()), seed=seed, device="cuda")[:, :int(lens.sum())].cpu().numpy()
    torch.cuda.synchronize()
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    return [np.ascontiguousarray(mat[:, s:s + L]) for s, L in zip(starts, lens)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fixed-alignments", type=int, default=65536)
    ap.add_argument("--mle-alignments", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "orf_bench.json"))
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("orf_bench: no CUDA device")
    from phylocsfpp_b200 import capi, orf
    from phylocsfpp_b200.models import load_model
    model = load_model("29mammals", SPECIES12)
    dm = capi.DeviceModel(model)
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "model": "29mammals/12 species",
           "lengths": "30..600 log-uniform", "ref_row": 0, "cases": []}
    for strat, sname, n in ((capi.STRATEGY_FIXED, "fixed", args.fixed_alignments), (capi.STRATEGY_MLE, "mle", args.mle_alignments)):
        alns = workload(model, n, 777)
        refs = np.zeros(n, np.int32)
        cases = [("score_msa", lambda: dm.score_msa(alns, strat)),
                 ("regions_6_asis", lambda: dm.score_regions(alns, refs, strat, 6, orf.ASIS, 25)),
                 ("regions_6_atgstop_25", lambda: dm.score_regions(alns, refs, strat, 6, orf.ATGSTOP, 25))]
        for cname, fn in cases:
            out = fn()                                   # warm-up: scratch allocation, module load
            times, evals = [], []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                out = fn()                               # every call ends in a device synchronise and the D2H of its results
                times.append(time.perf_counter() - t0)
                if strat == capi.STRATEGY_MLE:
                    evals.append(dm.score_msa_stats()["evaluations"])
            nreg = n if cname == "score_msa" else len(out)
            t = float(np.median(times))
            row = {"strategy": sname, "case": cname, "alignments": n, "regions": int(nreg), "seconds_median": t,
                   "seconds_all": times, "alignments_per_s": n / t, "regions_per_s": nreg / t}
            if evals:
                row["mle_evaluations"] = int(evals[-1])
            res["cases"].append(row)
            print(json.dumps(row), flush=True)
    for sname in ("fixed", "mle"):
        c = {r["case"]: r for r in res["cases"] if r["strategy"] == sname}
        res[f"{sname}_time_ratio_6asis_vs_msa"] = c["regions_6_asis"]["seconds_median"] / c["score_msa"]["seconds_median"]
        res[f"{sname}_time_ratio_atgstop_vs_msa"] = c["regions_6_atgstop_25"]["seconds_median"] / c["score_msa"]["seconds_median"]
    c = {r["case"]: r for r in res["cases"] if r["strategy"] == "mle"}
    res["mle_evaluation_ratio_6asis_vs_msa"] = c["regions_6_asis"]["mle_evaluations"] / c["score_msa"]["mle_evaluations"]
    res["mle_evaluation_ratio_atgstop_vs_msa"] = c["regions_6_atgstop_25"]["mle_evaluations"] / c["score_msa"]["mle_evaluations"]
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))
    dm.close()


if __name__ == "__main__":
    main()
