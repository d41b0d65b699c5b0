#!/usr/bin/env python3
"""Writes tests/golden/ref-generated/digests.json: sha256 of what the reference's build-tracks writes for the synthetic MAFs of the
differential runs of tests/test_reference_build.py (ORACLE_CASES, CLI_CASES, ACCEPTANCE_CASES; seven wig files each), and of its
--model-info text (MODEL_INFO_MODELS, both sub-commands).

The reference binary is not part of the repository, so those tests compare against these digests.  They are computed here by the
implementations that reproduced the reference byte for byte on exactly these inputs when both ran side by side: the wig files by
the oracle + reader-mirror pipeline (CPU, no GPU needed), the --model-info text by phylocsfpp_b200/bin/phylocsf_b200.  The product's
FP64 path is held to the same digests on the GPU, so two independent implementations agree on every one of them.

  python tests/golden/make_ref_digests.py            # after __graft_entry__.build(); a few CPU-minutes
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile
from multiprocessing import get_context

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests import test_reference_build as T  # noqa: E402


def _build_tracks(case):
    kind, (model_name, cols, seed, extra) = case
    with tempfile.TemporaryDirectory() as tmp:
        maf = os.path.join(tmp, "in.maf")
        T.write_differential_maf(kind, maf, model_name, cols, seed)
        files = T.oracle_build_tracks_for(model_name, maf, extra)
    return f"{model_name}-{seed}", {n: hashlib.sha256(files[n]).hexdigest() for n in T.WIGS}


def main():
    cases = ([("acceptance", c + ([],)) for c in T.ACCEPTANCE_CASES] + [("cli", c) for c in T.CLI_CASES]
             + [("oracle", c) for c in T.ORACLE_CASES])
    with get_context("fork").Pool(min(len(cases), os.cpu_count() or 1)) as pool:
        build_tracks = dict(sorted(pool.map(_build_tracks, cases, chunksize=1)))
    model_info = {}
    for m in T.MODEL_INFO_MODELS:
        for tool in ("build-tracks", "score-msa"):
            out = subprocess.run([T.BIN, tool, "--model-info", m], capture_output=True, check=True).stdout
            model_info[f"{tool} {m}"] = hashlib.sha256(out).hexdigest()
    with open(T.DIGESTS, "w") as fh:
        json.dump({"build_tracks": build_tracks, "model_info": model_info}, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(T.DIGESTS, len(build_tracks), "build-tracks inputs,", len(model_info), "--model-info texts")


if __name__ == "__main__":
    main()
