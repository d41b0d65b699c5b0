#!/usr/bin/env python3
"""bench.py — MAF columns/sec of the PhyloCSF++ hot path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path (pack -> site-pattern keys/dedup -> Felsenstein pruning of both ECMs on
every codon window of both strands -> deciban scatter, plus the per-base BLS) over one batch of synthetic
alignment columns of BASELINE.json's config 3 shape: model 58mammals, 30 % missing cells, chromosome-scale
chain cut into batches of --cols columns (100 M columns = 12 such batches; every batch is larger than L2).

  value  columns/s with the batch resident in HBM (device-pointer C-ABI, CUDA events, max over ranks)
  e2e    columns/s through the host-buffer C-ABI call (pcsf_tracks): pinned host input, H2D, kernels, D2H
  --impl reference   the reference's own CPU implementation (oracle/_ref/phylocsf_ref = its unmodified sources compiled
                     against the GSL shim, OpenMP over all host cores; the oracle port only if that binary is missing),
                     MAF file -> 7 wig files on a bounded sample of the same workload

Launch: python bench.py --gpus N --steps K --warmup W   (N > 1: under torch.distributed.run, one rank per GPU).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "MAF columns/sec (6 frames, coding+noncoding ECM)"
UNIT = "columns/s"


def flops_per_pruning(nl: int) -> int:
    """SURVEY.md section 8(d): internal-child mat-vecs + Hadamard products + root dot."""
    return 2 * 64 * 64 * (nl - 2) + 64 * (nl - 1) + 128


def hbm_passes(tstats, nl, B, Wn):
    peak = 6458.7
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    alg = {"k_pack": ("ms_pack", 2 * nl * B),                       # ASCII in, codes out
           "k_keys_tracks": ("ms_hash", nl * B + 32 * B),           # codes in, two 128-bit keys per column out
           "dedup (insert/resolve/scan/finalize)": ("ms_dedup", 40 * 2 * Wn),
           "k_scatter_tracks": ("ms_scatter", 24 * 2 * Wn),
           "k_bls": ("ms_bls", nl * B + 8 * B)}
    out = {}
    for k, (key, nbytes) in alg.items():
        ms = tstats.get(key) or 0.0
        if ms > 0:
            gbs = nbytes / (ms * 1e-3) / 1e9
            out[k] = {"ms": ms, "bytes": nbytes, "gbs": gbs, "frac_of_hbm_peak": gbs / peak}
    return out


# ------------------------------------------------------------------------------------------------ CPU arm
_W = {}


def _cpu_init(model_name):
    from oracle import oracle as orc
    from phylocsfpp_b200.models import load_model
    m = load_model(model_name)
    _W["m"] = m
    _W["mc"] = orc.OracleModel(m.tree, m.S_c, m.f_c)
    _W["mnc"] = orc.OracleModel(m.tree, m.S_nc, m.f_nc)


def _cpu_chunk(seqs):
    """Reference path for one slice of columns: both strands' codon windows, both models, BLS."""
    from oracle import oracle as orc
    plus, minus = orc.window_codons(seqs)
    a = orc.run_tracks(_W["mc"], _W["mnc"], plus)
    b = orc.run_tracks(_W["mc"], _W["mnc"], minus)
    c = orc.bls(_W["m"].tree, seqs)[1]
    return float(a.sum() + b.sum() + c.sum())


def cpu_columns_per_sec(model_name, seqs_host: np.ndarray, ncores: int, pool=None):
    """Times the CPU path over seqs_host [nl, S]; returns (columns/s, seconds)."""
    import multiprocessing as mp
    S = seqs_host.shape[1]
    per = max(256, S // (ncores * 4))
    chunks = [np.ascontiguousarray(seqs_host[:, i:min(S, i + per + 2)]) for i in range(0, S - 2, per)]
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(ncores, initializer=_cpu_init, initargs=(model_name,))
        pool.map(_cpu_chunk, chunks[:ncores])  # warm: model build in every worker
    t0 = time.perf_counter()
    pool.map(_cpu_chunk, chunks)
    dt = time.perf_counter() - t0
    if own:
        pool.close()
    return S / dt, dt


REF_BIN = os.path.join(ROOT, "oracle", "_ref", "phylocsf_ref")


def ref_sample_shape(ncores: int, per_step: bool):
    """(chains, columns per chain) of the CPU sample: chains are the reference's unit of parallel work (a reader job owns the
    chains that start in its byte range, parallel_file_reader.hpp:281-350), so the sample is cut into 4 (2) chains per core;
    3000-4000 columns per chain keep the per-chain model instantiation (instance.hpp:449-646) near 10 % as on real chains."""
    return (2 * ncores, 3000) if per_step else (4 * ncores, 4000)


class RefSample:
    """The first S columns of the workload written as a MAF file (tmpfs when available) for the reference binary."""

    def __init__(self, model, mat: np.ndarray, chains: int, chain_cols: int):
        import tempfile
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from make_synth_maf import write_synth_maf
        self.S = chains * chain_cols
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        self.dir = tempfile.mkdtemp(prefix="pcsf_ref_", dir=base)
        self.maf = os.path.join(self.dir, "sample.maf")
        self.info = write_synth_maf(self.maf, model, self.S, seed=7, mat=mat, chain_cols=chain_cols, hole_p=0.0, ref_gap=0.0, alien_p=0.0)

    def run(self, model_name: str, threads: int) -> float:
        """One build-tracks run of the reference (power + 6 raw tracks); returns seconds."""
        import shutil
        out = os.path.join(self.dir, "out")
        shutil.rmtree(out, ignore_errors=True)
        t0 = time.perf_counter()
        subprocess.run([REF_BIN, "build-tracks", "--threads", str(threads), "--output", out, model_name, self.maf], check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        dt = time.perf_counter() - t0
        assert os.path.getsize(os.path.join(out, "PhyloCSFRaw+1.wig")) > 0
        return dt

    def close(self):
        import shutil
        shutil.rmtree(self.dir, ignore_errors=True)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}



# ------------------------------------------------------------------------------------------------ legs beyond config 3
SPECIES12 = "Human,Chimp,Mouse,Dog,Cow,Horse,Elephant,Armadillo,Rat,Rabbit,Cat,Megabat"


def kernel_sha16() -> str:
    """Hash of the sources of k_prune_tc5 (what a committed ncu capture is stamped with)."""
    import hashlib
    h = hashlib.sha256()
    for f in ("prune_tc5.cuh", "tc5.cuh"):
        h.update(open(os.path.join(ROOT, "phylocsfpp_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def n_tc5_gemms(tree) -> int:
    """GEMMs per pruning on the tcgen05 path: inner edges that are not cherries (a cherry's message is a table row)."""
    c1, c2, nl, n = tree.child1, tree.child2, tree.nl, tree.n
    cherries = sum(1 for i in range(nl, n - 1) if c1[c1[i]] < 0 and c1[c2[i]] < 0)
    return (nl - 2) - cherries


def _file_barrier(tag: str, rank: int, world: int, timeout: float = 3600.0):
    """A barrier that leaves the GPUs idle (an NCCL barrier spins a kernel on every device): ranks drop a file, rank 0 waits for all."""
    if world == 1:
        return
    base = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"pcsf_bar_{os.environ.get('MASTER_PORT', '0')}_{tag}")
    open(f"{base}.{rank}", "w").close()
    t0 = time.time()
    while not all(os.path.exists(f"{base}.{r}") for r in range(world)):
        if time.time() - t0 > timeout:
            raise SystemExit(f"file barrier {tag} timed out")
        time.sleep(0.02)


def leg_config4(total_cols, rank, world, local_rank, dist, torch, capi, precision_flag):
    """BASELINE config 4: build-tracks 100vertebrates on a 250 M-column chromosome, STRONG-scaled: rank r owns the column range
    [r T/N, (r+1) T/N), scores it in batches through pcsf_tracks (pinned host buffers, H2D + D2H inside) and writes the scores into
    its range of one host array that rank 0 ends up holding in column order (OrderedHostBuffer: the host-side ordered gather, no
    collective).  Timed region = all of that; max over ranks."""
    from concurrent.futures import ThreadPoolExecutor
    from phylocsfpp_b200.models import load_model
    from phylocsfpp_b200.shard import OrderedHostBuffer, column_ranges
    from phylocsfpp_b200.synth import synth_alignment
    model = load_model("100vertebrates")
    nl = model.nl
    Bc = 1 << 22
    lo, hi = column_ranges(total_cols, world, align=16)[rank]
    dev = torch.device("cuda", local_rank)
    dm = capi.DeviceModel(model, local_rank)
    seqs = synth_alignment(model, Bc, seed=4321 + rank, device=dev)
    ld = seqs.shape[1]
    h_seqs = torch.empty((nl, ld), dtype=torch.uint8, pin_memory=True)
    h_seqs.copy_(seqs)
    del seqs
    outs = [[torch.empty(Bc, dtype=torch.float64, pin_memory=True) for _ in range(3)] for _ in range(2)]
    nbytes = 3 * total_cols * 8
    path = os.path.join(OrderedHostBuffer.pick_dir(nbytes), f"pcsf_cfg4_{os.environ.get('MASTER_PORT', '0')}.bin")
    if rank == 0:
        OrderedHostBuffer(path, 3, total_cols, create=True).close()
    if world > 1:
        dist.barrier()
    buf = OrderedHostBuffer(path, 3, total_cols)
    buf.prefault(lo, hi)          # the output array exists and is mapped before the clock starts, like the pinned input / output buffers
    lib = capi.load()
    st = capi.TracksStats()
    flags = capi.TRACKS_SCORES | capi.TRACKS_BLS | precision_flag
    pool = ThreadPoolExecutor(1)

    def run(do_store):
        pending = [None, None]
        k = 0
        for c0 in range(lo, hi, Bc):
            n = min(Bc, hi - c0)
            o = outs[k & 1]
            if pending[k & 1] is not None:
                pending[k & 1].result()
            capi._check(lib.pcsf_tracks(dm.h, h_seqs.data_ptr(), n, ld, flags, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), None, st))

            def store(o=o, c0=c0, n=n):
                buf.write(0, c0, o[0].numpy()[:max(n - 2, 0)])
                buf.write(1, c0, o[1].numpy()[:max(n - 2, 0)])
                buf.write(2, c0, o[2].numpy()[:n])
            pending[k & 1] = pool.submit(store) if do_store else None
            k += 1
        for f in pending:
            if f is not None:
                f.result()
        return k

    # warm-up: one batch (allocations inside the library, page faults of the mapping are part of the timed run as in production)
    hi_saved, hi = hi, min(hi, lo + Bc)
    run(False)
    hi = hi_saved
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    n_calls = run(True)
    t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
    sec = float(t.item())
    out = None
    if rank == 0:
        # every range has been written (first, last and a sample of columns of every rank's range are finite scores)
        probe = []
        for r in range(world):
            rlo, rhi = column_ranges(total_cols, world, align=16)[r]
            if rhi > rlo:
                probe += [rlo, rhi - 1] + list(range(rlo, rhi, max(1, (rhi - rlo) // 50)))
        bl = np.asarray(buf.arr[2, probe])
        assert np.isfinite(bl).all() and (bl != 0).any()
        out = {"workload": f"build-tracks 100vertebrates, {total_cols} synthetic columns (30% missing cells), strong-scaled over {world} GPU(s): "
                           f"one column range per rank in batches of {Bc} (the rank's synthetic batch is re-used for every batch; 419 MB > L2), "
                           "scores gathered in column order into one host array on rank 0 (file-backed mapping, no collective)",
               "columns": total_cols, "seconds": sec, "columns_per_s": total_cols / sec, "n_gpus": world, "scaling": "strong",
               "calls_per_rank": n_calls, "h2d_bytes": nl * total_cols, "d2h_bytes": 24 * total_cols,
               "ordered_output": {"path_dir": os.path.dirname(path), "bytes": nbytes, "checksum_bls_probe": float(bl.sum())},
               "precision": "tc5" if precision_flag else "f64", "timing": "wall clock around the whole leg, max over ranks (host work is part of it)"}
    buf.close(unlink=(rank == 0))
    pool.shutdown()
    dm.close()
    return out


def leg_config5(total_aln, rank, world, local_rank, dist, torch, capi):
    """BASELINE config 5: score-msa --strategy mle, 29mammals reduced to 12 species, synthetic single-block alignments of 30..600
    columns (log-uniform), strong-scaled: every rank scores its share through pcsf_score_msa (host blob in, host scores out)."""
    from phylocsfpp_b200.models import load_model
    from phylocsfpp_b200.synth import synth_alignment
    model = load_model("29mammals", SPECIES12)
    nl = model.nl
    dev = torch.device("cuda", local_rank)
    dm = capi.DeviceModel(model, local_rank)
    batch = 65536
    share = (total_aln + world - 1) // world
    n_calls = max(1, (share + batch - 1) // batch)
    share = n_calls * batch
    g = torch.Generator(device="cpu")
    g.manual_seed(99 + rank)
    lens = torch.exp(torch.rand(batch, generator=g, dtype=torch.float64) * (np.log(600.0) - np.log(30.0)) + np.log(30.0)).to(torch.int64)
    starts = torch.cumsum(lens, 0) - lens
    Ltot = int(lens.sum())
    mat = synth_alignment(model, Ltot, seed=777 + rank, device=dev)[:, :Ltot]          # [nl, Ltot] on the device
    lens_d, starts_d = lens.to(dev), starts.to(dev)
    offs_d = starts_d * nl                                                             # alignment i is a contiguous [nl][len_i] block
    aln_of_col = torch.repeat_interleave(torch.arange(batch, device=dev), lens_d)
    col_in_aln = torch.arange(Ltot, device=dev) - starts_d[aln_of_col]
    blob_d = torch.empty(nl * Ltot, dtype=torch.uint8, device=dev)
    for s_ in range(nl):
        blob_d[offs_d[aln_of_col] + s_ * lens_d[aln_of_col] + col_in_aln] = mat[s_]
    blob = torch.empty(nl * Ltot, dtype=torch.uint8, pin_memory=True)
    blob.copy_(blob_d)
    del blob_d, mat, aln_of_col, col_in_aln
    offs = (starts * nl).contiguous()
    phylo = torch.empty(batch, dtype=torch.float32, pin_memory=True)
    anc = torch.empty(batch, dtype=torch.float32, pin_memory=True)
    bls = torch.empty(batch, dtype=torch.float32, pin_memory=True)
    lib = capi.load()

    def call():
        capi._check(lib.pcsf_score_msa(dm.h, capi.STRATEGY_MLE, batch, blob.data_ptr(), offs.data_ptr(), lens.data_ptr(),
                                       phylo.data_ptr(), anc.data_ptr(), bls.data_ptr()))

    call()          # warm-up (scratch allocation)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(n_calls):
        call()
    t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item())
    stats = dm.score_msa_stats()
    out = None
    if rank == 0:
        # one instrumented call: CUDA-event time per kernel -> rooflines of the batched P(t) construction and of the MLE pruning
        dm.set_timing(True)
        call()
        ts = dm.score_msa_stats()
        dm.set_timing(False)
        n = model.tree.n
        flop_expm = ts["evaluations"] * (n - 1) * (2 * 64 ** 3 + 64 ** 2)
        codons = float((lens // 3).sum())
        flop_prune = ts["evaluations"] / max(1, 2 * batch) * 2 * codons * flops_per_pruning(nl)      # evaluations x codons of the alignment (mean)
        peak = 37.16
        try:
            peak = json.load(open(os.path.join(ROOT, "profiles", "peaks_fp64.json")))["micro"]["dmma_tflops"]
        except Exception:
            pass
        finite = int(torch.isfinite(phylo).sum())
        out = {"workload": f"score-msa --strategy mle --comp-anc 1 --species <12 of 29mammals>, {share * world} synthetic single-block alignments "
                           f"of 30..600 columns (log-uniform, mean {Ltot / batch:.0f}), strong-scaled over {world} GPU(s) in calls of {batch} "
                           "(the rank's batch is re-used for every call), host blob in / host scores out through pcsf_score_msa",
               "alignments": share * world, "seconds": sec, "alignments_per_s": share * world / sec, "columns_per_s": Ltot * n_calls * world / sec,
               "n_gpus": world, "scaling": "strong", "mean_evaluations_per_alignment": stats["evaluations"] / batch,
               "rounds_per_call": stats["rounds"], "slots": stats["slots"], "finite_scores_in_last_batch": finite,
               "roofline": {"k_mle_expm": {"bound": "tensor", "unit": "TFLOP/s", "flop": flop_expm, "ms": ts["ms_expm"],
                                           "achieved": flop_expm / max(ts["ms_expm"], 1e-9) / 1e9, "peak": peak,
                                           "frac": flop_expm / max(ts["ms_expm"], 1e-9) / 1e9 / peak,
                                           "note": "(n-1)(2*64^3+64^2) flop per evaluation (SURVEY 8d), FP64 DMMA peak of profiles/peaks_fp64.json"},
                            "k_prune<true>": {"bound": "tensor", "unit": "TFLOP/s", "flop": flop_prune, "ms": ts["ms_prune"],
                                              "achieved": flop_prune / max(ts["ms_prune"], 1e-9) / 1e9, "peak": peak,
                                              "frac": flop_prune / max(ts["ms_prune"], 1e-9) / 1e9 / peak},
                            "ms_step": ts["ms_step"], "ms_plan": ts["ms_plan"]}}
    dm.close()
    return out


def leg_cli(cols, rank, world, local_rank, torch, n_files=4):
    """The drop-in command line at BASELINE config 3's size: phylocsf_b200 build-tracks --gpus N --precision tc5 on `n_files` chromosome
    MAF files in tmpfs (58mammals, cols / n_files columns each), MAF text -> 7 wig files.  Rank 0 runs the process (it deals chain
    groups to all N devices itself); the other ranks keep their GPUs idle."""
    import shutil
    import tempfile
    from phylocsfpp_b200.models import load_model
    from phylocsfpp_b200.synth import synth_alignment
    out = None
    if rank == 0:
        BIN = os.path.join(ROOT, "phylocsfpp_b200", "bin", "phylocsf_b200")
        model = load_model("58mammals")
        base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 4 * 58 * cols else None
        tmp = tempfile.mkdtemp(prefix="pcsf_cli_", dir=base)
        try:
            dev = torch.device("cuda", local_rank)
            per = cols // n_files
            piece = 1 << 23
            t_gen = time.perf_counter()
            procs, mafs = [], []
            for f in range(n_files):
                mbin = os.path.join(tmp, f"m{f}.bin")
                # [nl][per] row-major, written piece by piece through a memmap (the pieces are column ranges)
                mm = np.lib.format.open_memmap(mbin + ".npy", mode="w+", dtype=np.uint8, shape=(model.nl, per))
                for c0 in range(0, per, piece):
                    n = min(piece, per - c0)
                    mm[:, c0:c0 + n] = synth_alignment(model, n, seed=5000 + 100 * f + c0 // piece, device=dev)[:, :n].cpu().numpy()
                off = mm.offset
                del mm
                maf = os.path.join(tmp, f"chr{f + 1}.maf")
                mafs.append(maf)
                procs.append(subprocess.Popen([BIN, "matrix-to-maf", "--chain", str(25_000_000), "--chrom", f"chr{f + 1}", "--skip-bytes", str(off), "58mammals",
                                               mbin + ".npy", str(per), maf], stdout=subprocess.DEVNULL))
            for pr in procs:
                if pr.wait() != 0:
                    raise SystemExit("matrix-to-maf failed")
            for f in range(n_files):
                os.unlink(os.path.join(tmp, f"m{f}.bin.npy"))
            torch.cuda.empty_cache()
            t_gen = time.perf_counter() - t_gen
            threads = os.cpu_count() or 1
            best = None
            for rep in range(2):
                t0 = time.perf_counter()
                r = subprocess.run([BIN, "build-tracks", "--threads", str(threads), "--gpus", str(world), "--precision", "tc5", "--output",
                                    os.path.join(tmp, "out")] + ["58mammals"] + mafs, check=True, capture_output=True, text=True,
                                   env=dict(os.environ, PCSF_HOST_STATS="1"))
                dt = time.perf_counter() - t0
                js = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
                st = js[0]
                for extra in js[1:]:
                    st.update(extra)
                if best is None or dt < best[0]:
                    best = (dt, st)
            wig_bytes = sum(os.path.getsize(os.path.join(tmp, "out", f)) for f in os.listdir(os.path.join(tmp, "out")))
            maf_bytes = sum(os.path.getsize(m) for m in mafs)
            ncols = per * n_files
            out = {"workload": f"phylocsf_b200 build-tracks --gpus {world} --precision tc5 --threads {threads} on {n_files} synthetic 58mammals chromosome MAF files "
                               f"({ncols} columns, {maf_bytes} bytes, tmpfs; blocks of 120 columns, 30% missing cells) -> PhyloCSFpower.wig + 6 PhyloCSFRaw wigs ({wig_bytes} bytes)",
                   "columns": ncols, "process_seconds": best[0], "columns_per_s": ncols / best[0], "tool_seconds": best[1]["seconds"],
                   "columns_per_s_tool": ncols / best[1]["seconds"], "n_gpus": world, "host_threads": threads,
                   "tool_stats": best[1], "generate_seconds": t_gen,
                   "note": "process_seconds = the whole command (exec -> exit: CUDA context, model preparation, scan, scoring, 7 files written); tool_seconds = inside main after option parsing; best of 2 runs"}
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    _file_barrier("cli", rank, world)
    return out


DUMP_LIMIT = 64 << 20
DUMP_SAMPLE = 1 << 21


def dump_outputs(outdir: str, arrays: dict) -> None:
    """Writes each 1-D float64 device tensor as outdir/<name>.npy.  When the arrays together exceed DUMP_LIMIT bytes, each one is
    cut to DUMP_SAMPLE positions drawn (sorted, without replacement) from a generator seeded with 0, so that two runs with the same
    arguments write the same positions and can be compared element for element."""
    import torch
    os.makedirs(outdir, exist_ok=True)
    full = sum(a.numel() * a.element_size() for a in arrays.values()) <= DUMP_LIMIT
    for name, a in arrays.items():
        if not full and a.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.numel(), DUMP_SAMPLE, replace=False))
            a = a[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(outdir, name + ".npy"), a.cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="58mammals")
    ap.add_argument("--cols", type=int, default=1 << 23, help="alignment columns per step (per GPU)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="columns of the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-port", action="store_true", help="time the oracle port instead of the reference binary on the CPU legs")
    ap.add_argument("--no-dedup", action="store_true")
    ap.add_argument("--chunk-cols", type=int, default=0, help="dedup / pipeline chunk of the library in columns (0 = the library's default, 2 Mi)")
    ap.add_argument("--config4-cols", type=int, default=250_000_000, help="columns of the strong-scaled 100vertebrates leg (0 = skip)")
    ap.add_argument("--config5-alignments", type=int, default=1_000_000, help="alignments of the strong-scaled MLE leg (0 = skip)")
    ap.add_argument("--cli-cols", type=int, default=100_000_000, help="columns of the MAF files of the command-line leg, four chromosome files (0 = skip)")
    ap.add_argument("--precision", default="tc5", choices=["f64", "tc5"],
                    help="tc5: tcgen05/TMEM split-TF32 path (fastest path inside the 1e-3 deciban contract); "
                         "f64: FP64 DMMA path (parity anchor, byte-identical wig text)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed on rank 0 (plus / minus decibans per window, bls per column) as "
                         "DIR/<name>.npy, float64; above 64 MiB in all, the same seeded sample of positions of every array")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 arm")

    # stdout carries exactly one JSON line: libraries that write to fd 1 (NCCL prints its version banner there at
    # communicator creation) are sent to stderr instead
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncores = os.cpu_count() or 1

    from phylocsfpp_b200.models import load_model
    model = load_model(args.model)
    nl = model.nl
    workload = (f"build-tracks {args.model} on synthetic hg38.100way-shaped alignment columns, 30% missing cells, "
                f"batches of {args.cols} columns (100M-column chain = {-(-100_000_000 // args.cols)} batches)")

    if args.impl == "reference":
        # rank 0 only: the reference's own CPU implementation on a bounded sample per step
        if rank != 0:
            return
        import torch
        from phylocsfpp_b200.synth import synth_alignment
        if os.path.exists(REF_BIN) and not args.cpu_port:
            chains, chain_cols = ref_sample_shape(ncores, per_step=True)
            S = args.cpu_sample or chains * chain_cols
            chains = max(1, S // chain_cols)
            seqs = synth_alignment(model, chains * chain_cols, seed=1234, device="cpu")[:, :chains * chain_cols].numpy()
            smp = RefSample(model, seqs, chains, chain_cols)
            S = smp.S
            for _ in range(args.warmup):
                smp.run(args.model, ncores)
            t = sum(smp.run(args.model, ncores) for _ in range(args.steps))
            smp.close()
            kind = "reference"
            sample = (f"{S} columns per step of the same synthetic workload as a MAF file of {chains} chains x {chain_cols} columns "
                      f"({smp.info['blocks']} blocks, {smp.info['bytes']} bytes, tmpfs), the reference's unmodified build-tracks "
                      f"(oracle/_ref, GSL shim, -O3 -fopenmp) --threads {ncores}: MAF parse + 6 raw tracks + power track + wig text")
        else:
            import multiprocessing as mp
            S = args.cpu_sample or 6000 * ncores
            seqs = synth_alignment(model, S, seed=1234, device="cpu")[:, :S].numpy()
            pool = mp.get_context("fork").Pool(ncores, initializer=_cpu_init, initargs=(args.model,))
            pool.map(_cpu_chunk, [np.ascontiguousarray(seqs[:, :64])] * ncores)
            for _ in range(args.warmup):
                cpu_columns_per_sec(args.model, seqs, ncores, pool)
            t = 0.0
            for _ in range(args.steps):
                t += cpu_columns_per_sec(args.model, seqs, ncores, pool)[1]
            pool.close()
            kind = "port"
            sample = f"{S} columns per step of the same synthetic workload, oracle port of the reference path, {ncores} processes"
        v = S * args.steps / t
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "sample_columns_per_step": S, "phylogenetic_model": args.model},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": ncores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}), file=json_out, flush=True)
        return

    import torch
    import torch.distributed as dist
    from phylocsfpp_b200 import capi
    from phylocsfpp_b200.synth import synth_alignment

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: phylocsfpp_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    B = args.cols
    Wn = B - 2
    dm = capi.DeviceModel(model, local_rank)
    if args.chunk_cols:
        dm.set_chunk_columns(args.chunk_cols)
    seqs = synth_alignment(model, B, seed=1234 + rank, device=dev)     # [nl, ld] resident in HBM
    ld = seqs.shape[1]
    plus = torch.empty(Wn, dtype=torch.float64, device=dev)
    minus = torch.empty(Wn, dtype=torch.float64, device=dev)
    bls = torch.empty(B, dtype=torch.float64, device=dev)
    flags = (capi.TRACKS_SCORES | capi.TRACKS_BLS | (capi.TRACKS_NO_DEDUP if args.no_dedup else 0)
             | {"f64": 0, "tc5": capi.TRACKS_TC5}[args.precision])
    stream = torch.cuda.current_stream()

    def step():
        dm.tracks_device(seqs.data_ptr(), B, ld, flags, plus.data_ptr(), minus.data_ptr(), bls.data_ptr(), 0, stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    stats = dm.tracks_device_finish(stream.cuda_stream)

    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    stats = dm.tracks_device_finish(stream.cuda_stream)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    t_ms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = world * B * args.steps / (ms_max / 1e3)
    checksum = float(plus[::4097].sum().item() + minus[::4099].sum().item() + bls[::4111].sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"plus": plus, "minus": minus, "bls": bls})

    # ---- e2e through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region)
    h_seqs = torch.empty((nl, ld), dtype=torch.uint8, pin_memory=True)
    h_seqs.copy_(seqs)
    h_plus = torch.empty(Wn, dtype=torch.float64, pin_memory=True)
    h_minus = torch.empty(Wn, dtype=torch.float64, pin_memory=True)
    h_bls = torch.empty(B, dtype=torch.float64, pin_memory=True)
    lib = capi.load()
    st = capi.TracksStats()

    def e2e_step():
        capi._check(lib.pcsf_tracks(dm.h, h_seqs.data_ptr(), B, ld, flags, h_plus.data_ptr(), h_minus.data_ptr(),
                                    h_bls.data_ptr(), None, st))

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    n_e2e = max(1, min(args.steps, 3))
    for _ in range(n_e2e):
        e2e_step()
    torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = world * B * n_e2e / float(t_e2e.item())
    assert abs(float(h_bls[::4111].sum()) - float(bls[::4111].sum().item())) < 1e-6

    # ---- per-kernel durations (CUDA events on the launching stream, one extra instrumented step)
    dm.set_timing(True)
    step()
    tstats = dm.tracks_device_finish(stream.cuda_stream)
    dm.set_timing(False)

    # one instrumented step of the other precisions, for the side-by-side the north star asks for
    other = {}
    if rank == 0:
        base = flags & ~capi.TRACKS_TC5
        dm.set_timing(True)
        for pname, pflag in (("f64", 0), ("tc5", capi.TRACKS_TC5)):
            if pname == args.precision:
                continue
            dm.tracks_device(seqs.data_ptr(), B, ld, base | pflag, plus.data_ptr(), minus.data_ptr(), bls.data_ptr(), 0, stream.cuda_stream)
            o = dm.tracks_device_finish(stream.cuda_stream)
            other[pname] = {"ms_prune_per_step": o["ms_prune"],
                            "columns_per_s_kernels_only": B / (1e-3 * sum(o[k] for k in ("ms_pack", "ms_hash", "ms_dedup", "ms_prune", "ms_scatter", "ms_bls")))}
        dm.set_timing(False)

    out = None
    if rank == 0:
        F = flops_per_pruning(nl)
        n_prune_launch = max(1, tstats["n_chunks"])
        flop_per_launch = tstats["n_unique"] * 2 * F / n_prune_launch
        ms_per_launch = tstats["ms_prune"] / n_prune_launch
        achieved = flop_per_launch / (ms_per_launch * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "profiles", "peaks_fp64.json")))
        except Exception:
            pass
        traffic = None
        traffic_note = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_prune_traffic.json")))
            traffic = tj.get({"f64": "dram_bytes_per_launch", "f32": "dram_bytes_per_launch_f32", "tc5": "dram_bytes_per_launch_tc5"}[args.precision])
            cap_cols = tj.get("tc5_columns_per_captured_launch") if args.precision == "tc5" else None
            if traffic and cap_cols:
                # the ncu --set full capture ran on a smaller batch; DRAM traffic of this kernel (codon ids in, log z out) is linear
                # in the columns of a launch.  The capture is stamped with the hash of the kernel's sources (tools/ncu_traffic_stamp.py):
                # a kernel edited since then gets no traffic figure rather than a stale one.
                traffic = traffic * (B / n_prune_launch) / cap_cols
                traffic_note = f"dram__bytes_read+write of one ncu --set full capture ({tj.get('tc5_source')}) at {cap_cols} columns per launch, scaled to {B // n_prune_launch}"
                if args.precision == "tc5" and tj.get("tc5_kernel_sha16") != kernel_sha16():
                    traffic, traffic_note = None, "the committed ncu capture predates the current kernel sources (profiles/ncu_prune_traffic.json: tc5_kernel_sha16)"
        except Exception:
            pass
        if args.precision == "f64":
            kernel, dtype = "k_prune", "f64"
            peak = peaks.get("micro", {}).get("dmma_tflops", 37.16)
            peak_source = ("FP64 DMMA (mma.sync.m8n8k4.f64) register-loop peak measured on this pool "
                           "(profiles/peaks_fp64.json); MEASURED_PEAKS.json carries no FP64 figure")
            executed = achieved
        else:
            # executed tensor flops per pruning: every inner edge is a (window x 64 x 64) product done as 3 TF32 products
            # (hi*hi, hi*lo, lo*hi) on either tensor path; leaf edges are gathers (no tensor work) on both
            kernel, dtype = "k_prune_tc5", "tf32x3/f32"
            peak = peaks.get("tf32_tflops", 764.2)
            peak_source = ("dense TF32 tensor peak = cuBLAS TF32 GEMM 8192^3 measured on this pool (profiles/peaks_fp64.json; "
                           "MEASURED_PEAKS.json carries bf16 only: 1605 TFLOP/s burst, TF32 is half rate); `achieved` counts "
                           "ALGORITHMIC flops (one FP product per term), `executed_tflops` what the tensor pipe ran")
            # executed tensor flops: three TF32 products per GEMM edge; cherry edges are table rows (no tensor work)
            mult = (3.0 * 8192 * n_tc5_gemms(model.tree)) / F
            executed = achieved * mult
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic",
            "config": {"workload": workload, "phylogenetic_model": args.model, "leaves": nl, "columns_per_step_per_gpu": B,
                       "precision": args.precision,
                       "missing_fraction": 0.30, "l2_policy": "inputs larger than L2 (%.0f MB per step)" % (nl * B / 1e6),
                       "dedup": not args.no_dedup, "unique_pattern_ratio": tstats["n_unique"] / max(1, tstats["n_windows"]),
                       "sharding": "independent column batches per rank, no collective"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": nl * B, "d2h_bytes_per_step": 8 * (2 * Wn + B),
                    "steps": n_e2e, "api": "pcsf_tracks (C-ABI, pinned host buffers)"},
            "gpu_launches": stats["n_launches"] * args.steps,
            "clocks": clocks,
            "roofline": {"kernel": kernel, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "executed_tflops": executed,
                         "executed_frac": executed / peak, "peak_source": peak_source,
                         "flop_per_launch": flop_per_launch, "ms_per_launch": ms_per_launch,
                         "prunings_per_launch": tstats["n_unique"] * 2 / n_prune_launch},
            "stages_ms": {k: tstats[k] for k in ("ms_pack", "ms_hash", "ms_dedup", "ms_prune", "ms_scatter", "ms_bls")},
            # the HBM-bound passes around the pruning kernel: ALGORITHMIC bytes (DESIGN.md section 4) / measured time, against
            # MEASURED_PEAKS.json's copy bandwidth
            "hbm_passes": hbm_passes(tstats, nl, B, Wn),
            "checksum": checksum,
            "other_precisions": other,
        }
        if world == 1 and not args.no_cpu_baseline:
            if os.path.exists(REF_BIN) and not args.cpu_port:
                chains, chain_cols = ref_sample_shape(ncores, per_step=False)
                if args.cpu_sample:
                    chains = max(1, args.cpu_sample // chain_cols)
                smp = RefSample(model, seqs[:, :chains * chain_cols].cpu().numpy(), chains, chain_cols)
                dt = smp.run(args.model, ncores)
                smp.close()
                out["cpu_baseline"] = {
                    "value": smp.S / dt, "unit": UNIT, "cores": ncores, "kind": "reference", "seconds": dt,
                    "sample": f"first {smp.S} columns of the step's batch as a MAF file of {chains} chains x {chain_cols} columns "
                              f"({smp.info['blocks']} blocks, tmpfs), the reference's unmodified build-tracks (oracle/_ref, GSL shim, "
                              f"-O3 -fopenmp) --threads {ncores}: MAF parse + 6 raw tracks + power track + wig text"}
            else:
                S = args.cpu_sample or 3000 * ncores
                v, dt = cpu_columns_per_sec(args.model, seqs[:, :S].cpu().numpy(), ncores)
                out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": ncores, "kind": "port", "seconds": dt,
                                       "sample": f"first {S} columns of the step's batch, oracle port of the reference path, "
                                                 f"{ncores} processes"}
    # ---- the other BASELINE configs and the command line, on the same box in the same run (all ranks take part)
    dm.close()
    del seqs, plus, minus, bls, h_seqs, h_plus, h_minus, h_bls
    torch.cuda.empty_cache()
    pflag = capi.TRACKS_TC5 if args.precision == "tc5" else 0
    legs = {}
    if args.config4_cols > 0:
        legs["config4"] = leg_config4(args.config4_cols, rank, world, local_rank, dist, torch, capi, pflag)
    if args.config5_alignments > 0:
        legs["config5"] = leg_config5(args.config5_alignments, rank, world, local_rank, dist, torch, capi)
    if args.cli_cols > 0:
        legs["cli"] = leg_cli(args.cli_cols, rank, world, local_rank, torch)
    if rank == 0:
        out.update(legs)
        print(json.dumps(out), file=json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
