"""The build-tracks kernels through every door the callers use, not only DeviceModel.tracks.

DeviceModel.tracks calls pcsf_tracks with pageable buffers and ld == L.  bench.py times pcsf_tracks_device on the legacy default
stream with several calls queued before one pcsf_tracks_device_finish; its e2e and config-4 legs and the command line pass
page-locked buffers, config 4 with ld > L.  Those paths differ in what they pack and when: segment by segment with a 2-column halo
on an H2D stream (pcsf_capi.cu, pcsf_tracks_device: the `seg` branch), a D2H copy per chunk on a copy stream behind ev_chunk, timing
mode without segments, PCSF_LEGACY_STREAM=1 without copy streams.

Every window is computed on its own and deterministically on both precisions (tcgen05 with and without dedup is bit-identical,
reverse-complement symmetry holds bit for bit: test_gpu_tracks.py), so every variant here must reproduce the anchor of its precision
bit for bit: pcsf_tracks with one dedup chunk and pageable buffers, itself checked against the oracle.  Pattern indices are checked
against a vectorised restatement of the first-occurrence rule per dedup chunk.

Each variant runs on a fresh handle that first scores a decoy input of the same shape, so that its scratch (packed codes, scores
on the device) holds another input's values: a missing halo or a copy that races its kernel then shows as a wrong score instead of
reading back the right one left over from an earlier call.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi
from phylocsfpp_b200.models import load_model
from tests.util import pattern_index_reference, random_alignment

ONE_CHUNK = 1 << 23            # the largest dedup chunk pcsf_set_chunk_columns accepts
DEFAULT_CHUNK = 1 << 21        # the library's default
JUNK = np.frombuffer(b"R\x00\xff", np.uint8)     # outside ACGTacgt.-Nn: written into the pitch padding [L, ld)
ENTRIES = ("pageable", "alloc_pinned", "register_host", "device_legacy", "device_side")


# ---- CPU-side restatements -----------------------------------------------------------------------------------------------------

def restate_pattern_index(plus: np.ndarray, minus: np.ndarray, chunk: int, dedup: bool = True):
    """pattern_index[2*o + strand] and the unique count of every dedup chunk, for codon-id matrices plus / minus [nl, W]: within a
    chunk, the rank of the first occurrence of the window's leaf-state column (np.unique over the columns viewed as np.void); with
    dedup off, the window's index within its chunk."""
    nl, W = plus.shape
    keys = np.empty((2 * W, nl), np.uint8)
    keys[0::2] = plus.T
    keys[1::2] = minus.T
    rows = keys.view(np.dtype((np.void, nl))).reshape(-1)
    out = np.empty(2 * W, np.uint32)
    counts = []
    for c0 in range(0, W, chunk):
        c1 = min(W, c0 + chunk)
        n = 2 * (c1 - c0)
        if not dedup:
            out[2 * c0:2 * c1] = np.arange(n, dtype=np.uint32)
            counts.append(n)
            continue
        _, first, inverse = np.unique(rows[2 * c0:2 * c1], return_index=True, return_inverse=True)
        rank = np.empty(len(first), np.uint32)
        rank[np.argsort(first, kind="stable")] = np.arange(len(first), dtype=np.uint32)
        out[2 * c0:2 * c1] = rank[inverse.reshape(-1)]
        counts.append(len(first))
    return out, np.array(counts, np.int64)


@pytest.mark.parametrize("L,chunk", [(3, 64), (200, 1 << 22), (333, 64), (700, 7), (1500, 701), (1500, 4095)])
def test_restatement_matches_pattern_index_reference(L, chunk):
    """The vectorised restatement against the loop in tests/util.pattern_index_reference, on inputs with repeated patterns."""
    seqs = random_alignment(12, L, seed=L + chunk, gap=0.5, conserve=0.97)
    plus, minus = orc.window_codons(seqs)
    got, counts = restate_pattern_index(plus, minus, chunk)
    ref = pattern_index_reference(plus, minus, chunk)
    assert np.array_equal(got, ref)
    W = L - 2
    expect = [int(ref[2 * c0:2 * min(W, c0 + chunk)].max()) + 1 for c0 in range(0, W, chunk)]
    assert counts.tolist() == expect
    if W > 1:
        assert counts.sum() < 2 * W, "this input must contain repeated site patterns"
    nd, nd_counts = restate_pattern_index(plus, minus, chunk, dedup=False)
    assert nd_counts.sum() == 2 * W and all(nd[2 * c0] == 0 for c0 in range(0, W, chunk))


def oracle_sample(model, seqs: np.ndarray, idx: np.ndarray):
    """Oracle decibans of the '+' and '-' windows at column offsets idx: the sampled windows' 3 columns side by side, every third
    window of that matrix."""
    sub = np.ascontiguousarray(seqs[:, (idx[:, None] + np.arange(3)).reshape(-1)])
    plus, minus = orc.window_codons(sub)
    mc = orc.OracleModel(model.tree, model.S_c, model.f_c)
    mnc = orc.OracleModel(model.tree, model.S_nc, model.f_nc)
    return orc.run_tracks(mc, mnc, plus[:, 0::3]), orc.run_tracks(mc, mnc, minus[:, 0::3])


def oracle_bls_at(model, seqs: np.ndarray, cols: np.ndarray) -> np.ndarray:
    """Per-base branch length score of the columns `cols` (a column's score depends on that column only)."""
    return orc.bls(model.tree, np.ascontiguousarray(seqs[:, cols]))[1]


# ---- the raw entry points ------------------------------------------------------------------------------------------------------

def _flags(tc5: bool, dedup: bool = True, scores: bool = True, bls: bool = True) -> int:
    return ((capi.TRACKS_SCORES if scores else 0) | (capi.TRACKS_BLS if bls else 0) | (0 if dedup else capi.TRACKS_NO_DEDUP)
            | (capi.TRACKS_TC5 if tc5 else 0))


def _padded(seqs: np.ndarray, ld: int) -> np.ndarray:
    """[nl, ld] copy of seqs with bytes outside the alphabet in the padding [L, ld)."""
    nl, L = seqs.shape
    out = np.empty((nl, ld), np.uint8)
    out[:, :L] = seqs
    if ld > L:
        out[:, L:] = np.resize(JUNK, (nl, ld - L))
    return out


class _HostBuffers:
    """Input [nl, ld] and outputs of one pcsf_tracks call in pageable, pcsf_alloc_pinned or pcsf_register_host memory."""

    def __init__(self, kind: str, nl: int, L: int, ld: int):
        self.kind = kind
        W = max(L - 2, 0)
        sizes = [nl * ld, 8 * W, 8 * W, 8 * L, 8 * W]            # seqs, plus, minus, bls, pattern_index
        self.total = sum(-(-s // 64) * 64 for s in sizes) + 64
        lib = capi.load()
        if kind == "alloc_pinned":
            self.ptr = lib.pcsf_alloc_pinned(self.total)
            assert self.ptr, lib.pcsf_last_error()
            raw = np.frombuffer((C.c_ubyte * self.total).from_address(self.ptr), np.uint8)
        else:
            self._keep = np.empty(self.total + 4096, np.uint8)
            off = (-self._keep.ctypes.data) % 4096
            raw = self._keep[off:off + self.total]
            self.ptr = raw.ctypes.data
            if kind == "register_host":
                capi._check(lib.pcsf_register_host(C.c_void_p(self.ptr), C.c_size_t(self.total)))
        views, o = [], 0
        for s in sizes:
            views.append(raw[o:o + s])
            o += -(-s // 64) * 64
        self.seqs = views[0].reshape(nl, ld)
        self.plus, self.minus, self.bls = views[1].view(np.float64), views[2].view(np.float64), views[3].view(np.float64)
        self.pat = views[4].view(np.uint32)

    def close(self):
        lib = capi.load()
        if self.kind == "alloc_pinned" and self.ptr:
            lib.pcsf_free_pinned(C.c_void_p(self.ptr))
        elif self.kind == "register_host" and self.ptr:
            capi._check(lib.pcsf_unregister_host(C.c_void_p(self.ptr)))
        self.ptr = None


def run_host(dm, seqs: np.ndarray, ld: int, flags: int, kind: str = "pageable", patterns: bool = True):
    """pcsf_tracks on buffers of `kind`; returns plus, minus, bls, pattern_index and stats (copies, the buffers are released)."""
    nl, L = seqs.shape
    W = max(L - 2, 0)
    hb = _HostBuffers(kind, nl, L, ld)
    try:
        hb.seqs[:] = _padded(seqs, ld)
        for a in (hb.plus, hb.minus, hb.bls):
            a[:] = np.nan
        hb.pat[:] = 0xFFFFFFFF
        st = capi.TracksStats()
        capi._check(capi.load().pcsf_tracks(dm.h, hb.seqs.ctypes.data, L, ld, flags, hb.plus.ctypes.data, hb.minus.ctypes.data,
                                            hb.bls.ctypes.data, hb.pat.ctypes.data if patterns else None, C.byref(st)))
        return dict(plus=hb.plus[:W].copy(), minus=hb.minus[:W].copy(), bls=hb.bls[:L].copy(),
                    pattern_index=hb.pat[:2 * W].copy() if patterns else None, stats=st.as_dict())
    finally:
        hb.close()


class _DeviceCall:
    """Device buffers of one pcsf_tracks_device call: input [nl, ld] at `offset` bytes past a 256-byte aligned allocation,
    outputs filled with NaN / 0xFFFFFFFF so that a window the call never writes cannot pass."""

    def __init__(self, seqs: np.ndarray, ld: int, offset: int = 0):
        import torch
        nl, L = seqs.shape
        W = max(L - 2, 0)
        self.L, self.ld = L, ld
        self.flat = torch.empty(nl * ld + offset + 16, dtype=torch.uint8, device="cuda")
        self.flat[offset:offset + nl * ld].copy_(torch.from_numpy(_padded(seqs, ld).reshape(-1)))
        self.d_seqs = self.flat.data_ptr() + offset
        self.plus = torch.full((max(W, 1),), float("nan"), dtype=torch.float64, device="cuda")
        self.minus = torch.full((max(W, 1),), float("nan"), dtype=torch.float64, device="cuda")
        self.bls = torch.full((max(L, 1),), float("nan"), dtype=torch.float64, device="cuda")
        self.pat = torch.full((max(2 * W, 1),), -1, dtype=torch.int32, device="cuda")
        torch.cuda.current_stream().synchronize()       # the copy and the fills are done before any stream reads the buffers

    def enqueue(self, dm, flags: int, stream_handle: int):
        dm.tracks_device(self.d_seqs, self.L, self.ld, flags, self.plus.data_ptr(), self.minus.data_ptr(), self.bls.data_ptr(),
                         self.pat.data_ptr(), stream_handle)

    def result(self, stats=None):
        W = max(self.L - 2, 0)
        return dict(plus=self.plus[:W].cpu().numpy(), minus=self.minus[:W].cpu().numpy(), bls=self.bls[:self.L].cpu().numpy(),
                    pattern_index=self.pat[:2 * W].cpu().numpy().view(np.uint32), stats=stats)


def _stream(kind: str):
    """(torch stream or None, handle): the legacy default stream is handle 0, as bench.py passes it."""
    import torch
    if kind == "device_legacy":
        return None, 0
    torch.cuda.current_stream().synchronize()        # buffers the caller filled on the current stream are ready
    s = torch.cuda.Stream()
    return s, s.cuda_stream


def run_device(dm, seqs: np.ndarray, ld: int, flags: int, kind: str = "device_legacy", offset: int = 0):
    """One pcsf_tracks_device call and its finish on the legacy default stream or on a side stream."""
    call = _DeviceCall(seqs, ld, offset)
    s, handle = _stream(kind)
    call.enqueue(dm, flags, handle)
    stats = dm.tracks_device_finish(handle)
    return call.result(stats)


def run_entry(dm, kind: str, seqs: np.ndarray, ld: int, flags: int, offset: int = 0):
    if kind in ("device_legacy", "device_side"):
        return run_device(dm, seqs, ld, flags, kind, offset)
    assert offset == 0
    return run_host(dm, seqs, ld, flags, kind)


def fresh_handle(model, chunk: int, timing: bool = False):
    dm = capi.DeviceModel(model)
    dm.set_chunk_columns(chunk)
    dm.set_timing(timing)
    return dm


def anchors(model, seqs: np.ndarray):
    """The FP64 and tcgen05 anchors: pcsf_tracks, one dedup chunk, pageable buffers, ld == L, each on a fresh handle."""
    out = {}
    for tc5 in (False, True):
        dm = fresh_handle(model, ONE_CHUNK)
        out[tc5] = run_host(dm, seqs, seqs.shape[1], _flags(tc5))
        dm.close()
    return out


def check_anchors(model, seqs: np.ndarray, anc, n_sample: int = 2048, seed: int = 0):
    """Anchors against the oracle on sampled windows (FP64 1e-6, tcgen05 2e-4 decibans) and the tcgen05 anchor against the FP64
    one on every window (2e-4); BLS bit-exact on sampled columns; pattern indices against the restatement of one chunk."""
    nl, L = seqs.shape
    W = L - 2
    rng = np.random.default_rng(seed)
    idx = np.unique(np.concatenate([[0, W - 1], rng.integers(0, W, min(n_sample, W))]))
    ref_p, ref_m = oracle_sample(model, seqs, idx)
    cols = np.unique(np.concatenate([[0, L - 1], rng.integers(0, L, min(n_sample, L))]))
    ref_b = oracle_bls_at(model, seqs, cols)
    f64, t5 = anc[False], anc[True]
    assert max(np.abs(f64["plus"][idx] - ref_p).max(), np.abs(f64["minus"][idx] - ref_m).max()) <= 1e-6
    assert max(np.abs(t5["plus"][idx] - ref_p).max(), np.abs(t5["minus"][idx] - ref_m).max()) <= 2e-4
    assert max(np.abs(t5["plus"] - f64["plus"]).max(), np.abs(t5["minus"] - f64["minus"]).max()) <= 2e-4
    for a in (f64, t5):
        assert np.array_equal(a["bls"][cols], ref_b), "BLS must be bit-exact"
        assert np.isfinite(a["plus"]).all() and np.isfinite(a["minus"]).all()
    plus, minus = orc.window_codons(seqs)
    pidx, counts = restate_pattern_index(plus, minus, ONE_CHUNK)
    for a in (f64, t5):
        assert np.array_equal(a["pattern_index"], pidx)
        assert a["stats"]["n_windows"] == 2 * W and a["stats"]["n_chunks"] == 1 and a["stats"]["n_unique"] == counts.sum()


def check_variant(res, anchor, seqs: np.ndarray, chunk: int, dedup: bool, timing: bool = False, codons=None):
    """A variant reproduces its precision's anchor bit for bit; pattern indices and stats follow its own dedup chunks."""
    nl, L = seqs.shape
    W = L - 2
    for k in ("plus", "minus", "bls"):
        assert np.array_equal(res[k], anchor[k]), f"{k} differs from the anchor at {np.flatnonzero(res[k] != anchor[k])[:8]}"
    plus, minus = codons if codons is not None else orc.window_codons(seqs)
    pidx, counts = restate_pattern_index(plus, minus, chunk, dedup)
    if chunk >= W and dedup:
        assert np.array_equal(pidx, anchor["pattern_index"])
    assert np.array_equal(res["pattern_index"], pidx)
    st = res["stats"]
    assert st["n_windows"] == 2 * W and st["n_chunks"] == -(-W // chunk) and st["n_unique"] == counts.sum()
    ms = [st[k] for k in ("ms_pack", "ms_hash", "ms_dedup", "ms_prune", "ms_scatter", "ms_bls")]
    if timing:
        assert st["ms_prune"] > 0 and min(ms) >= 0, st
    else:
        assert all(v == 0 for v in ms), st


# ---- 1 + 2: anchors and the invariance matrix ----------------------------------------------------------------------------------

MATRIX_L = 4099 + 2            # 4099 windows: 6 chunks of 701 (the last of 594), 2 of 4095 (the last of 4)


@pytest.fixture(scope="module")
def matrix_input():
    model = load_model("12flies")
    seqs = random_alignment(model.nl, MATRIX_L, seed=2024, gap=0.5, conserve=0.97)
    decoy = random_alignment(model.nl, MATRIX_L, seed=2025, gap=0.3, conserve=0.7)
    anc = anchors(model, seqs)
    return model, seqs, decoy, anc, orc.window_codons(seqs)


@pytest.mark.gpu
def test_anchors_against_oracle(matrix_input):
    """pcsf_tracks, one chunk, pageable, ld == L (pcsf_capi.cu pcsf_tracks -> pcsf_tracks_device, non-segmented run_pack) on
    both precisions, against the oracle; the anchors every variant below must reproduce."""
    model, seqs, _, anc, _ = matrix_input
    check_anchors(model, seqs, anc)
    assert anc[False]["stats"]["n_unique"] < 2 * (MATRIX_L - 2), "this input must contain repeated site patterns"


# (entry point, tcgen05, dedup, chunk columns, ld mode, device base offset, timing, PCSF_LEGACY_STREAM)
#   ld mode: "L"; "16" = L rounded up to 16; "junk" = L + 37; padding bytes are R, 0x00, 0xFF
MATRIX = [
    ("pageable", False, True, 0, "L", 0, False, False),
    ("pageable", True, False, 701, "junk", 0, False, False),        # segmented: 6 chunks, k_keys_tracks_unaligned (no dedup: unused)
    ("pageable", False, True, 4095, "16", 0, True, False),          # timing: no segments, per-stage events
    ("alloc_pinned", True, True, 701, "junk", 0, False, False),     # segmented page-locked, unaligned keys, ld > L
    ("alloc_pinned", False, False, 4095, "16", 0, False, False),
    ("alloc_pinned", True, True, 0, "L", 0, True, False),
    ("alloc_pinned", False, True, 701, "junk", 0, False, True),     # legacy stream: one H2D, non-piped D2H
    ("register_host", False, True, 4095, "junk", 0, False, False),
    ("register_host", True, False, 0, "L", 0, False, False),
    ("register_host", True, True, 4095, "16", 0, False, True),
    ("device_legacy", False, True, 701, "L", 3, True, False),       # misaligned base: every row goes through k_pack's table path
    ("device_legacy", True, True, 4095, "16", 0, False, False),
    ("device_legacy", True, False, 0, "junk", 8, False, True),
    ("device_side", False, False, 0, "junk", 15, False, False),
    ("device_side", True, True, 701, "junk", 1, False, False),
    ("device_side", False, True, 4095, "L", 0, False, True),
    ("device_side", True, True, 0, "16", 0, True, False),
]


def _ld(mode: str, L: int) -> int:
    return {"L": L, "16": (L + 15) // 16 * 16, "junk": L + 37}[mode]


@pytest.mark.gpu
@pytest.mark.parametrize("entry,tc5,dedup,chunk,ld_mode,offset,timing,legacy", MATRIX,
                         ids=[f"{e}-{'tc5' if t else 'f64'}-{'dedup' if d else 'nodedup'}-c{c or 'default'}-ld{m}-off{o}"
                              f"{'-timing' if ti else ''}{'-legacy' if lg else ''}" for e, t, d, c, m, o, ti, lg in MATRIX])
def test_entry_point_matrix(matrix_input, monkeypatch, entry, tc5, dedup, chunk, ld_mode, offset, timing, legacy):
    """Each variant equals the anchor of its precision bit for bit.  Reaches:
    - segmented page-locked and pageable pcsf_tracks (pcsf_capi.cu:654 `segmented`; :518-533 H2D segments on h2d_stream behind
      ev_h2d[c] with the row pitch ld > L; :558-575 run_pack_segment with its 2-column halo; :593 D2H per chunk behind ev_chunk);
    - k_keys_tracks_unaligned (kernels.cuh:180, launched at pcsf_capi.cu:326-330): chunks of 701 and 4095 start at columns that
      are not multiples of 4;
    - ld > L with R, 0x00 and 0xFF in [L, ld) (the H2D copy at :530 and k_pack read [0, L) of each row only);
    - pcsf_tracks_device on the legacy default stream and on a side stream, the base 1 to 15 bytes past an aligned address
      (k_pack's per-row `vec` test, kernels.cuh:31, sends such rows to the table path, kernels.cuh:75-91);
    - timing mode (pcsf_capi.cu:654 `!m->timing`: no segments; event synchronisation at :319 and :580);
    - PCSF_LEGACY_STREAM=1 (pcsf_capi.cu:221: no own, copy or h2d stream; pcsf_tracks' non-piped D2H at :670)."""
    model, seqs, decoy, anc, codons = matrix_input
    if legacy:
        monkeypatch.setenv("PCSF_LEGACY_STREAM", "1")         # read in pcsf_model_create
    L = seqs.shape[1]
    ld = _ld(ld_mode, L)
    eff_chunk = chunk or DEFAULT_CHUNK
    dm = fresh_handle(model, chunk, timing)
    flags = _flags(tc5, dedup)
    run_entry(dm, entry, decoy, ld, flags, offset)             # the scratch now holds another input's codes and scores
    res = run_entry(dm, entry, seqs, ld, flags, offset)
    dm.close()
    check_variant(res, anc[tc5], seqs, eff_chunk, dedup, timing, codons)


@pytest.mark.gpu
def test_chunks_of_64_with_every_tail():
    """Chunks of 64 columns with L = 64 k + 2 + r, r = 1..15: the last chunk has r windows, and for r <= 13 the previous segment's
    halo already reached L (pcsf_capi.cu:558-565: the empty segment is not packed again).  Every r on another entry point and
    precision, page-locked and device entries included, against fresh anchors of the same input."""
    model = load_model("12flies")
    for r in range(1, 16):
        L = 64 * 6 + 2 + r
        seqs = random_alignment(model.nl, L, seed=700 + r, gap=0.5, conserve=0.9)
        decoy = random_alignment(model.nl, L, seed=800 + r)
        anc = anchors(model, seqs)
        check_anchors(model, seqs, anc, n_sample=64, seed=r)
        entry = ENTRIES[r % len(ENTRIES)]
        tc5, dedup = bool(r & 1), r % 3 != 0
        ld = _ld(("L", "16", "junk")[r % 3], L)
        offset = r if entry.startswith("device") else 0
        dm = fresh_handle(model, 64)
        run_entry(dm, entry, decoy, ld, _flags(tc5, dedup), offset)
        res = run_entry(dm, entry, seqs, ld, _flags(tc5, dedup), offset)
        dm.close()
        check_variant(res, anc[tc5], seqs, 64, dedup)


@pytest.mark.gpu
def test_one_chunk_of_more_than_4_mi_windows():
    """One dedup chunk of 2.3 Mi columns (4.6 M windows, 1147 scan blocks): k_scan_sums sums several block totals per thread
    (kernels.cuh:320-337, `per = (nblocks + 1023) / 1024` = 2), which needs a chunk of more than 2 Mi columns
    (pcsf_set_chunk_columns allows 8 Mi).  Anchors against the oracle and the restated pattern indices, then the device entry on a
    side stream with the same chunk, and page-locked pcsf_tracks with the default chunk (2 segments, no multi-sum)."""
    model = load_model("12flies")
    L = (1 << 21) + 250_000
    seqs = random_alignment(model.nl, L, seed=4, gap=0.5, conserve=0.97)
    W = L - 2
    assert 2 * W > 1024 * 4096
    anc = anchors(model, seqs)
    check_anchors(model, seqs, anc, n_sample=2048, seed=4)
    codons = orc.window_codons(seqs)
    assert anc[False]["stats"]["n_unique"] < 2 * W, "dedup must have work to do"
    dm = fresh_handle(model, ONE_CHUNK)
    res = run_device(dm, seqs, L + 37, _flags(True), "device_side", offset=5)
    dm.close()
    check_variant(res, anc[True], seqs, ONE_CHUNK, True, codons=codons)
    dm = fresh_handle(model, 0)
    res = run_host(dm, seqs, (L + 15) // 16 * 16, _flags(False), "alloc_pinned")
    dm.close()
    check_variant(res, anc[False], seqs, DEFAULT_CHUNK, True, codons=codons)


# ---- 3: the benchmark's shapes -------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_config3_shape_every_path():
    """bench.py's timed shape: 58mammals, synth_alignment on the device, 8 Mi + 5 columns, tcgen05 + BLS, several
    pcsf_tracks_device calls queued on the legacy default stream before one finish (bench.py `step`), the same on a side stream,
    and page-locked pcsf_tracks (segmented, 5 dedup chunks of 2 Mi: H2D segments at pcsf_capi.cu:518-533, per-chunk D2H behind
    ev_chunk at :590-597).  The three
    tcgen05 runs are bit-identical, within 3e-4 decibans of the FP64 path on every window with bit-identical BLS; 4096 sampled
    windows against the oracle (FP64 1e-6, tcgen05 3e-4)."""
    import torch
    from phylocsfpp_b200.synth import synth_alignment
    model = load_model("58mammals")
    nl = model.nl
    B = (1 << 23) + 5
    W = B - 2
    d_seqs = synth_alignment(model, B, seed=1234, device="cuda")
    ld = d_seqs.shape[1]
    flags = _flags(True)

    def queued(kind, n_calls=3):
        dm = capi.DeviceModel(model)
        plus = torch.full((W,), float("nan"), dtype=torch.float64, device="cuda")
        minus = torch.full((W,), float("nan"), dtype=torch.float64, device="cuda")
        bls = torch.full((B,), float("nan"), dtype=torch.float64, device="cuda")
        s, handle = _stream(kind)
        for _ in range(n_calls):
            dm.tracks_device(d_seqs.data_ptr(), B, ld, flags, plus.data_ptr(), minus.data_ptr(), bls.data_ptr(), 0, handle)
        st = dm.tracks_device_finish(handle)
        dm.close()
        assert st["n_windows"] == 2 * W and st["n_chunks"] == 5
        return plus.cpu().numpy(), minus.cpu().numpy(), bls.cpu().numpy()

    legacy = queued("device_legacy")
    side = queued("device_side")
    h_seqs = torch.empty((nl, ld), dtype=torch.uint8, pin_memory=True)
    h_seqs.copy_(d_seqs)
    decoy = torch.empty((nl, ld), dtype=torch.uint8, pin_memory=True)
    decoy.copy_(synth_alignment(model, B, seed=99, device="cuda"))
    outs = [torch.full((n,), float("nan"), dtype=torch.float64, pin_memory=True) for n in (W, W, B)]
    dm = capi.DeviceModel(model)
    lib = capi.load()
    st = capi.TracksStats()
    for src in (decoy, h_seqs):
        capi._check(lib.pcsf_tracks(dm.h, src.data_ptr(), B, ld, flags, *[o.data_ptr() for o in outs], None, C.byref(st)))
    dm.close()
    assert st.n_chunks == 5
    pinned = tuple(o.numpy().copy() for o in outs)
    for name, got in (("side stream", side), ("page-locked", pinned)):
        for k in range(3):
            assert np.array_equal(got[k], legacy[k]), f"{name}: {('plus', 'minus', 'bls')[k]} differs from the legacy-stream run"
    dm = capi.DeviceModel(model)
    f_plus = torch.empty(W, dtype=torch.float64, device="cuda")
    f_minus = torch.empty(W, dtype=torch.float64, device="cuda")
    f_bls = torch.empty(B, dtype=torch.float64, device="cuda")
    dm.tracks_device(d_seqs.data_ptr(), B, ld, _flags(False), f_plus.data_ptr(), f_minus.data_ptr(), f_bls.data_ptr(), 0, 0)
    dm.tracks_device_finish(0)
    dm.close()
    f64 = f_plus.cpu().numpy(), f_minus.cpu().numpy(), f_bls.cpu().numpy()
    d = max(np.abs(legacy[0] - f64[0]).max(), np.abs(legacy[1] - f64[1]).max())
    print(f"config 3 shape, {2 * W} windows: tcgen05 max |delta| vs FP64 = {d:.3e} decibans")
    assert d <= 3e-4
    assert np.array_equal(legacy[2], f64[2])
    seqs = h_seqs.numpy()[:, :B]
    rng = np.random.default_rng(3)
    idx = np.unique(np.concatenate([[0, W - 1], rng.integers(0, W, 4096)]))
    ref_p, ref_m = oracle_sample(model, seqs, idx)
    assert max(np.abs(f64[0][idx] - ref_p).max(), np.abs(f64[1][idx] - ref_m).max()) <= 1e-6
    assert max(np.abs(legacy[0][idx] - ref_p).max(), np.abs(legacy[1][idx] - ref_m).max()) <= 3e-4
    cols = np.unique(np.concatenate([[0, B - 1], rng.integers(0, B, 4096)]))
    assert np.array_equal(f64[2][cols], oracle_bls_at(model, seqs, cols))


@pytest.mark.gpu
def test_config4_last_batch_with_ld_above_L():
    """bench.py's config 4: 100vertebrates, a page-locked [nl][4 Mi] buffer, tcgen05; the last batch of a 250 M-column run on one
    GPU is L = 2,536,064 < ld (pcsf_tracks segmented over 2 chunks, pcsf_capi.cu:530 copying [0, L) of each row with the pitch ld).
    Bit-identical to a contiguous pageable call on the same columns."""
    import torch
    from phylocsfpp_b200.synth import synth_alignment
    model = load_model("100vertebrates")
    nl = model.nl
    Bc = 1 << 22
    L = 250_000_000 % Bc
    assert L == 2_536_064
    d_seqs = synth_alignment(model, Bc, seed=4321, device="cuda")
    ld = d_seqs.shape[1]
    h_seqs = torch.empty((nl, ld), dtype=torch.uint8, pin_memory=True)
    h_seqs.copy_(d_seqs)
    del d_seqs
    h_seqs[:, L:] = torch.from_numpy(np.resize(JUNK, (nl, ld - L)))       # the rest of the buffer is not this batch's input
    W = L - 2
    outs = [torch.full((n,), float("nan"), dtype=torch.float64, pin_memory=True) for n in (Bc, Bc, Bc)]
    dm = capi.DeviceModel(model)
    st = capi.TracksStats()
    capi._check(capi.load().pcsf_tracks(dm.h, h_seqs.data_ptr(), L, ld, _flags(True), *[o.data_ptr() for o in outs], None,
                                        C.byref(st)))
    dm.close()
    assert st.n_chunks == 2 and st.n_windows == 2 * W
    got = outs[0].numpy()[:W], outs[1].numpy()[:W], outs[2].numpy()[:L]
    dm = capi.DeviceModel(model)
    ref = dm.tracks(np.ascontiguousarray(h_seqs.numpy()[:, :L]), tc5=True)
    dm.close()
    for k, name in enumerate(("plus", "minus", "bls")):
        assert np.array_equal(got[k], ref[name]), name
    assert np.isfinite(got[0]).all() and np.isfinite(got[1]).all()


# ---- 4: queued calls of different sizes ----------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["device_legacy", "device_side"])
def test_queued_calls_of_growing_and_shrinking_size(kind):
    """A small, a large and a small pcsf_tracks_device call queued on one stream before one finish, each with its own outputs: the
    large one grows the scratch (DevBuf::reserve, pcsf_capi.cu:43, frees and reallocates) while the first is still queued.  Every
    output equals its own anchor.  The stats finish returns describe the last call (n_windows, n_chunks, and n_unique from the last
    call's chunk counters)."""
    import torch
    model = load_model("12flies")
    sizes = (1000, 300_000, 777)
    inputs = [random_alignment(model.nl, L, seed=40 + i, gap=0.5, conserve=0.95) for i, L in enumerate(sizes)]
    dm = fresh_handle(model, 65536)
    calls = [_DeviceCall(x, x.shape[1] + 5, offset=i) for i, x in enumerate(inputs)]
    s, handle = _stream(kind)
    for c, tc5 in zip(calls, (True, False, True)):
        c.enqueue(dm, _flags(tc5), handle)
    stats = dm.tracks_device_finish(handle)
    torch.cuda.synchronize()
    dm.close()
    for seqs, c, tc5 in zip(inputs, calls, (True, False, True)):
        anc = anchors(model, seqs)
        res = c.result()
        for k in ("plus", "minus", "bls"):
            assert np.array_equal(res[k], anc[tc5][k]), (seqs.shape[1], k)
        plus, minus = orc.window_codons(seqs)
        assert np.array_equal(res["pattern_index"], restate_pattern_index(plus, minus, 65536)[0])
    L = sizes[-1]
    plus, minus = orc.window_codons(inputs[-1])
    assert stats["n_windows"] == 2 * (L - 2) and stats["n_chunks"] == 1
    assert stats["n_unique"] == restate_pattern_index(plus, minus, 65536)[1].sum()


# ---- 5: bad characters ---------------------------------------------------------------------------------------------------------

ACCEPTED = {c: c for c in b"ACGTN"} | {ord("a"): ord("A"), ord("c"): ord("C"), ord("g"): ord("G"), ord("t"): ord("T"),
                                         ord("n"): ord("N"), ord("-"): ord("N"), ord("."): ord("N")}


@pytest.mark.gpu
def test_every_byte_at_a_simd_and_a_table_position():
    """Each of the 256 byte values once at column 20 (k_pack's SIMD-compare path, kernels.cuh:61-74: 16-byte aligned row, a full
    16-byte vector) and once at column L - 3 of L = 70 (the table path, kernels.cuh:75-91: the last partial vector).  Exactly the
    bytes in ACGTacgt.-Nn are accepted, each scored as its canonical byte (A C G T, or N); every other byte gives
    PCSF_ERR_BAD_CHAR, and the handle scores the next call normally."""
    model = load_model("12flies")
    L = 70
    base = random_alignment(model.nl, L, seed=1, gap=0.0, conserve=0.8)
    dm = capi.DeviceModel(model)
    clean = run_host(dm, base, L, _flags(False))
    for col in (20, L - 3):
        canon = {}
        for b in set(ACCEPTED.values()):
            s = base.copy()
            s[4, col] = b
            canon[b] = run_host(dm, s, L, _flags(False))
        for b in range(256):
            s = base.copy()
            s[4, col] = b
            if b in ACCEPTED:
                res = run_host(dm, s, L, _flags(False))
                want = canon[ACCEPTED[b]]
                for k in ("plus", "minus", "bls", "pattern_index"):
                    assert np.array_equal(res[k], want[k]), (col, chr(b), k)
            else:
                with pytest.raises(capi.PcsfError) as ei:
                    run_host(dm, s, L, _flags(False))
                assert ei.value.status == capi.PCSF_ERR_BAD_CHAR, (col, b)
        assert np.array_equal(run_host(dm, base, L, _flags(False))["plus"], clean["plus"])
    dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["alloc_pinned", "register_host"])
def test_bad_byte_in_a_later_segment(kind):
    """Page-locked pcsf_tracks over 7 chunks of 64 (segmented: every segment is packed by run_pack_segment, pcsf_capi.cu:565, right
    before its chunk is pruned): a bad byte in segment 1, or in the last partial segment, gives PCSF_ERR_BAD_CHAR; the same buffer
    without it then scores PCSF_OK (the flag was cleared)."""
    model = load_model("12flies")
    L = 64 * 6 + 2 + 9
    seqs = random_alignment(model.nl, L, seed=17)
    dm = fresh_handle(model, 64)
    good = run_host(dm, seqs, L + 11, _flags(True), kind)
    for col in (64 * 2 + 5, L - 1):
        s = seqs.copy()
        s[7, col] = ord("R")
        with pytest.raises(capi.PcsfError) as ei:
            run_host(dm, s, L + 11, _flags(True), kind)
        assert ei.value.status == capi.PCSF_ERR_BAD_CHAR
        again = run_host(dm, seqs, L + 11, _flags(True), kind)
        assert np.array_equal(again["plus"], good["plus"]) and again["stats"]["n_chunks"] == 7
    dm.close()


@pytest.mark.gpu
def test_bad_bytes_only_in_the_pitch_padding():
    """Bytes outside the alphabet in [L, ld) only are never read: PCSF_OK from pcsf_tracks (pageable and page-locked, segmented)
    and from pcsf_tracks_device."""
    model = load_model("12flies")
    L = 500
    seqs = random_alignment(model.nl, L, seed=23)
    dm = fresh_handle(model, 64)
    for kind in ("pageable", "alloc_pinned"):
        run_host(dm, seqs, L + 37, _flags(False), kind)
    run_device(dm, seqs, L + 37, _flags(False), "device_side", offset=2)
    dm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["device_legacy", "device_side"])
def test_bad_call_queued_before_a_good_one(kind):
    """A pcsf_tracks_device call with a bad character queued before a clean one, then one finish (how bench.py queues its steps):
    PCSF_ERR_BAD_CHAR.  The flag covers every call since the last finish (pcsf_tracks_device_finish reads and clears it,
    pcsf_capi.cu:612-613; no call clears it before packing).  It does not leak: a clean device call, pcsf_score_msa and pcsf_tracks
    afterwards give PCSF_OK, and a score-msa call between a bad device call and its finish neither reports nor swallows it
    (score_regions_core reads a flag of its own)."""
    import torch
    model = load_model("12flies")
    L = 300
    good = random_alignment(model.nl, L, seed=5)
    bad = good.copy()
    bad[2, 100] = ord("R")
    dm = capi.DeviceModel(model)
    flags = _flags(True)
    calls = [_DeviceCall(bad, L), _DeviceCall(good, L)]
    s, handle = _stream(kind)
    for c in calls:
        c.enqueue(dm, flags, handle)
    with pytest.raises(capi.PcsfError) as ei:
        dm.tracks_device_finish(handle)
    assert ei.value.status == capi.PCSF_ERR_BAD_CHAR
    # nothing left over: clean calls of every kind on the same handle
    ok = run_device(dm, good, L, flags, kind)
    assert np.array_equal(ok["plus"], calls[1].result()["plus"])
    phylo, _, _ = dm.score_msa([good[:, :297]])
    assert np.isfinite(phylo).all()
    run_host(dm, good, L, flags, "pageable")
    # a score-msa call between a bad device call and its finish (after the device call has run: one handle's scratch serves one
    # call at a time)
    c = _DeviceCall(bad, L)
    c.enqueue(dm, flags, handle)
    torch.cuda.synchronize()
    dm.score_msa([good[:, :297]])
    with pytest.raises(capi.PcsfError) as ei:
        dm.tracks_device_finish(handle)
    assert ei.value.status == capi.PCSF_ERR_BAD_CHAR
    # and a bad score-msa batch leaves the tracks flag alone
    with pytest.raises(capi.PcsfError) as ei:
        dm.score_msa([bad[:, :297]])
    assert ei.value.status == capi.PCSF_ERR_BAD_CHAR
    run_device(dm, good, L, flags, kind)
    dm.score_msa([good[:, :297]])
    dm.close()
