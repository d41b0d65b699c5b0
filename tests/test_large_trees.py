"""Trees of 129 to 512 leaves on the CPU: the generated trees (tests/large_tree_shapes.py), the FP64 pruning program and shared
memory a model of each gets, the eight-word BLS program against the oracle bit for bit, the leaf limit, and the register budget of
the large-tree kernels.  No GPU needed."""
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from phylocsfpp_b200 import capi, newick
from phylocsfpp_b200.models import load_model
from tests import large_tree_shapes as lt
from tests import tree_shapes as ts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def tree_dir(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("large_trees"))
    for t in lt.ALL:
        lt.write_model(d, t.spec)
    lt.write_model(d, lt.TOO_LARGE)
    return d


@pytest.fixture(scope="module")
def check_exe(tmp_path_factory):
    import __graft_entry__ as g
    exe = os.path.join(str(tmp_path_factory.mktemp("ltc")), "large_tree_check")
    subprocess.run([g.NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-o", exe,
                    os.path.join(ROOT, "tools", "large_tree_check.cu")], check=True, capture_output=True)
    return exe


def _stats(exe, prefix, masks=None):
    r = subprocess.run([exe, prefix] + ([masks] if masks else []), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    head = dict((k.strip(), int(v)) for k, v in re.findall(r"([a-z0-9 _]+?) (\d+)(?:,|$)", lines[0]))
    return head, lines[1:]


def test_large_shapes_do_not_touch_the_128_leaf_suite():
    """The shapes of the existing suite stay what they were; the large ones are a list of their own."""
    assert max(s.nl for s in ts.BY_NAME.values()) == 128
    assert not set(ts.BY_NAME) & set(lt.BY_NAME)
    assert sorted({t.nl for t in lt.LARGE}) == [129, 192, 256, 257, 470, 512]
    assert {t.spec.shape for t in lt.LARGE} == {"balanced", "caterpillar", "yule"}


@pytest.mark.parametrize("name", list(lt.BY_NAME))
def test_large_tree_round_trips(tree_dir, name):
    """Each tree parses back with its leaf count, loads as an external model, has its stated FP64 stack depth (Strahler number - 1),
    and the branch lengths are the intended mix.  The recursive generator and parsers stay within Python's default recursion limit."""
    t = lt.BY_NAME[name]
    prefix = os.path.join(tree_dir, name)
    with open(prefix + ".nh") as fh:
        flat = newick.flatten(newick.parse(fh.read()))
    assert flat.nl == t.nl and flat.n == 2 * t.nl - 1
    assert sorted(flat.labels[:flat.nl]) == [f"s{i:03d}" for i in range(t.nl)]
    m = load_model(prefix)
    assert m.nl == t.nl and (m.tree.child1 == flat.child1).all() and (m.tree.branch_len == flat.branch_len).all()
    _, need = newick.strahler_order(flat)
    assert need[flat.n - 1] - 1 == t.max_stack
    bl = flat.branch_len_f64[:-1]
    if t.spec.long_only:
        assert (bl >= 2.5).all() and (bl <= 8.0).all()
    else:
        assert (bl == 1e-4).any() and ((bl >= 0.01) & (bl <= 0.3)).any() and (bl >= 2.5).any()
    assert ts.newick_text(t.spec) == ts.newick_text(t.spec)


@pytest.mark.parametrize("name", list(lt.BY_NAME))
def test_large_tree_program_fits_shared_memory(tree_dir, check_exe, name):
    """prepare_model's FP64 program of each tree has the stated size and stack depth, no tcgen05 program, and k_prune_scaled's shared
    memory at 4 compute warps (stack, exponent stack, leaf ids, program, P stages) fits the 227 KiB opt-in limit."""
    t = lt.BY_NAME[name]
    head, _ = _stats(check_exe, os.path.join(tree_dir, name))
    assert (head["nl"], head["program ops"], head["max_stack"], head["tc5 steps"]) == (t.nl, t.ops, t.max_stack, 0), head
    assert head["smem 4 warps"] == t.smem4 <= lt.SMEM_LIMIT, head


def _boundary_masks(nl, rng, n):
    """Presence patterns (bool [n, nl]): uniform at several densities, and patterns whose present leaves sit within a few leaves of
    the 64-leaf word boundaries 64, 128, 192 and 256 (and of the last leaf), so that collapsed subtrees and left / right leaf sets
    straddle two words."""
    out = []
    for i in range(n):
        kind = i % 4
        if kind == 0:
            m = rng.random(nl) < rng.choice([0.02, 0.3, 0.7, 0.97])
        else:
            m = np.zeros(nl, bool)
            for b in (64, 128, 192, 256, nl - 1):
                if b < nl:
                    lo, hi = max(0, b - 8), min(nl, b + 8)
                    m[lo:hi] = rng.random(hi - lo) < (0.5 if kind == 1 else 0.15)
            if kind == 3:
                m |= rng.random(nl) < 0.05
        out.append(m)
    out += [np.ones(nl, bool), np.zeros(nl, bool), np.eye(1, nl, 0, dtype=bool)[0], np.eye(1, nl, min(64, nl - 1), dtype=bool)[0]]
    return np.array(out)


@pytest.mark.parametrize("name", ["balanced129", "yule192", "caterpillar256", "yule257", "balanced470", "yule512", "balanced512"])
def test_wide_bls_program_matches_the_oracle(tree_dir, check_exe, tmp_path, name):
    """The BLS program k_bls<8> runs (eight-word masks, collapsed subtrees whose first leaf is stored past bit 8 of the flags) gives
    the oracle's compute_bls_score per-base doubles bit for bit on presence patterns around every word boundary."""
    t = lt.BY_NAME[name]
    prefix = os.path.join(tree_dir, name)
    masks = _boundary_masks(t.nl, np.random.default_rng(t.nl), 400)
    path = tmp_path / "masks.txt"
    path.write_text("".join("".join("1" if x else "0" for x in m) + "\n" for m in masks))
    head, lines = _stats(check_exe, prefix, str(path))
    assert head["bls tables"] >= 1 and len(lines) == len(masks)
    got = np.array([float.fromhex(s) for s in lines])
    seqs = np.where(masks.T, ord("A"), ord("N")).astype(np.uint8)        # column c = mask c
    ref = orc.bls(load_model(prefix).tree, seqs)[1]
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    assert (got > 0).sum() > len(masks) // 2


def test_more_than_512_leaves_is_refused(tree_dir):
    """pcsf_model_create refuses a 513-leaf tree with PCSF_ERR_UNSUPPORTED (before it looks for a device), naming the limit."""
    model = load_model(os.path.join(tree_dir, lt.TOO_LARGE.name))
    assert model.nl == 513
    with pytest.raises(capi.PcsfError) as ei:
        capi.DeviceModel(model)
    assert ei.value.status == capi.PCSF_ERR_UNSUPPORTED
    assert "513" in str(ei.value) and "512" in str(ei.value)


def test_large_tree_kernels_do_not_spill(tmp_path):
    """k_prune_scaled (both instantiations) and k_bls<8> compile for sm_100a without local memory: no stack frame, no spills."""
    import __graft_entry__ as g
    out = subprocess.run([g.NVCC] + [f for f in g.NVCC_FLAGS if f != "-shared"] + ["-c", "-Xptxas", "-v", "-o", str(tmp_path / "capi.o"),
                          os.path.join(g.CSRC, "pcsf_capi.cu")], capture_output=True, text=True, check=True).stderr
    props = re.findall(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       out)
    seen = []
    for name, frame, st, ld in props:
        if "k_prune_scaled" in name or "k_blsILi8E" in name:
            seen.append(name)
            assert (int(frame), int(st), int(ld)) == (0, 0, 0), (name, frame, st, ld)
    assert len(seen) == 3, seen
