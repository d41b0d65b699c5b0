"""The generated trees of tests/tree_shapes.py on the CPU: the generator itself, and the tcgen05 step program on every tree.

The GPU suite (tests/test_gpu_tree_shapes.py) runs both pruning kernels on these trees; this file pins that the trees have the
shapes it relies on and that the host-side program the tcgen05 kernel interprets is right for each of them.
"""
import os
import re
import subprocess

import pytest

from phylocsfpp_b200 import newick
from phylocsfpp_b200.models import load_model
from tests import tree_shapes as ts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = list(ts.BY_NAME.values())


@pytest.fixture(scope="module")
def tree_dir(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("trees"))
    for spec in ALL:
        ts.write_model(d, spec)
    return d


@pytest.fixture(scope="module")
def tc5_check_exe(tmp_path_factory):
    exe = os.path.join(str(tmp_path_factory.mktemp("tc5chk")), "tc5_program_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tools", "tc5_program_check.cpp")], check=True)
    return exe


@pytest.mark.parametrize("name", [s.name for s in ALL])
def test_generated_tree_round_trips(tree_dir, name):
    """Each tree parses back through newick.parse / flatten with its leaf count, loads as an external model, has its stated
    FP64 stack depth (Strahler number - 1), and its branch lengths are the intended mix."""
    spec = ts.BY_NAME[name]
    prefix = os.path.join(tree_dir, name)
    with open(prefix + ".nh") as fh:
        t = newick.flatten(newick.parse(fh.read()))
    assert t.nl == spec.nl and t.n == 2 * spec.nl - 1
    assert sorted(t.labels[:t.nl]) == [f"s{i:03d}" for i in range(spec.nl)]
    m = load_model(prefix)
    assert m.nl == spec.nl and (m.tree.child1 == t.child1).all() and (m.tree.branch_len == t.branch_len).all()
    _, need = newick.strahler_order(t)
    if spec.fp64_depth is not None:
        assert need[t.n - 1] - 1 == spec.fp64_depth
    bl = t.branch_len_f64[:-1]
    assert t.branch_len_f64[-1] == 0.0 and (bl > 0).all()
    if spec.long_only:
        assert (bl >= 2.5).all() and (bl <= 8.0).all()
    elif spec.nl >= 63:
        assert (bl == 1e-4).any() and ((bl >= 0.01) & (bl <= 0.3)).any() and (bl >= 2.5).any()
    assert ts.newick_text(spec) == ts.newick_text(spec), "the generator must be deterministic"


@pytest.mark.parametrize("name", [s.name for s in ALL])
def test_tcgen05_step_program_on_generated_trees(tree_dir, tc5_check_exe, name):
    """The tcgen05 step program (chain starts, GEMM steps, leaf and cherry sources, pushes / pops) interpreted on the host in
    FP64 equals the plain Felsenstein recursion, and its FP32-class emulation stays inside 2e-4 decibans: the bounds of
    test_host_logic.py::test_tcgen05_step_program_on_the_cpu, here on program shapes the built-in models do not have (no step
    at all, starts made of cherries, 125 steps, stack depth 5).  The program's shape is the one stated in tree_shapes.py."""
    spec = ts.BY_NAME[name]
    r = subprocess.run([tc5_check_exe, os.path.join(tree_dir, name), "", "60"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    d64 = float(re.search(r"max \|d log z\| = (\S+)", r.stdout).group(1))
    d32 = float(re.search(r"max \|d\| = (\S+) decibans", r.stdout).group(1))
    assert d64 < 1e-11 and d32 < 2e-4, r.stdout
    m = re.search(r"nl (\d+), gemm steps (\d+) .* direct leaves (\d+), cherries (\d+), pushes \d+, stack depth (\d+)", r.stdout)
    nl, steps, leaves, cherries, depth = map(int, m.groups())
    assert nl == spec.nl and leaves + 2 * cherries == nl
    if spec.tc5_steps is not None:
        assert (steps, leaves, cherries, depth) == (spec.tc5_steps, spec.tc5_leaves, spec.tc5_cherries, spec.tc5_depth), r.stdout
