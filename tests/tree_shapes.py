"""Deterministic species trees of 2 to 128 leaves for the pruning kernels, written as external models.

A generated model is `<dir>/<name>.nh` next to copies of 58mammals_coding.ECM / 58mammals_noncoding.ECM, so that
`load_model(prefix)` and the command line's `<model>` argument both accept it.  Branch lengths mix very short (1e-4: P is
nearly the identity), ordinary (0.01 to 0.3) and long (2.5 to 8: P is nearly stationary) values.

Shapes:
  balanced     leaves split as evenly as possible at every node (ceil / floor)
  leafcherry   (leaf, (leaf, leaf))
  caterpillar  ((((l, l), l), l), ...): one cherry at the bottom, every other inner node has a leaf child
  yule         random joins of two subtrees at a time (fixed seed per tree)
"""
from __future__ import annotations

import os
import shutil
from dataclasses import dataclass
from typing import Optional

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ECM_PREFIX = os.path.join(ROOT, "phylocsfpp_b200", "data", "models", "58mammals")


@dataclass(frozen=True)
class Shape:
    shape: str
    nl: int
    long_only: bool = False      # every branch long (2.5 to 8)
    tc5_fits: bool = True        # k_prune_tc5's shared memory holds the tree (pcsf_tracks accepts PCSF_TRACKS_TC5)
    # the tcgen05 program of the tree (csrc/model_prep.hpp: prepare_tc5_program) and the FP64 program's stack depth
    tc5_steps: Optional[int] = None
    tc5_leaves: Optional[int] = None
    tc5_cherries: Optional[int] = None
    tc5_depth: Optional[int] = None
    fp64_depth: Optional[int] = None

    @property
    def name(self) -> str:
        return f"{self.shape}{self.nl}" + ("long" if self.long_only else "")


# The trees the suite runs.  Counts of the balanced and caterpillar trees follow from their shape; those of the Yule trees are
# what the fixed seeds give.
SHAPES = [
    Shape("balanced", 2, tc5_steps=0, tc5_leaves=2, tc5_cherries=0, tc5_depth=0, fp64_depth=0),
    Shape("leafcherry", 3, tc5_steps=0, tc5_leaves=1, tc5_cherries=1, tc5_depth=0, fp64_depth=0),
    Shape("balanced", 4, tc5_steps=0, tc5_leaves=0, tc5_cherries=2, tc5_depth=0, fp64_depth=1),
    Shape("caterpillar", 63, tc5_steps=60, tc5_leaves=61, tc5_cherries=1, tc5_depth=0, fp64_depth=0),
    Shape("caterpillar", 64, tc5_steps=61, tc5_leaves=62, tc5_cherries=1, tc5_depth=0, fp64_depth=0),
    Shape("caterpillar", 65, tc5_steps=62, tc5_leaves=63, tc5_cherries=1, tc5_depth=0, fp64_depth=0),
    Shape("balanced", 63, tc5_steps=30, tc5_leaves=1, tc5_cherries=31, tc5_depth=4, fp64_depth=4),
    Shape("balanced", 64, tc5_steps=30, tc5_leaves=0, tc5_cherries=32, tc5_depth=4, fp64_depth=5),
    Shape("balanced", 65, tc5_steps=31, tc5_leaves=1, tc5_cherries=32, tc5_depth=4, fp64_depth=5),
    Shape("yule", 65, tc5_steps=40, tc5_leaves=19, tc5_cherries=23, tc5_depth=3, fp64_depth=3),
    Shape("yule", 100, tc5_steps=67, tc5_leaves=38, tc5_cherries=31, tc5_depth=3, fp64_depth=3),
    Shape("caterpillar", 120, tc5_steps=117, tc5_leaves=118, tc5_cherries=1, tc5_depth=0, fp64_depth=0),
    Shape("balanced", 125, tc5_steps=62, tc5_leaves=3, tc5_cherries=61, tc5_depth=5, fp64_depth=5),
    Shape("caterpillar", 128, False, False, tc5_steps=125, tc5_leaves=126, tc5_cherries=1, tc5_depth=0, fp64_depth=0),
    Shape("balanced", 128, False, False, tc5_steps=62, tc5_leaves=0, tc5_cherries=64, tc5_depth=5, fp64_depth=6),
    Shape("yule", 128, False, False, tc5_steps=81, tc5_leaves=38, tc5_cherries=45, tc5_depth=3, fp64_depth=3),
]
# the tcgen05 path's shared-memory budget: the longest caterpillar that fits, the shortest that does not, the smallest balanced
# tree that does not, and a 127-leaf tree (none fits: the codon-id block alone is 2 x nl x 128 bytes)
BUDGET_SHAPES = [Shape("caterpillar", 123), Shape("caterpillar", 124, False, False), Shape("balanced", 126, False, False),
                 Shape("balanced", 127, False, False)]
# all-certain columns on long branches: the reference's unscaled FP64 product comes close to underflow
LONG_CATERPILLAR = Shape("caterpillar", 128, True, False)

BY_NAME = {s.name: s for s in SHAPES + BUDGET_SHAPES + [LONG_CATERPILLAR]}


def _seed(spec: Shape) -> int:
    return {"balanced": 1, "leafcherry": 2, "caterpillar": 3, "yule": 4}[spec.shape] * 1000 + spec.nl + 500 * spec.long_only


def topology(spec: Shape):
    """Nested tuples of leaf numbers 0..nl-1 (a leaf is an int)."""
    nl = spec.nl
    if spec.shape == "balanced":
        def bal(lo, hi):
            if hi - lo == 1:
                return lo
            mid = lo + (hi - lo + 1) // 2
            return (bal(lo, mid), bal(mid, hi))
        return bal(0, nl)
    if spec.shape == "leafcherry":
        assert nl == 3
        return (0, (1, 2))
    if spec.shape == "caterpillar":
        t = (0, 1)
        for i in range(2, nl):
            t = (t, i)
        return t
    if spec.shape == "yule":
        rng = np.random.default_rng(_seed(spec))
        pool = list(range(nl))
        while len(pool) > 1:
            i, j = sorted(rng.choice(len(pool), size=2, replace=False).tolist())
            b = pool.pop(j)
            a = pool.pop(i)
            pool.append((a, b))
        return pool[0]
    raise ValueError(spec.shape)


def newick_text(spec: Shape) -> str:
    rng = np.random.default_rng(_seed(spec) + 7)

    def length() -> float:
        u = rng.random()
        if spec.long_only or u >= 0.85:
            return float(rng.uniform(2.5, 8.0))
        if u < 0.15:
            return 1e-4
        return float(rng.uniform(0.01, 0.3))

    def walk(t) -> str:
        if isinstance(t, int):
            s = f"s{t:03d}"
        else:
            s = f"({walk(t[0])},{walk(t[1])})"
        return f"{s}:{length():.6f}"      # the Newick readers take [0-9.]+ lengths: no exponent

    root = topology(spec)
    return f"({walk(root[0])},{walk(root[1])});\n"


def write_model(directory: str, spec: Shape) -> str:
    """Writes <directory>/<name>.nh and the two ECM files next to it; returns the model prefix."""
    prefix = os.path.join(directory, spec.name)
    with open(prefix + ".nh", "w") as fh:
        fh.write(newick_text(spec))
    for kind in ("coding", "noncoding"):
        shutil.copyfile(f"{ECM_PREFIX}_{kind}.ECM", f"{prefix}_{kind}.ECM")
    return prefix
