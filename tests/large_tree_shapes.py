"""Deterministic species trees of 129 to 512 leaves, written as external models by tests/tree_shapes.py's generator (same branch-length
mix, same 58mammals ECMs).  Trees above 128 leaves run the rescaled FP64 pruning (k_prune_scaled) and the eight-word BLS masks
(k_bls<8>), and have no tcgen05 path.

Each shape states the FP64 pruning program's size and stack depth and the shared memory k_prune_scaled needs for it at 4 compute
warps (csrc/kernels.cuh: prune_smem_bytes, which for these trees includes 128 bytes per warp and stack level for the exponents of the
stacked partials).  A balanced tree has the largest Strahler number for its leaf count, so balanced512 is the largest shared-memory
footprint of any tree the library accepts; it fits the 227 KiB (232,448 bytes) a CTA may opt in to.
"""
from __future__ import annotations

from dataclasses import dataclass

from tests.tree_shapes import Shape, write_model  # noqa: F401  (write_model is this module's writer too)

SMEM_LIMIT = 227 * 1024


@dataclass(frozen=True)
class Large:
    spec: Shape
    ops: int            # FP64 pruning program (GATHER / GEMM / PUSH / POP ops + END)
    max_stack: int      # sibling partials alive at once (Strahler number - 1)
    smem4: int          # prune_smem_bytes at 4 compute warps

    @property
    def name(self) -> str:
        return self.spec.name

    @property
    def nl(self) -> int:
        return self.spec.nl


LARGE = [
    Large(Shape("balanced", 129), 383, 6, 174_912),
    Large(Shape("caterpillar", 129), 257, 0, 89_936),
    Large(Shape("yule", 129), 339, 3, 124_048),
    Large(Shape("balanced", 192), 509, 6, 177_440),
    Large(Shape("caterpillar", 192), 383, 0, 92_448),
    Large(Shape("yule", 192), 507, 4, 143_632),
    Large(Shape("balanced", 256), 765, 7, 197_408),
    Large(Shape("caterpillar", 256), 511, 0, 95_008),
    Large(Shape("yule", 256), 667, 4, 146_320),
    Large(Shape("balanced", 257), 767, 7, 197_440),
    Large(Shape("caterpillar", 257), 513, 0, 95_056),
    Large(Shape("yule", 257), 679, 4, 146_400),
    Large(Shape("balanced", 470), 1365, 7, 206_656),
    Large(Shape("caterpillar", 470), 939, 0, 103_568),
    Large(Shape("yule", 470), 1257, 5, 172_432),
    Large(Shape("balanced", 512), 1533, 8, 225_568),
    Large(Shape("caterpillar", 512), 1023, 0, 105_248),
    Large(Shape("yule", 512), 1365, 4, 157_312),
]
# every branch long (2.5 to 8): all-certain columns underflow the reference's unscaled FP64 product
LONG_CATERPILLAR_512 = Large(Shape("caterpillar", 512, True, False), 1023, 0, 105_248)
# one leaf past PCSF_MAX_LEAVES
TOO_LARGE = Shape("caterpillar", 513)

ALL = LARGE + [LONG_CATERPILLAR_512]
BY_NAME = {t.name: t for t in ALL}
