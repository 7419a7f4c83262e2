"""Regenerate tests/golden/host_vectors_ref.npz: the UNMODIFIED reference's geometry, hull and manifold functions on the
seeded inputs of tests/test_host_cpu.py (the product's s2MakeRoundedBox is compared with the reference's box polygon
given a radius) (needs oracle/_ref, built by `make -C oracle ref`).

    python tests/golden/make_host_vectors.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref  # noqa: E402
from test_host_cpu import GOLDEN, box_with_radius, hull_outputs, manifold_outputs, polygon_factory_outputs  # noqa: E402


def main():
    R = ref.load()
    np.savez_compressed(GOLDEN, polygon_factories=polygon_factory_outputs(R, box_with_radius), hull=hull_outputs(R),
                        manifolds=manifold_outputs(R))
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")


if __name__ == "__main__":
    main()
