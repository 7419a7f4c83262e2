"""Regenerate tests/golden/lockstep/*.npz from the UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref`).

    python tests/golden/make_lockstep.py

Every test module listed below names its reference runs in REFERENCE_RUNS (name -> function of the reference library
returning the arrays to store): the scene scripts live next to the tests that replay them on the product.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import lockstep  # noqa: E402
from oracle import ref  # noqa: E402

TEST_MODULES = ("test_e2e_gpu", "test_api_lifecycle_gpu")


def main():
    R = ref.load()
    for module_name in TEST_MODULES:
        for name, run in __import__(module_name).REFERENCE_RUNS.items():
            print("wrote", lockstep.save(name, run(R)))


if __name__ == "__main__":
    main()
