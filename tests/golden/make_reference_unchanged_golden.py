"""Golden data of tests/test_reference_unchanged.py, so that its comparisons run without the reference:

    python tests/golden/make_reference_unchanged_golden.py      -> tests/golden/reference_unchanged.npz

It records the mirrors' products on the tests' seeded weights and inputs (model forward and gradients, losses, BEV label
images, batch products / losses / gradients / Adam step of the training step, mix3D merge).  Run it only where
tests/test_reference_unchanged.py passes against a checkout of the reference at oracle/_ref/, so that what it records
equals the reference's results (bit for bit where those tests compare bit for bit, within their bounds elsewhere)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import test_reference_unchanged as t  # noqa: E402


def main():
    out = t.golden_products()
    np.savez_compressed(t.GOLDEN, **out)
    print({k: getattr(v, "shape", v) for k, v in out.items()})


if __name__ == "__main__":
    main()
