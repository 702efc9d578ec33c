#!/usr/bin/env python
"""Record the activation taps of the original BitNetMCU kernels, for tests/test_taps.py.  Needs a checkout of that project (REF, also
read by oracle/Makefile, which builds its unmodified kernels into oracle/_ref):

    REF=<BitNetMCU checkout> python tests/golden/make_reference_taps.py

What it writes (small, committed, read by the tests wherever they run):

  reference_taps.npz   per fixture model and tap t, "<model>/tap<t>": int8 [266, width] -- the row layer_in holds after the t-th
                       tap-producing ReLUNorm of BitMnistInference (include/bitnetmcu_b200.h section 7), run through the unmodified
                       reference kernels (tests/test_taps.py chain_taps), on the 10 test digits then the 256 xorshift32 images of
                       golden.npz
"""
import os
import sys

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(OUT))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import test_taps as T  # noqa: E402
from conftest import load_model, model_names  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main():
    O.build(quiet=True)
    ref = O.Reference()
    d = np.load(os.path.join(OUT, "digits.npz"))
    imgs = T.fixture_images((d["images"], d["labels"]))
    out = {}
    for name in model_names():
        _, _, taps = T.chain_taps(ref, load_model(name), imgs)
        out.update({f"{name}/tap{t}": tap for t, tap in enumerate(taps)})
    np.savez_compressed(os.path.join(OUT, "reference_taps.npz"), **out)


if __name__ == "__main__":
    main()
