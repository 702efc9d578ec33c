#!/usr/bin/env python
"""Record what the original BitNetMCU project computes, for the tests that compare against it.  Needs a checkout of that
project (REF, also read by oracle/Makefile, which builds its unmodified kernels into oracle/_ref):

    REF=<BitNetMCU checkout> python tests/golden/make_reference_vectors.py

What it writes (small, committed, read by the tests wherever they run):

  reference_vectors.npz   outputs of the unmodified reference kernels on the seeded inputs of tests/test_oracle_golden.py
                          (its *_cases / whole_model_images generators): processfclayer per encoding and shape, ReLUNorm,
                          processconv33ReLU / processmaxpool22, and whole-model inference -- labels of every image, logits of the
                          first LOGITS_HEAD images and the CRC-32 of all logits
  shipped_headers.json    per shipped model header: the fixture under models/ that holds it and what the header parser reads
                          from it (tests/test_packer_header.py header_fingerprint)
"""
import glob
import json
import os
import sys

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(OUT))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
REF = os.environ["REF"]

import test_oracle_golden as T  # noqa: E402
import test_packer_header as TP  # noqa: E402
from conftest import load_model, model_names  # noqa: E402
from bitnetmcu_b200 import model as M  # noqa: E402
from oracle import oracle as O  # noqa: E402


def reference_vectors(ref):
    out = {}
    for enc in T.FCLAYER_ENCODINGS:
        for n_in, n_out, act, w in T.fclayer_cases(enc):
            out[f"fclayer/{enc}/{n_in}x{n_out}"] = ref.fclayer(act, w, enc, n_in, n_out)
    outs, pos = zip(*(ref.relunorm(x) for x in T.relunorm_cases()))
    out["relunorm/out"], out["relunorm/pos"] = np.concatenate(outs), np.array(pos, dtype=np.int32)
    conv, pool = {}, {}
    for xy, act, w in T.conv_pool_cases():
        conv.setdefault(xy, []).append(ref.conv33relu(act, w, xy, 4))
        if xy % 2 == 0:
            pool.setdefault(xy, []).append(ref.maxpool22(act, xy))
    out.update({f"conv/{xy}": np.stack(v) for xy, v in conv.items()})
    out.update({f"pool/{xy}": np.stack(v) for xy, v in pool.items()})
    for name in T.WHOLE_MODELS:
        m = load_model(name)
        lo, la = ref.infer(m, T.whole_model_images(m))
        out[f"model/{name}/logits_head"] = lo[:T.LOGITS_HEAD]
        out[f"model/{name}/logits_crc32"] = np.uint32(T.logits_crc32(lo))
        out[f"model/{name}/labels"] = la.astype(np.uint8)
    return out


def shipped_headers():
    """Every shipped model header, matched to the fixture model its parse equals (the one named after it, when several do)."""
    fixtures = {name: TP.header_fingerprint(load_model(name)) for name in model_names()}
    heads = [os.path.join(REF, "BitNetMCU_model_fc.h"), os.path.join(REF, "BitNetMCU_model_cnn.h")] + \
        sorted(glob.glob(os.path.join(REF, "mcu", "BitNetMCU_model_*.h")))
    out = {}
    for h in heads:
        parsed = TP.header_fingerprint(M.parse_header(h))
        same = [name for name, fp in sorted(fixtures.items()) if fp == parsed]
        own = os.path.basename(h)[len("BitNetMCU_model_"):-len(".h")]
        out[os.path.relpath(h, REF)] = {"fixture": own if own in same else same[0], "parsed": parsed}
    return out


def main():
    O.build(quiet=True)
    np.savez_compressed(os.path.join(OUT, "reference_vectors.npz"), **reference_vectors(O.Reference()))
    with open(os.path.join(OUT, "shipped_headers.json"), "w") as f:   # one header per line
        f.write("{\n" + ",\n".join(f" {json.dumps(h)}: {json.dumps(v)}" for h, v in shipped_headers().items()) + "\n}\n")


if __name__ == "__main__":
    main()
