"""Activation taps on FC 4bitsym-64 (tests/golden/models/fc.bnm) at batch 2^20, one GPU, one run: plain fused launches, fused launches
that also store every tap, and the layer-by-layer path with every tap.  Device events around `--steps` launches after `--warmup`; the
images alternate between two 256 MB buffers (twice the L2), so every launch reads them from HBM.

Algorithmic bytes per image: 256 image + 40 logits = 296 plain; + 3 hidden rows x 64 = 488 with taps (labels are not requested).  The
share of the HBM roofline uses the measured copy bandwidth of profiles/README.md (6 592.9 GB/s).  Prints one JSON object (and writes
it to --out) with the card's name and power limit next to the numbers."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bitnetmcu_b200 import _lib  # noqa: E402
from bitnetmcu_b200.engine import Engine  # noqa: E402
from bitnetmcu_b200.model import Model  # noqa: E402

HBM_GBS = 6592.9
BYTES_PLAIN, BYTES_TAPS = 256 + 40, 256 + 40 + 3 * 64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "unavailable"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n = a.batch
    dev = torch.device("cuda", 0)
    model = Model.load(os.path.join(ROOT, "tests", "golden", "models", "fc.bnm"))
    fused = Engine(model, path=_lib.PATH_TCGEN05)
    layered = Engine(model, path=_lib.PATH_LAYERS)
    g = torch.Generator(device=dev).manual_seed(0)
    x = [torch.randint(-128, 128, (n, 256), dtype=torch.int8, device=dev, generator=g) for _ in range(2)]
    lo = torch.empty((n, 10), dtype=torch.int32, device=dev)
    taps = [torch.empty((n, s), dtype=torch.int8, device=dev) for _, s in fused.tap_shapes()]
    taps2 = [torch.empty_like(t) for t in taps]
    lo2 = torch.empty_like(lo)

    def timed(fn):
        for i in range(a.warmup):
            fn(i)
        torch.cuda.synchronize(dev)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(a.steps):
            fn(i)
        t1.record()
        torch.cuda.synchronize(dev)
        return t0.elapsed_time(t1) / a.steps * 1e3   # us per launch

    legs = {
        "fused_plain": (lambda i: fused.infer_device(x[i & 1], lo), BYTES_PLAIN),
        "fused_taps": (lambda i: fused.infer_device_taps(x[i & 1], lo, None, taps), BYTES_TAPS),
        "layered_taps": (lambda i: layered.infer_device_taps(x[i & 1], lo2, None, taps2), BYTES_TAPS),
    }
    out = {"model": "fc (4bitsym 256-64-64-64-10)", "batch": n, "steps": a.steps, "warmup": a.warmup, "card": card(),
           "hbm_gbs_denominator": HBM_GBS}
    for name, (fn, bpi) in legs.items():
        us = timed(fn)
        out[name] = {"us_per_launch": round(us, 2), "images_per_s": round(n / us * 1e6), "bytes_per_image": bpi,
                     "hbm_fraction": round(bpi * n / us / 1e3 / HBM_GBS, 4)}
    # the three legs computed the same thing on the last buffer they saw
    fused.infer_device(x[(a.steps - 1) & 1], lo)
    fused.infer_device_taps(x[(a.steps - 1) & 1], lo2, None, taps)
    torch.cuda.synchronize(dev)
    out["fused_taps_equal_layered_taps"] = all(torch.equal(p[:, :64], q[:, :64]) for p, q in zip(taps, taps2))
    out["fused_taps_logits_equal_plain"] = bool(torch.equal(lo, lo2))
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
