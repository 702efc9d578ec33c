# compute-sanitizer target (memcheck, racecheck): one ragged taps launch (148 x 128 + 77 images) per form of the fused kernel and of
# the layered path, checked against each other.  Run: compute-sanitizer --tool memcheck python tools/taps_sanitize.py  (from the repository root)
import os, sys, numpy as np, torch
sys.path.insert(0, os.getcwd())
from bitnetmcu_b200 import _lib
from bitnetmcu_b200.engine import Engine
from bitnetmcu_b200.model import Model
n = 148 * 128 + 77
x = torch.from_numpy(np.random.default_rng(1).integers(-128, 128, size=(n, 256)).astype(np.int8)).cuda()
for name in ("fc", "2bitsym96", "binary160", "cnn_letters", "ternary64", "cnn"):
    res = []
    for path in (_lib.PATH_TCGEN05, _lib.PATH_LAYERS):
        e = Engine(Model.load(f"tests/golden/models/{name}.bnm"), path=path)
        lo = torch.empty((n, e.n_classes), dtype=torch.int32, device="cuda")
        la = torch.empty(n, dtype=torch.int32, device="cuda")
        taps = [torch.zeros((n, s), dtype=torch.int8, device="cuda") for _, s in e.tap_shapes()]
        e.infer_device_taps(x, lo, la, taps)
        torch.cuda.synchronize()
        res.append((lo.cpu(), la.cpu(), [t[:, :w].cpu() for t, (w, _) in zip(taps, e.tap_shapes())]))
        e.close()
    ok = torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]) and all(torch.equal(a, b) for a, b in zip(res[0][2], res[1][2]))
    print(name, "fused == layered:", ok)
    assert ok
