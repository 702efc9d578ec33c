"""Activation taps (include/bitnetmcu_b200.h section 7): every hidden layer's int8 row out of the engine, bit-exact with the rows the
reference's BitMnistInference leaves in layer_in after each ReLUNorm (BitNetMCU_MNIST_dll.c:80,102-109).

The checker is ``chain_taps``: BitMnistInference restated one image at a time over the four single-item kernels of the oracle (or of
the unmodified reference, which tests/golden/make_reference_taps.py records into reference_taps.npz)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_model, model_names, xorshift_images

TAPS_NPZ = os.path.join(GOLDEN, "reference_taps.npz")

# (width, stride) of every tap for a few fixture models: the header's definition written out
EXPECTED_SHAPES = {
    "fc": [(64, 64)] * 3,
    "1k": [(16, 32)] * 2,
    "ternary64": [(64, 96)] * 3,
    "cnn": [(256, 256), (96, 96), (64, 64)],
    "cnn_16small": [(64, 64), (64, 64), (48, 64)],
}


def chain_taps(kern, model, images):
    """BitMnistInference (dll.c:48-121) image by image through ``kern``'s processconv33ReLU / processmaxpool22 / processfclayer /
    ReLUNorm -> (logits int32 [n, n_classes], labels uint32 [n], [int8 [n, width] per tap]): the rows layer_in holds after each
    tap-producing ReLUNorm."""
    from bitnetmcu_b200 import model as M
    imgs = np.ascontiguousarray(images, dtype=np.int8).reshape(-1, model.img_bytes)
    n = imgs.shape[0]
    fc = model.fc_layers
    cnn = model.model_class == M.MODEL_CNNMNIST
    t0 = 1 if cnn else 0
    taps = [np.zeros((n, w), dtype=np.int8) for w, _ in model.tap_shapes()]
    logits = np.zeros((n, model.n_classes), dtype=np.int32)
    labels = np.zeros(n, dtype=np.uint32)
    front = [l for l in model.layers if l.kind != M.LAYER_FC]   # conv, conv, pool, conv, pool (dll.c:64-77)
    for i in range(n):
        act = imgs[i]
        if cnn:
            pooled = []
            for c in range(model.channels):
                x = imgs[i].astype(np.int32)
                for l in front:
                    if l.kind == M.LAYER_CONV33:
                        x = kern.conv33relu(x, np.asarray(l.weights).reshape(-1, 9)[c], l.n_in, 4)
                    else:
                        x = kern.maxpool22(x, l.n_in)
                pooled.append(x)
            act, _ = kern.relunorm(np.concatenate(pooled))   # dll.c:80
            taps[0][i] = act
        for l, L in enumerate(fc):
            a = np.zeros(max(L.n_in, act.size), dtype=np.int8)   # ternary n_in is padded with zero trits: those bytes are never used
            a[:act.size] = act
            out = kern.fclayer(a, L.weights, L.bitperweight, L.n_in, L.n_out)
            act, pos = kern.relunorm(out)
            if l + 1 < len(fc):
                taps[t0 + l][i] = act
        logits[i], labels[i] = out, pos
    return logits, labels, taps


def fixture_images(digits):
    """The 10 reference digits, then the 256 xorshift32 images golden.npz uses."""
    return np.concatenate([digits[0], xorshift_images(256)])


@pytest.fixture(scope="module")
def reference_taps():
    return dict(np.load(TAPS_NPZ))


@pytest.fixture(scope="module")
def oracle_taps(oracle, digits):
    """chain_taps over the oracle's kernels, per fixture model, on fixture_images (computed once per module)."""
    imgs = fixture_images(digits)
    return {name: chain_taps(oracle, load_model(name), imgs) for name in model_names()}


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_fixture_covers_every_model(reference_taps):
    for name in model_names():
        shapes = load_model(name).tap_shapes()
        for t, (w, _) in enumerate(shapes):
            assert reference_taps[f"{name}/tap{t}"].shape == (266, w)
        assert f"{name}/tap{len(shapes)}" not in reference_taps


@pytest.mark.parametrize("name", model_names())
def test_oracle_taps_equal_reference(oracle_taps, reference_taps, name):
    logits, labels, taps = oracle_taps[name]
    for t, tap in enumerate(taps):
        assert np.array_equal(tap, reference_taps[f"{name}/tap{t}"]), (name, t)


@pytest.mark.parametrize("name", model_names())
def test_chain_logits_equal_oracle_inference(oracle, oracle_taps, digits, name):
    logits, labels, _ = oracle_taps[name]
    want_lo, want_la = oracle.infer(load_model(name), fixture_images(digits))
    assert np.array_equal(logits, want_lo)
    assert np.array_equal(labels, want_la)


def test_model_tap_shapes():
    for name, want in EXPECTED_SHAPES.items():
        assert load_model(name).tap_shapes() == want, name
    for name in model_names():
        m = load_model(name)
        shapes = m.tap_shapes()
        assert len(shapes) == len(m.fc_layers) - 1 + (1 if m.model_class == 1 else 0)
        assert all(w <= s and s % 16 == 0 for w, s in shapes)


def _write_test_data_header(path, images, labels):
    with open(path, "w") as f:
        for i in range(images.shape[0]):
            f.write(f"int8_t input_data_{i}[256] = {{" + ", ".join(str(int(v)) for v in images[i]) + "};\n")
            f.write(f"uint8_t label_{i} = {int(labels[i])};\n")


def _build_activations(tmp, name):
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.pack import write_header
    write_header(load_model(name), os.path.join(tmp, "BitNetMCU_model.h"))
    d = np.load(os.path.join(GOLDEN, "digits.npz"))
    _write_test_data_header(os.path.join(tmp, "BitNetMCU_MNIST_test_data.h"), d["images"], d["labels"])
    libdir = os.path.dirname(_lib.LIB_PATH)
    common = ["-I" + tmp, "-I" + os.path.join(ROOT, "include"), "-L" + libdir, "-lbitnetmcu_b200", "-Wl,-rpath," + libdir]
    dll = os.path.join(tmp, "Bitnet_inf.dll")
    exe = os.path.join(tmp, "activations")
    subprocess.run(["gcc", "-Wall", "-Werror", "-fPIC", "-shared", "-D_DLL", "-o", dll, os.path.join(ROOT, "host", "bitnetmcu_b200_dll.c")] + common,
                   check=True)
    subprocess.run(["gcc", "-Wall", "-Werror", "-o", exe, os.path.join(ROOT, "host", "bitnetmcu_b200_activations.c"), dll,
                    "-Wl,-rpath," + tmp] + common, check=True)
    return dll, exe, d


@pytest.mark.parametrize("name", ["fc", "cnn"])
def test_shim_exports_printactivations_and_program_compiles(built, tmp_path, name):
    dll, _, _ = _build_activations(str(tmp_path), name)
    out = subprocess.run(["nm", "-D", "--defined-only", dll], capture_output=True, text=True, check=True).stdout
    assert " T printactivations" in out


def test_printactivations_format(built, tmp_path):
    """printactivations is plain C with no device work: "%d, " per value, a newline after every 16."""
    dll, _, _ = _build_activations(str(tmp_path), "fc")
    vals = np.arange(-3, 37, dtype=np.int8).astype(np.uint8)
    prog = tmp_path / "p.py"
    prog.write_text(
        "import ctypes as C, numpy as np, sys\n"
        f"lib = C.CDLL({dll!r})\n"
        f"v = np.array({vals.tolist()}, dtype=np.uint8)\n"
        "lib.printactivations(C.c_void_p(v.ctypes.data), C.c_int32(v.size))\n")
    out = subprocess.run(["python", str(prog)], capture_output=True, text=True, check=True).stdout
    assert out == render_activations(vals)   # uint8, as the reference declares the row


def render_activations(row):
    """What printactivations prints for one row."""
    s = ""
    for j, v in enumerate(row):
        s += f"{int(v)}, "
        if (j + 1) % 16 == 0:
            s += "\n"
    return s


# ---------------------------------------------------------------------------------------------------------------- GPU
def _device_taps(eng, imgs, taps_wanted=None, sentinel=0x5A, extra_rows=3):
    """bnm_infer_batch_device_taps on torch buffers -> (logits, labels, [int8 [n, stride] or None per tap]) on the host; tap buffers
    have extra_rows rows past n, filled with sentinel and checked untouched."""
    import torch
    n = imgs.shape[0]
    dev = torch.device("cuda", eng.device)
    x = torch.from_numpy(np.ascontiguousarray(imgs)).to(dev)
    lo = torch.empty((n, eng.n_classes), dtype=torch.int32, device=dev)
    la = torch.empty(n, dtype=torch.int32, device=dev)
    shapes = eng.tap_shapes()
    wanted = range(len(shapes)) if taps_wanted is None else taps_wanted
    full = [torch.full((n + extra_rows, s), sentinel, dtype=torch.int8, device=dev) if t in wanted else None for t, (_, s) in enumerate(shapes)]
    eng.infer_device_taps(x, lo, la, [b[:n] if b is not None else None for b in full])
    torch.cuda.synchronize(dev)
    out = []
    for b in full:
        if b is None:
            out.append(None)
            continue
        h = b.cpu().numpy()
        assert (h[n:] == sentinel).all(), "rows at or beyond n were written"
        out.append(h[:n])
    return lo.cpu().numpy(), la.cpu().numpy().astype(np.uint32), out


def _check(eng, imgs, want_taps, plain=None):
    lo, la, taps = _device_taps(eng, imgs)
    p_lo, p_la = plain if plain is not None else eng.infer(imgs)
    assert np.array_equal(lo, p_lo) and np.array_equal(la, p_la), "logits / labels differ from the plain call"
    for t, ((w, _), tap) in enumerate(zip(eng.tap_shapes(), taps)):
        assert np.array_equal(tap[:, :w], want_taps[t]), (t, np.argwhere(tap[:, :w] != want_taps[t])[:4])
    return lo, la, taps


@pytest.mark.gpu
@pytest.mark.parametrize("name", model_names())
def test_taps_all_fixture_models(built, oracle_taps, reference_taps, digits, name):
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    m = load_model(name)
    imgs = fixture_images(digits)
    want_lo, want_la, want = oracle_taps[name]
    for t, w in enumerate(want):
        assert np.array_equal(w, reference_taps[f"{name}/tap{t}"])
    frontends = [_lib.CNN_CUDA_CORES, _lib.CNN_TENSOR_CORES] if m.model_class == 1 else [None]
    for path in (_lib.PATH_TCGEN05, _lib.PATH_LAYERS):
        for fe in frontends:
            e = Engine(m, path=path)
            if fe == _lib.CNN_TENSOR_CORES and m.channels % 16:
                e.close()
                continue
            if fe is not None:
                e.set_option(_lib.OPT_CNN_FRONTEND, fe)
            assert e.tap_shapes() == m.tap_shapes()
            assert e.n_taps == len(m.tap_shapes())
            _check(e, imgs, want, plain=(want_lo, want_la))
            lo, la, taps = e.infer_taps(imgs)   # host entry
            assert np.array_equal(lo, want_lo) and np.array_equal(la, want_la)
            assert all(np.array_equal(a, b) for a, b in zip(taps, want)), (name, path, fe)
            e.close()


# the fused kernel's forms: kSmemA, kFourWG, the +128 residual plane, stride > round_up(width, 32), kManyClasses
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["binary160", "2bitsym96", "rand_fp130_64", "ternary64", "cnn_letters", "fc"])
@pytest.mark.parametrize("n", [1, 127, 128, 129, 148 * 128 + 1, 2 ** 16 + 37])
def test_taps_forms_and_batch_sizes(built, oracle, name, n):
    """Ragged and multi-tile batches: fused taps equal the layered path's (itself pinned to the oracle above) and, on a sample of
    rows, the oracle's chain; rows at or beyond n are never written."""
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    m = load_model(name)
    imgs = np.random.default_rng(n).integers(-128, 128, size=(n, 256)).astype(np.int8)
    want_lo, want_la = oracle.infer(m, imgs)
    lay = Engine(m, path=_lib.PATH_LAYERS)
    l_lo, l_la, l_taps = _device_taps(lay, imgs)
    lay.close()
    assert np.array_equal(l_lo, want_lo) and np.array_equal(l_la, want_la)
    sample = np.unique(np.r_[0, n - 1, np.arange(0, n, max(1, n // 24))])
    _, _, c_taps = chain_taps(oracle, m, imgs[sample])
    for t, (w, _) in enumerate(m.tap_shapes()):
        assert np.array_equal(l_taps[t][sample, :w], c_taps[t])
    fused = Engine(m, path=_lib.PATH_TCGEN05)
    _check(fused, imgs, [tap[:, :w] for tap, (w, _) in zip(l_taps, m.tap_shapes())], plain=(want_lo, want_la))
    fused.close()


_ODD_CHAINS = [(4, (256, 96, 64, 37)), (4, (256, 160, 160, 17)), (12, (256, 48, 250)), (16, (256, 16, 16, 10)), (20, (64, 224, 32, 20)),
               (4, (256, 64, 64, 64, 64, 64, 64, 64, 10)), (20, (256, 160, 144, 10)), (64, (128, 176, 176, 176, 7)), (2, (256, 96, 96, 10)),
               (64, (256, 48, 40, 10))]


@pytest.mark.gpu
@pytest.mark.parametrize("enc,widths", _ODD_CHAINS)
def test_taps_odd_width_chains(built, oracle, enc, widths):
    """16-column tails, widths that are not multiples of 32, the 8-layer maximum, > 16 classes."""
    from bitnetmcu_b200 import _lib, pack as P
    from bitnetmcu_b200.engine import Engine
    m = P.random_fc_model(enc, widths, seed=enc + sum(widths))
    m.img_bytes = widths[0]
    imgs = np.random.default_rng(sum(widths)).integers(-128, 128, size=(3 * 128 + 29, widths[0])).astype(np.int8)
    want_lo, want_la, want = chain_taps(oracle, m, imgs)
    for path in (_lib.PATH_TCGEN05, _lib.PATH_LAYERS):
        e = Engine(m, path=path)
        assert e.tap_shapes() == m.tap_shapes()
        _check(e, imgs, want, plain=(want_lo, want_la))
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fc", "cnn", "binary160"])
def test_taps_subsets(built, oracle_taps, digits, name):
    """Each tap alone, and none: the other buffers stay untouched, logits and labels stay those of the plain call."""
    from bitnetmcu_b200.engine import Engine
    m = load_model(name)
    imgs = fixture_images(digits)
    want_lo, want_la, want = oracle_taps[name]
    e = Engine(m)
    for subset in [[t] for t in range(e.n_taps)] + [[]]:
        lo, la, taps = _device_taps(e, imgs, taps_wanted=subset)
        assert np.array_equal(lo, want_lo) and np.array_equal(la, want_la), subset
        for t, tap in enumerate(taps):
            if t in subset:
                assert np.array_equal(tap[:, :want[t].shape[1]], want[t]), (subset, t)
            else:
                assert tap is None
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fc", "cnn"])
def test_host_entry_crosses_chunks(built, name):
    """bnm_infer_batch_taps with 128-image chunks equals the device entry."""
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    m = load_model(name)
    imgs = np.random.default_rng(7).integers(-128, 128, size=(1000 + 5, 256)).astype(np.int8)
    e = Engine(m)
    d_lo, d_la, d_taps = _device_taps(e, imgs)
    e.set_option(_lib.OPT_CHUNK_IMAGES, 128)
    lo, la, taps = e.infer_taps(imgs)
    assert np.array_equal(lo, d_lo) and np.array_equal(la, d_la)
    for t, (w, _) in enumerate(e.tap_shapes()):
        assert np.array_equal(taps[t], d_taps[t][:, :w])
    e.close()


@pytest.mark.gpu
def test_taps_between_independent_launches(built, oracle):
    """Mode 2 (independent launches), then a taps call, then mode 2 again, all on one stream: all three results are right (the taps
    launch is a plain launch and the launch after it keeps its grid-dependency wait)."""
    import torch
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    m = load_model("fc")
    e = Engine(m)
    e.set_option(_lib.OPT_LAUNCH_OVERLAP, 2)
    dev = torch.device("cuda", 0)
    n = 148 * 128 * 2 + 3
    rng = np.random.default_rng(3)
    h = [rng.integers(-128, 128, size=(n, 256)).astype(np.int8) for _ in range(3)]
    x = [torch.from_numpy(a).to(dev) for a in h]
    lo = [torch.empty((n, 10), dtype=torch.int32, device=dev) for _ in range(3)]
    la = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3)]
    taps = [torch.empty((n, s), dtype=torch.int8, device=dev) for _, s in e.tap_shapes()]
    torch.cuda.synchronize(dev)
    e.infer_device(x[0], lo[0], la[0])
    e.infer_device_taps(x[1], lo[1], la[1], taps)
    e.infer_device(x[2], lo[2], la[2])
    torch.cuda.synchronize(dev)
    for k in range(3):
        want_lo, want_la = oracle.infer(m, h[k])
        assert np.array_equal(lo[k].cpu().numpy(), want_lo), k
        assert np.array_equal(la[k].cpu().numpy().astype(np.uint32), want_la), k
    sample = np.arange(0, n, 997)
    _, _, want = chain_taps(oracle, m, h[1][sample])
    for t, (w, _) in enumerate(e.tap_shapes()):
        assert np.array_equal(taps[t].cpu().numpy()[sample, :w], want[t])
    e.close()


@pytest.mark.gpu
def test_taps_rejections(built):
    """Float input has no taps; a tap the model does not have and a misaligned buffer are argument errors."""
    import torch
    from bitnetmcu_b200 import _lib
    from bitnetmcu_b200.engine import Engine
    e = Engine(load_model("fc"))
    dev = torch.device("cuda", 0)
    n = 4
    lo = torch.empty((n, 10), dtype=torch.int32, device=dev)
    taps = [torch.empty((n, s), dtype=torch.int8, device=dev) for _, s in e.tap_shapes()]
    with pytest.raises(_lib.BnmError, match="float input has no taps"):
        e.infer_device_taps(torch.zeros((n, 256), dtype=torch.float32, device=dev), lo, None, taps)
    x = torch.zeros((n, 256), dtype=torch.int8, device=dev)
    lib = _lib.load()
    tt = _lib.BnmTaps()
    tt.act[e.n_taps] = taps[0].data_ptr()
    assert lib.bnm_infer_batch_device_taps(e.handle, C.c_void_p(x.data_ptr()), n, C.c_void_p(lo.data_ptr()), None, C.byref(tt), None) == -1
    tt = _lib.BnmTaps()
    tt.act[0] = taps[0].data_ptr() + 8
    assert lib.bnm_infer_batch_device_taps(e.handle, C.c_void_p(x.data_ptr()), n, C.c_void_p(lo.data_ptr()), None, C.byref(tt), None) == -1
    assert lib.bnm_model_tap_width(e.handle, e.n_taps) == 0 and lib.bnm_model_tap_stride(e.handle, e.n_taps) == 0
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fc", "cnn"])
def test_activations_program_stdout(built, tmp_path, reference_taps, name):
    """host/bitnetmcu_b200_activations.c prints, per digit, what the reference's commented printactivations lines would print."""
    _, exe, d = _build_activations(str(tmp_path), name)
    out = subprocess.run([exe], capture_output=True, text=True, check=True, timeout=120).stdout
    m = load_model(name)
    want = ""
    for i in range(10):
        for t in range(len(m.tap_shapes())):
            want += f"L{t + 1} activations:  \n" + render_activations(reference_taps[f"{name}/tap{t}"][i])
        want += f"label: {int(d['labels'][i])} predicted: {int(d['labels'][i])}\n"
    assert out == want
