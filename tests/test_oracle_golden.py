"""Pin the oracle (oracle/bitnet_oracle.c) against the reference: golden vectors made by the unmodified
reference kernels (tests/golden/make_golden.py), the reference's own label KAT, exhaustive decode sweeps, and
random function-level comparisons against the reference's outputs stored by tests/golden/make_reference_vectors.py."""
import json
import os
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, load_model, model_names, xorshift_images
from bitnetmcu_b200 import model as M
from bitnetmcu_b200 import pack as P


@pytest.mark.parametrize("name", model_names())
def test_oracle_matches_golden_logits(oracle, golden, digits, name):
    m = load_model(name)
    imgs, _ = digits
    lo, la = oracle.infer(m, imgs, threads=1)
    assert np.array_equal(lo, golden[name + "/digits_logits"])
    assert np.array_equal(la, golden[name + "/digits_labels"])
    xs = oracle.xorshift_images(256)
    lo, la = oracle.infer(m, xs, threads=2)
    assert np.array_equal(lo, golden[name + "/xs_logits"])
    assert np.array_equal(la, golden[name + "/xs_labels"])


def test_reference_label_kat(oracle, digits):
    """BitNetMCU_MNIST_test.c:17-40: predicted == label for both shipped models (config #1)."""
    imgs, labels = digits
    kat = json.load(open(os.path.join(GOLDEN, "kat.json")))
    assert kat["reference_labels"] == labels.tolist() == kat["dll_fc_labels"] == kat["dll_cnn_labels"]
    for name in ("fc", "cnn", "12k", "12k_FP130", "1k", "cnn_48", "cnn_32", "cnn_16", "binary160"):
        _, la = oracle.infer(load_model(name), imgs)
        assert la.tolist() == labels.tolist(), name


def test_survey_kats(oracle):
    """SURVEY.md 8c synthetic KAT: CRC-32 of the first 1000x10 logits, label sums."""
    kat = json.load(open(os.path.join(GOLDEN, "kat.json")))
    xs = oracle.xorshift_images(1000)
    assert xs[0, :8].tolist() == kat["xorshift_first_pixels"] == [122, -81, -96, -22, -45, 98, -104, 56]
    assert np.array_equal(xs[:4], xorshift_images(4))
    lo, la = oracle.infer(load_model("fc"), xs)
    assert lo[0].tolist() == kat["fc_xs_logits0"]
    assert "%08x" % zlib.crc32(lo.astype("<i4").tobytes()) == kat["fc_xs_crc32_first1000"] == "fc621bad"
    assert int(la.sum()) == kat["fc_xs_sum_labels_1000"] == 4064
    xs = oracle.xorshift_images(40000)
    _, la = oracle.infer(load_model("cnn"), xs)
    assert int(la.sum()) == kat["cnn_xs_sum_labels_40000"] == 303886


def test_relunorm_probed_vectors(oracle):
    """SURVEY.md 8a row a2, probed against the reference."""
    cases = [([127, 128, 255, 256, -3], [32, 32, 64, 64, 0], 3), ([255, 254, 253, 127, 1], [127, 127, 127, 64, 1], 0),
             ([1000, 509, 510, -1, 1], [125, 64, 64, 0, 0], 0), ([-5, -1, -7], [0, 0, 0], 1), ([5, 9, 9, 2], None, 1),
             ([], [], 255)]
    for x, want, pos in cases:
        out, p = oracle.relunorm(np.array(x, dtype=np.int32))
        assert p == pos
        if want is not None:
            assert out.tolist() == want


def test_decode_tables(oracle):
    """nibble/code -> weight tables of SURVEY.md 8a, through the packed-word decoder."""
    for enc, want in [(M.ENC_4BITSYM, [1, 3, 5, 7, 9, 11, 13, 15, -1, -3, -5, -7, -9, -11, -13, -15]),
                      (M.ENC_4BIT, [0, 1, 2, 3, 4, 5, 6, 7, -8, -7, -6, -5, -4, -3, -2, -1]),
                      (M.ENC_FP130, [1, 2, 4, 8, 16, 32, 64, 128, -1, -2, -4, -8, -16, -32, -64, -128])]:
        codes = np.arange(16, dtype=np.uint32).reshape(1, 16)
        dense = oracle.decode_fc(P.pack_codes(codes, 4), enc, 16, 1)
        assert dense[0].tolist() == want
        assert P.INT_LUT[enc].tolist() == want
    dense = oracle.decode_fc(P.pack_codes(np.tile(np.arange(4, dtype=np.uint32), 4).reshape(1, 16), 2), M.ENC_2BITSYM, 16, 1)
    assert dense[0, :4].tolist() == [1, 3, -1, -3]
    dense = oracle.decode_fc(np.array([0x80000001], dtype=np.uint32), M.ENC_BINARY, 32, 1)
    assert dense[0, 0] == 1 and dense[0, 1] == -1 and dense[0, 31] == 1
    dense = oracle.decode_fc(np.array([0x7F80FF01], dtype=np.uint32), M.ENC_8BIT, 4, 1)
    assert dense[0].tolist() == [127, -128, -1, 1]
    # NF4: zeros in the reference (inference.c:202); LUT only as the documented extension
    w = P.pack_codes(np.arange(16, dtype=np.uint32).reshape(1, 16), 4)
    assert not oracle.decode_fc(w, M.ENC_NF4, 16, 1).any()
    assert oracle.decode_fc(w, M.ENC_NF4, 16, 1, nf4_extension=True)[0].tolist() == P.NF4_INT_LUT.tolist()


def test_ternary_all_words(oracle):
    """Every one of the 65536 raw uint16 words decodes deterministically (0xFFFF -> all 0, 0x0000 -> all +1),
    and all 59049 trit codes round-trip through pack -> decode (SURVEY.md 8c)."""
    words = np.arange(65536, dtype=np.uint16)
    dense = oracle.decode_fc(words, M.ENC_TERNARY, 10, 65536)
    assert np.array_equal(dense, P.unpack_ternary(words, 65536, 10))
    assert not dense[0xFFFF].any() and (dense[0] == 1).all()
    idx = np.arange(59049)
    trits = np.stack([(idx // 3 ** (9 - j)) % 3 for j in range(10)], axis=1) - 1
    packed, n_in = P.pack_ternary(trits)
    assert n_in == 10
    assert np.array_equal(oracle.decode_fc(packed, M.ENC_TERNARY, 10, 59049), trits)


# ---- comparisons with the unmodified reference kernels: their outputs on these seeded inputs are stored in
# golden/reference_vectors.npz (written by golden/make_reference_vectors.py, which calls the same *_cases generators) ---

FCLAYER_ENCODINGS = [1, 2, 4, 12, 16, 20, 36, 64, 3]
WHOLE_MODELS = ["fc", "cnn", "cnn_48", "binary160", "ternary64", "rand_fp130_64", "rand_nf4_64", "1k"]
LOGITS_HEAD = 80   # rows stored in full per model: the MNIST-like, all -128, all 127 and all-zero images


def fclayer_cases(enc):
    """(n_in, n_out, activations, weights) of one fully connected layer per shape."""
    rng = np.random.default_rng(enc)
    for n_in, n_out in [(256, 64), (64, 10), (160, 160), (320, 7)]:
        if enc == 64:
            n_in = (n_in + 9) // 10 * 10
            w = rng.integers(0, 65536, size=n_out * n_in // 10, dtype=np.uint32).astype(np.uint16)
        else:
            w = rng.integers(0, 2 ** 32, size=n_out * n_in // 4 + 4, dtype=np.uint64).astype(np.uint32)
        act = rng.integers(-128, 128, size=n_in + 16).astype(np.int8)
        yield n_in, n_out, act, w


def relunorm_cases():
    rng = np.random.default_rng(7)
    for trial in range(300):
        n = int(rng.integers(1, 300))
        scale = int(rng.choice([1, 100, 20000, 500000, 4000000]))
        x = rng.integers(-scale, scale + 1, size=n).astype(np.int32)
        if trial % 7 == 0:
            x = -np.abs(x) - 1
        if trial % 11 == 0:
            x[rng.integers(0, n)] = 2 ** (7 + trial % 20) - 1
        yield x


def conv_pool_cases():
    """(xy, activations, 3x3 weights), twenty per image size."""
    rng = np.random.default_rng(9)
    for xy in (16, 14, 6, 4, 3):
        for _ in range(20):
            act = rng.integers(-20000, 20000, size=xy * xy).astype(np.int32)
            w = rng.integers(-128, 128, size=9).astype(np.int8)
            yield xy, act, w


def whole_model_images(m):
    rng = np.random.default_rng(11)
    n = 3000 if m.model_class == M.MODEL_FCMNIST else 600
    imgs = rng.integers(-128, 128, size=(n, 256)).astype(np.int8)
    imgs[:50] = np.clip(imgs[:50], -20, 127)          # MNIST-like background
    imgs[50:60] = -128
    imgs[60:70] = 127
    imgs[70:80] = 0
    return imgs


def logits_crc32(logits):
    return zlib.crc32(np.ascontiguousarray(logits, dtype="<i4").tobytes())


@pytest.mark.parametrize("enc", FCLAYER_ENCODINGS)
def test_fclayer_vs_reference(oracle, reference_vectors, enc):
    for n_in, n_out, act, w in fclayer_cases(enc):
        want = reference_vectors[f"fclayer/{enc}/{n_in}x{n_out}"]
        assert np.array_equal(oracle.fclayer(act, w, enc, n_in, n_out), want), (n_in, n_out)


def test_relunorm_vs_reference(oracle, reference_vectors):
    want_out, want_pos = reference_vectors["relunorm/out"], reference_vectors["relunorm/pos"]
    at = 0
    for trial, x in enumerate(relunorm_cases()):
        a, pa = oracle.relunorm(x)
        assert pa == want_pos[trial] and np.array_equal(a, want_out[at:at + x.size]), trial
        at += x.size
    assert at == want_out.size


def test_conv_pool_vs_reference(oracle, reference_vectors):
    seen = {}
    for xy, act, w in conv_pool_cases():
        k = seen[xy] = seen.get(xy, -1) + 1
        assert np.array_equal(oracle.conv33relu(act, w, xy, 4), reference_vectors[f"conv/{xy}"][k]), (xy, k)
        if xy % 2 == 0:
            assert np.array_equal(oracle.maxpool22(act, xy), reference_vectors[f"pool/{xy}"][k]), (xy, k)


@pytest.mark.parametrize("name", WHOLE_MODELS)
def test_whole_model_vs_reference_random(oracle, reference_vectors, name):
    """Labels of every image and logits of the first LOGITS_HEAD are stored; the full logits array by its CRC-32."""
    m = load_model(name)
    lo, la = oracle.infer(m, whole_model_images(m))
    assert np.array_equal(lo[:LOGITS_HEAD], reference_vectors[f"model/{name}/logits_head"])
    assert logits_crc32(lo) == int(reference_vectors[f"model/{name}/logits_crc32"])
    assert np.array_equal(la, reference_vectors[f"model/{name}/labels"])
