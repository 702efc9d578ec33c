"""Host logic either side of the path: the BitNetMCU_model.h parser, the exportquant-compatible packer, the BNM1 blob."""
import json
import os
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, load_model, model_names
from bitnetmcu_b200 import model as M
from bitnetmcu_b200 import pack as P


@pytest.mark.parametrize("enc", [M.ENC_BINARY, M.ENC_2BITSYM, M.ENC_4BITSYM, M.ENC_4BIT, M.ENC_8BIT, M.ENC_FP130, M.ENC_NF4])
def test_pack_unpack_roundtrip_and_oracle_decode(oracle, enc):
    rng = np.random.default_rng(enc)
    bits = P.CODE_BITS[enc]
    codes = rng.integers(0, 1 << bits, size=(24, 64), dtype=np.uint32)
    words = P.pack_codes(codes, bits)
    assert words.dtype == np.uint32 and words.size == 24 * 64 * bits // 32      # no interleaved zero words (exportquant.py:105,187 defect)
    assert np.array_equal(P.unpack_codes(words, bits, 24, 64), codes)
    layer = M.Layer(kind=M.LAYER_FC, name="L1", bitperweight=enc, n_in=64, n_out=24, weights=words)
    want = P.INT_LUT[enc][codes]
    assert np.array_equal(P.decode_int_weights(layer, nf4_extension=True), want)
    assert np.array_equal(oracle.decode_fc(words, enc, 64, 24, nf4_extension=True), want)
    assert np.array_equal(P.codes_from_int_weights(enc, want), codes) or enc == M.ENC_NF4  # NF4 LUT has no duplicates either
    # first weight of a row sits in the most significant bits (inference.c tests bit 31 and shifts left)
    assert (words[0] >> (32 - bits)) == codes[0, 0]


def test_encode_levels_matches_exporter_tables():
    assert P.encode_levels("Binary", np.array([[-1, 1, 1, -1]])).tolist() == [[0, 1, 1, 0]]
    assert P.encode_levels("2bitsym", np.array([[-1.5, -0.5, 0.5, 1.5]])).tolist() == [[3, 2, 0, 1]]
    lv = np.array([[-7.5, -0.5, 0.5, 7.5]])
    assert P.encode_levels("4bitsym", lv).tolist() == [[15, 8, 0, 7]]
    assert P.INT_LUT[M.ENC_4BITSYM][P.encode_levels("4bitsym", lv)].tolist() == [[-15, -1, 1, 15]]   # C sees 2|w| (SURVEY.md section 4)
    assert P.encode_levels("4bit", np.array([[-8.0, -1.0, 0.0, 7.0]])).tolist() == [[8, 15, 0, 7]]
    assert P.encode_levels("8bit", np.array([[-128.0, -1.0, 127.0]])).tolist() == [[128, 255, 127]]
    assert P.encode_levels("FP130", np.array([[1.0, 128.0, -2.0, -128.0]])).tolist() == [[0, 7, 9, 15]]
    assert P.encode_levels("NF4", np.array([[-1.0, 0.0, 1.0, 0.08]])).tolist() == [[0, 7, 15, 8]]
    for q in ("Binary", "NF4"):
        assert P.encode_levels(q, np.array([[1.0, -1.0]])).dtype == np.uint32


def test_ternary_padding_and_header_size():
    rng = np.random.default_rng(0)
    trits = rng.integers(-1, 2, size=(8, 256))
    layer = P.fc_layer_from_trits("L1", trits)
    assert layer.n_in == 260 and layer.weights.dtype == np.uint16 and layer.weights.size == 8 * 26   # padded to x10 (exportquant.py:132-137,166)
    dec = P.decode_int_weights(layer)
    assert np.array_equal(dec[:, :256], trits) and not dec[:, 256:].any()


def test_write_header_parses_back_and_keeps_results(oracle, tmp_path, digits):
    imgs, _ = digits
    for name in ("fc", "cnn_48", "ternary64", "binary160", "12k_FP130"):
        m = load_model(name)
        path = os.path.join(tmp_path, name + ".h")
        P.write_header(m, path)
        text = open(path).read()
        assert "#define MODEL_" in text and "#ifndef BITNETMCU_MODEL_H" in text
        m2 = M.parse_header(path)
        assert m2.model_class == m.model_class and len(m2.layers) == len(m.layers)
        assert np.array_equal(oracle.infer(m2, imgs)[0], oracle.infer(m, imgs)[0])


def test_parser_discovers_layers_by_scanning_names():
    """The current exporter names FC layers L3/L5/L7/L9 (module enumeration index), shipped headers L1..L4 (SURVEY section 7)."""
    text = """
    #define MODEL_FCMNIST
    #define L3_active
    #define L3_bitperweight 4
    #define L3_incoming_weights 8 // trailing comment
    #define L3_outgoing_weights 2
    const uint32_t L3_weights[] = {0x12345678, 0x9abcdef0,}; //first channel is topmost bit
    /* block comment #define L5_active */
    #define L9_active
    #define L9_bitperweight 16
    #define L9_incoming_weights 4
    #define L9_outgoing_weights 1
    const uint32_t L9_weights[] = { 0x7f80ff01 };
    """
    m = M.parse_header_text(text)
    assert [l.name for l in m.layers] == ["L3", "L9"] and m.n_classes == 1
    assert m.layers[0].weights.tolist() == [0x12345678, 0x9ABCDEF0]
    with pytest.raises(ValueError):
        M.parse_header_text("#define L1_active\n")                       # '#error No model defined'
    with pytest.raises(ValueError):
        M.parse_header_text(text.replace("0x9abcdef0,", ""))             # array shorter than the reference would read


@pytest.mark.parametrize("name", model_names())
def test_blob_roundtrip(name):
    m = load_model(name)
    m2 = M.Model.from_blob(m.to_blob())
    assert m2.model_class == m.model_class and m2.img_bytes == m.img_bytes
    for a, b in zip(m.layers, m2.layers):
        assert (a.kind, a.bitperweight, a.n_in, a.n_out) == (b.kind, b.bitperweight, b.n_in, b.n_out)
        assert (a.weights is None) == (b.weights is None)
        if a.weights is not None:
            assert a.weights.dtype == b.weights.dtype and np.array_equal(a.weights, b.weights)


def header_fingerprint(m):
    """What a header parse yields, in JSON form: class, MACs per image, and per layer its shape and the CRC-32 of its weights."""
    return {"model_class": m.model_class, "macs_per_image": m.macs_per_image,
            "layers": [[l.name, l.kind, l.bitperweight, l.n_in, l.n_out, l.in_channels, l.groups,
                        None if l.weights is None else zlib.crc32(np.ascontiguousarray(l.weights).tobytes())] for l in m.layers]}


def test_parser_on_every_shipped_reference_header(tmp_path):
    """The reference ships eleven model headers (ten distinct models: the CNN one twice) and a test-data header.
    golden/shipped_headers.json records what the parser read from each model header
    (tests/golden/make_reference_vectors.py): every fixture model is exactly that parse, and so is the parse of the header
    written for it.  The test digits, written in the test-data header's hex layout, parse back unchanged."""
    shipped = json.load(open(os.path.join(GOLDEN, "shipped_headers.json")))
    assert len(shipped) == 11
    for header, want in shipped.items():
        m = load_model(want["fixture"])
        assert header_fingerprint(m) == want["parsed"], header
        assert m.fc_layers and m.macs_per_image > 0
        path = os.path.join(tmp_path, os.path.basename(header))
        P.write_header(m, path)
        assert header_fingerprint(M.parse_header(path)) == want["parsed"], header
    d = np.load(os.path.join(GOLDEN, "digits.npz"))
    path = os.path.join(tmp_path, "BitNetMCU_MNIST_test_data.h")
    with open(path, "w") as f:
        for i, (img, label) in enumerate(zip(d["images"], d["labels"])):
            rows = [", ".join("0x%02X" % v for v in img[r:r + 16].view(np.uint8)) for r in range(0, 256, 16)]
            f.write(f"int8_t input_data_{i}[256] = {{\n" + ",\n".join(rows) + "\n};\n" + f"uint8_t label_{i} = {int(label)};\n")
    imgs, labels = M.parse_test_data_header(path)
    assert imgs.shape == (10, 256) and labels.tolist() == [3, 2, 0, 9, 0, 6, 9, 2, 7, 7] and imgs[0, 0] == -20   # 0xEC narrowed to int8
    assert np.array_equal(imgs, d["images"])


def test_blob_roundtrip_names_layers_like_the_reference_harness():
    """ADVICE r1: the BNM1 blob stores no layer names; Model.load assigns the names the reference's dll.c compiles against
    (FC: L1.., CNN: L2, L4, L6, L7, L9, L11, L13, L15 -- BitNetMCU_MNIST_dll.c:48-121), so write_header output links unchanged."""
    from bitnetmcu_b200.model import Model
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    fc = Model.load(os.path.join(root, "tests", "golden", "models", "fc.bnm"))
    assert [l.name for l in fc.layers] == ["L1", "L2", "L3", "L4"]
    cnn = Model.load(os.path.join(root, "tests", "golden", "models", "cnn_48.bnm"))
    assert [l.name for l in cnn.layers] == ["L2", "L4", "L6", "L7", "L9", "L11", "L13", "L15"]
    again = Model.from_blob(cnn.to_blob())
    assert [l.name for l in again.layers] == [l.name for l in cnn.layers]
