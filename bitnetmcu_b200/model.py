"""Packed-model container for the BitNetMCU hot path: header parser, runtime descriptor, blob format.

The reference selects its model at compile time by naming a generated header ``BitNetMCU_model.h``
(/root/reference/Makefile:2, BitNetMCU_MNIST_dll.c:4).  The layout contract is the header that
``export_to_hfile`` writes (/root/reference/exportquant.py:49-263) and the shipped samples
(/root/reference/BitNetMCU_model_fc.h:8-25, BitNetMCU_model_cnn.h:12-34,126-132,195-201):

* ``#define MODEL_<class>``, ``Lk_bitperweight`` (an encoding *id*: 1,2,4,12,16,20,36,64),
  ``Lk_incoming_weights`` / ``Lk_outgoing_weights`` and ``const uint32_t Lk_weights[]`` with the first
  weight of a row in the most-significant bits (ternary: ``const uint16_t``, 10 trits per word);
* conv layers: ``Lk_in_channels/out_channels/incoming_x/groups`` + ``const int8_t Lk_weights[]`` in
  ``[C][1][3][3]`` order; max-pool layers: macros only.

This module parses such a header *without a C compiler* into a runtime descriptor (the engine needs a
runtime model, SURVEY.md section 5 "Config / flags"), discovers layers by scanning ``L<k>_`` names rather
than assuming ``L1..L4`` (current exporter emits ``L3/L5/L7/L9``, SURVEY.md section 7), and (de)serialises
the descriptor to a flat little-endian blob (``.bnm``) that the C-ABI ``bnm_model_load_blob`` reads and
that ships as the test fixtures under ``tests/golden/models``.
"""
from __future__ import annotations

import re
import struct
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

# layer kinds / model classes -- numbering shared with include/bitnetmcu_b200.h
LAYER_FC = 0
LAYER_CONV33 = 1
LAYER_MAXPOOL22 = 2
MODEL_FCMNIST = 0
MODEL_CNNMNIST = 1

# encoding ids written by exportquant.py:106-159 ("QuantID") and switched on in inference.c:96-201
ENC_BINARY = 1
ENC_2BITSYM = 2
ENC_4BITSYM = 4
ENC_4BIT = 12
ENC_8BIT = 16
ENC_FP130 = 20
ENC_NF4 = 36  # exported by the reference but NOT decoded by its C engine (inference.c:202)
ENC_TERNARY = 64

ENC_NAMES = {
    ENC_BINARY: "Binary", ENC_2BITSYM: "2bitsym", ENC_4BITSYM: "4bitsym", ENC_4BIT: "4bit",
    ENC_8BIT: "8bit", ENC_FP130: "FP130", ENC_NF4: "NF4", ENC_TERNARY: "Ternary",
}
# weights per 32-bit word (ternary: 10 per 16-bit word)
ENC_WEIGHTS_PER_WORD = {ENC_BINARY: 32, ENC_2BITSYM: 16, ENC_4BITSYM: 8, ENC_4BIT: 8, ENC_FP130: 8,
                        ENC_NF4: 8, ENC_8BIT: 4}

BLOB_MAGIC = b"BNM1"
_BLOB_HDR = struct.Struct("<4sIII")
_BLOB_LAYER = struct.Struct("<IiIIIIII")


@dataclass
class Layer:
    kind: int
    name: str                       # "L1", "L11", ...
    bitperweight: int = 0           # FC: encoding id; conv: 8
    n_in: int = 0                   # FC: incoming_weights ; conv/pool: incoming_x
    n_out: int = 0                  # FC: outgoing_weights ; conv: out_channels ; pool: outgoing_x
    in_channels: int = 0
    groups: int = 0
    weights: Optional[np.ndarray] = None   # uint32 / uint16 (ternary) / int8 (conv)

    def weight_bytes(self) -> bytes:
        return b"" if self.weights is None else np.ascontiguousarray(self.weights).tobytes()

    def expected_words(self) -> int:
        """Number of array elements the reference reads for this layer (inference.c:88-208)."""
        if self.kind == LAYER_CONV33:
            return self.n_out * 9
        if self.kind != LAYER_FC:
            return 0
        if self.bitperweight == ENC_TERNARY:
            return self.n_out * (self.n_in // 10)
        wpw = ENC_WEIGHTS_PER_WORD.get(self.bitperweight)
        if wpw is None:
            return 0 if self.weights is None else int(self.weights.size)
        return self.n_out * ((self.n_in + wpw - 1) // wpw)


@dataclass
class Model:
    model_class: int
    layers: List[Layer] = field(default_factory=list)
    img_bytes: int = 256            # 16x16 int8 image (BitNetMCU_MNIST_dll.c:68)
    source: str = ""

    # ---- views -------------------------------------------------------------------------------
    @property
    def fc_layers(self) -> List[Layer]:
        return [l for l in self.layers if l.kind == LAYER_FC]

    @property
    def conv_layers(self) -> List[Layer]:
        return [l for l in self.layers if l.kind == LAYER_CONV33]

    @property
    def n_classes(self) -> int:
        return self.fc_layers[-1].n_out

    @property
    def channels(self) -> int:
        return self.conv_layers[0].n_out if self.conv_layers else 0

    @property
    def macs_per_image(self) -> int:
        """Integer multiply-accumulates per image (SURVEY.md 8d)."""
        macs = sum(l.n_in * l.n_out for l in self.fc_layers)
        if self.model_class == MODEL_CNNMNIST:
            xy = self.conv_layers[0].n_in
            o1, o2, o3 = (xy - 2) ** 2, (xy - 4) ** 2, ((xy - 4) // 2 - 2) ** 2
            macs += self.channels * 9 * (o1 + o2 + o3)
        return macs

    def tap_shapes(self) -> List[Tuple[int, int]]:
        """(width, stride) of every activation tap (include/bitnetmcu_b200.h section 7), from the layer table alone: the CNN
        features (C*4 values, rows of round_up(C*4, 16) bytes) for CNN models, then per hidden FC layer its n_out values in rows
        of round_up(n_in of the next layer, 32) bytes."""
        fc = self.fc_layers
        shapes = []
        if self.model_class == MODEL_CNNMNIST:
            shapes.append((self.channels * 4, -(-self.channels * 4 // 16) * 16))
        shapes += [(fc[l].n_out, -(-fc[l + 1].n_in // 32) * 32) for l in range(len(fc) - 1)]
        return shapes

    def describe(self) -> str:
        parts = []
        for l in self.layers:
            if l.kind == LAYER_FC:
                parts.append(f"{l.name}:fc[{ENC_NAMES.get(l.bitperweight, l.bitperweight)}]{l.n_in}->{l.n_out}")
            elif l.kind == LAYER_CONV33:
                parts.append(f"{l.name}:conv33x{l.n_out}@{l.n_in}")
            else:
                parts.append(f"{l.name}:pool@{l.n_in}")
        return ("CNNMNIST " if self.model_class == MODEL_CNNMNIST else "FCMNIST ") + " ".join(parts)

    def validate(self) -> None:
        if not self.fc_layers:
            raise ValueError("model has no fully connected layer")
        for l in self.layers:
            if l.kind in (LAYER_FC, LAYER_CONV33):
                if l.weights is None:
                    raise ValueError(f"{l.name}: no weight array")
                need = l.expected_words()
                if l.weights.size < need:
                    raise ValueError(f"{l.name}: weight array has {l.weights.size} elements, reference reads {need}")
        if self.model_class == MODEL_CNNMNIST:
            kinds = [l.kind for l in self.layers if l.kind != LAYER_FC]
            if kinds != [LAYER_CONV33, LAYER_CONV33, LAYER_MAXPOOL22, LAYER_CONV33, LAYER_MAXPOOL22]:
                raise ValueError("CNN front-end must be conv,conv,pool,conv,pool (BitNetMCU_MNIST_dll.c:64-80)")
            c = self.channels
            if any(cl.n_out != c for cl in self.conv_layers):
                raise ValueError("all conv layers must have the same channel count")

    # ---- blob --------------------------------------------------------------------------------
    def to_blob(self) -> bytes:
        """Flat little-endian blob: header | layer table | 16-byte aligned weight data."""
        self.validate()
        table_end = _BLOB_HDR.size + _BLOB_LAYER.size * len(self.layers)
        data = bytearray()
        entries = []
        for l in self.layers:
            raw = l.weight_bytes()
            off = 0
            if raw:
                pad = (-(table_end + len(data))) % 16
                data += b"\0" * pad
                off = table_end + len(data)
                data += raw
            entries.append(_BLOB_LAYER.pack(l.kind, l.bitperweight, l.n_in, l.n_out, l.in_channels, l.groups,
                                            off, len(raw)))
        return _BLOB_HDR.pack(BLOB_MAGIC, self.model_class, len(self.layers), self.img_bytes) + b"".join(entries) + bytes(data)

    @staticmethod
    def reference_layer_names(model_class: int, kinds: List[int]) -> List[str]:
        """The ``L<k>`` names the reference's harnesses compile against (the blob does not store names): FC models
        ``L1..Ln`` (BitNetMCU_MNIST_dll.c:95-121, BitNetMCU_model_fc.h), CNN models the module-enumeration indices of the
        shipped header -- conv L2, conv L4, pool L6, conv L7, pool L9, then FC L11, L13, L15, ...
        (BitNetMCU_MNIST_dll.c:64-90, BitNetMCU_model_cnn.h)."""
        if model_class == MODEL_CNNMNIST and kinds[:5] == [LAYER_CONV33, LAYER_CONV33, LAYER_MAXPOOL22, LAYER_CONV33, LAYER_MAXPOOL22]:
            return ["L2", "L4", "L6", "L7", "L9"] + [f"L{11 + 2 * i}" for i in range(len(kinds) - 5)]
        return [f"L{i + 1}" for i in range(len(kinds))]

    @staticmethod
    def from_blob(blob: bytes, source: str = "") -> "Model":
        magic, cls, n_layers, img_bytes = _BLOB_HDR.unpack_from(blob, 0)
        if magic != BLOB_MAGIC:
            raise ValueError("not a BNM1 model blob")
        m = Model(model_class=cls, img_bytes=img_bytes, source=source)
        for i in range(n_layers):
            kind, bpw, n_in, n_out, in_ch, groups, off, nbytes = _BLOB_LAYER.unpack_from(
                blob, _BLOB_HDR.size + i * _BLOB_LAYER.size)
            w = None
            if nbytes:
                dt = np.int8 if kind == LAYER_CONV33 else (np.uint16 if bpw == ENC_TERNARY else np.uint32)
                w = np.frombuffer(blob, dtype=dt, count=nbytes // np.dtype(dt).itemsize, offset=off).copy()
            m.layers.append(Layer(kind=kind, name=f"L{i}", bitperweight=bpw, n_in=n_in, n_out=n_out,
                                  in_channels=in_ch, groups=groups, weights=w))
        for l, name in zip(m.layers, Model.reference_layer_names(cls, [l.kind for l in m.layers])):
            l.name = name
        m.validate()
        return m

    def save(self, path: str) -> None:
        with open(path, "wb") as f:
            f.write(self.to_blob())

    @staticmethod
    def load(path: str) -> "Model":
        with open(path, "rb") as f:
            return Model.from_blob(f.read(), source=path)


# ---------------------------------------------------------------------------------------------------
# header parser
# ---------------------------------------------------------------------------------------------------
_RE_DEFINE = re.compile(r"^\s*#\s*define\s+(\w+)(?:[ \t]+([^\n/]*?))?\s*(?://.*)?$", re.M)
_RE_ARRAY = re.compile(r"const\s+(u?int(?:8|16|32)_t)\s+(\w+)\s*\[\s*\]\s*=\s*\{(.*?)\}\s*;", re.S)
_RE_LAYER = re.compile(r"^L(\d+)_(\w+)$")
_CTYPE = {"uint32_t": np.uint32, "uint16_t": np.uint16, "int8_t": np.int8, "uint8_t": np.uint8,
          "int32_t": np.int32, "int16_t": np.int16}


def _strip_comments(text: str) -> str:
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def _parse_array(ctype: str, body: str) -> np.ndarray:
    toks = [t for t in re.split(r"[\s,]+", body.strip()) if t]
    vals = [int(t, 0) for t in toks]
    dt = _CTYPE[ctype]
    info = np.iinfo(dt)
    # C narrowing of out-of-range initialisers (e.g. 0xEC for int8_t, BitNetMCU_MNIST_test_data.h:2)
    arr = np.array(vals, dtype=np.int64)
    if info.min < 0:
        span = 1 << (8 * np.dtype(dt).itemsize)
        arr = ((arr + (span >> 1)) % span) - (span >> 1)
    return arr.astype(dt)


def parse_header_text(text: str, source: str = "") -> Model:
    clean = _strip_comments(text)
    defines: Dict[str, str] = {}
    for m in _RE_DEFINE.finditer(clean):
        defines[m.group(1)] = (m.group(2) or "").strip()
    arrays = {m.group(2): _parse_array(m.group(1), m.group(3)) for m in _RE_ARRAY.finditer(clean)}

    if "MODEL_CNNMNIST" in defines:
        model_class = MODEL_CNNMNIST
    elif "MODEL_FCMNIST" in defines:
        model_class = MODEL_FCMNIST
    else:
        raise ValueError(f"{source or 'header'}: neither MODEL_FCMNIST nor MODEL_CNNMNIST defined "
                         "(BitNetMCU_MNIST_dll.c:122 '#error No model defined')")

    per_layer: Dict[int, Dict[str, str]] = {}
    for name, val in defines.items():
        lm = _RE_LAYER.match(name)
        if lm:
            per_layer.setdefault(int(lm.group(1)), {})[lm.group(2)] = val

    model = Model(model_class=model_class, source=source)
    for k in sorted(per_layer):
        d = per_layer[k]
        if "active" not in d:
            continue
        lname = f"L{k}"
        ltype = d.get("type", "")
        if ltype == "BitConv2d":
            model.layers.append(Layer(kind=LAYER_CONV33, name=lname, bitperweight=int(d.get("bitperweight", 8)),
                                      n_in=int(d["incoming_x"]), n_out=int(d["out_channels"]),
                                      in_channels=int(d.get("in_channels", 1)), groups=int(d.get("groups", 1)),
                                      weights=arrays.get(f"{lname}_weights")))
            if int(d.get("kernel_size", 3)) != 3:
                raise ValueError(f"{lname}: only 3x3 kernels exist in the reference (inference.c:238)")
        elif ltype == "MaxPool2d":
            model.layers.append(Layer(kind=LAYER_MAXPOOL22, name=lname, n_in=int(d["incoming_x"]),
                                      n_out=int(d.get("outgoing_x", int(d["incoming_x"]) // 2))))
        elif "bitperweight" in d and "incoming_weights" in d:
            model.layers.append(Layer(kind=LAYER_FC, name=lname, bitperweight=int(d["bitperweight"]),
                                      n_in=int(d["incoming_weights"]), n_out=int(d["outgoing_weights"]),
                                      weights=arrays.get(f"{lname}_weights")))
    model.validate()
    return model


def parse_header(path: str) -> Model:
    with open(path, "r") as f:
        return parse_header_text(f.read(), source=path)


def parse_test_data_header(path: str):
    """``BitNetMCU_MNIST_test_data.h``: returns (images int8 [n,256], labels uint8 [n])."""
    with open(path, "r") as f:
        clean = _strip_comments(f.read())
    imgs, labels = {}, {}
    for m in re.finditer(r"(u?int8_t)\s+input_data_(\d+)\s*\[\s*\d*\s*\]\s*=\s*\{(.*?)\}\s*;", clean, re.S):
        imgs[int(m.group(2))] = _parse_array("int8_t", m.group(3))
    for m in re.finditer(r"u?int8_t\s+label_(\d+)\s*=\s*(\d+)\s*;", clean):
        labels[int(m.group(1))] = int(m.group(2))
    idx = sorted(imgs)
    return np.stack([imgs[i] for i in idx]).astype(np.int8), np.array([labels[i] for i in idx], dtype=np.uint8)
