"""Host-side mirror of the reference interface for the hot path, on top of the C ABI.

Reference                                              here
-------------------------------------------------------------------------------------------------
lib.Inference(ptr) per image (test_inference.py:146)   Engine.infer(images) / Engine.inference(image)
processfclayer / ReLUNorm / processconv33ReLU /        processfclayer / relunorm / conv33relu / maxpool22
processmaxpool22 (BitNetMCU_inference.h:15-60)         (same argument meaning, batched over a leading axis)
model = whichever header is named BitNetMCU_model.h    Engine(Model) from parse_header() / a .bnm blob

Nothing here computes on the CPU: every call goes through libbitnetmcu_b200.so (hand-written sm_100a CUDA).
torch is used only as plumbing for device memory / streams in ``infer_device``.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .model import Model


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else C.c_void_p(a.ctypes.data)


class Engine:
    """One packed model resident on one GPU."""

    def __init__(self, model: Model, device: int = 0, path: int = _lib.PATH_AUTO, nf4_extension: bool = False):
        self.lib = _lib.load()
        if self.lib.bnm_device_count() == 0:
            raise _lib.BnmError("no CUDA device: bitnetmcu_b200 has no CPU fallback")
        self.model = model
        blob = model.to_blob()
        self._blob = (C.c_char * len(blob)).from_buffer_copy(blob)
        h = C.c_void_p()
        _lib.check(self.lib.bnm_model_load_blob(self._blob, len(blob), device, C.byref(h)), "bnm_model_load_blob")
        self.handle = h
        self.device = device
        self.n_classes = int(self.lib.bnm_model_n_classes(h))
        self.img_bytes = int(self.lib.bnm_model_img_bytes(h))
        if nf4_extension:
            self.set_option(_lib.OPT_NF4_EXTENSION, 1)
        if path != _lib.PATH_AUTO:
            self.set_option(_lib.OPT_PATH, path)

    def close(self) -> None:
        if getattr(self, "handle", None):
            self.lib.bnm_model_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, option: int, value: int) -> None:
        _lib.check(self.lib.bnm_model_set_option(self.handle, option, int(value)), "bnm_model_set_option")

    @property
    def active_path(self) -> int:
        return int(self.lib.bnm_model_active_path(self.handle))

    def launch_count(self, n: int) -> int:
        return int(self.lib.bnm_infer_launch_count(self.handle, n))

    # ---- batched inference over host arrays (H2D / kernels / D2H pipelined inside the library) -----------
    def infer(self, images: np.ndarray, want_labels: bool = True, out_logits: Optional[np.ndarray] = None,
              out_labels: Optional[np.ndarray] = None) -> Tuple[np.ndarray, Optional[np.ndarray]]:
        imgs = np.ascontiguousarray(images, dtype=np.int8).reshape(-1, self.img_bytes)
        n = imgs.shape[0]
        logits = out_logits if out_logits is not None else np.empty((n, self.n_classes), dtype=np.int32)
        labels = out_labels if out_labels is not None else (np.empty(n, dtype=np.uint32) if want_labels else None)
        _lib.check(self.lib.bnm_infer_batch(self.handle, _ptr(imgs), n, _ptr(logits), _ptr(labels)), "bnm_infer_batch")
        return logits, labels

    def inference(self, image: np.ndarray) -> int:
        """``uint32_t Inference(int8_t *input)`` (BitNetMCU_MNIST_dll.c:24): predicted class of one image."""
        _, labels = self.infer(np.asarray(image, dtype=np.int8).reshape(1, self.img_bytes))
        return int(labels[0])

    # ---- device pointers (torch tensors as plumbing) ---------------------------------------------------
    def infer_device(self, images, logits, labels=None, stream: Optional[int] = None) -> None:
        """images: torch.int8 [n, img_bytes] on this GPU; logits: torch.int32 [n, n_classes]; labels: torch.int32/uint32 [n]
        or None.  Asynchronous on ``stream`` (a cudaStream_t as int; default: torch's current stream).

        With ``OPT_LAUNCH_OVERLAP`` = 2 a launch whose buffers differ from the previous call's is NOT ordered against earlier
        work on the stream (include/bitnetmcu_b200.h): its images must already be complete when the previous call was
        enqueued.  Chains such as ``quantize_images_device`` -> ``infer_device`` on one stream need mode 0 or 1."""
        import torch
        n = images.shape[0]
        if stream is None:
            stream = torch.cuda.current_stream(images.device).cuda_stream
        assert images.is_contiguous() and logits.is_contiguous() and images.dtype == torch.int8 and logits.dtype == torch.int32
        assert images.shape[1] == self.img_bytes and tuple(logits.shape) == (n, self.n_classes)
        lab_ptr = None
        if labels is not None:
            assert labels.is_contiguous() and labels.element_size() == 4 and labels.numel() == n
            lab_ptr = C.c_void_p(labels.data_ptr())
        _lib.check(self.lib.bnm_infer_batch_device(self.handle, C.c_void_p(images.data_ptr()), n, C.c_void_p(logits.data_ptr()),
                                                   lab_ptr, C.c_void_p(stream)), "bnm_infer_batch_device")


    # ---- activation taps: the int8 rows between the layers (include/bitnetmcu_b200.h section 7) -------------
    @property
    def n_taps(self) -> int:
        """Taps of this model: one per hidden FC layer, plus the CNN features (tap 0) for CNN models."""
        return int(self.lib.bnm_model_n_taps(self.handle))

    def tap_shapes(self) -> List[Tuple[int, int]]:
        """(width, stride) per tap: real int8 values per row, and bytes between rows of a tap buffer."""
        return [(int(self.lib.bnm_model_tap_width(self.handle, t)), int(self.lib.bnm_model_tap_stride(self.handle, t)))
                for t in range(self.n_taps)]

    def infer_taps(self, images: np.ndarray) -> Tuple[np.ndarray, np.ndarray, List[np.ndarray]]:
        """As ``infer``, plus every tap: (logits int32 [n, n_classes], labels uint32 [n], [int8 [n, width] per tap])."""
        imgs = np.ascontiguousarray(images, dtype=np.int8).reshape(-1, self.img_bytes)
        n = imgs.shape[0]
        logits = np.empty((n, self.n_classes), dtype=np.int32)
        labels = np.empty(n, dtype=np.uint32)
        bufs = [np.empty((n, stride), dtype=np.int8) for _, stride in self.tap_shapes()]
        taps = _lib.BnmTaps()
        for t, b in enumerate(bufs):
            taps.act[t] = b.ctypes.data
        _lib.check(self.lib.bnm_infer_batch_taps(self.handle, _ptr(imgs), n, _ptr(logits), _ptr(labels), C.byref(taps)),
                   "bnm_infer_batch_taps")
        return logits, labels, [b[:, :w] for b, (w, _) in zip(bufs, self.tap_shapes())]

    def infer_device_taps(self, images, logits, labels, taps: Sequence, stream: Optional[int] = None) -> None:
        """As ``infer_device``, plus the taps: ``taps[t]`` is a torch.int8 [n, stride of t] tensor on this GPU, or None when tap t
        is not wanted.  Only int8 images: float input has no taps."""
        import torch
        n = images.shape[0]
        if images.dtype != torch.int8:
            raise _lib.BnmError(f"activation taps need int8 images (got {images.dtype}): float input has no taps")
        if stream is None:
            stream = torch.cuda.current_stream(images.device).cuda_stream
        assert images.is_contiguous() and logits.is_contiguous() and logits.dtype == torch.int32
        assert images.shape[1] == self.img_bytes and tuple(logits.shape) == (n, self.n_classes)
        assert len(taps) <= _lib.MAX_TAPS
        lab_ptr = None
        if labels is not None:
            assert labels.is_contiguous() and labels.element_size() == 4 and labels.numel() == n
            lab_ptr = C.c_void_p(labels.data_ptr())
        shapes = self.tap_shapes()
        tt = _lib.BnmTaps()
        for t, b in enumerate(taps):
            if b is None:
                continue
            assert t < len(shapes), f"tap {t}: the model has {len(shapes)} taps"
            assert b.dtype == torch.int8 and b.is_contiguous() and tuple(b.shape) == (n, shapes[t][1]), \
                f"tap {t}: want a contiguous torch.int8 [{n}, {shapes[t][1]}] tensor"
            tt.act[t] = b.data_ptr()
        _lib.check(self.lib.bnm_infer_batch_device_taps(self.handle, C.c_void_p(images.data_ptr()), n, C.c_void_p(logits.data_ptr()),
                                                        lab_ptr, C.byref(tt), C.c_void_p(stream)), "bnm_infer_batch_device_taps")

    def inference_quantized(self, input_data: np.ndarray) -> np.ndarray:
        """``QuantizedModel.inference_quantized`` (/root/reference/BitNetMCU.py:420-535) on the GPU: float32 images [n, img_bytes]
        -> float64 logits [n, n_classes] with the Python emulator's normalisation rules (not the C engine's): what
        ``np.argmax`` is taken of in test_inference.py:153-154 and exportquant.py:537-559."""
        x = np.ascontiguousarray(input_data, dtype=np.float32).reshape(-1, self.img_bytes)
        out = np.empty((x.shape[0], self.n_classes), dtype=np.float64)
        _lib.check(self.lib.bnm_emulate_inference_quantized(self.handle, _ptr(x), x.shape[0], _ptr(out)), "bnm_emulate_inference_quantized")
        return out

    def infer_device_f32(self, images, logits, labels=None, stream: Optional[int] = None) -> None:
        """images: torch.float32 [n, img_bytes] on this GPU (un-normalised pixels, as test_inference.py:140 sees them) -> logits
        torch.int32 [n, n_classes], labels [n].  FC models: one kernel with the input scaling fused into its load stage."""
        import torch
        n = images.shape[0]
        if stream is None:
            stream = torch.cuda.current_stream(images.device).cuda_stream
        assert images.is_contiguous() and images.dtype == torch.float32 and images.shape[1] == self.img_bytes
        assert logits.is_contiguous() and logits.dtype == torch.int32 and tuple(logits.shape) == (n, self.n_classes)
        lab_ptr = C.c_void_p(labels.data_ptr()) if labels is not None else None
        _lib.check(self.lib.bnm_infer_batch_device_f32(self.handle, C.c_void_p(images.data_ptr()), n, C.c_void_p(logits.data_ptr()), lab_ptr,
                                                       C.c_void_p(stream)), "bnm_infer_batch_device_f32")

    def infer_tensor(self, images):
        """images: torch.int8 [n, img_bytes] on this engine's GPU -> (logits torch.int32 [n, n_classes], labels torch.int32 [n]) on
        the same GPU, asynchronous on torch's current stream (device memory end to end; plumbing for ``dist.sharded_infer``)."""
        import torch
        n = images.shape[0]
        logits = torch.empty((n, self.n_classes), dtype=torch.int32, device=images.device)
        labels = torch.empty(n, dtype=torch.int32, device=images.device)
        if n:
            self.infer_device(images.contiguous(), logits, labels)
        return logits, labels


# ---- the four reference kernels, batched (host arrays) --------------------------------------------------------

def processfclayer(activations: np.ndarray, weights: np.ndarray, bits_per_weight: int, n_input: int, n_output: int,
                   nf4_extension: bool = False) -> np.ndarray:
    """inference.c:88-208 over a batch: activations int8 [n, n_input] -> int32 [n, n_output]."""
    lib = _lib.load()
    act = np.ascontiguousarray(activations, dtype=np.int8).reshape(-1, n_input)
    w = np.ascontiguousarray(weights)
    out = np.empty((act.shape[0], n_output), dtype=np.int32)
    _lib.check(lib.bnm_processfclayer_batch(_ptr(act), _ptr(w), bits_per_weight, n_input, n_output, _ptr(out), act.shape[0],
                                            int(nf4_extension)), "bnm_processfclayer_batch")
    return out


def relunorm(x: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """inference.c:23-72 over a batch: int32 [n, n_input] -> (int8 [n, n_input], argmax uint32 [n])."""
    lib = _lib.load()
    x = np.ascontiguousarray(x, dtype=np.int32)
    x2 = x.reshape(-1, x.shape[-1]) if x.ndim > 1 else x.reshape(1, -1)
    out = np.empty(x2.shape, dtype=np.int8)
    pos = np.empty(x2.shape[0], dtype=np.uint32)
    _lib.check(lib.bnm_relunorm_batch(_ptr(x2), _ptr(out), _ptr(pos), x2.shape[1], x2.shape[0]), "bnm_relunorm_batch")
    return out, pos


def conv33relu(activations: np.ndarray, weights: np.ndarray, xy: int, n_shift: int = 4) -> np.ndarray:
    """inference.c:238-277 over a batch: int32 [n, xy*xy], int8 [n_w, 9] (item i uses weights[i % n_w])."""
    lib = _lib.load()
    a = np.ascontiguousarray(activations, dtype=np.int32).reshape(-1, xy * xy)
    w = np.ascontiguousarray(weights, dtype=np.int8).reshape(-1, 9)
    out = np.empty((a.shape[0], (xy - 2) * (xy - 2)), dtype=np.int32)
    _lib.check(lib.bnm_conv33relu_batch(_ptr(a), _ptr(w), w.shape[0], xy, n_shift, _ptr(out), a.shape[0]), "bnm_conv33relu_batch")
    return out


def maxpool22(activations: np.ndarray, xy: int) -> np.ndarray:
    """inference.c:300-322 over a batch: int32 [n, xy*xy] -> int32 [n, (xy/2)^2]."""
    lib = _lib.load()
    a = np.ascontiguousarray(activations, dtype=np.int32).reshape(-1, xy * xy)
    out = np.empty((a.shape[0], (xy // 2) * (xy // 2)), dtype=np.int32)
    _lib.check(lib.bnm_maxpool22_batch(_ptr(a), xy, _ptr(out), a.shape[0]), "bnm_maxpool22_batch")
    return out


def quantize_images(images: np.ndarray) -> np.ndarray:
    """The step right before the path (test_inference.py:140-141): float32 [n, elems] -> int8 [n, elems],
    ``np.round(x * (127 / max(|x|.max(-1), 1e-5))).clip(-128, 127)`` computed on the GPU, bit-identical to NumPy float32."""
    lib = _lib.load()
    x = np.ascontiguousarray(images, dtype=np.float32)
    x2 = x.reshape(-1, x.shape[-1]) if x.ndim > 1 else x.reshape(1, -1)
    out = np.empty(x2.shape, dtype=np.int8)
    _lib.check(lib.bnm_quantize_images(_ptr(x2), x2.shape[0], x2.shape[1], _ptr(out)), "bnm_quantize_images")
    return out


def quantize_images_device(images, out, stream: Optional[int] = None) -> None:
    """Device-buffer form: images torch.float32 [n, elems] -> out torch.int8 [n, elems] on the same GPU, asynchronous on
    ``stream`` (default: torch's current stream), so it chains with ``Engine.infer_device`` without a host pass."""
    import torch
    lib = _lib.load()
    assert images.is_contiguous() and out.is_contiguous() and images.dtype == torch.float32 and out.dtype == torch.int8
    assert images.dim() == 2 and tuple(out.shape) == tuple(images.shape)
    if stream is None:
        stream = torch.cuda.current_stream(images.device).cuda_stream
    _lib.check(lib.bnm_quantize_images_device(C.c_void_p(images.data_ptr()), images.shape[0], images.shape[1],
                                              C.c_void_p(out.data_ptr()), C.c_void_p(stream)), "bnm_quantize_images_device")
