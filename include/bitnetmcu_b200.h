/*
 * bitnetmcu_b200.h -- C ABI of the B200-native BitNetMCU inference engine (libbitnetmcu_b200.so).
 *
 * Drop-in boundary for ONE path of cpldcpu/BitNetMCU: processfclayer + ReLUNorm + the per-channel
 * conv/maxpool loop of BitNetMCU_inference.c, chained as BitMnistInference does.  Host code stays
 * plain C; everything behind these entry points is hand-written sm_100a CUDA.  There is NO CPU
 * fallback: every compute entry fails (negative return / aborts, see below) without a CUDA device.
 *
 * Section 1 keeps the reference's own symbols, signatures and semantics
 *   (/root/reference/BitNetMCU_inference.h:15,31,45,60) so code written against the reference links
 *   unchanged; each call copies its small host buffers to the GPU, runs the kernel on one item and
 *   copies the result back.
 * Section 2 is the model container: the packed-weight layout of exportquant.py / BitNetMCU_model.h
 *   (/root/reference/exportquant.py:68-84,182-207,222-259) as a runtime descriptor.
 * Section 3 is the batched entry the reference lacks (its caller loops lib.Inference() per image,
 *   /root/reference/test_inference.py:136-150): millions of 16x16 int8 images per call.
 * Section 4 exposes the four kernels batched, for parity tests and partial integration.
 *
 * Pointers are plain host (or, where the name says _device, CUDA device) pointers; sizes are element
 * counts unless named *_bytes.  All-integer arithmetic: results are bit-exact with the reference.
 */
#ifndef BITNETMCU_B200_H
#define BITNETMCU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNM_API __attribute__((visibility("default")))
#define BNM_VERSION 100

/* ---------------------------------------------------------------------------------------------
 * 1. Reference-compatible kernels (host pointers, one item per call).
 *    Same names/signatures as BitNetMCU_inference.h so they replace BitNetMCU_inference.c at link time.
 *    The reference has no error reporting (SURVEY.md 8b); on a CUDA failure these print the reason to
 *    stderr and abort() -- they never fall back to a CPU implementation.
 * ------------------------------------------------------------------------------------------- */

/* replaces BitNetMCU_inference.c:23-72 (proto BitNetMCU_inference.h:15).  Returns argmax (first max; 255 if n==0);
 * output[i] = x<0 ? 0 : min(127,(x+rounding)>>shift).  input/output may alias (dll.c:80). */
BNM_API uint32_t ReLUNorm(int32_t *input, int8_t *output, uint32_t n_input);

/* replaces BitNetMCU_inference.c:88-208 (proto BitNetMCU_inference.h:31).  bits_per_weight is the encoding id
 * 1,2,4,12,16,20,64; any other id (incl. 36 = NF4) yields zeros exactly like inference.c:202. */
BNM_API void processfclayer(int8_t *activations, const uint32_t *weights, int32_t bits_per_weight,
                            uint32_t n_input, uint32_t n_output, int32_t *output);

/* replaces BitNetMCU_inference.c:238-277 (proto BitNetMCU_inference.h:45); in-place allowed; returns end pointer */
BNM_API int32_t *processconv33ReLU(int32_t *activations, const int8_t *weights, uint32_t xy_input,
                                   uint32_t n_shift, int32_t *output);

/* replaces BitNetMCU_inference.c:300-322 (proto BitNetMCU_inference.h:60); in-place allowed; returns end pointer */
BNM_API int32_t *processmaxpool22(int32_t *activations, uint32_t xy_input, int32_t *output);

/* ---------------------------------------------------------------------------------------------
 * 2. Model container
 * ------------------------------------------------------------------------------------------- */
enum { BNM_LAYER_FC = 0, BNM_LAYER_CONV33 = 1, BNM_LAYER_MAXPOOL22 = 2 };
enum { BNM_MODEL_FCMNIST = 0, BNM_MODEL_CNNMNIST = 1 };            /* #define MODEL_FCMNIST / MODEL_CNNMNIST */
/* encoding ids = Lk_bitperweight (exportquant.py:106-159, inference.c:96-201) */
enum { BNM_ENC_BINARY = 1, BNM_ENC_2BITSYM = 2, BNM_ENC_4BITSYM = 4, BNM_ENC_4BIT = 12, BNM_ENC_8BIT = 16,
       BNM_ENC_FP130 = 20, BNM_ENC_NF4 = 36, BNM_ENC_TERNARY = 64 };

typedef struct bnm_layer {
    uint32_t kind;          /* BNM_LAYER_*                                                           */
    int32_t  bitperweight;  /* FC: Lk_bitperweight (encoding id) ; conv: 8                           */
    uint32_t n_in;          /* FC: Lk_incoming_weights ; conv/pool: Lk_incoming_x                    */
    uint32_t n_out;         /* FC: Lk_outgoing_weights ; conv: Lk_out_channels ; pool: Lk_outgoing_x */
    uint32_t in_channels;   /* conv: Lk_in_channels                                                  */
    uint32_t groups;        /* conv: Lk_groups                                                       */
    const void *weights;    /* FC: const uint32_t Lk_weights[] (uint16_t for Ternary) ; conv: const int8_t Lk_weights[] */
    size_t   weight_bytes;  /* sizeof(Lk_weights)                                                    */
} bnm_layer;

typedef struct bnm_model bnm_model;   /* opaque; weights decoded and resident on one GPU */

/* execution path of the FC chain */
enum {
    BNM_PATH_AUTO = 0,     /* fused tcgen05 kernel when the model shape is supported, else BNM_PATH_LAYERS */
    BNM_PATH_LAYERS = 1,   /* one CUDA-core (dp4a) kernel per layer + ReLUNorm kernel; any shape          */
    BNM_PATH_TCGEN05 = 2   /* fused persistent kernel: TMA -> tcgen05.mma kind::i8 -> in-TMEM ReLUNorm     */
};
enum { BNM_OPT_PATH = 1, BNM_OPT_NF4_EXTENSION = 2, BNM_OPT_CHUNK_IMAGES = 3, BNM_OPT_LAUNCH_OVERLAP = 4, BNM_OPT_CNN_FRONTEND = 5 };
/* BNM_OPT_CNN_FRONTEND (CNN models, the conv/pool loop of BitNetMCU_MNIST_dll.c:64-80): 0 (default) conv1 on the tensor cores
 * (tcgen05, depthwise tail fed from TMEM) when the channel count is a multiple of 16 and <= 128, else the CUDA-core kernel;
 * 1 CUDA-core kernel; 2 tensor-core kernel or fail.  Results are identical. */
/* BNM_OPT_LAUNCH_OVERLAP (fused kernel, consecutive bnm_infer_batch_device calls on one stream):
 *   0  (default) plain launches, ordinary stream semantics.
 *   1  programmatic dependent launch with a grid-dependency wait: the next launch's prologue (barriers, TMEM, weights) runs
 *      under the tail of the previous one; inputs are read and outputs written only after the previous kernel has
 *      completed.  Ordinary stream semantics.  Measured erratic on B200 (-2 % ... +7 % against mode 0 for builds that
 *      differ in one instruction), hence not the default.
 *   2  the caller declares consecutive launches independent -- the images / logits / labels of one call are not the
 *      buffers of the call right before it (e.g. double-buffered batches), exactly what issuing them on two streams would
 *      promise.  The next launch's tiles then start on each SM as the previous launch leaves it (-6 ... -9 % per step).
 *      CONTRACT: an independent launch executes no grid-dependency wait, so it is ordered against NOTHING enqueued before it
 *      on the stream -- neither the previous bnm launch nor a producer kernel / copy that writes `images`.  The images of
 *      call k must therefore be complete before call k-1 was enqueued (resident inputs, or produced on another stream and
 *      joined by an event before call k-1).  The library keeps ordinary stream semantics (the wait) for every launch where it
 *      can see the promise broken: the first launch after the option is set, a launch on another stream than the one before,
 *      and a launch that reuses the images, logits or labels pointer of the one before.  Producer -> inference chains on one
 *      stream (bnm_quantize_images_device then bnm_infer_batch_device) belong to mode 0 or 1.
 *      Only launches that fill the GPU (>= one 128-image tile per SM) trigger early, and every launch occupies its SM
 *      exclusively (more than half of the shared memory): at most two consecutive launches are ever in flight together.
 *      CNN models are held at mode 1 (the front-end kernel really feeds the FC kernel). */
BNM_API int bnm_version(void);
BNM_API const char *bnm_last_error(void);           /* thread-local text of the last failure */
BNM_API int bnm_device_count(void);                 /* 0 when no CUDA device is usable        */

/* Build a model on `device` from a layer table (the macros/arrays of a BitNetMCU_model.h; see
 * include/bitnetmcu_b200_model.h for the plain-C glue).  FC models: 1..8 FC layers.  CNN models:
 * conv,conv,pool,conv,pool then FC layers (BitNetMCU_MNIST_dll.c:48-91).  Returns 0 or a negative code. */
BNM_API int bnm_model_create(int model_class, const bnm_layer *layers, uint32_t n_layers, uint32_t img_bytes,
                             int device, bnm_model **out);
/* Same, from the flat BNM1 blob written by bitnetmcu_b200.model.Model.to_blob(). */
BNM_API int bnm_model_load_blob(const void *blob, size_t blob_bytes, int device, bnm_model **out);
BNM_API void bnm_model_destroy(bnm_model *m);
BNM_API uint32_t bnm_model_n_classes(const bnm_model *m);
BNM_API uint32_t bnm_model_img_bytes(const bnm_model *m);
BNM_API int bnm_model_set_option(bnm_model *m, int option, int64_t value);
BNM_API int64_t bnm_model_get_option(const bnm_model *m, int option);
/* which path bnm_infer_* will take with the current options (BNM_PATH_LAYERS or BNM_PATH_TCGEN05) */
BNM_API int bnm_model_active_path(const bnm_model *m);

/* ---------------------------------------------------------------------------------------------
 * 3. Batched inference (the hot path)
 * ------------------------------------------------------------------------------------------- */

/* images: int8 [n][img_bytes] row-major (what Inference() takes, n times).  logits: int32 [n][n_classes]
 * = layer_out after the last processfclayer (dll.c:89,115; the reference computes but never returns them).
 * labels: uint32 [n] = the value Inference() returns (argmax of the last ReLUNorm), may be NULL.
 * Host version: buffers are ordinary (ideally pinned, see bnm_host_alloc) host memory; the call streams them
 * through the GPU in chunks with copies overlapped and returns when the results are in `logits`/`labels`. */
BNM_API int bnm_infer_batch(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels);

/* Device version: pointers are device memory on the model's GPU (images 16-byte, logits 8-byte aligned); asynchronous on `stream`
 * (a cudaStream_t, NULL = default stream).  No host synchronisation. */
BNM_API int bnm_infer_batch_device(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels,
                                   void *stream);
/* Fused result exchange (SURVEY.md 8e; the reference has none -- its caller collects one label per call,
 * /root/reference/test_inference.py:146-150): as bnm_infer_batch_device, and the kernel's epilogue ALSO stores row i of this call
 * at row (row_offset + i) of every destination buffer: labels uint32 [rows], logits int32 [rows][n_classes].  Destinations
 * are device pointers valid on the model's GPU -- typically buffers of the peer GPUs of the box mapped through CUDA IPC
 * (bnm_ipc_export / bnm_ipc_open) or same-process P2P (bnm_enable_peer_access), so that the all-gather of the batch-sharded
 * results rides under the compute over NVLink instead of running as a collective after it.  Visibility at the destination
 * follows stream completion of this call on the source plus whatever cross-rank synchronisation the caller uses.
 * Only the fused tcgen05 path supports it. */
#define BNM_MAX_GATHER_DST 8
typedef struct bnm_gather {
    uint32_t n_labels_dst, n_logits_dst;
    uint32_t *labels_dst[BNM_MAX_GATHER_DST];
    int32_t *logits_dst[BNM_MAX_GATHER_DST];   /* 8-byte aligned */
    size_t row_offset;
    uint32_t labels_u8;   /* non-zero: labels_dst are uint8 [rows] buffers (one byte per label, n_classes <= 255): a quarter of the NVLink traffic */
    uint32_t reserved;
} bnm_gather;
BNM_API int bnm_infer_batch_device_gather(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels,
                                          const bnm_gather *gather, void *stream);
/* device memory that can be exported to the other processes of the box (cudaMalloc), CUDA IPC handles (64 bytes) */
BNM_API int bnm_device_alloc(int device, size_t bytes, void **out);
BNM_API void bnm_device_free(void *p);
BNM_API int bnm_ipc_export(const void *dev_ptr, void *handle64);
BNM_API int bnm_ipc_open(int device, const void *handle64, void **out);
BNM_API int bnm_ipc_close(void *p);
BNM_API int bnm_enable_peer_access(int device, int peer);   /* same-process multi-GPU */

/* number of kernels bnm_infer_batch_device launches for n images with the current options */
BNM_API int bnm_infer_launch_count(const bnm_model *m, size_t n);

BNM_API void *bnm_host_alloc(size_t bytes);         /* pinned host memory (cudaHostAlloc) */
BNM_API void bnm_host_free(void *p);

/* ---------------------------------------------------------------------------------------------
 * 4. The four kernels, batched (host pointers; n items per call, each item laid out like one reference call)
 * ------------------------------------------------------------------------------------------- */
/* activations int8 [n][n_input] -> output int32 [n][n_output]; weights = one packed layer */
BNM_API int bnm_processfclayer_batch(const int8_t *activations, const uint32_t *weights, int32_t bits_per_weight,
                                     uint32_t n_input, uint32_t n_output, int32_t *output, size_t n, int nf4_extension);
/* input int32 [n][n_input] -> output int8 [n][n_input], argmax uint32 [n] (may be NULL) */
BNM_API int bnm_relunorm_batch(const int32_t *input, int8_t *output, uint32_t *argmax, uint32_t n_input, size_t n);
/* activations int32 [n][xy*xy], weights int8 [n_w][9] with item i using weights[(i % n_w)] -> output int32 [n][(xy-2)^2] */
BNM_API int bnm_conv33relu_batch(const int32_t *activations, const int8_t *weights, uint32_t n_w, uint32_t xy_input,
                                 uint32_t n_shift, int32_t *output, size_t n);
/* activations int32 [n][xy*xy] -> output int32 [n][(xy/2)^2] */
BNM_API int bnm_maxpool22_batch(const int32_t *activations, uint32_t xy_input, int32_t *output, size_t n);

/* ---------------------------------------------------------------------------------------------
 * 5. Input quantisation, the step right before the path (the reference does it in Python per image:
 *    /root/reference/test_inference.py:140-141, BitNetMCU.py:435-436):
 *        scale = 127 / max(max|x|, 1e-5);  q = round_half_even(x * scale) clipped to [-128, 127]      (all float32)
 *    images float32 [n][elems] -> int8 [n][elems]; bit-identical to the NumPy expression.
 * ------------------------------------------------------------------------------------------- */
/* Float images straight to logits / labels (device buffers, asynchronous on `stream`): for FC models on the fused path (image rows of
 * <= 256 elements, <= 16 classes) this is ONE kernel -- four extra warps read the float rows, reduce the row maximum, quantise and write
 * the int8 rows into the shared-memory stage the tensor core reads, so a float image costs 1 024 B of HBM traffic once.  Other models:
 * the scaling kernel into a scratch buffer, then bnm_infer_batch_device.  Results are those of bnm_quantize_images + bnm_infer_batch. */
BNM_API int bnm_infer_batch_device_f32(bnm_model *m, const float *images, size_t n, int32_t *logits, uint32_t *labels, void *stream);
BNM_API int bnm_quantize_images(const float *images, size_t n, uint32_t elems, int8_t *out);                       /* host buffers */
BNM_API int bnm_quantize_images_device(const float *images, size_t n, uint32_t elems, int8_t *out, void *stream);  /* device buffers */

/* ---------------------------------------------------------------------------------------------
 * 6. Emulation mode: QuantizedModel.inference_quantized of the reference on the GPU
 *    (/root/reference/BitNetMCU.py:420-535; what exportquant.py:537-559 and test_inference.py:153-154 call per image).
 *    images float32 [n][img_bytes] (host) -> float64 [n][n_classes] (host): the emulator's logits, i.e. WITH its normalisation
 *    rules (rescale = 2^floor(log2(127/max)), np.round; per-image conv renormalisation), which differ from the C engine's by
 *    design (SURVEY.md section 4).  Exact for Binary / Ternary / 2bitsym / 4bitsym / 8bit / FP130 weights; the reference's
 *    "4bit" levels carry a +0.01 offset (BitNetMCU.py:159) and NF4 levels are non-dyadic: those two are approximated by the
 *    engine's integer weights (statistical parity only).
 * ------------------------------------------------------------------------------------------- */
BNM_API int bnm_emulate_inference_quantized(bnm_model *m, const float *images, size_t n, double *logits);

/* ---------------------------------------------------------------------------------------------
 * 7. Activation taps: the int8 rows between the layers (what the reference's printactivations() dumps, dll.c:29-37,102-109)
 *
 *    A tap is the int8 row that a ReLUNorm of BitMnistInference writes into layer_in and the next layer then reads.  Taps are
 *    numbered in chain order: for CNN models tap 0 is the C*4 features after the front-end's ReLUNorm (dll.c:80; channel-major,
 *    four pooled values per channel); then, for both model classes, one tap per hidden FC layer (every FC layer but the last,
 *    whose normalised row the reference never uses).  An FC model with L layers has L-1 taps, a CNN model L; at most 8.
 *    Tap t has
 *      width   real values: C*4 for the CNN features, the producing layer's n_out for a hidden FC row;
 *      stride  bytes between rows: round_up(C*4, 16) for the CNN features, round_up(n_in of the next layer, 32) for a hidden FC
 *              row (Ternary layers pad n_in to a multiple of 10: a 64-wide hidden row of a ternary chain has stride 96).
 *    Bytes between width and stride are unspecified (the next layer multiplies them by zero weights).
 *
 *    The _taps calls compute exactly what bnm_infer_batch[_device] computes (bit-identical logits and labels) and also store
 *    every requested tap: act[t] = int8 [n][stride of t], 16-byte aligned, or NULL when tap t is not wanted; taps == NULL or all
 *    entries NULL is the plain call.  Not for float input or the fused gather (BNM_E_UNSUPPORTED).  A taps launch is a plain
 *    launch (ordinary stream semantics) whatever BNM_OPT_LAUNCH_OVERLAP says: a debugging path, not a throughput path.
 * ------------------------------------------------------------------------------------------- */
#define BNM_MAX_TAPS 8
typedef struct bnm_taps { int8_t *act[BNM_MAX_TAPS]; } bnm_taps;   /* NULL entry = tap not wanted */
BNM_API uint32_t bnm_model_n_taps(const bnm_model *m);
BNM_API uint32_t bnm_model_tap_width(const bnm_model *m, uint32_t t);    /* 0 when t >= n_taps */
BNM_API uint32_t bnm_model_tap_stride(const bnm_model *m, uint32_t t);   /* 0 when t >= n_taps */
/* device buffers on the model's GPU, asynchronous on `stream` (as bnm_infer_batch_device) */
BNM_API int bnm_infer_batch_device_taps(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels,
                                        const bnm_taps *taps, void *stream);
/* host buffers (as bnm_infer_batch; tap rows at the same strides), one stream, chunks of BNM_OPT_CHUNK_IMAGES images */
BNM_API int bnm_infer_batch_taps(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels,
                                 const bnm_taps *taps);

#ifdef __cplusplus
}
#endif
#endif /* BITNETMCU_B200_H */
