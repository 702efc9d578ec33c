// kernels.h -- internal launch interface between the C-ABI layer (capi.cu) and the CUDA kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace bnm {

constexpr int kMaxFcLayers = 8;
constexpr int kTileM = 128;  // images per MMA tile / per CTA tile of the layer kernels
constexpr int kMaxGatherDst = 8;   // destination buffers of the fused result exchange (one box: 8 GPUs)

// destinations of the fused result exchange: layout of bnm_gather (include/bitnetmcu_b200.h)
struct GatherDst {
    uint32_t n_labels_dst, n_logits_dst;
    uint32_t *labels_dst[kMaxGatherDst];
    int32_t *logits_dst[kMaxGatherDst];
    size_t row_offset;
    uint32_t labels_u8, reserved;
};

// One fully connected layer, decoded once at model build into dense int8 planes (K3 "weight pre-decode").
struct FcLayerDev {
    int32_t enc = 0;
    uint32_t n_in = 0, n_out = 0;   // as in the model header (Lk_incoming_weights / Lk_outgoing_weights)
    uint32_t k_pad = 0;             // n_in rounded up to 32 (one tcgen05 kind::i8 K-step), zero padded
    uint32_t n_pad = 0;             // n_out rounded up to 16 (UMMA N granularity), zero padded
    int8_t *dense_a = nullptr;      // [n_pad][k_pad] row-major int8: clamp(w, -128, 127)
    int8_t *dense_b = nullptr;      // [n_pad][k_pad] residual plane w - clamp(w) (only FP130's +128), or null
    int4 *quad_a = nullptr;         // dp4a layout [(n_pad/4)][k_pad/4] of int4 = 4 outputs x 4 k (layer kernels)
    int4 *quad_b = nullptr;
};

// ---- weight decode (packed exportquant words -> dense planes); returns whether plane B is needed via *d_flag
void launch_decode_fc(const void *d_packed, int32_t enc, uint32_t n_in, uint32_t n_out, uint32_t k_pad, uint32_t n_pad,
                      int8_t *dense_a, int8_t *dense_b, int4 *quad_a, int4 *quad_b, int nf4_extension, int *d_flag,
                      cudaStream_t st);

// ---- layer-by-layer CUDA-core path (any shape)
// act int8 [n][act_stride] (zero padded to >= k_pad) -> out int32 [n][n_out]
// false: the layer needs more shared memory than an SM has (n_in above ~1.8k)
bool launch_fc_dp4a(const int8_t *act, uint32_t act_stride, const FcLayerDev &L, int32_t *out, size_t n, cudaStream_t st);
// in int32 [n][n_in] -> out int8 [n][out_stride] (zero padded), argmax uint32 [n]; out / argmax may be null
void launch_relunorm(const int32_t *in, uint32_t n_in, int8_t *out, uint32_t out_stride, uint32_t *argmax, size_t n,
                     cudaStream_t st);
void launch_conv33relu(const int32_t *act, const int8_t *w, uint32_t n_w, uint32_t xy, uint32_t n_shift, int32_t *out,
                       size_t n, cudaStream_t st);
void launch_maxpool22(const int32_t *act, uint32_t xy, int32_t *out, size_t n, cudaStream_t st);
// fused CNN front-end (dll.c:64-80): images int8 [n][256] -> features int8 [n][feat_stride] after ReLUNorm over C*4
// returns false if the geometry is not the 16x16 / conv,conv,pool,conv,pool one
// frontend: 0 = tensor-core kernel when the shape is covered, else CUDA cores; 1 = CUDA cores (k_cnn_frontend16); 2 = tensor cores only
bool launch_cnn_frontend(const int8_t *images, const int8_t *w1, const int8_t *w2, const int8_t *w3, uint32_t channels,
                         uint32_t xy, int8_t *features, uint32_t feat_stride, size_t n, int sm_count, int frontend, int *d_err,
                         bool conv3_fits_u16, cudaStream_t st);
// conv3_fits_u16: the pooled conv2 outputs (conv3's inputs) cannot exceed 65535 for this model's conv1 / conv2 weights
// (cnn_conv3_fits_u16, computed once per model): conv3 may then run on IDP.2A
bool cnn_conv3_fits_u16(const int8_t *w1, const int8_t *w2, uint32_t channels);
bool cnn_frontend_tc_supported(uint32_t channels, uint32_t xy);

// same front-end with conv1 on tcgen05 and the depthwise tail fed from TMEM (cnn_tcgen05.cu); false when the shape is not
// covered (channels not a multiple of 16, > 128, or geometry other than 16x16)
bool launch_cnn_frontend_tc(const int8_t *images, const int8_t *w1, const int8_t *w2, const int8_t *w3, uint32_t channels,
                            uint32_t xy, int8_t *features, uint32_t feat_stride, size_t n, int sm_count, int *d_err,
                            bool conv3_fits_u16, cudaStream_t st);

// emulation mode (BitNetMCU.py:420-535): normalisation rules of the reference's Python emulator, see generic_kernels.cu
void launch_relunorm_emul(const int32_t *in, uint32_t n_in, int level_shift, int8_t *out, uint32_t out_stride, size_t n, cudaStream_t st);
void launch_expand_image(const int8_t *img, int32_t *planes, uint32_t C, uint32_t elems, size_t n, cudaStream_t st);
void launch_conv_renorm(int32_t *planes, uint32_t elems_per_image, size_t n, cudaStream_t st);
void launch_i32_to_i8(const int32_t *in, uint32_t n_in, int8_t *out, uint32_t out_stride, size_t n, cudaStream_t st);

// input quantisation ahead of the path (test_inference.py:140-141): float [n][elems] -> int8 [n][elems]
void launch_quantize_images(const float *in, uint32_t elems, int8_t *out, size_t n, cudaStream_t st);

// ---- fused tcgen05 FC chain (fc_tcgen05.cu)
struct FcChainPlan;  // opaque, owned by the model
FcChainPlan *fc_chain_plan_create(const FcLayerDev *layers, int n_layers, uint32_t in_bytes, int device, int sm_count,
                                  char *err, size_t err_len);
void fc_chain_plan_destroy(FcChainPlan *p);
// 0 plain launches, 1 programmatic dependent launch (inputs read after the previous kernel completed), 2 launches declared independent
void fc_chain_plan_set_overlap(FcChainPlan *p, int mode);
// activation taps of the fused chain: act[l] = int8 [n][k_pad of layer l + 1] receiving hidden layer l's ReLUNorm rows (null: not
// wanted; bytes past the layer's n_pad are not written), l < n_layers - 1
struct FcTaps { int8_t *act[kMaxFcLayers]; };
// images int8 [n][in_bytes] (device, 16B aligned) -> logits int32 [n][n_classes], labels uint32 [n] (may be null)
// gather (may be null): extra destination buffers every row is also stored to (peer memory), fused into the epilogue
// taps (may be null; not with gather): a plain launch (mode 0) that also stores the hidden layers' rows
int fc_chain_launch(FcChainPlan *p, const int8_t *in, size_t n, int32_t *logits, uint32_t *labels, const GatherDst *gather,
                    cudaStream_t st, const FcTaps *taps = nullptr);

// float32 images [n][in_bytes] (elements) -> logits / labels with the input scaling of test_inference.py:140-141 fused into the
// kernel's load stage; supported for image rows of up to 256 elements and up to 16 classes
bool fc_chain_float_input_supported(const FcChainPlan *p);
int fc_chain_launch_f32(FcChainPlan *p, const float *in, size_t n, int32_t *logits, uint32_t *labels, cudaStream_t st);

}  // namespace bnm
