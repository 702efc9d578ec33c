// capi.cu -- the C ABI of include/bitnetmcu_b200.h: model container, batched inference (device + host
// pipelined), the four reference-named kernels and their batched forms.  No CPU compute path exists here:
// every entry needs a CUDA device and reports (or, for the reference-named symbols, aborts on) failure.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/bitnetmcu_b200.h"
#include "kernels.h"

using namespace bnm;

// -----------------------------------------------------------------------------------------------
// errors
// -----------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CU_TRY(expr)                                                                                       \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess) return fail(-100 - (int)e_, "%s failed: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

enum { BNM_E_ARG = -1, BNM_E_NODEV = -2, BNM_E_UNSUPPORTED = -3, BNM_E_CUDA = -4 };

static uint32_t round_up(uint32_t v, uint32_t m) { return (v + m - 1) / m * m; }

// -----------------------------------------------------------------------------------------------
// model
// -----------------------------------------------------------------------------------------------
struct FcLayerHost {
    int32_t enc;
    uint32_t n_in, n_out;
    void *d_packed;
    size_t packed_bytes;
};

struct PipeSlot {
    cudaStream_t stream = nullptr;
    int8_t *d_images = nullptr;
    int32_t *d_logits = nullptr;
    uint32_t *d_labels = nullptr;
    int8_t *d_feat = nullptr;    // CNN models: this slot's own feature buffer, so that the slots' chunks may overlap in time
};

struct bnm_model {
    int device = 0, sm_count = 0;
    int model_class = 0;
    uint32_t img_bytes = 256, n_classes = 0;
    std::vector<FcLayerHost> fc_host;
    std::vector<FcLayerDev> fc;
    // CNN front-end
    uint32_t channels = 0, xy0 = 0, feat_stride = 0;
    int8_t *d_conv[3] = {nullptr, nullptr, nullptr};
    // options
    int opt_path = BNM_PATH_AUTO;
    int nf4_ext = 0;
    size_t chunk_images = 1 << 16;   // host pipeline chunk
    int launch_overlap = 0;
    int cnn_frontend = 0;            // BNM_OPT_CNN_FRONTEND
    bool conv3_fits_u16 = false;     // static range of conv3's inputs for this model's weights (cnn_conv3_fits_u16)
    std::vector<int8_t> h_conv[3];   // host copies of the conv weights (range analysis)
    int *d_err = nullptr;            // error word of the bounded device-side waits
    // fused plan
    FcChainPlan *plan = nullptr;
    std::string plan_err;
    // device scratch (grow-only): layered path accumulators / activations, CNN features
    size_t scratch_n = 0;
    int32_t *d_acc = nullptr;
    int8_t *d_act[2] = {nullptr, nullptr};
    int8_t *d_feat = nullptr;
    uint32_t max_kpad = 0, max_nout = 0;
    // host pipeline
    PipeSlot slots[3];
    size_t slot_n = 0;
    // small-batch path of bnm_infer_batch (the reference's own calling pattern: one image per Inference() call,
    // test_inference.py:146-150): pinned staging buffers, one stream, one synchronisation
    int8_t *small_h_in = nullptr, *small_d_in = nullptr;     // [kSmallBatch][img_bytes]
    int32_t *small_h_out = nullptr, *small_d_out = nullptr;  // logits [n][n_classes] then labels [n]
    int8_t *d_f32_scratch = nullptr;   // bnm_infer_batch_device_f32 fallback: quantised images
    size_t f32_scratch_n = 0;
    int small_zero_copy = 1;   // 0: H2D + D2H copies; 1 (default, measured fastest: 14.3 vs 20.1 / 16.8 us per call): the kernel writes results
                               // straight into mapped pinned host memory; 2: ... and reads the images from it (TMA over PCIe)
};
static const size_t kSmallBatch = 1024;

static void free_fc_dev(bnm_model *m) {
    for (auto &L : m->fc) {
        cudaFree(L.dense_a);
        cudaFree(L.dense_b);
        cudaFree(L.quad_a);
        cudaFree(L.quad_b);
    }
    m->fc.clear();
    if (m->plan) fc_chain_plan_destroy(m->plan);
    m->plan = nullptr;
}

static int effective_overlap(const bnm_model *m) {
    // the CNN front-end writes the features the FC kernel reads: there the dependency is real, never declare it away
    return m->model_class == BNM_MODEL_CNNMNIST && m->launch_overlap == 2 ? 1 : m->launch_overlap;
}

// decode all FC layers into int8 planes and (re)build the fused plan
static int build_fc_dev(bnm_model *m) {
    free_fc_dev(m);
    int *d_flag = nullptr;
    CU_TRY(cudaMalloc(&d_flag, sizeof(int)));
    m->max_kpad = round_up(std::max(m->img_bytes, m->feat_stride), 32);
    m->max_nout = 0;
    for (auto &H : m->fc_host) {
        FcLayerDev L;
        L.enc = H.enc;
        L.n_in = H.n_in;
        L.n_out = H.n_out;
        L.k_pad = round_up(H.n_in, 32);
        L.n_pad = round_up(H.n_out, 16);
        size_t plane = (size_t)L.k_pad * L.n_pad;
        int flag = 0;
        cudaError_t e = cudaMalloc(&L.dense_a, plane);
        if (e == cudaSuccess) e = cudaMalloc(&L.dense_b, plane);
        if (e == cudaSuccess) e = cudaMalloc(&L.quad_a, plane);
        if (e == cudaSuccess) e = cudaMalloc(&L.quad_b, plane);
        if (e == cudaSuccess) e = cudaMemset(d_flag, 0, sizeof(int));
        if (e == cudaSuccess) {
            launch_decode_fc(H.d_packed, H.enc, H.n_in, H.n_out, L.k_pad, L.n_pad, L.dense_a, L.dense_b, L.quad_a, L.quad_b,
                             m->nf4_ext, d_flag, 0);
            e = cudaMemcpy(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost);
        }
        if (e != cudaSuccess) {   // nothing half-built stays behind
            cudaFree(L.dense_a); cudaFree(L.dense_b); cudaFree(L.quad_a); cudaFree(L.quad_b);
            cudaFree(d_flag);
            free_fc_dev(m);
            return fail(BNM_E_CUDA, "weight decode of an FC layer failed: %s", cudaGetErrorString(e));
        }
        if (!flag) {   // no residual plane needed (everything but FP130 layers that contain +128)
            cudaFree(L.dense_b);
            cudaFree(L.quad_b);
            L.dense_b = nullptr;
            L.quad_b = nullptr;
        }
        m->max_kpad = std::max(m->max_kpad, L.k_pad);
        m->max_nout = std::max(m->max_nout, L.n_out);
        m->fc.push_back(L);
    }
    cudaFree(d_flag);
    m->n_classes = m->fc.back().n_out;
    // fused plan (may legitimately be unavailable for exotic shapes: the layered path then serves the model)
    char err[256] = {0};
    uint32_t in_bytes = m->model_class == BNM_MODEL_CNNMNIST ? m->feat_stride : m->img_bytes;
    m->plan = fc_chain_plan_create(m->fc.data(), (int)m->fc.size(), in_bytes, m->device, m->sm_count, err, sizeof(err));
    m->plan_err = err;
    fc_chain_plan_set_overlap(m->plan, effective_overlap(m));
    // scratch must be re-sized for the new widths
    m->scratch_n = 0;
    return 0;
}

static int ensure_scratch(bnm_model *m, size_t n, bool layered) {
    if (n <= m->scratch_n && (!layered || m->d_acc)) return 0;
    n = std::max(n, m->scratch_n);
    cudaFree(m->d_acc);
    cudaFree(m->d_act[0]);
    cudaFree(m->d_act[1]);
    cudaFree(m->d_feat);
    m->d_acc = nullptr; m->d_act[0] = m->d_act[1] = nullptr; m->d_feat = nullptr;
    m->scratch_n = 0;
    if (layered) {   // int32 accumulators + ping-pong int8 activations of the layer-by-layer path; the fused path needs neither
        CU_TRY(cudaMalloc(&m->d_acc, n * (size_t)std::max(m->max_nout, 1u) * sizeof(int32_t)));
        for (int i = 0; i < 2; i++) {
            CU_TRY(cudaMalloc(&m->d_act[i], n * (size_t)m->max_kpad));
            CU_TRY(cudaMemset(m->d_act[i], 0, n * (size_t)m->max_kpad));
        }
    }
    if (m->model_class == BNM_MODEL_CNNMNIST) {
        CU_TRY(cudaMalloc(&m->d_feat, n * (size_t)m->feat_stride));
        CU_TRY(cudaMemset(m->d_feat, 0, n * (size_t)m->feat_stride));
    }
    m->scratch_n = n;
    return 0;
}

static int require_device_index(int device);
extern "C" int bnm_version(void) { return BNM_VERSION; }
extern "C" const char *bnm_last_error(void) { return g_err.c_str(); }
extern "C" int bnm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int bnm_model_create(int model_class, const bnm_layer *layers, uint32_t n_layers, uint32_t img_bytes, int device,
                                bnm_model **out) {
    if (!out || !layers || n_layers == 0) return fail(BNM_E_ARG, "bnm_model_create: null argument");
    *out = nullptr;
    if (model_class != BNM_MODEL_FCMNIST && model_class != BNM_MODEL_CNNMNIST)
        return fail(BNM_E_ARG, "unknown model class %d (expected MODEL_FCMNIST=0 / MODEL_CNNMNIST=1)", model_class);
    int ndev = bnm_device_count();
    if (ndev == 0) return fail(BNM_E_NODEV, "no CUDA device: this engine has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(BNM_E_ARG, "device %d out of range (have %d)", device, ndev);
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(BNM_E_UNSUPPORTED, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);

    bnm_model *m = new bnm_model();
    m->device = device;
    m->sm_count = prop.multiProcessorCount;
    m->model_class = model_class;
    m->img_bytes = img_bytes ? img_bytes : 256;
    int rc = 0;
    uint32_t n_conv = 0;
    std::vector<uint32_t> front;   // kinds of the non-FC layers, in order
    for (uint32_t i = 0; i < n_layers && rc == 0; i++) {
        const bnm_layer &L = layers[i];
        if (L.kind == BNM_LAYER_FC) {
            if (!L.weights || L.n_in == 0 || L.n_out == 0) { rc = fail(BNM_E_ARG, "FC layer %u: empty", i); break; }
            // the reference reads n_out * ceil(n_in/wpw) words (ternary: n_out*(n_in/10) uint16) -- inference.c:88-208
            size_t need = 0;
            switch (L.bitperweight) {
            case BNM_ENC_BINARY: need = (size_t)L.n_out * ((L.n_in + 31) / 32) * 4; break;
            case BNM_ENC_2BITSYM: need = (size_t)L.n_out * ((L.n_in + 15) / 16) * 4; break;
            case BNM_ENC_4BITSYM: case BNM_ENC_4BIT: case BNM_ENC_FP130: case BNM_ENC_NF4: need = (size_t)L.n_out * ((L.n_in + 7) / 8) * 4; break;
            case BNM_ENC_8BIT: need = (size_t)L.n_out * ((L.n_in + 3) / 4) * 4; break;
            case BNM_ENC_TERNARY: need = (size_t)L.n_out * (L.n_in / 10) * 2; break;
            default: need = 0; break;   // unknown id: decoded as zeros like inference.c:202, nothing is read
            }
            if (L.weight_bytes < need) { rc = fail(BNM_E_ARG, "FC layer %u: %zu weight bytes, reference reads %zu", i, L.weight_bytes, need); break; }
            FcLayerHost H{L.bitperweight, L.n_in, L.n_out, nullptr, std::max<size_t>(need, 16)};
            if (cudaMalloc(&H.d_packed, H.packed_bytes + 16) != cudaSuccess) { rc = fail(BNM_E_CUDA, "cudaMalloc failed"); break; }
            cudaMemset(H.d_packed, 0, H.packed_bytes + 16);
            if (need) cudaMemcpy(H.d_packed, L.weights, need, cudaMemcpyHostToDevice);
            m->fc_host.push_back(H);
        } else if (L.kind == BNM_LAYER_CONV33) {
            front.push_back(L.kind);
            if (n_conv == 3) { rc = fail(BNM_E_UNSUPPORTED, "more than three conv layers"); break; }
            if (!L.weights || L.weight_bytes < (size_t)L.n_out * 9) { rc = fail(BNM_E_ARG, "conv layer %u: needs %u int8 weights", i, L.n_out * 9); break; }
            if (n_conv == 0) { m->channels = L.n_out; m->xy0 = L.n_in; }
            else if (L.n_out != m->channels) { rc = fail(BNM_E_UNSUPPORTED, "conv layers must share the channel count (dll.c:66)"); break; }
            if (cudaMalloc(&m->d_conv[n_conv], (size_t)L.n_out * 9) != cudaSuccess) { rc = fail(BNM_E_CUDA, "cudaMalloc failed"); break; }
            cudaMemcpy(m->d_conv[n_conv], L.weights, (size_t)L.n_out * 9, cudaMemcpyHostToDevice);
            m->h_conv[n_conv].assign(static_cast<const int8_t *>(L.weights), static_cast<const int8_t *>(L.weights) + (size_t)L.n_out * 9);
            n_conv++;
        } else if (L.kind == BNM_LAYER_MAXPOOL22) {
            front.push_back(L.kind);
        } else {
            rc = fail(BNM_E_ARG, "layer %u: unknown kind %u", i, L.kind);
        }
    }
    if (rc == 0 && (m->fc_host.empty() || m->fc_host.size() > (size_t)kMaxFcLayers)) rc = fail(BNM_E_UNSUPPORTED, "model needs 1..%d FC layers", kMaxFcLayers);
    if (rc == 0 && model_class == BNM_MODEL_CNNMNIST) {
        const uint32_t want[5] = {BNM_LAYER_CONV33, BNM_LAYER_CONV33, BNM_LAYER_MAXPOOL22, BNM_LAYER_CONV33, BNM_LAYER_MAXPOOL22};
        if (front.size() != 5 || memcmp(front.data(), want, sizeof(want)) != 0)
            rc = fail(BNM_E_UNSUPPORTED, "CNN front-end must be conv,conv,pool,conv,pool (BitNetMCU_MNIST_dll.c:64-80)");
        else if (m->xy0 != 16 || m->img_bytes != 256)
            rc = fail(BNM_E_UNSUPPORTED, "CNN input must be 16x16 int8 (the reference hard-codes it, BitNetMCU_MNIST_dll.c:68)");
        else {
            uint32_t f = ((m->xy0 - 4) / 2 - 2) / 2;   // 16 -> 2
            m->feat_stride = round_up(m->channels * f * f, 16);
            m->conv3_fits_u16 = cnn_conv3_fits_u16(m->h_conv[0].data(), m->h_conv[1].data(), m->channels);
        }
    }
    if (rc == 0 && model_class == BNM_MODEL_FCMNIST && !front.empty()) rc = fail(BNM_E_ARG, "MODEL_FCMNIST with conv/pool layers");
    if (rc == 0) rc = build_fc_dev(m);
    if (rc == 0 && (cudaMalloc(&m->d_err, sizeof(int)) != cudaSuccess || cudaMemset(m->d_err, 0, sizeof(int)) != cudaSuccess)) rc = fail(BNM_E_CUDA, "cudaMalloc failed");
    if (rc == 0) {
        if (const char *e = getenv("BNM_CNN_FRONTEND")) m->cnn_frontend = std::max(0, std::min(2, atoi(e)));   // development override, read once per model
        for (auto &s : m->slots)
            if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) { rc = fail(BNM_E_CUDA, "cudaStreamCreate failed"); break; }
    }
    if (rc != 0) { std::string keep = g_err; bnm_model_destroy(m); g_err = keep; return rc; }
    *out = m;
    return 0;
}

extern "C" int bnm_model_load_blob(const void *blob, size_t bytes, int device, bnm_model **out) {
    // layout written by bitnetmcu_b200.model.Model.to_blob(): "BNM1" | class | n_layers | img_bytes | table | data
    if (!blob || bytes < 16 || memcmp(blob, "BNM1", 4) != 0) return fail(BNM_E_ARG, "not a BNM1 model blob");
    const uint8_t *b = static_cast<const uint8_t *>(blob);
    uint32_t hdr[3];
    memcpy(hdr, b + 4, 12);
    const uint32_t cls = hdr[0], n_layers = hdr[1], img_bytes = hdr[2];
    if (n_layers == 0 || n_layers > 64 || 16 + (size_t)n_layers * 32 > bytes) return fail(BNM_E_ARG, "corrupt model blob (layer table)");
    std::vector<bnm_layer> layers(n_layers);
    for (uint32_t i = 0; i < n_layers; i++) {
        uint32_t e[8];
        memcpy(e, b + 16 + (size_t)i * 32, 32);
        if ((size_t)e[6] + e[7] > bytes) return fail(BNM_E_ARG, "corrupt model blob (layer %u data)", i);
        layers[i] = bnm_layer{e[0], (int32_t)e[1], e[2], e[3], e[4], e[5], e[7] ? b + e[6] : nullptr, e[7]};
    }
    return bnm_model_create((int)cls, layers.data(), n_layers, img_bytes, device, out);
}

extern "C" void bnm_model_destroy(bnm_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    free_fc_dev(m);
    for (auto &H : m->fc_host) cudaFree(H.d_packed);
    for (auto &p : m->d_conv) cudaFree(p);
    cudaFree(m->d_acc);
    cudaFree(m->d_act[0]);
    cudaFree(m->d_act[1]);
    cudaFree(m->d_feat);
    cudaFree(m->d_err);
    cudaFree(m->small_d_in);
    cudaFree(m->small_d_out);
    cudaFree(m->d_f32_scratch);
    if (m->small_h_in) cudaFreeHost(m->small_h_in);
    if (m->small_h_out) cudaFreeHost(m->small_h_out);
    for (auto &s : m->slots) {
        cudaFree(s.d_images);
        cudaFree(s.d_logits);
        cudaFree(s.d_labels);
        cudaFree(s.d_feat);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    delete m;
}

extern "C" uint32_t bnm_model_n_classes(const bnm_model *m) { return m ? m->n_classes : 0; }
extern "C" uint32_t bnm_model_img_bytes(const bnm_model *m) { return m ? m->img_bytes : 0; }

extern "C" int bnm_model_active_path(const bnm_model *m) {
    if (!m) return 0;
    if (m->opt_path == BNM_PATH_LAYERS) return BNM_PATH_LAYERS;
    return m->plan ? BNM_PATH_TCGEN05 : BNM_PATH_LAYERS;
}

extern "C" int bnm_model_set_option(bnm_model *m, int option, int64_t value) {
    if (!m) return fail(BNM_E_ARG, "null model");
    CU_TRY(cudaSetDevice(m->device));
    switch (option) {
    case BNM_OPT_PATH:
        if (value < BNM_PATH_AUTO || value > BNM_PATH_TCGEN05) return fail(BNM_E_ARG, "bad path %lld", (long long)value);
        if (value == BNM_PATH_TCGEN05 && !m->plan) return fail(BNM_E_UNSUPPORTED, "fused tcgen05 path unavailable for this model: %s", m->plan_err.c_str());
        m->opt_path = (int)value;
        return 0;
    case BNM_OPT_NF4_EXTENSION:
        if ((value != 0) == (m->nf4_ext != 0)) return 0;
        m->nf4_ext = value != 0;
        CU_TRY(cudaDeviceSynchronize());
        return build_fc_dev(m);
    case BNM_OPT_CHUNK_IMAGES:
        if (value < 128) return fail(BNM_E_ARG, "chunk must be >= 128 images");
        m->chunk_images = (size_t)value;
        return 0;
    case BNM_OPT_CNN_FRONTEND:
        if (value < 0 || value > 2) return fail(BNM_E_ARG, "CNN front-end must be 0 (auto), 1 (CUDA cores) or 2 (tensor cores)");
        if (value == 2 && !(m->model_class == BNM_MODEL_CNNMNIST && cnn_frontend_tc_supported(m->channels, m->xy0)))
            return fail(BNM_E_UNSUPPORTED, "tensor-core CNN front-end needs a 16x16 CNN model with a multiple of 16 (<= 128) channels");
        m->cnn_frontend = (int)value;
        return 0;
    case BNM_OPT_LAUNCH_OVERLAP:
        if (value < 0 || value > 2) return fail(BNM_E_ARG, "launch overlap mode must be 0, 1 or 2");
        m->launch_overlap = (int)value;
        fc_chain_plan_set_overlap(m->plan, effective_overlap(m));
        return 0;
    default:
        return fail(BNM_E_ARG, "unknown option %d", option);
    }
}
extern "C" int64_t bnm_model_get_option(const bnm_model *m, int option) {
    if (!m) return -1;
    switch (option) {
    case BNM_OPT_PATH: return m->opt_path;
    case BNM_OPT_NF4_EXTENSION: return m->nf4_ext;
    case BNM_OPT_CHUNK_IMAGES: return (int64_t)m->chunk_images;
    case BNM_OPT_LAUNCH_OVERLAP: return m->launch_overlap;
    case BNM_OPT_CNN_FRONTEND: return m->cnn_frontend;
    default: return -1;
    }
}

// -----------------------------------------------------------------------------------------------
// batched inference, device pointers
// -----------------------------------------------------------------------------------------------
static const size_t kLayeredChunk = 1 << 17;   // images per pass of the layer-by-layer path (bounds its scratch)
static const size_t kFusedCnnChunk = 1 << 20;  // fused path, CNN models: images per front-end + FC launch pair (256 B of features each)

// FC chain, one CUDA-core kernel per layer: input int8 [n][in_stride].  taps (may be null): a requested hidden row is written
// straight into its tap buffer (at the next layer's k_pad, the stride the next layer reads) instead of the ping-pong scratch.
static int run_fc_layers(bnm_model *m, const int8_t *in, uint32_t in_stride, size_t n, int32_t *logits, uint32_t *labels, cudaStream_t st,
                         const FcTaps *taps = nullptr) {
    const int8_t *act = in;
    uint32_t stride = in_stride;
    const size_t nl = m->fc.size();
    for (size_t l = 0; l < nl; l++) {
        const bool last = l + 1 == nl;
        int32_t *acc = last ? logits : m->d_acc;
        if (!launch_fc_dp4a(act, stride, m->fc[l], acc, n, st))
            return fail(BNM_E_UNSUPPORTED, "FC layer %zu: %u inputs need more shared memory than an SM has (layer kernel stages 128 rows)", l, m->fc[l].n_in);
        if (last) {
            if (labels) launch_relunorm(acc, m->fc[l].n_out, nullptr, 0, labels, n, st);
        } else {
            int8_t *next = taps && taps->act[l] ? taps->act[l] : m->d_act[l & 1];
            uint32_t next_stride = m->fc[l + 1].k_pad;
            launch_relunorm(acc, m->fc[l].n_out, next, next_stride, nullptr, n, st);
            act = next;
            stride = next_stride;
        }
    }
    return 0;
}

// CNN front-end into feat (int8 [n][feat_stride])
static int run_cnn_front(bnm_model *m, const int8_t *images, size_t n, int8_t *feat, cudaStream_t st) {
    if (launch_cnn_frontend(images, m->d_conv[0], m->d_conv[1], m->d_conv[2], m->channels, m->xy0, feat, m->feat_stride, n,
                            m->sm_count, m->cnn_frontend, m->d_err, m->conv3_fits_u16, st))
        return 0;
    return fail(BNM_E_UNSUPPORTED, "CNN front-end: %u channels at %ux%u not supported by the selected kernel (the reference hard-codes 16x16, dll.c:68)",
                m->channels, m->xy0, m->xy0);
}

extern "C" int bnm_infer_launch_count(const bnm_model *m, size_t n) {
    if (!m || n == 0) return 0;
    const bool fused = bnm_model_active_path(m) == BNM_PATH_TCGEN05;
    const bool cnn = m->model_class == BNM_MODEL_CNNMNIST;
    if (fused && !cnn) return 1;
    const size_t chunk_images = fused ? kFusedCnnChunk : kLayeredChunk;
    size_t chunks = (n + chunk_images - 1) / chunk_images;
    int per = cnn ? 1 : 0;
    per += fused ? 1 : (int)(2 * m->fc.size());   // fc + relunorm per layer (last relunorm = labels)
    return (int)(chunks * per);
}

static uint32_t n_taps(const bnm_model *m) { return (uint32_t)m->fc.size() - 1 + (m->model_class == BNM_MODEL_CNNMNIST ? 1 : 0); }
static uint32_t tap_stride(const bnm_model *m, uint32_t t) {
    const uint32_t t0 = m->model_class == BNM_MODEL_CNNMNIST ? 1 : 0;
    return t < t0 ? m->feat_stride : m->fc[t - t0 + 1].k_pad;
}

// slot_feat: a caller-owned feature buffer for n images (the host pipeline's per-slot buffers); null = the model's own scratch
// taps: checked by check_taps, at least one entry set (null: none)
static int infer_device_impl(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels, const GatherDst *gather, void *stream,
                             int8_t *slot_feat = nullptr, const bnm_taps *taps = nullptr) {
    if (!m || (n && (!images || !logits))) return fail(BNM_E_ARG, "bnm_infer_batch_device: null argument");
    if (n == 0) return 0;
    if ((uintptr_t)images & 15) return fail(BNM_E_ARG, "the device image buffer must be 16-byte aligned (TMA)");
    if ((uintptr_t)logits & 7) return fail(BNM_E_ARG, "the device logits buffer must be 8-byte aligned (64-bit row stores)");
    CU_TRY(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool fused = bnm_model_active_path(m) == BNM_PATH_TCGEN05;
    const bool cnn = m->model_class == BNM_MODEL_CNNMNIST;
    if (gather && !fused) return fail(BNM_E_UNSUPPORTED, "the fused result exchange needs the tcgen05 path (model: %s)", m->plan_err.c_str());
    if (gather && taps) return fail(BNM_E_UNSUPPORTED, "activation taps are not available with the fused result exchange");
    const uint32_t t0 = cnn ? 1 : 0;   // FC layer l's row is tap t0 + l
    // FC taps of the images from row b on
    auto fc_taps_at = [&](size_t b, FcTaps &ft) -> const FcTaps * {
        if (!taps) return nullptr;
        for (size_t l = 0; l < (size_t)kMaxFcLayers; l++) {
            const uint32_t t = t0 + (uint32_t)l;
            ft.act[l] = l + 1 < m->fc.size() && taps->act[t] ? taps->act[t] + b * tap_stride(m, t) : nullptr;
        }
        return &ft;
    };
    FcTaps ft;
    if (fused && !cnn) {
        int rc = fc_chain_launch(m->plan, images, n, logits, labels, gather, st, fc_taps_at(0, ft));
        return rc ? fail(BNM_E_CUDA, "fused FC kernel launch failed (%d): %s", rc, cudaGetErrorString(cudaGetLastError())) : 0;
    }
    const size_t chunk = slot_feat ? n : std::min(n, fused ? kFusedCnnChunk : kLayeredChunk);
    int rc = (slot_feat && fused) ? 0 : ensure_scratch(m, chunk, !fused);
    if (rc) return rc;
    int8_t *feat = slot_feat ? slot_feat : m->d_feat;
    for (size_t b = 0; b < n; b += chunk) {
        const size_t nb = std::min(chunk, n - b);
        const int8_t *img = images + b * m->img_bytes;
        int32_t *lg = logits + b * m->n_classes;
        uint32_t *lb = labels ? labels + b : nullptr;
        const int8_t *fc_in = img;
        uint32_t fc_stride = m->img_bytes;
        if (cnn) {
            // tap 0 requested: the front-end writes the features straight into it and the FC chain reads them from there
            int8_t *f = taps && taps->act[0] ? taps->act[0] + b * m->feat_stride : feat;
            rc = run_cnn_front(m, img, nb, f, st);
            if (rc) return rc;
            fc_in = f;
            fc_stride = m->feat_stride;
        }
        if (fused) {
            GatherDst gchunk;
            if (gather) { gchunk = *gather; gchunk.row_offset += b; }
            rc = fc_chain_launch(m->plan, fc_in, nb, lg, lb, gather ? &gchunk : nullptr, st, fc_taps_at(b, ft));
            if (rc) return fail(BNM_E_CUDA, "fused FC kernel launch failed (%d)", rc);
        } else {
            rc = run_fc_layers(m, fc_in, fc_stride, nb, lg, lb, st, fc_taps_at(b, ft));
            if (rc) return rc;
        }
    }
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail(BNM_E_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

extern "C" int bnm_infer_batch_device(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels, void *stream) {
    return infer_device_impl(m, images, n, logits, labels, nullptr, stream);
}

extern "C" int bnm_infer_batch_device_gather(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels,
                                             const bnm_gather *gather, void *stream) {
    static_assert(sizeof(bnm_gather) == sizeof(GatherDst), "bnm_gather and GatherDst must share their layout");
    if (gather && (gather->n_labels_dst > BNM_MAX_GATHER_DST || gather->n_logits_dst > BNM_MAX_GATHER_DST))
        return fail(BNM_E_ARG, "at most %d gather destinations", BNM_MAX_GATHER_DST);
    if (gather)
        for (uint32_t d = 0; d < gather->n_logits_dst; d++)
            if ((uintptr_t)gather->logits_dst[d] & 7) return fail(BNM_E_ARG, "gather logits buffers must be 8-byte aligned");
    return infer_device_impl(m, images, n, logits, labels, reinterpret_cast<const GatherDst *>(gather), stream);
}

// -----------------------------------------------------------------------------------------------
// activation taps (section 7 of the header)
// -----------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16) == cudaSuccess ? 0 : -1; }
    template <class T> T *as() { return static_cast<T *>(p); }
};

extern "C" uint32_t bnm_model_n_taps(const bnm_model *m) { return m ? n_taps(m) : 0; }
extern "C" uint32_t bnm_model_tap_width(const bnm_model *m, uint32_t t) {
    if (!m || t >= n_taps(m)) return 0;
    const uint32_t t0 = m->model_class == BNM_MODEL_CNNMNIST ? 1 : 0;
    return t < t0 ? m->channels * 4 : m->fc[t - t0].n_out;
}
extern "C" uint32_t bnm_model_tap_stride(const bnm_model *m, uint32_t t) { return m && t < n_taps(m) ? tap_stride(m, t) : 0; }

// 0: taps usable for this call; *any = some entry is set
static int check_taps(const bnm_model *m, const bnm_taps *taps, bool device, bool *any) {
    *any = false;
    if (!taps) return 0;
    const uint32_t nt = n_taps(m);
    for (uint32_t t = 0; t < BNM_MAX_TAPS; t++) {
        if (!taps->act[t]) continue;
        if (t >= nt) return fail(BNM_E_ARG, "tap %u requested, the model has %u taps", t, nt);
        if (device && ((uintptr_t)taps->act[t] & 15)) return fail(BNM_E_ARG, "tap %u: the device buffer must be 16-byte aligned", t);
        *any = true;
    }
    // the fused kernel stores a hidden row n_pad = round_up(n_out, 16) bytes wide: it has to fit the stride the next layer reads
    const uint32_t t0 = m->model_class == BNM_MODEL_CNNMNIST ? 1 : 0;
    for (uint32_t t = t0; *any && t < nt; t++)
        if (taps->act[t] && m->fc[t - t0].n_pad > tap_stride(m, t))
            return fail(BNM_E_UNSUPPORTED, "tap %u: FC layer %u has %u outputs, the next layer reads %u", t, t - t0, m->fc[t - t0].n_out,
                        m->fc[t - t0 + 1].n_in);
    return 0;
}

extern "C" int bnm_infer_batch_device_taps(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels,
                                           const bnm_taps *taps, void *stream) {
    static_assert(BNM_MAX_TAPS == kMaxFcLayers, "a CNN model with 8 FC layers has 8 taps");
    if (!m) return fail(BNM_E_ARG, "bnm_infer_batch_device_taps: null model");
    bool any = false;
    if (int rc = check_taps(m, taps, true, &any)) return rc;
    return infer_device_impl(m, images, n, logits, labels, nullptr, stream, nullptr, any ? taps : nullptr);
}

extern "C" int bnm_infer_batch_taps(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels, const bnm_taps *taps) {
    if (!m) return fail(BNM_E_ARG, "bnm_infer_batch_taps: null model");
    bool any = false;
    if (int rc = check_taps(m, taps, false, &any)) return rc;
    if (!any) return bnm_infer_batch(m, images, n, logits, labels);
    if (n && (!images || !logits)) return fail(BNM_E_ARG, "bnm_infer_batch_taps: null argument");
    if (n == 0) return 0;
    CU_TRY(cudaSetDevice(m->device));
    const size_t chunk = std::min(n, m->chunk_images);
    const uint32_t nt = n_taps(m);
    DevBuf d_img, d_log, d_lab, d_tap[BNM_MAX_TAPS];
    bnm_taps dt{};
    if (d_img.alloc(chunk * m->img_bytes) || d_log.alloc(chunk * m->n_classes * sizeof(int32_t)) || d_lab.alloc(chunk * sizeof(uint32_t)))
        return fail(BNM_E_CUDA, "cudaMalloc failed");
    for (uint32_t t = 0; t < nt; t++) {
        if (!taps->act[t]) continue;
        if (d_tap[t].alloc(chunk * tap_stride(m, t))) return fail(BNM_E_CUDA, "cudaMalloc failed");
        dt.act[t] = d_tap[t].as<int8_t>();
    }
    cudaStream_t st = m->slots[0].stream;
    for (size_t b = 0; b < n; b += chunk) {
        const size_t nb = std::min(chunk, n - b);
        CU_TRY(cudaMemcpyAsync(d_img.p, images + b * m->img_bytes, nb * m->img_bytes, cudaMemcpyHostToDevice, st));
        int rc = infer_device_impl(m, d_img.as<int8_t>(), nb, d_log.as<int32_t>(), labels ? d_lab.as<uint32_t>() : nullptr, nullptr, st, nullptr, &dt);
        if (rc) { cudaStreamSynchronize(st); return rc; }
        CU_TRY(cudaMemcpyAsync(logits + b * m->n_classes, d_log.p, nb * m->n_classes * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        if (labels) CU_TRY(cudaMemcpyAsync(labels + b, d_lab.p, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        for (uint32_t t = 0; t < nt; t++)
            if (dt.act[t])
                CU_TRY(cudaMemcpyAsync(taps->act[t] + b * tap_stride(m, t), dt.act[t], nb * tap_stride(m, t), cudaMemcpyDeviceToHost, st));
    }
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

// -----------------------------------------------------------------------------------------------
// peer memory plumbing for the fused result exchange: cudaMalloc'd buffers exported / opened through CUDA IPC
// -----------------------------------------------------------------------------------------------
extern "C" int bnm_device_alloc(int device, size_t bytes, void **out) {
    if (!out) return fail(BNM_E_ARG, "bnm_device_alloc: null argument");
    *out = nullptr;
    if (int rc = require_device_index(device)) return rc;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaMalloc(out, bytes ? bytes : 16));
    return 0;
}
extern "C" void bnm_device_free(void *p) { if (p) cudaFree(p); }
extern "C" int bnm_ipc_export(const void *dev_ptr, void *handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    if (!dev_ptr || !handle64) return fail(BNM_E_ARG, "bnm_ipc_export: null argument");
    cudaIpcMemHandle_t h;
    CU_TRY(cudaIpcGetMemHandle(&h, const_cast<void *>(dev_ptr)));
    memcpy(handle64, &h, 64);
    return 0;
}
extern "C" int bnm_ipc_open(int device, const void *handle64, void **out) {
    if (!handle64 || !out) return fail(BNM_E_ARG, "bnm_ipc_open: null argument");
    *out = nullptr;
    if (int rc = require_device_index(device)) return rc;
    CU_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    CU_TRY(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
extern "C" int bnm_ipc_close(void *p) {
    if (!p) return 0;
    CU_TRY(cudaIpcCloseMemHandle(p));
    return 0;
}
// same-process multi-GPU callers: let `device` read / write memory of `peer` directly
extern "C" int bnm_enable_peer_access(int device, int peer) {
    if (int rc = require_device_index(device)) return rc;
    if (int rc = require_device_index(peer)) return rc;
    if (device == peer) return 0;
    int can = 0;
    CU_TRY(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) return fail(BNM_E_UNSUPPORTED, "device %d cannot access device %d (no P2P path)", device, peer);
    CU_TRY(cudaSetDevice(device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return 0; }
    CU_TRY(e);
    return 0;
}

// -----------------------------------------------------------------------------------------------
// batched inference, host pointers: chunks round-robin over three streams so H2D, kernels and D2H overlap
// -----------------------------------------------------------------------------------------------
// n <= kSmallBatch images: staging buffers allocated once, one stream, one synchronisation per call
static int infer_small(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels) {
    const size_t in_bytes = kSmallBatch * (size_t)m->img_bytes, out_ints = kSmallBatch * ((size_t)m->n_classes + 1);
    if (!m->small_h_in) {
        if (const char *e = getenv("BNM_SMALL_ZC")) m->small_zero_copy = std::max(0, std::min(2, atoi(e)));   // development knob, read once per model
        CU_TRY(cudaHostAlloc(reinterpret_cast<void **>(&m->small_h_in), in_bytes, cudaHostAllocMapped));
        CU_TRY(cudaHostAlloc(reinterpret_cast<void **>(&m->small_h_out), out_ints * 4, cudaHostAllocMapped));
        CU_TRY(cudaMalloc(&m->small_d_in, in_bytes));
        CU_TRY(cudaMalloc(&m->small_d_out, out_ints * 4));
    }
    cudaStream_t st = m->slots[0].stream;
    memcpy(m->small_h_in, images, n * (size_t)m->img_bytes);
    const int8_t *d_in = m->small_d_in;
    int32_t *d_out = m->small_d_out;
    if (m->small_zero_copy >= 2) CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(const_cast<int8_t **>(&d_in)), m->small_h_in, 0));
    else CU_TRY(cudaMemcpyAsync(m->small_d_in, m->small_h_in, n * (size_t)m->img_bytes, cudaMemcpyHostToDevice, st));
    if (m->small_zero_copy >= 1) CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(&d_out), m->small_h_out, 0));
    const size_t n_log = n * (size_t)m->n_classes;
    uint32_t *d_lab = reinterpret_cast<uint32_t *>(d_out + n_log);
    int rc = bnm_infer_batch_device(m, d_in, n, d_out, labels ? d_lab : nullptr, st);
    if (rc) return rc;
    if (m->small_zero_copy == 0) CU_TRY(cudaMemcpyAsync(m->small_h_out, m->small_d_out, (n_log + (labels ? n : 0)) * 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    memcpy(logits, m->small_h_out, n_log * 4);
    if (labels) memcpy(labels, m->small_h_out + n_log, n * 4);
    return 0;
}

extern "C" int bnm_infer_batch(bnm_model *m, const int8_t *images, size_t n, int32_t *logits, uint32_t *labels) {
    if (!m || (n && (!images || !logits))) return fail(BNM_E_ARG, "bnm_infer_batch: null argument");
    if (n == 0) return 0;
    CU_TRY(cudaSetDevice(m->device));
    if (n <= kSmallBatch && n <= m->chunk_images) return infer_small(m, images, n, logits, labels);
    const size_t chunk = std::min(n, m->chunk_images);
    if (m->slot_n < chunk) {
        CU_TRY(cudaDeviceSynchronize());
        for (auto &s : m->slots) {
            cudaFree(s.d_images); cudaFree(s.d_logits); cudaFree(s.d_labels); cudaFree(s.d_feat);
            s.d_images = nullptr; s.d_logits = nullptr; s.d_labels = nullptr; s.d_feat = nullptr;
            if (m->model_class == BNM_MODEL_CNNMNIST) {
                CU_TRY(cudaMalloc(&s.d_feat, chunk * (size_t)m->feat_stride));
                CU_TRY(cudaMemset(s.d_feat, 0, chunk * (size_t)m->feat_stride));
            }
            CU_TRY(cudaMalloc(&s.d_images, chunk * (size_t)m->img_bytes));
            CU_TRY(cudaMalloc(&s.d_logits, chunk * (size_t)m->n_classes * sizeof(int32_t)));
            CU_TRY(cudaMalloc(&s.d_labels, chunk * sizeof(uint32_t)));
        }
        m->slot_n = chunk;
    }
    // the layer-by-layer path shares one scratch arena (accumulators / activations): its chunks must not overlap in time -> one
    // stream.  The fused path has no shared state (CNN models: one feature buffer per slot) and uses all three.
    const bool shared_scratch = bnm_model_active_path(m) != BNM_PATH_TCGEN05;
    size_t k = 0;
    for (size_t b = 0; b < n; b += chunk, k++) {
        const size_t nb = std::min(chunk, n - b);
        PipeSlot &s = m->slots[shared_scratch ? 0 : k % 3];
        CU_TRY(cudaMemcpyAsync(s.d_images, images + b * m->img_bytes, nb * (size_t)m->img_bytes, cudaMemcpyHostToDevice, s.stream));
        int rc = infer_device_impl(m, s.d_images, nb, s.d_logits, labels ? s.d_labels : nullptr, nullptr, s.stream, shared_scratch ? nullptr : s.d_feat);
        if (rc) return rc;
        CU_TRY(cudaMemcpyAsync(logits + b * m->n_classes, s.d_logits, nb * (size_t)m->n_classes * sizeof(int32_t), cudaMemcpyDeviceToHost, s.stream));
        if (labels) CU_TRY(cudaMemcpyAsync(labels + b, s.d_labels, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    }
    for (auto &s : m->slots) CU_TRY(cudaStreamSynchronize(s.stream));
    return 0;
}

extern "C" void *bnm_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); fail(BNM_E_CUDA, "cudaHostAlloc(%zu) failed", bytes); return nullptr; }
    return p;
}
extern "C" void bnm_host_free(void *p) { if (p) cudaFreeHost(p); }

// -----------------------------------------------------------------------------------------------
// the four kernels, batched over host buffers
// -----------------------------------------------------------------------------------------------
static int require_device() {
    if (bnm_device_count() == 0) return fail(BNM_E_NODEV, "no CUDA device: this engine has no CPU fallback");
    return 0;
}
static int require_device_index(int device) {
    const int n = bnm_device_count();
    if (n == 0) return fail(BNM_E_NODEV, "no CUDA device: this engine has no CPU fallback");
    if (device < 0 || device >= n) return fail(BNM_E_ARG, "device %d out of range (have %d)", device, n);
    return 0;
}

extern "C" int bnm_processfclayer_batch(const int8_t *activations, const uint32_t *weights, int32_t enc, uint32_t n_input,
                                        uint32_t n_output, int32_t *output, size_t n, int nf4_extension) {
    if (int rc = require_device()) return rc;
    if (n == 0 || n_output == 0) return 0;
    if (!activations || !weights || !output) return fail(BNM_E_ARG, "bnm_processfclayer_batch: null argument");
    size_t need = 0;
    switch (enc) {
    case BNM_ENC_BINARY: need = (size_t)n_output * ((n_input + 31) / 32) * 4; break;
    case BNM_ENC_2BITSYM: need = (size_t)n_output * ((n_input + 15) / 16) * 4; break;
    case BNM_ENC_4BITSYM: case BNM_ENC_4BIT: case BNM_ENC_FP130: case BNM_ENC_NF4: need = (size_t)n_output * ((n_input + 7) / 8) * 4; break;
    case BNM_ENC_8BIT: need = (size_t)n_output * ((n_input + 3) / 4) * 4; break;
    case BNM_ENC_TERNARY: need = (size_t)n_output * (n_input / 10) * 2; break;
    default: need = 0;
    }
    FcLayerDev L;
    L.enc = enc; L.n_in = n_input; L.n_out = n_output;
    L.k_pad = round_up(std::max(n_input, 1u), 32);
    L.n_pad = round_up(n_output, 16);
    const size_t plane = (size_t)L.k_pad * L.n_pad;
    DevBuf packed, da, db, qa, qb, flag, act, out;
    if (packed.alloc(need + 16) || da.alloc(plane) || db.alloc(plane) || qa.alloc(plane) || qb.alloc(plane) || flag.alloc(4) ||
        act.alloc(n * (size_t)L.k_pad) || out.alloc(n * (size_t)n_output * 4))
        return fail(BNM_E_CUDA, "cudaMalloc failed");
    CU_TRY(cudaMemset(packed.p, 0, need + 16));
    if (need) CU_TRY(cudaMemcpy(packed.p, weights, need, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(flag.p, 0, 4));
    L.dense_a = da.as<int8_t>(); L.quad_a = qa.as<int4>();
    launch_decode_fc(packed.p, enc, n_input, n_output, L.k_pad, L.n_pad, L.dense_a, db.as<int8_t>(), L.quad_a, qb.as<int4>(), nf4_extension,
                     flag.as<int>(), 0);
    int f = 0;
    CU_TRY(cudaMemcpy(&f, flag.p, 4, cudaMemcpyDeviceToHost));
    if (f) { L.dense_b = db.as<int8_t>(); L.quad_b = qb.as<int4>(); }
    CU_TRY(cudaMemset(act.p, 0, n * (size_t)L.k_pad));
    // Ternary layers declare n_input padded to a multiple of 10 with zero trits (exportquant.py:132-137,166) and the
    // reference never reads the activations under a zero trit (inference.c:128): a caller may hand in a 256-byte row for
    // n_input = 260.  Read exactly what the reference can read: up to the last non-zero trit of any row.
    uint32_t valid_in = n_input;
    if (enc == BNM_ENC_TERNARY) {
        const uint16_t *w16 = reinterpret_cast<const uint16_t *>(weights);
        const uint32_t wpr = n_input / 10;
        valid_in = 0;
        for (uint32_t o = 0; o < n_output; o++)
            for (uint32_t g = wpr; g-- > 0;) {
                if (g * 10 + 10 <= valid_in) break;
                uint32_t c = w16[(size_t)o * wpr + g];
                for (uint32_t j = 0; j < 10; j++) {
                    c *= 3u;
                    if (!(c & 0x20000u)) valid_in = std::max(valid_in, g * 10 + j + 1);
                    c &= 0xFFFFu;
                }
            }
    }
    if (valid_in) CU_TRY(cudaMemcpy2D(act.p, L.k_pad, activations, n_input, valid_in, n, cudaMemcpyHostToDevice));
    if (!launch_fc_dp4a(act.as<int8_t>(), L.k_pad, L, out.as<int32_t>(), n, 0))
        return fail(BNM_E_UNSUPPORTED, "processfclayer: n_input %u needs more shared memory than an SM has (layer kernel stages 128 rows)", n_input);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(output, out.p, n * (size_t)n_output * 4, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int bnm_relunorm_batch(const int32_t *input, int8_t *output, uint32_t *argmax, uint32_t n_input, size_t n) {
    if (int rc = require_device()) return rc;
    if (n == 0) return 0;
    if (n_input == 0) {   // inference.c:24-37: nothing is scanned, position stays 255
        if (argmax) for (size_t i = 0; i < n; i++) argmax[i] = 255;
        return 0;
    }
    if (!input) return fail(BNM_E_ARG, "bnm_relunorm_batch: null input");
    DevBuf in, out, am;
    if (in.alloc(n * (size_t)n_input * 4) || out.alloc(n * (size_t)n_input) || am.alloc(n * 4)) return fail(BNM_E_CUDA, "cudaMalloc failed");
    CU_TRY(cudaMemcpy(in.p, input, n * (size_t)n_input * 4, cudaMemcpyHostToDevice));   // copied first: output may alias input
    launch_relunorm(in.as<int32_t>(), n_input, output ? out.as<int8_t>() : nullptr, n_input, am.as<uint32_t>(), n, 0);
    CU_TRY(cudaGetLastError());
    if (argmax) CU_TRY(cudaMemcpy(argmax, am.p, n * 4, cudaMemcpyDeviceToHost));
    else CU_TRY(cudaDeviceSynchronize());
    if (output) CU_TRY(cudaMemcpy(output, out.p, n * (size_t)n_input, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int bnm_conv33relu_batch(const int32_t *activations, const int8_t *weights, uint32_t n_w, uint32_t xy, uint32_t n_shift,
                                    int32_t *output, size_t n) {
    if (int rc = require_device()) return rc;
    if (n == 0 || xy < 3) return 0;
    if (!activations || !weights || !output || n_w == 0) return fail(BNM_E_ARG, "bnm_conv33relu_batch: null argument");
    const size_t in_el = n * (size_t)xy * xy, out_el = n * (size_t)(xy - 2) * (xy - 2);
    DevBuf in, w, out;
    if (in.alloc(in_el * 4) || w.alloc((size_t)n_w * 9) || out.alloc(out_el * 4)) return fail(BNM_E_CUDA, "cudaMalloc failed");
    CU_TRY(cudaMemcpy(in.p, activations, in_el * 4, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(w.p, weights, (size_t)n_w * 9, cudaMemcpyHostToDevice));
    launch_conv33relu(in.as<int32_t>(), w.as<int8_t>(), n_w, xy, n_shift, out.as<int32_t>(), n, 0);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(output, out.p, out_el * 4, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int bnm_maxpool22_batch(const int32_t *activations, uint32_t xy, int32_t *output, size_t n) {
    if (int rc = require_device()) return rc;
    if (n == 0 || xy < 2) return 0;
    if (!activations || !output) return fail(BNM_E_ARG, "bnm_maxpool22_batch: null argument");
    const size_t in_el = n * (size_t)xy * xy, out_el = n * (size_t)(xy / 2) * (xy / 2);
    DevBuf in, out;
    if (in.alloc(in_el * 4) || out.alloc(out_el * 4)) return fail(BNM_E_CUDA, "cudaMalloc failed");
    CU_TRY(cudaMemcpy(in.p, activations, in_el * 4, cudaMemcpyHostToDevice));
    launch_maxpool22(in.as<int32_t>(), xy, out.as<int32_t>(), n, 0);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(output, out.p, out_el * 4, cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int bnm_quantize_images_device(const float *images, size_t n, uint32_t elems, int8_t *out, void *stream) {
    if (int rc = require_device()) return rc;
    if (n == 0 || elems == 0) return 0;
    if (!images || !out) return fail(BNM_E_ARG, "bnm_quantize_images_device: null argument");
    launch_quantize_images(images, elems, out, n, static_cast<cudaStream_t>(stream));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail(BNM_E_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
}

// float images -> logits / labels on the device.  FC models on the fused path (rows of <= 256 elements, <= 16 classes): ONE kernel, the
// input scaling fused into its load stage.  Everything else: the scaling kernel into a scratch buffer, then the ordinary path.
extern "C" int bnm_infer_batch_device_f32(bnm_model *m, const float *images, size_t n, int32_t *logits, uint32_t *labels, void *stream) {
    if (!m || (n && (!images || !logits))) return fail(BNM_E_ARG, "bnm_infer_batch_device_f32: null argument");
    if (n == 0) return 0;
    if ((uintptr_t)images & 15) return fail(BNM_E_ARG, "the device image buffer must be 16-byte aligned");
    if ((uintptr_t)logits & 7) return fail(BNM_E_ARG, "the device logits buffer must be 8-byte aligned (64-bit row stores)");
    CU_TRY(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool fused_fc = bnm_model_active_path(m) == BNM_PATH_TCGEN05 && m->model_class == BNM_MODEL_FCMNIST;
    if (fused_fc && fc_chain_float_input_supported(m->plan)) {
        int rc = fc_chain_launch_f32(m->plan, images, n, logits, labels, st);
        return rc ? fail(BNM_E_CUDA, "fused float-input kernel launch failed (%d): %s", rc, cudaGetErrorString(cudaGetLastError())) : 0;
    }
    if (m->f32_scratch_n < n) {
        cudaFree(m->d_f32_scratch);
        m->d_f32_scratch = nullptr; m->f32_scratch_n = 0;
        CU_TRY(cudaMalloc(&m->d_f32_scratch, n * (size_t)m->img_bytes));
        m->f32_scratch_n = n;
    }
    launch_quantize_images(images, m->img_bytes, m->d_f32_scratch, n, st);
    return bnm_infer_batch_device(m, m->d_f32_scratch, n, logits, labels, stream);
}

extern "C" int bnm_quantize_images(const float *images, size_t n, uint32_t elems, int8_t *out) {
    if (int rc = require_device()) return rc;
    if (n == 0 || elems == 0) return 0;
    if (!images || !out) return fail(BNM_E_ARG, "bnm_quantize_images: null argument");
    DevBuf in, q;
    if (in.alloc(n * (size_t)elems * 4) || q.alloc(n * (size_t)elems)) return fail(BNM_E_CUDA, "cudaMalloc failed");
    CU_TRY(cudaMemcpy(in.p, images, n * (size_t)elems * 4, cudaMemcpyHostToDevice));
    launch_quantize_images(in.as<float>(), elems, q.as<int8_t>(), n, 0);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(out, q.p, n * (size_t)elems, cudaMemcpyDeviceToHost));
    return 0;
}

// -----------------------------------------------------------------------------------------------
// Emulation mode (SURVEY.md 8f rank 4): QuantizedModel.inference_quantized of the reference (BitNetMCU.py:420-535) on the GPU --
// float images in, float64 "logits" out, with the EMULATOR's normalisation rules (power-of-two rescale to max <= 127 with
// round-half-even for BitLinear, per-image renormalisation of every conv output) instead of the C engine's.  It reuses the
// engine's integer kernels (decoded weights, dp4a layers, conv / pool); weight levels are the engine's integers divided by
// level_scale (2 for 2bitsym / 4bitsym), so every intermediate is an exact dyadic rational and the result equals NumPy's.
// -----------------------------------------------------------------------------------------------
static int level_shift_of(int32_t enc) { return (enc == BNM_ENC_2BITSYM || enc == BNM_ENC_4BITSYM) ? 1 : 0; }

extern "C" int bnm_emulate_inference_quantized(bnm_model *m, const float *images, size_t n, double *logits) {
    if (!m || (n && (!images || !logits))) return fail(BNM_E_ARG, "bnm_emulate_inference_quantized: null argument");
    if (n == 0) return 0;
    CU_TRY(cudaSetDevice(m->device));
    const bool cnn = m->model_class == BNM_MODEL_CNNMNIST;
    const uint32_t C = m->channels, elems = m->img_bytes;
    const size_t chunk = std::min<size_t>(n, cnn ? 2048 : 65536);
    const size_t nl = m->fc.size();
    uint32_t max_nout = 1, max_kpad = round_up(std::max(m->img_bytes, m->feat_stride), 32);
    for (auto &L : m->fc) { max_nout = std::max(max_nout, L.n_out); max_kpad = std::max(max_kpad, L.k_pad); }
    DevBuf d_f, d_q, d_acc, d_a0, d_a1, d_p0, d_p1;
    if (d_f.alloc(chunk * elems * 4) || d_q.alloc(chunk * elems) || d_acc.alloc(chunk * (size_t)max_nout * 4) || d_a0.alloc(chunk * (size_t)max_kpad) ||
        d_a1.alloc(chunk * (size_t)max_kpad) || (cnn && (d_p0.alloc(chunk * C * 256 * 4) || d_p1.alloc(chunk * C * 256 * 4))))
        return fail(BNM_E_CUDA, "cudaMalloc failed (emulation scratch)");
    CU_TRY(cudaMemset(d_a0.p, 0, chunk * (size_t)max_kpad));
    CU_TRY(cudaMemset(d_a1.p, 0, chunk * (size_t)max_kpad));
    std::vector<int32_t> h_acc(chunk * (size_t)m->n_classes);
    cudaStream_t st = 0;
    for (size_t b = 0; b < n; b += chunk) {
        const size_t nb = std::min(chunk, n - b);
        CU_TRY(cudaMemcpy(d_f.p, images + b * elems, nb * elems * 4, cudaMemcpyHostToDevice));
        launch_quantize_images(d_f.as<float>(), elems, d_q.as<int8_t>(), nb, st);   // BitNetMCU.py:435-436
        const int8_t *act = d_q.as<int8_t>();
        uint32_t stride = elems;
        if (cnn) {
            // conv (ReLU, no shift) -> per-image renormalisation, pools in between (BitNetMCU.py:459-526), planes [(image, channel)][xy*xy]
            int32_t *p0 = d_p0.as<int32_t>(), *p1 = d_p1.as<int32_t>();
            launch_expand_image(d_q.as<int8_t>(), p0, C, 256, nb, st);
            launch_conv33relu(p0, m->d_conv[0], C, 16, 0, p1, nb * C, st);
            launch_conv_renorm(p1, C * 196, nb, st);
            launch_conv33relu(p1, m->d_conv[1], C, 14, 0, p0, nb * C, st);
            launch_conv_renorm(p0, C * 144, nb, st);
            launch_maxpool22(p0, 12, p1, nb * C, st);
            launch_conv33relu(p1, m->d_conv[2], C, 6, 0, p0, nb * C, st);
            launch_conv_renorm(p0, C * 16, nb, st);
            launch_maxpool22(p0, 4, p1, nb * C, st);
            launch_i32_to_i8(p1, C * 4, d_a1.as<int8_t>(), m->feat_stride, nb, st);   // flatten (C, 2, 2) -> features (BitNetMCU.py:443-445)
            act = d_a1.as<int8_t>();
            stride = m->feat_stride;
        }
        for (size_t l = 0; l < nl; l++) {
            if (!launch_fc_dp4a(act, stride, m->fc[l], d_acc.as<int32_t>(), nb, st)) return fail(BNM_E_UNSUPPORTED, "FC layer %zu too wide for the layer kernel", l);
            if (l + 1 == nl) break;   // no renormalisation for the last layer (BitNetMCU.py:528-530)
            int8_t *next = (l & 1) ? d_a1.as<int8_t>() : d_a0.as<int8_t>();   // CNN features sit in d_a1 and are dead once layer 0 has run
            const uint32_t next_stride = m->fc[l + 1].k_pad;
            launch_relunorm_emul(d_acc.as<int32_t>(), m->fc[l].n_out, level_shift_of(m->fc[l].enc), next, next_stride, nb, st);
            act = next;
            stride = next_stride;
        }
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaMemcpy(h_acc.data(), d_acc.p, nb * (size_t)m->n_classes * 4, cudaMemcpyDeviceToHost));
        const double inv = 1.0 / (double)(1 << level_shift_of(m->fc[nl - 1].enc));
        for (size_t i = 0; i < nb * (size_t)m->n_classes; i++) logits[b * m->n_classes + i] = (double)h_acc[i] * inv;
    }
    return 0;
}

// -----------------------------------------------------------------------------------------------
// reference-named symbols (BitNetMCU_inference.h:15-60): one item, abort on failure -- never a CPU path
// -----------------------------------------------------------------------------------------------
static void die(const char *fn) {
    fprintf(stderr, "bitnetmcu_b200: %s failed: %s\n", fn, g_err.c_str());
    abort();
}

extern "C" uint32_t ReLUNorm(int32_t *input, int8_t *output, uint32_t n_input) {
    uint32_t pos = 255;
    if (bnm_relunorm_batch(input, output, &pos, n_input, 1) != 0) die("ReLUNorm");
    return pos;
}
extern "C" void processfclayer(int8_t *activations, const uint32_t *weights, int32_t bits_per_weight, uint32_t n_input,
                               uint32_t n_output, int32_t *output) {
    if (bnm_processfclayer_batch(activations, weights, bits_per_weight, n_input, n_output, output, 1, 0) != 0) die("processfclayer");
}
extern "C" int32_t *processconv33ReLU(int32_t *activations, const int8_t *weights, uint32_t xy_input, uint32_t n_shift, int32_t *output) {
    if (bnm_conv33relu_batch(activations, weights, 1, xy_input, n_shift, output, 1) != 0) die("processconv33ReLU");
    return output + (size_t)(xy_input - 2) * (xy_input - 2);
}
extern "C" int32_t *processmaxpool22(int32_t *activations, uint32_t xy_input, int32_t *output) {
    if (bnm_maxpool22_batch(activations, xy_input, output, 1) != 0) die("processmaxpool22");
    return output + (size_t)(xy_input / 2) * (xy_input / 2);
}
