// fc_tcgen05.cu -- the hot path: the whole processfclayer -> ReLUNorm chain of BitMnistInference
// (/root/reference/BitNetMCU_MNIST_dll.c:95-121, kernels inference.c:88-208 + 23-72) as ONE persistent
// sm_100a kernel.  Per 128-image tile:
//
//   TMA (cp.async.bulk.tensor, SWIZZLE_128B, evict-first)  images  HBM -> smem ring
//   layer 1   tcgen05.mma kind::i8  A = smem image tile, B = decoded int8 weights (smem)  -> D int32 in TMEM
//   ReLUNorm  tcgen05.ld (thread = image row): max -> shift -> clamp(x+r,0,cap)>>shift -> int8x4 pack
//             -> tcgen05.st back into TMEM as the next layer's A operand (no smem / HBM round trip)
//   layer l>1 tcgen05.mma kind::i8  A = TMEM (.ts form), B = smem weights                 -> D int32 in TMEM
//   last      int32 logits: thread-local argmax (first maximum via packed keys) + 64-bit stores straight to HBM
//
// Several warpgroups (128 threads = 128 TMEM lanes each) run this chain on different tiles so the tensor
// pipe, the TMEM<->register traffic and the integer ALU work of the ReLUNorm epilogues overlap.
// Weights of every encoding are pre-decoded once per model into int8 planes (kernels.h FcLayerDev); FP130's
// +128 does not fit s8 and is carried by a second residual plane accumulated by extra MMAs into the same D.
// All arithmetic is integer: results are bit-exact with the reference.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.h"
#include "sm100_ptx.cuh"

namespace bnm {

constexpr int kMaxWG = 4;        // epilogue warpgroups: three with 2 tile slots each (6 x (64 D + 16 A) = 480 of the 512 TMEM columns),
                                 // or four with one slot each when only 4..5 slots fit (kFourWG instantiations)
constexpr int kMaxWG2 = 3;       // ... of the two-slot form
constexpr int kMaxStages = 7;
constexpr uint32_t kFloatQuantWarps = 8;    // float-input path: quantiser warps per CTA
constexpr uint32_t kFloatWG = 2;            // ... next to two epilogue warpgroups (four tiles in flight are plenty at 1 kB per image): 576 threads
constexpr uint32_t kFloatRowsPerWarp = 128 / kFloatQuantWarps;   // rows of every tile per quantiser warp
constexpr uint32_t kFloatGroupRows = 4;     // rows per bulk copy of a quantiser warp (4 kB for 256-element rows) = rows per pass

struct ChainParams {
    int n_layers;
    uint32_t n_pad[kMaxFcLayers];     // UMMA N of layer l (multiple of 16)
    uint32_t n_real[kMaxFcLayers];    // real outputs
    uint32_t k_steps[kMaxFcLayers];   // K/32 MMA steps per plane
    uint32_t planes[kMaxFcLayers];    // 1, or 2 when the residual plane exists
    uint32_t b_off[kMaxFcLayers];     // smem byte offset (from weight base) of the layer's first [n_pad x 32B] tile
    uint32_t idesc[kMaxFcLayers];
    uint32_t in_atoms;                // layer-1 A: 128-byte SW128 atoms per row (TMA boxes per tile)
    uint32_t stage_bytes;             // in_atoms * 128 rows * 128 B
    uint32_t n_stages, n_wg, n_slots;
    uint32_t w_bytes;                 // weight image bytes (multiple of 16)
    uint32_t off_w;                   // smem offset (from the 1024-aligned base) of the weight image
    uint32_t tmem_wg_cols, tmem_a_off;
    uint32_t off_a, a_slot_bytes;     // kSmemA: the hidden layers' int8 activations live in shared memory (one [128 x K] buffer per slot)
    uint32_t n_classes;
    uint32_t n_tiles;
    const uint8_t *w_image;
    int32_t *logits;
    uint32_t *labels;
    size_t n;
    int *err;
    int32_t kadd[16];                 // argmax key offsets of the (single) logits chunk: 15-j for real classes, -2^30 for padding
    long long *trace;                 // diagnostics: clock64 per phase of CTA 0 / warpgroup 0 (null in production)
    uint32_t stagger_cycles;          // tuning knob (BNM_STAGGER_NS): warpgroup g starts no earlier than g * this after kernel entry
    uint32_t wait_prior_grid;         // programmatic dependent launch: read inputs only after the previous kernel has completed
    uint32_t early_trigger;           // let the next launch's CTAs take over SMs as this launch's CTAs leave (full grids only)
    // result exchange fused into the epilogue (SURVEY.md 8e): besides logits / labels, row i of this launch is also stored at row
    // row0 + i of every destination buffer -- peer GPUs' memory mapped through CUDA IPC / P2P, written over NVLink
    uint32_t n_lab_dst, n_log_dst;
    uint32_t *lab_dst[kMaxGatherDst];
    int32_t *log_dst[kMaxGatherDst];
    size_t row0;
    uint32_t lab_u8;                  // gather launches: lab_dst are uint8 buffers (one byte per label)
    const float *fimages;             // float-input launches (fc_chain_kernel<..., kFloatIn>): float32 [n][in_elems] instead of the int8 tensor map
    uint32_t in_elems;                // real elements per image row (<= 256 for the float path)
    uint32_t off_fring;               // float-input launches: smem offset of the quantiser warps' float rings (8 warps x 2 slots x 4 kB)
    uint32_t off_gstage;              // gather launches: smem offset of the per-warp staging rows for the bulk peer stores (0: none)
    // activation taps (fc_chain_kernel<..., kTaps>): hidden layer l's int8 ReLUNorm row of image i is also stored at
    // tap[l] + i * tap_stride[l] (null: not wanted).  The stride is the next layer's k_pad, set at plan creation.
    int8_t *tap[kMaxFcLayers];
    uint32_t tap_stride[kMaxFcLayers];
};

struct FcChainPlan {
    ChainParams p{};
    uint8_t *d_w_image = nullptr;
    int *d_err = nullptr;             // error word of the bounded device-side waits: mapped pinned host memory, readable after a trap
    int *h_err = nullptr;
    size_t smem_bytes = 0;
    uint32_t in_bytes = 0;
    int threads = 0;
    int sm_count = 0;
    int device = 0;
    int overlap = 0;                  // BNM_OPT_LAUNCH_OVERLAP: 0 plain launch, 1 dependent launch + wait, 2 independent launches
    // gather launches (fused result exchange) stage each warp's 32 logits rows in shared memory and push them to the peers with
    // one bulk copy per destination (full NVLink packets instead of 8-byte scattered stores): their own ring depth and layout
    uint32_t g_n_stages = 0, g_off_w = 0, g_off_gstage = 0;
    size_t g_smem_bytes = 0;
    // wide models (kSmemA launches): activations in shared memory, accumulator-only TMEM slots -> one more tile slot
    uint32_t sa_n_wg = 0, sa_n_stages = 0, sa_off_w = 0, sa_off_a = 0, sa_a_slot_bytes = 0, sa_tmem_wg_cols = 0;
    size_t sa_smem_bytes = 0;
    // float-input launches: fewer int8 stages, the freed shared memory holds the quantiser warps' float rings
    uint32_t f_n_stages = 0, f_off_w = 0, f_off_fring = 0;
    size_t f_smem_bytes = 0;
    // launch-path state (nothing on the launch path reads the environment or re-encodes a known tensor map)
    struct TmapSlot { const void *ptr = nullptr; size_t n = 0; CUtensorMap map; };
    TmapSlot tmaps[4];                // tensor maps of the most recent (pointer, n) pairs: double/triple-buffered callers hit every time
    unsigned tmap_next = 0;
    std::string trace_path;           // BNM_TRACE (diagnostics build path), read once at plan creation
    int stagger_override = -1;        // BNM_STAGGER_NS in cycles, read once at plan creation (-1: not set)
    // mode 2 bookkeeping: the buffers of the previous launch on this plan (the promise "consecutive launches are independent" is
    // checked as far as the library can see it: a launch that reuses a buffer of the one before keeps the grid-dependency wait)
    const void *prev_in = nullptr, *prev_logits = nullptr, *prev_labels = nullptr;
    cudaStream_t prev_stream = nullptr;
    bool prev_valid = false;
};

// ---------------------------------------------------------------------------------------------------
// weight image: every MMA K-step reads one [n_pad x 32 B] tile in the no-swizzle K-major canonical layout
// (8-row x 16-byte core matrices; LBO = 128 B between the two K halves, SBO = 256 B between 8-row groups)
// ---------------------------------------------------------------------------------------------------
__global__ void k_build_b_image(const int8_t *__restrict__ dense, uint32_t k_pad_src, uint32_t n_pad, uint32_t k_steps,
                                uint8_t *__restrict__ image) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = (size_t)n_pad * k_steps * 32;
    if (idx >= total) return;
    uint32_t n = idx / (k_steps * 32), k = idx % (k_steps * 32);
    uint8_t v = k < k_pad_src ? (uint8_t)dense[(size_t)n * k_pad_src + k] : 0;
    uint32_t kb = k & 31;
    size_t off = (size_t)(k >> 5) * n_pad * 32 + (n >> 3) * 256 + (kb >> 4) * 128 + (n & 7) * 16 + (kb & 15);
    image[off] = v;
}

// ---------------------------------------------------------------------------------------------------
// ReLUNorm pieces (inference.c:23-72), thread = one image row
// ---------------------------------------------------------------------------------------------------
struct NormCoef { int rounding, cap; uint32_t mult; };

__device__ __forceinline__ NormCoef norm_coef(int row_max_relu) {
    // shift = bit length of (max >> 7) (inference.c:41-47).  row_max_relu = max(row max, 0): a negative row
    // maximum zeroes every output whatever the shift, so taking the maximum over relu'd values is equivalent.
    const uint32_t shift = 32u - (uint32_t)__clz(row_max_relu >> 7);
    NormCoef c;
    c.rounding = (int)((1u << shift) >> 1);                 // inference.c:51
    c.cap = (int)((128u << shift) - 1u);                    // (cap >> shift) == 127: the clip of inference.c:60-64
    c.mult = 1u << (24u - shift);                           // u * mult puts (u >> shift) into byte 3
    return c;
}
// four int32 accumulators -> four int8 (0..127) packed little-endian.  1 VIADDMNMX.RELU + 1 IMAD per element,
// 3 PRMT per four.
__device__ __forceinline__ uint32_t norm_pack4(uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, const NormCoef &c) {
    uint32_t z0, z1, z2, z3;
    // mul.lo via asm so the power-of-two multiply stays an IMAD (FMA pipe) instead of a shift on the ALU pipe
    asm("mul.lo.u32 %0, %1, %2;" : "=r"(z0) : "r"((uint32_t)__viaddmin_s32_relu((int)x0, c.rounding, c.cap)), "r"(c.mult));
    asm("mul.lo.u32 %0, %1, %2;" : "=r"(z1) : "r"((uint32_t)__viaddmin_s32_relu((int)x1, c.rounding, c.cap)), "r"(c.mult));
    asm("mul.lo.u32 %0, %1, %2;" : "=r"(z2) : "r"((uint32_t)__viaddmin_s32_relu((int)x2, c.rounding, c.cap)), "r"(c.mult));
    asm("mul.lo.u32 %0, %1, %2;" : "=r"(z3) : "r"((uint32_t)__viaddmin_s32_relu((int)x3, c.rounding, c.cap)), "r"(c.mult));
    uint32_t lo = __byte_perm(z0, z1, 0x0073), hi = __byte_perm(z2, z3, 0x0073);
    return __byte_perm(lo, hi, 0x5410);
}
__device__ __forceinline__ int max16(const uint32_t (&v)[16], int m) {
    int m2 = 0;   // two interleaved chains; every value is compared against 0 anyway (relu'd maximum)
#pragma unroll
    for (int j = 0; j < 16; j += 4) {
        m = __vimax3_s32(m, (int)v[j], (int)v[j + 1]);
        m2 = __vimax3_s32(m2, (int)v[j + 2], (int)v[j + 3]);
    }
    return max(m, m2);
}

// activation taps: a thread's packed int8 words also go to its image's row in global memory.  Nothing in the kernel reads
// them back, so a plain generic-proxy store with a streaming hint needs no barrier.
__device__ __forceinline__ void st_global_cs_v4(int8_t *p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.cs.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d));
}

// hidden-layer epilogue, the common 64-wide case: one TMEM load of the whole row, one TMEM store of the 16 packed words.
// kTaps: tap (null: this row is not wanted) receives the same 16 words.
template <bool kTaps>
__device__ __forceinline__ void relunorm_tmem64(uint32_t d_addr, uint32_t a_addr, int8_t *tap) {
    uint32_t v[64];
    tmem_ld_x64(d_addr, v);
    tmem_ld_wait();
    int mc[4];   // four independent max chains (ILP), merged at the end
#pragma unroll
    for (int c = 0; c < 4; c++) {
        int m = 0, m2 = 0;
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
            m = __vimax3_s32(m, (int)v[16 * c + j], (int)v[16 * c + j + 1]);
            m2 = __vimax3_s32(m2, (int)v[16 * c + j + 2], (int)v[16 * c + j + 3]);
        }
        mc[c] = max(m, m2);
    }
    const NormCoef k = norm_coef(max(__vimax3_s32(mc[0], mc[1], mc[2]), mc[3]));
    // (an IMAD.HI + I2IP.S8.SAT formulation that moves shift/round/clip to the FMA pipe is bit-exact too but measured
    //  slower in this kernel for every ALU/FMA split: tools/requant_bench.cu, profiles/r1_micro_requant.txt)
#pragma unroll
    for (int h = 0; h < 2; h++) {   // two 8-word stores keep the register peak below the 128-register budget
        uint32_t w[8];
#pragma unroll
        for (int q = 0; q < 8; q++) w[q] = norm_pack4(v[32 * h + 4 * q], v[32 * h + 4 * q + 1], v[32 * h + 4 * q + 2], v[32 * h + 4 * q + 3], k);
        tmem_st_x8(a_addr + 8 * h, w);
        if (kTaps && tap) {
            st_global_cs_v4(tap + 32 * h, w[0], w[1], w[2], w[3]);
            st_global_cs_v4(tap + 32 * h + 16, w[4], w[5], w[6], w[7]);
        }
    }
    tmem_st_wait();
}

// hidden-layer epilogue for every other width: D[tmem, n_pad columns] -> A[tmem, n_pad/4 columns] in two passes over
// TMEM (row maximum first, then requantise), 32 columns at a time -- wide layers (Binary-160) would not fit the
// register budget in one pass, narrow ones (16..48) do not need it.
template <bool kTaps>
__device__ __forceinline__ void relunorm_tmem(uint32_t d_addr, uint32_t a_addr, uint32_t n_pad, int8_t *tap) {
    {
        int m = 0;
        const uint32_t n32 = n_pad & ~31u;   // 32-column chunks, then at most one 16-column tail
#pragma unroll 1
        for (uint32_t c = 0; c < n32; c += 32) {
            uint32_t v[32];
            tmem_ld_x32(d_addr + c, v);
            tmem_ld_wait();
            m = max16(reinterpret_cast<const uint32_t (&)[16]>(v[0]), m);
            m = max16(reinterpret_cast<const uint32_t (&)[16]>(v[16]), m);
        }
        if (n32 < n_pad) {
            uint32_t v[16];
            tmem_ld_x16(d_addr + n32, v);
            tmem_ld_wait();
            m = max16(v, m);
        }
        const NormCoef k = norm_coef(m);
#pragma unroll 1
        for (uint32_t c = 0; c < n32; c += 32) {
            uint32_t v[32], w[8];
            tmem_ld_x32(d_addr + c, v);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 8; q++) w[q] = norm_pack4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3], k);
            tmem_st_x8(a_addr + (c >> 2), w);
            if (kTaps && tap) {
                st_global_cs_v4(tap + c, w[0], w[1], w[2], w[3]);
                st_global_cs_v4(tap + c + 16, w[4], w[5], w[6], w[7]);
            }
        }
        if (n32 < n_pad) {
            uint32_t v[16], w[4];
            tmem_ld_x16(d_addr + n32, v);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 4; q++) w[q] = norm_pack4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3], k);
            tmem_st_x4(a_addr + (n32 >> 2), w);
            if (kTaps && tap) st_global_cs_v4(tap + n32, w[0], w[1], w[2], w[3]);
        }
    }
    tmem_st_wait();
}

// hidden-layer epilogue of the kSmemA form: as relunorm_tmem, but the int8 row goes to shared memory in the no-swizzle K-major
// layout of the weight tiles (per 32-byte K-step a [128 rows x 32 B] block: 8-row groups 256 B apart, the two 16-byte K-chunks
// of a group 128 B apart), where the next layer's MMAs read it as their A operand (SS form).
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// 32-column chunks of a TMEM row, software-pipelined: the load of chunk c+1 is in flight while f works on chunk c (the
// tcgen05.ld latency otherwise sits in front of every chunk: with one slot per warpgroup nothing else hides it)
template <typename F>
__device__ __forceinline__ void for_chunks32_pipelined(uint32_t d_addr, uint32_t n32, F f) {
    if (n32 == 0) return;
    uint32_t va[32], vb[32];
    tmem_ld_x32(d_addr, va);
    tmem_ld_wait();
    uint32_t c = 0;
#pragma unroll 1
    while (true) {
        if (c + 32 < n32) tmem_ld_x32(d_addr + c + 32, vb);
        f(va, c);
        c += 32;
        if (c >= n32) break;
        tmem_ld_wait();
        if (c + 32 < n32) tmem_ld_x32(d_addr + c + 32, va);
        f(vb, c);
        c += 32;
        if (c >= n32) break;
        tmem_ld_wait();
    }
}
template <bool kTaps>
__device__ __forceinline__ void relunorm_smem(uint32_t d_addr, uint32_t a_slot_addr, uint32_t row, uint32_t n_pad, int8_t *tap) {
    int m = 0;
    const uint32_t n32 = n_pad & ~31u;
    for_chunks32_pipelined(d_addr, n32, [&](const uint32_t (&v)[32], uint32_t) {
        m = max16(reinterpret_cast<const uint32_t (&)[16]>(v[0]), m);
        m = max16(reinterpret_cast<const uint32_t (&)[16]>(v[16]), m);
    });
    if (n32 < n_pad) {
        uint32_t v[16];
        tmem_ld_x16(d_addr + n32, v);
        tmem_ld_wait();
        m = max16(v, m);
    }
    const NormCoef k = norm_coef(m);
    const uint32_t a_row = a_slot_addr + (row >> 3) * 256 + (row & 7) * 16;
    for_chunks32_pipelined(d_addr, n32, [&](const uint32_t (&v)[32], uint32_t c) {
        uint32_t w[8];
#pragma unroll
        for (int q = 0; q < 8; q++) w[q] = norm_pack4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3], k);
        st_shared_v4(a_row + c * 128, w[0], w[1], w[2], w[3]);            // K-step c / 32: block of 4096 B
        st_shared_v4(a_row + c * 128 + 128, w[4], w[5], w[6], w[7]);
        if (kTaps && tap) {
            st_global_cs_v4(tap + c, w[0], w[1], w[2], w[3]);
            st_global_cs_v4(tap + c + 16, w[4], w[5], w[6], w[7]);
        }
    });
    if (n32 < n_pad) {   // (the K-step's second chunk multiplies zero weights)
        uint32_t v[16], w[4];
        tmem_ld_x16(d_addr + n32, v);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; q++) w[q] = norm_pack4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3], k);
        st_shared_v4(a_row + n32 * 128, w[0], w[1], w[2], w[3]);
        if (kTaps && tap) st_global_cs_v4(tap + n32, w[0], w[1], w[2], w[3]);
    }
    fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
}

// ---------------------------------------------------------------------------------------------------
// the kernel
//
// Roles (one CTA per SM, persistent over image tiles):
//   * n_wg epilogue warpgroups (4 warps = the 4 TMEM lane quarters).  Every warp owns 32 image rows and works
//     alone: it never synchronises with the other warps of its group.
//   * n_wg issuer warps, one per warpgroup: they wait for "operand ready", issue the tcgen05.mma batch of the next
//     layer and commit it to an mbarrier.  tcgen05.mma issue + commit blocks the issuing warp for roughly the MMA
//     pipeline latency (~450 cycles, tools/umma_tput.cu), so it lives in its own warp, off the epilogue's path.
//   * every warpgroup runs kSlots tiles at once ("slots", each with its own TMEM accumulator + activation columns):
//     while the MMAs of slot X are in flight the epilogue warps requantise slot Y, so the integer ALU work of
//     ReLUNorm -- the real limiter of this kernel -- is never parked behind tensor-pipe latency.
// Barriers: full[2][stage] (TMA tile landed), mma[g][slot] (MMA batch complete -> epilogue may read D),
//           ready[g][slot] (128 arrivals: every epilogue thread has written A / finished reading D -> issuer may go on).
// ---------------------------------------------------------------------------------------------------
constexpr int kMaxSlots = 2;
constexpr uint32_t kFullBars = 8;           // "tile landed" barriers per ring stage: >= slots / gcd(slots, stages) for every shape (ring comment in the kernel)
constexpr uint32_t kReadyArrivals = 128;   // every epilogue thread arrives
static_assert(kFullBars >= (uint32_t)(kMaxWG * kMaxSlots) && (kFullBars & (kFullBars - 1)) == 0,
              "kFullBars must cover slots / gcd(slots, stages) for every launch shape (and be a power of two)");

// layer-1 MMAs: A = image tile in smem (SWIZZLE_128B K-major), B = weight tiles.  Whole warp converged so that all
// descriptor arithmetic stays in the uniform datapath; only the tcgen05 instructions are predicated on one lane.
__device__ __forceinline__ void issue_layer1(const ChainParams &P, uint32_t a_stage_addr, uint32_t w_base, uint32_t d_tmem, bool leader) {
    const uint64_t a0 = make_smem_desc(a_stage_addr, 0, 1024, UMMA_LAYOUT_SW128);
    const uint64_t b0 = make_smem_desc(w_base + P.b_off[0], 128, 256, UMMA_LAYOUT_NONE);
    const uint32_t b_step = (P.n_pad[0] * 32) >> 4, nk = P.k_steps[0], idesc = P.idesc[0];
    uint32_t bo = 0;
    for (uint32_t pl = 0; pl < P.planes[0]; pl++)
        for (uint32_t k = 0; k < nk; k++, bo += b_step) {
            // K advance inside a SW128 atom: +32 B (>>4 = 2); next atom: +16384 B (>>4 = 1024)
            const uint64_t ad = a0 + (uint64_t)((k >> 2) * 1024 + (k & 3) * 2);
            if (leader) umma_i8_ss(d_tmem, ad, b0 + bo, idesc, bo != 0);
        }
}
// layer l > 1: A = int8 activations in TMEM (written by the ReLUNorm epilogue), B = weight tiles
__device__ __forceinline__ void issue_layer_ts(const ChainParams &P, int l, uint32_t w_base, uint32_t d_tmem, uint32_t a_tmem, bool leader) {
    const uint64_t b0 = make_smem_desc(w_base + P.b_off[l], 128, 256, UMMA_LAYOUT_NONE);
    const uint32_t b_step = (P.n_pad[l] * 32) >> 4, nk = P.k_steps[l], idesc = P.idesc[l];
    uint32_t bo = 0;
    for (uint32_t pl = 0; pl < P.planes[l]; pl++)
        for (uint32_t k = 0; k < nk; k++, bo += b_step)
            if (leader) umma_i8_ts(d_tmem, a_tmem + k * 8, b0 + bo, idesc, bo != 0);
}

// layer l > 1, kSmemA form: A = int8 activations in shared memory (relunorm_smem), B = weight tiles
__device__ __forceinline__ void issue_layer_ss(const ChainParams &P, int l, uint32_t w_base, uint32_t d_tmem, uint32_t a_smem, bool leader) {
    const uint64_t a0 = make_smem_desc(a_smem, 128, 256, UMMA_LAYOUT_NONE);
    const uint64_t b0 = make_smem_desc(w_base + P.b_off[l], 128, 256, UMMA_LAYOUT_NONE);
    const uint32_t b_step = (P.n_pad[l] * 32) >> 4, nk = P.k_steps[l], idesc = P.idesc[l];
    uint32_t bo = 0;
    for (uint32_t pl = 0; pl < P.planes[l]; pl++)
        for (uint32_t k = 0; k < nk; k++, bo += b_step)
            if (leader) umma_i8_ss(d_tmem, a0 + (uint64_t)(k * (4096 >> 4)), b0 + bo, idesc, bo != 0);
}

// kManyClasses: more than 16 classes (chunked logits / argmax epilogue).  A template parameter, like kGather, so that the common
// kernel stays below the 32 kB instruction cache: the gather variant at 41 kB ran 9 % slower for code size alone.
// kFloatIn: the input scaling of the reference's caller (test_inference.py:140-141: scale = 127 / max(max|x|, 1e-5), q = round-half-even
// (x * scale) clipped to int8, all float32) is fused into the load stage: eight extra warps fetch float32 rows from HBM (1 kB per
// image, bulk async copies into a small ring), reduce each row's absolute maximum, quantise and write the int8 row
// straight into the shared-memory image stage in the SWIZZLE_128B layout the layer-1 MMA expects -- the place of the TMA load.
// Float input then costs 1 024 B of HBM traffic per image once, instead of 1 024 + 256 (quantise kernel) + 256 (this kernel).
// kSmemA: wide models -- the hidden layers' activations go through shared memory instead of TMEM columns (relunorm_smem), so
// that a tile slot is the accumulator alone and one more slot fits (Binary-160: 3 x 160 columns instead of 2 x 208).
// kTaps: the hidden layers' int8 rows are also stored to P.tap[l] (activation taps), from the registers that already hold them.
template <int kSlots, bool kTrace, bool kGather, bool kManyClasses, bool kFloatIn = false, bool kFourWG = false, bool kSmemA = false,
          bool kTaps = false>
__global__ void __launch_bounds__(kFloatIn ? kFloatWG * 160 + 32 * kFloatQuantWarps : (kFourWG ? kMaxWG : kMaxWG2) * 160, 1)
fc_chain_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ ChainParams P) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[kFullBars][kMaxStages], bar_mma[kMaxWG][kMaxSlots], bar_ready[kMaxWG][kMaxSlots];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(8) uint64_t bar_w;   // weight image landed (one bulk async copy, no generic-proxy writes)
    __shared__ __align__(8) uint64_t bar_fload[kFloatQuantWarps][2];   // kFloatIn: a quantiser warp's ring slot has landed (bulk async copy)
    __shared__ __align__(8) uint64_t bar_free[kMaxStages];   // kFloatIn: the layer-1 MMAs of a stage's tile are done, the quantiser warps may refill it

    const long long t_entry = clock64();
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    const uint32_t warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler (uniform datapath)
    if (kTrace && P.trace && blockIdx.x == 0 && tid == 0) P.trace[1020] = clock64();   // kernel entry
    // Programmatic dependent launch: the next kernel in the stream may take over each SM as soon as this CTA leaves it (it
    // cannot co-reside: every launch asks for more than half of the SM's shared memory, fc_chain_plan_create), so its launch
    // latency and prologue -- and, when the caller
    // declares consecutive launches independent, its first tiles -- overlap the ragged end of this one.
    // Only when the grid fills the GPU (one CTA per SM): then launch k+1 can start no CTA before the matching CTA of launch k
    // has left, and launch k+2 none before all of launch k are gone -- at most two consecutive launches ever overlap.  A
    // smaller grid leaves SMs free, where later launches could pile up next to earlier ones; it triggers at completion.
    if (P.early_trigger) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t n_wg = P.n_wg, n_st = P.n_stages;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;   // SWIZZLE_128B tiles need 1024-byte alignment
    uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));

    const uint32_t tile0 = blockIdx.x, tile_step = gridDim.x;
    const uint32_t my_tiles = tile0 < P.n_tiles ? (P.n_tiles - tile0 + tile_step - 1) / tile_step : 0;
    const uint32_t n_virt = n_wg * kSlots;                 // tiles in flight per CTA
    const uint32_t n_rounds = (my_tiles + n_virt - 1) / n_virt;
    const uint32_t w_base = smem_base + P.off_w;

    // Image tile i of this CTA lives in ring stage i % n_st and belongs to slot (i % n_virt) = warpgroup (i % n_virt) / kSlots.
    // (Handing consecutive tiles to different warpgroups instead was measured 3 % slower: the warpgroups then start in
    // lockstep and compete for the ALU pipe at the same moments; the staggered start of this mapping keeps them out of
    // phase.  Three slots on two warpgroups: 15 % slower.)  The first n_st loads are
    // issued during setup, right after the weight copy has been requested; afterwards the warp that
    // has just seen the layer-1 MMAs of tile i complete (stage free) refills the stage with tile i + n_st.  Ring round
    // u = i / n_st signals barrier bar_full[u % kFullBars][s], phase parity (u / kFullBars) & 1.  A parity wait is only
    // unambiguous if it starts after the barrier's previous phase has completed: the wait for tile j (same barrier as tile
    // j - kFullBars n_st, other parity) must come after that tile has landed.  What is certain when the issuer gets to tile j:
    // its slot's earlier tiles j - a n_virt have landed, and with a tile every earlier tile of the same STAGE (a stage's loads
    // are requested one after the other).  The latest same-stage tile among them is j - m n_st with m = n_virt / gcd(n_virt,
    // n_st) -- 1 when every slot keeps its stage (6 slots on 6 stages), 6 for the gather launches (6 slots on 5 stages), 4 for
    // the four-warpgroup form (4 on 5), 3 for the shared-memory-activation form (3 on 2).  So kFullBars >= m for every shape:
    // 8 covers all of them (n_virt <= 8).  Two barriers per stage, the original scheme, were only safe for m = 1: a development
    // shape with 8 slots on 6 stages lost a phase under launch overlap and trapped on a bounded wait (tests/test_ring_protocol.py
    // replays the protocol on a discrete-event model with adversarial load latencies).
    const uint64_t l2_policy = policy_evict_first();   // images are read exactly once
    auto issue_tile_load = [&](uint32_t i) {
        const uint32_t s = i % n_st;
        uint64_t *bar = &bar_full[(i / n_st) & (kFullBars - 1)][s];
        mbar_arrive_expect_tx(bar, P.stage_bytes);
        const int32_t row = (int32_t)((tile0 + i * tile_step) * kTileM);
        for (uint32_t a = 0; a < P.in_atoms; a++)
            tma_load_2d_hint(smem + s * P.stage_bytes + a * 16384, &tmap_in, (int32_t)(a * 128), row, bar, l2_policy);
    };

    // ---------------- one-time setup
    // The first issuer warp initialises the barriers (one lane each); its lane 0 then starts the weight copy and issues the
    // first image loads.  Nobody executes a generic->async proxy fence -- measured: that fence, executed by a thread that has TMA loads in
    // flight, waits for them to land (~3 us per launch).
    if (kTrace && P.trace && tid == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); P.trace[1024 + 2 * blockIdx.x] = (long long)gt; }
    const bool setup_thread = tid == n_wg * 128;
    if (warp == n_wg * 4) {
        // barrier init, at most three barriers per lane (29 mbarrier.init in a row by one thread took ~1100 cycles of every launch)
        constexpr uint32_t kNFull = kFullBars * kMaxStages, kNSlot = kMaxWG * kMaxSlots;
#pragma unroll
        for (uint32_t b = lane; b <= kNFull + 2 * kNSlot; b += 32) {
            if (b < kNFull) { if ((b % kMaxStages) < n_st) mbar_init(&bar_full[b / kMaxStages][b % kMaxStages], kFloatIn ? kFloatQuantWarps : 1); }
            else if (b < kNFull + kNSlot) mbar_init(&bar_mma[0][0] + (b - kNFull), 1);
            else if (b < kNFull + 2 * kNSlot) mbar_init(&bar_ready[0][0] + (b - kNFull - kNSlot), kReadyArrivals);
            else mbar_init(&bar_w, 1);
        }
        if (kFloatIn && lane < n_st) mbar_init(&bar_free[lane], 1);
        if (kFloatIn && lane >= 8 && lane < 8 + 2 * kFloatQuantWarps) mbar_init(&bar_fload[(lane - 8) >> 1][lane & 1], 1);
        fence_mbar_init();
        __syncwarp();
    }
    if (setup_thread) {
        if (kTrace && P.trace && blockIdx.x == 0) P.trace[1016] = clock64();   // barriers initialised
        // weight image -> smem with bulk async copies (same bytes for every CTA; L2-resident after the first wave).  The
        // async proxy writes them, so the tensor core may read them as soon as bar_w completes: no staging loop, no
        // generic->async proxy fence in the prologue.  The weights were written at model build, long before any kernel that
        // may still be running ahead of this one, so they are fetched before the grid dependency is resolved.
        mbar_arrive_expect_tx(&bar_w, P.w_bytes);
        for (uint32_t off = 0; off < P.w_bytes; off += 32768)
            bulk_load_1d(smem + P.off_w + off, P.w_image + off, min(32768u, P.w_bytes - off), &bar_w);
        // Everything this kernel reads or writes besides the weights may belong to the kernel launched before it: wait until
        // that one has completed and flushed (no-op without a programmatic dependency).  Every other access of this CTA
        // happens after a barrier that these loads complete, i.e. after this wait.
        if (P.wait_prior_grid) asm volatile("griddepcontrol.wait;" ::: "memory");
        if (!kFloatIn)
            for (uint32_t i = 0; i < n_st && i < my_tiles; i++) issue_tile_load(i);
        if (kTrace && P.trace && blockIdx.x == 0) P.trace[1017] = clock64();   // first loads issued
    } else if (warp == 1) {
        tmem_alloc<512>(&tmem_base_s);
        if (kTrace && P.trace && blockIdx.x == 0 && lane == 0) P.trace[1018] = clock64();   // TMEM allocated
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    if (kTrace && P.trace && blockIdx.x == 0 && tid == 0) P.trace[1021] = clock64();   // prologue done

    if (warp >= n_wg * 4 && warp < n_wg * 5) {
        // ======================= MMA issuer warp of warpgroup g =======================
        const uint32_t g = warp - n_wg * 4;
        const bool leader = elect_one();
        uint32_t ready_phase = 0;   // one phase bit per slot
        mbar_wait(&bar_w, 0, P.err, 6);   // weight tiles are in shared memory
        if (P.stagger_cycles) {   // keep the warpgroups out of phase (they would otherwise compete for the ALU pipe in lockstep)
            const long long t_go = t_entry + (long long)g * P.stagger_cycles;
            while (clock64() < t_go) __nanosleep(64);
        }
        for (uint32_t r = 0; r < n_rounds; r++)
            for (int l = 0; l < P.n_layers; l++)
#pragma unroll 1
                for (int q = 0; q < kSlots; q++) {
                    const uint32_t v = g * kSlots + q;
                    const uint32_t i = r * n_virt + v;
                    if (i >= my_tiles) continue;
                    const uint32_t d_tmem = tmem_base + v * P.tmem_wg_cols, a_tmem = d_tmem + P.tmem_a_off;
                    if (r != 0 || l != 0) {   // previous epilogue step of this slot: A written / D drained by all 4 warps
                        mbar_wait(&bar_ready[g][q], (ready_phase >> q) & 1, P.err, 4);
                        ready_phase ^= 1u << q;
                    }
                    if (l == 0) {
                        const uint32_t s = i % n_st;
                        mbar_wait(&bar_full[(i / n_st) & (kFullBars - 1)][s], (i / (kFullBars * n_st)) & 1, P.err, 2);
                        tc_fence_after();
                        issue_layer1(P, smem_base + s * P.stage_bytes, w_base, d_tmem, leader);
                    } else {
                        tc_fence_after();
                        if (kSmemA) issue_layer_ss(P, l, w_base, d_tmem, smem_base + P.off_a + v * P.a_slot_bytes, leader);
                        else issue_layer_ts(P, l, w_base, d_tmem, a_tmem, leader);
                    }
                    if (leader) umma_commit(&bar_mma[g][q]);
                    __syncwarp();
                }
    } else if (warp < n_wg * 4) {
        // ======================= epilogue warps =======================
        const uint32_t g = warp >> 2, quarter = warp & 3;
        const uint32_t lane_sel = (quarter * 32) << 16;
        // slot-0 constants in registers; slot q adds a multiple (the slot loop stays rolled: one copy of the code in the I-cache)
        const uint32_t slot_cols = P.tmem_wg_cols;
        const uint32_t d_tm0 = tmem_base + g * kSlots * slot_cols + lane_sel;
        const uint32_t bar_mma0 = smem_u32(&bar_mma[g][0]), bar_ready0 = smem_u32(&bar_ready[g][0]);
        const uint32_t a_off = P.tmem_a_off;
        const int n_layers = P.n_layers;
        uint32_t mma_phase = 0;   // one phase bit per slot
        const bool tracing = kTrace && P.trace != nullptr && blockIdx.x == 0 && warp == 0 && lane == 0;
        uint32_t trace_n = 0;
#define BNM_TRACE_POINT() do { if (kTrace && tracing && trace_n < 1000) P.trace[trace_n++] = clock64(); } while (0)

        const uint32_t i_first = g * kSlots, i_slot = 1;
        for (uint32_t r = 0, i0 = i_first; r < n_rounds; r++, i0 += n_virt)
            for (int l = 0; l < n_layers; l++) {
                const uint32_t n_pad_l = P.n_pad[l];
#pragma unroll 1
                for (int q = 0; q < kSlots; q++) {
                    const uint32_t i = i0 + q * i_slot;
                    if (i >= my_tiles) continue;
                    const uint32_t d_tm = d_tm0 + q * slot_cols;
                    BNM_TRACE_POINT();   // step start
                    mbar_wait_a(bar_mma0 + q * 8, (mma_phase >> q) & 1, P.err, 3);
                    mma_phase ^= 1u << q;
                    tc_fence_after();
                    BNM_TRACE_POINT();   // MMAs of layer l+1 complete
                    if (l + 1 < n_layers) {
                        if (l == 0 && quarter == 1 && i + n_st < my_tiles && elect_one()) {   // stage is free
                            if (kFloatIn) mbar_arrive(&bar_free[i % n_st]);
                            else issue_tile_load(i + n_st);
                        }
                        int8_t *tap = nullptr;
                        if (kTaps) {   // rows of a ragged last tile at or beyond n store nothing
                            const size_t img = (size_t)(tile0 + i * tile_step) * kTileM + quarter * 32 + lane;
                            if (P.tap[l] && img < P.n) tap = P.tap[l] + img * P.tap_stride[l];
                        }
                        if (kSmemA) relunorm_smem<kTaps>(d_tm, smem_base + P.off_a + (g * kSlots + q) * P.a_slot_bytes, quarter * 32 + lane, n_pad_l, tap);
                        else if (n_pad_l == 64) relunorm_tmem64<kTaps>(d_tm, d_tm + a_off, tap);
                        else relunorm_tmem<kTaps>(d_tm, d_tm + a_off, n_pad_l, tap);
                        // this thread's reads of D and writes of A are complete: tell the issuer (128 fire-and-forget arrivals per
                        // step; measured faster than syncwarp + one elected arrival: fewer instructions)
                        tc_fence_before();
                        mbar_arrive_a(bar_ready0 + q * 8);
                    } else {
                        // ---- logits + label (dll.c:115-116: the last ReLUNorm's argmax is what Inference() returns).
                        // argmax = first maximum (strict '>' from -INT32_MAX / 255, inference.c:32-37), computed as a max over
                        // keys x*16 + (15-j): equal x -> the smaller j wins.  |x| < 2^27 is guaranteed by the plan (n_in <= 1024,
                        // int8 x int8) so the key cannot overflow; padded columns get -2^30 and can never win.
                        const uint32_t tile = tile0 + i * tile_step;
                        const size_t img = (size_t)tile * kTileM + quarter * 32 + lane;
                        const bool full_tile = (size_t)(tile + 1) * kTileM <= P.n;   // warp-uniform
                        const uint32_t ncls = P.n_classes;
                        int32_t *dst = P.logits + img * ncls;
                        uint32_t pos;
                        if (!kManyClasses) {
                            uint32_t x[16];
                            tmem_ld_x16(d_tm, x);
                            tmem_ld_wait();
                            // the logits now live in registers: the accumulator is free, so the issuer may start the next tile's
                            // layer-1 MMAs (the longest batch) while this warp is still busy with argmax + stores
                            tc_fence_before();
                            mbar_arrive_a(bar_ready0 + q * 8);
                            int key = INT32_MIN;
#pragma unroll
                            for (int j = 0; j < 16; j += 2)
                                key = __vimax3_s32(key, (int)x[j] * 16 + P.kadd[j], (int)x[j + 1] * 16 + P.kadd[j + 1]);
                            pos = 15 - (key & 15);
                            if (full_tile || img < P.n) {
                                auto store_row = [&](int32_t *d) {
                                    if ((ncls & 1) == 0) {   // rows are 8-byte aligned: 64-bit stores straight to HBM (write-combined in L2)
#pragma unroll
                                        for (int j = 0; j < 16; j += 2)
                                            if ((uint32_t)j < ncls) *reinterpret_cast<int2 *>(d + j) = make_int2((int)x[j], (int)x[j + 1]);
                                    } else {
#pragma unroll
                                        for (int j = 0; j < 16; j++)
                                            if ((uint32_t)j < ncls) d[j] = (int)x[j];
                                    }
                                };
                                store_row(dst);
                                if (kGather && !P.off_gstage) {
#pragma unroll 1
                                    for (uint32_t d = 0; d < P.n_log_dst; d++) store_row(P.log_dst[d] + (P.row0 + img) * ncls);   // peers, over NVLink
                                }
                            }
                            if (kGather && P.off_gstage && P.n_log_dst) {
                                // peers: this warp's 32 rows are contiguous at every destination (32 x 4 ncls bytes).  Stage them in
                                // shared memory and push them with ONE bulk copy per destination -- full NVLink packets instead of
                                // 8-byte stores scattered at a 4 ncls stride.  (Compact code on purpose: the kernel's hot loop must
                                // keep fitting the instruction cache.)
                                int32_t *stg = reinterpret_cast<int32_t *>(smem + P.off_gstage) + warp * 32 * ncls;
#pragma unroll
                                for (int j = 0; j < 16; j++)
                                    if ((uint32_t)j < ncls) stg[lane * ncls + j] = (int)x[j];
                                const size_t row = P.row0 + (size_t)tile * kTileM + quarter * 32;
                                if (full_tile) {
                                    fence_proxy_async_smem();
                                    __syncwarp();
                                    if (elect_one()) {
#pragma unroll 1
                                        for (uint32_t d = 0; d < P.n_log_dst; d++) bulk_store_1d(P.log_dst[d] + row * ncls, stg, 128 * ncls);
                                        bulk_commit();
                                        bulk_wait_read<0>();   // the staging rows may be overwritten by this warp's next tile
                                    }
                                } else {   // ragged last tile: the valid rows, word by word (coalesced)
                                    __syncwarp();
                                    const size_t base_img = (size_t)tile * kTileM + quarter * 32;
                                    const uint32_t valid = base_img < P.n ? (uint32_t)min((size_t)32, P.n - base_img) * ncls : 0;
#pragma unroll 1
                                    for (uint32_t d = 0; d < P.n_log_dst; d++) {
                                        int32_t *pd = P.log_dst[d] + row * ncls;
#pragma unroll 1
                                        for (uint32_t idx = lane; idx < valid; idx += 32) pd[idx] = stg[idx];
                                    }
                                }
                                __syncwarp();
                            }
                        } else {
                            int best = -INT32_MAX;
                            pos = 255;
                            for (uint32_t c = 0; c < ncls; c += 16) {
                                uint32_t x[16];
                                tmem_ld_x16(d_tm + c, x);
                                tmem_ld_wait();
                                int key = INT32_MIN;
#pragma unroll
                                for (int j = 0; j < 16; j += 2) {
                                    const int k0 = c + j < ncls ? (int)x[j] * 16 + (15 - j) : INT32_MIN;
                                    const int k1 = c + j + 1 < ncls ? (int)x[j + 1] * 16 + (14 - j) : INT32_MIN;
                                    key = __vimax3_s32(key, k0, k1);
                                }
                                const int cx = key >> 4;
                                if (cx > best) { best = cx; pos = c + 15 - (key & 15); }
                                if (full_tile || img < P.n) {
#pragma unroll
                                    for (int j = 0; j < 16; j++)
                                        if (c + j < ncls) dst[c + j] = (int)x[j];
                                    if (kGather) {
#pragma unroll 1
                                        for (uint32_t d = 0; d < P.n_log_dst; d++) {
                                            int32_t *pd = P.log_dst[d] + (P.row0 + img) * ncls + c;
#pragma unroll
                                            for (int j = 0; j < 16; j++)
                                                if (c + j < ncls) pd[j] = (int)x[j];
                                        }
                                    }
                                }
                            }
                            tc_fence_before();
                            mbar_arrive_a(bar_ready0 + q * 8);
                        }
                        if (full_tile || img < P.n) {
                            if (P.labels) P.labels[img] = pos;
#pragma unroll 1
                            for (uint32_t d = 0; kGather && d < P.n_lab_dst; d++) {
                                if (P.lab_u8) reinterpret_cast<uint8_t *>(P.lab_dst[d])[P.row0 + img] = (uint8_t)pos;
                                else P.lab_dst[d][P.row0 + img] = pos;
                            }
                        }
                    }
                    BNM_TRACE_POINT();   // step end
                }
            }
    }

    if (kFloatIn && warp >= n_wg * 5) {
        // ======================= quantiser warps (float input): warp qw converts rows 16 qw .. 16 qw + 15 of every tile =======================
        // The float rows of a warp's share are contiguous in HBM: they are fetched four rows (4 kB) at a time by one bulk async copy
        // into the warp's own two-slot ring (64 kB in flight per SM: enough to cover the HBM latency).  A pass converts four rows at
        // once, eight lanes per row: a lane holds 32 of its row's floats (eight float4, visited in an order rotated by the row so that
        // the four rows never meet in a bank), so the row maximum needs three shuffles and every lane has 32 independent elements to
        // scale, round and pack.  The int8 words go straight into the image stage the layer-1 MMA reads.
        const uint32_t qw = warp - n_wg * 5;
        const uint32_t elems = P.in_elems, n_f4 = elems >> 2, row_words = P.in_atoms * 32;   // float4 per float row, 4-byte words per int8 row
        const float *src = P.fimages;
        uint8_t *ring = smem + P.off_fring + qw * (2 * kFloatGroupRows * 1024);
        uint64_t *fbar = &bar_fload[qw][0];
        constexpr uint32_t kGroupsPerTile = kFloatRowsPerWarp / kFloatGroupRows;
        const uint32_t n_groups = my_tiles * kGroupsPerTile;   // groups of rows of this warp, in order
        auto group_rows = [&](uint32_t gi, size_t &row) {   // first global row and number of valid rows of group gi
            const uint32_t i = gi / kGroupsPerTile, k = gi % kGroupsPerTile;
            row = (size_t)(tile0 + i * tile_step) * kTileM + qw * kFloatRowsPerWarp + k * kFloatGroupRows;
            return row < P.n ? (uint32_t)min((size_t)kFloatGroupRows, P.n - row) : 0u;
        };
        auto issue_group = [&](uint32_t gi) {
            size_t row;
            const uint32_t valid = group_rows(gi, row);
            if (lane == 0 && valid) {
                mbar_arrive_expect_tx(&fbar[gi & 1], valid * elems * 4);
                bulk_load_1d(ring + (gi & 1) * (kFloatGroupRows * 1024), src + row * elems, valid * elems * 4, &fbar[gi & 1]);
            }
        };
        const uint32_t u = lane >> 3, sub = lane & 7;   // row of the pass, position inside the row's eight-lane team
        uint32_t fphase = 0;   // one phase bit per ring slot
        if (n_groups > 0) issue_group(0);
        if (n_groups > 1) issue_group(1);
        for (uint32_t gi = 0; gi < n_groups; gi++) {
            const uint32_t i = gi / kGroupsPerTile, k = gi % kGroupsPerTile, s = i % n_st;
            if (k == 0 && i >= n_st) mbar_wait(&bar_free[s], ((i / n_st) - 1) & 1, P.err, 8);   // the tile that used this stage is through layer 1
            uint8_t *stage = smem + s * P.stage_bytes;
            size_t row;
            const uint32_t valid = group_rows(gi, row);
            const uint32_t slot = gi & 1;
            if (valid) {
                mbar_wait(&fbar[slot], (fphase >> slot) & 1, P.err, 9);
                fphase ^= 1u << slot;
            }
            const float4 *fr = reinterpret_cast<const float4 *>(ring + slot * (kFloatGroupRows * 1024)) + u * n_f4;
            const uint32_t r = qw * kFloatRowsPerWarp + k * kFloatGroupRows + u;   // this lane's row inside the tile
            float4 v[8];
            float m = 0.f;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t c = sub + 8 * ((j + u) & 7);
                v[j] = (u < valid && c < n_f4) ? fr[c] : make_float4(0.f, 0.f, 0.f, 0.f);
                m = fmaxf(m, fmaxf(fmaxf(fabsf(v[j].x), fabsf(v[j].y)), fmaxf(fabsf(v[j].z), fabsf(v[j].w))));
            }
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 4));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 2));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
            // test_inference.py:140-141 / BitNetMCU.py:435-436, every step one correctly rounded float32 operation
            const float scale = __fdiv_rn(127.0f, fmaxf(m, 1e-5f));
            auto q = [&](float x) { int d; asm("cvt.rni.sat.s8.f32 %0, %1;" : "=r"(d) : "f"(__fmul_rn(x, scale))); return (uint32_t)d; };   // round half to even, clip to int8
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t c = sub + 8 * ((j + u) & 7);   // word c of the int8 row (bytes 4c .. 4c+3)
                const uint32_t w = __byte_perm(__byte_perm(q(v[j].x), q(v[j].y), 0x0040), __byte_perm(q(v[j].z), q(v[j].w), 0x0040), 0x5410);
                // SWIZZLE_128B: 16-byte chunk jc of row r sits at chunk position jc ^ (r & 7) of the row's 128 bytes in its atom
                if (c < row_words)
                    *reinterpret_cast<uint32_t *>(stage + (c >> 5) * 16384 + r * 128 + ((((c & 31) >> 2) ^ (r & 7)) << 4) + (c & 3) * 4) = w;
            }
            __syncwarp();   // every lane has read its floats of this slot
            if (gi + 2 < n_groups) issue_group(gi + 2);
            if (k == kGroupsPerTile - 1) {
                fence_proxy_async_smem();   // the layer-1 MMAs (async proxy) read what these generic-proxy stores wrote
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_full[(i / n_st) & (kFullBars - 1)][s]);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (kTrace && P.trace && blockIdx.x == 0 && tid == 0) P.trace[1022] = clock64();   // all roles done
    if (kTrace && P.trace && tid == 0) {
        unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt)); P.trace[1025 + 2 * blockIdx.x] = (long long)gt;
        uint32_t smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); P.trace[1400 + blockIdx.x] = smid;
    }
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

static uint32_t round_up(uint32_t v, uint32_t m) { return (v + m - 1) / m * m; }

FcChainPlan *fc_chain_plan_create(const FcLayerDev *layers, int n_layers, uint32_t in_bytes, int device, int sm_count,
                                  char *err, size_t err_len) {
    auto fail = [&](const char *msg) -> FcChainPlan * { if (err) snprintf(err, err_len, "%s", msg); return nullptr; };
    if (n_layers < 1 || n_layers > kMaxFcLayers) return fail("fused path: 1..8 FC layers");
    if (in_bytes % 16 || in_bytes == 0 || in_bytes > 1024) return fail("fused path: input row must be a multiple of 16 bytes, <= 1024");
    if (!get_encode_fn()) return fail("cuTensorMapEncodeTiled not available");
    auto *plan = new FcChainPlan();
    ChainParams &p = plan->p;
    p.n_layers = n_layers;
    p.in_atoms = (in_bytes + 127) / 128;   // weights past the real input width multiply zero activations: dropped
    p.stage_bytes = p.in_atoms * 16384;
    uint32_t w_off = 0, d_cols = 0, a_cols = 0;
    for (int l = 0; l < n_layers; l++) {
        const FcLayerDev &L = layers[l];
        if (L.n_pad > 256) { delete plan; return fail("fused path: layer wider than 256 outputs"); }
        p.n_pad[l] = L.n_pad;
        p.n_real[l] = L.n_out;
        // K of layer l > 0: the activations past the previous layer's (padded) width are zero -- e.g. Ternary pads n_in to a
        // multiple of 10 with zero trits (64 -> 70, exportquant.py:132-137) -- so those K-steps are dropped, exactly
        p.k_steps[l] = l == 0 ? p.in_atoms * 4 : round_up(std::min(L.k_pad, layers[l - 1].n_pad), 32) / 32;
        p.planes[l] = L.dense_b ? 2 : 1;
        p.b_off[l] = w_off;
        p.idesc[l] = make_idesc_i8(128, L.n_pad);
        w_off += p.planes[l] * p.k_steps[l] * L.n_pad * 32;
        d_cols = std::max(d_cols, L.n_pad);
        if (l > 0) a_cols = std::max(a_cols, std::max(p.k_steps[l] * 32, layers[l - 1].n_pad) / 4);
    }
    p.w_bytes = w_off;
    p.n_classes = layers[n_layers - 1].n_out;
    for (int l = 0; l + 1 < n_layers; l++) p.tap_stride[l] = layers[l + 1].k_pad;
    p.tmem_a_off = round_up(d_cols, 32);
    p.tmem_wg_cols = p.tmem_a_off + round_up(std::max(a_cols, 1u), 16);
    if (p.tmem_wg_cols > 512) { delete plan; return fail("fused path: model does not fit the 512 TMEM columns"); }
    {   // Tiles in flight per CTA = n_wg warpgroups x n_slots slots, bounded by the 512 TMEM columns.  Measured on B200, us per
        // 2^20 images, warpgroups x slots: 4bitsym-64 2x1 93, 2x2 73.5, 3x1 72.2, 3x2 62.5, 4x1 63.6, four warpgroups with six slots
        // 64.0; 2bitsym-96 (four slots fit) 2x2 98.7, three warpgroups with four slots 95.7, 4x1 81.3.  Epilogue warps matter
        // more than slots until three warpgroups have two slots each; a fourth warpgroup then buys nothing.
        const uint32_t fit = 512 / p.tmem_wg_cols;
        if (fit >= 6) { p.n_wg = 3; p.n_slots = 2; }
        else { p.n_wg = std::min<uint32_t>(kMaxWG, fit); p.n_slots = 1; }
        if (const char *e = getenv("BNM_WG")) {                                                                   // tuning knobs
            p.n_wg = std::max(1, std::min<int>((int)std::min<uint32_t>(kMaxWG, fit), atoi(e)));
            p.n_slots = p.n_wg <= kMaxWG2 ? std::min<uint32_t>(kMaxSlots, fit / p.n_wg) : 1;
        }
        if (const char *e = getenv("BNM_SLOTS")) p.n_slots = p.n_wg <= kMaxWG2 ? std::max(1, std::min<int>((int)std::min<uint32_t>(kMaxSlots, fit / p.n_wg), atoi(e))) : 1;
    }
    const uint32_t smem_limit = 227 * 1024 - 1024 /*alignment slack*/ - 1024 /*static: barriers*/;
    p.off_w = 0;  // set below: stages first (1024-aligned), then weights
    uint32_t fixed = round_up(p.w_bytes, 128);
    if (fixed + 2 * p.stage_bytes > smem_limit) { delete plan; return fail("fused path: weights do not fit in shared memory"); }
    p.n_stages = std::min<uint32_t>(kMaxStages, (smem_limit - fixed) / p.stage_bytes);
    p.n_stages = std::min<uint32_t>(p.n_stages, 6);
    p.off_w = p.n_stages * p.stage_bytes;
    plan->smem_bytes = (size_t)p.off_w + round_up(p.w_bytes, 128) + 1024;
    // One CTA per SM is part of the launch-overlap contract (launch k+2 must never run next to launch k on an SM): registers and
    // TMEM do not enforce it (launch_dependents fires before tmem_alloc blocks), shared memory does once a CTA asks for more than
    // half of the SM's 227 kB.
    plan->smem_bytes = std::max<size_t>(plan->smem_bytes, 116 * 1024);
    if (in_bytes <= 256 && p.n_classes <= 16) {   // float-input path
        const uint32_t fring = kFloatQuantWarps * 2 * kFloatGroupRows * 1024;
        const uint32_t fixed_f = round_up(p.w_bytes, 128) + fring;
        if (fixed_f + 2 * p.stage_bytes <= smem_limit) {
            plan->f_n_stages = std::min<uint32_t>(4, (smem_limit - fixed_f) / p.stage_bytes);
            plan->f_off_w = plan->f_n_stages * p.stage_bytes;
            plan->f_off_fring = plan->f_off_w + round_up(p.w_bytes, 128);
            plan->f_smem_bytes = std::max<size_t>((size_t)plan->f_off_fring + fring + 1024, 116 * 1024);
        }
    }
    if (p.n_classes <= 16) {   // staged peer stores: 12 warps x 32 rows x 4 n_classes bytes next to the weights
        const uint32_t gstage = kMaxWG * 4 * 128 * p.n_classes;
        const uint32_t fixed_g = round_up(p.w_bytes, 128) + round_up(gstage, 128);
        if (fixed_g + 2 * p.stage_bytes <= smem_limit) {
            plan->g_n_stages = std::min<uint32_t>(p.n_stages, (smem_limit - fixed_g) / p.stage_bytes);
            plan->g_off_w = plan->g_n_stages * p.stage_bytes;
            plan->g_off_gstage = plan->g_off_w + round_up(p.w_bytes, 128);
            plan->g_smem_bytes = std::max<size_t>((size_t)plan->g_off_gstage + round_up(gstage, 128) + 1024, 116 * 1024);
        }
    }
    {   // wide models: with the activations in shared memory a slot is the accumulator alone -- used when that buys a third slot
        const uint32_t fit = 512 / p.tmem_wg_cols, acc_cols = round_up(d_cols, 32), acc_fit = 512 / acc_cols;
        uint32_t a_row = 0;
        for (int l = 1; l < n_layers; l++) a_row = std::max(a_row, p.k_steps[l] * 32);
        const uint32_t wg = std::min<uint32_t>(kMaxWG2, acc_fit), a_slot = kTileM * a_row;
        const uint32_t fixed_a = round_up(p.w_bytes, 128) + wg * a_slot;
        const char *knob = getenv("BNM_SMEM_A");   // tuning knob: 0 = never
        if (fit <= 2 && acc_fit > fit && n_layers > 1 && p.n_classes <= 16 && !(knob && atoi(knob) == 0) &&
            fixed_a + 2 * p.stage_bytes <= smem_limit) {
            plan->sa_n_wg = wg;
            plan->sa_tmem_wg_cols = acc_cols;
            plan->sa_a_slot_bytes = a_slot;
            plan->sa_n_stages = std::min<uint32_t>(6, (smem_limit - fixed_a) / p.stage_bytes);
            plan->sa_off_w = plan->sa_n_stages * p.stage_bytes;
            plan->sa_off_a = plan->sa_off_w + round_up(p.w_bytes, 128);
            plan->sa_smem_bytes = std::max<size_t>((size_t)plan->sa_off_a + wg * a_slot + 1024, 116 * 1024);
        }
    }
    if (getenv("BNM_VERBOSE"))   // diagnostics: the shapes this plan launches
        fprintf(stderr, "bitnetmcu_b200: fused FC plan: %u warpgroups x %u slots, %u TMEM columns per slot, %u stages, %u weight bytes; "
                        "smem-activation form: %u warpgroups, %u stages, %zu B smem\n", p.n_wg, p.n_slots, p.tmem_wg_cols, p.n_stages, p.w_bytes,
                plan->sa_n_wg, plan->sa_n_stages, plan->sa_smem_bytes);
    if (const char *e = getenv("BNM_TRACE")) plan->trace_path = e;                                   // diagnostics, read once
    if (const char *e = getenv("BNM_STAGGER_NS")) plan->stagger_override = (int)(atof(e) * 1.8);     // tuning knob; ~1.8 cycles per ns under load
    for (int j = 0; j < 16; j++) p.kadd[j] = (uint32_t)j < p.n_classes ? 15 - j : -(1 << 30);
    plan->threads = p.n_wg * 160;   // 4 epilogue warps + 1 issuer warp per warpgroup
    plan->in_bytes = in_bytes;
    plan->sm_count = sm_count;
    plan->device = device;

    // weight image
    if (cudaMalloc(&plan->d_w_image, p.w_bytes) != cudaSuccess || cudaHostAlloc(&plan->h_err, sizeof(int), cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(&plan->d_err, plan->h_err, 0) != cudaSuccess) {
        fc_chain_plan_destroy(plan);
        return fail("cudaMalloc failed (weight image)");
    }
    cudaMemset(plan->d_w_image, 0, p.w_bytes);
    *plan->h_err = 0;
    for (int l = 0; l < n_layers; l++) {
        const FcLayerDev &L = layers[l];
        for (uint32_t pl = 0; pl < p.planes[l]; pl++) {
            size_t total = (size_t)L.n_pad * p.k_steps[l] * 32;
            k_build_b_image<<<(unsigned)((total + 255) / 256), 256>>>(pl ? L.dense_b : L.dense_a, L.k_pad, L.n_pad, p.k_steps[l],
                                                                      plan->d_w_image + p.b_off[l] + (size_t)pl * p.k_steps[l] * L.n_pad * 32);
        }
    }
    if (cudaDeviceSynchronize() != cudaSuccess) { fc_chain_plan_destroy(plan); return fail("weight image kernel failed"); }
    p.w_image = plan->d_w_image;
    p.err = plan->d_err;
    const int smem_any = (int)std::max(std::max(plan->smem_bytes, plan->g_smem_bytes), std::max(plan->f_smem_bytes, plan->sa_smem_bytes));
    if (cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, true, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, false, false, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, true, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<2, false, false, true, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false, false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, true, false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess ||
        cudaFuncSetAttribute(fc_chain_kernel<1, false, false, false, false, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_any) != cudaSuccess) {
        fc_chain_plan_destroy(plan);
        return fail("cannot opt in to the required dynamic shared memory");
    }
    return plan;
}

void fc_chain_plan_set_overlap(FcChainPlan *p, int mode) {
    if (!p) return;
    p->overlap = mode;
    p->prev_valid = false;
    // Overlapped launches find HBM uncongested, all six first tiles of a CTA land within ~1 us and the three warpgroups
    // would run in lockstep, competing for the ALU pipe at the same moments (measured -3 %).  Start warpgroup g no earlier
    // than g x 2 us after kernel entry (a third of the ~6 us round).  Plain launches get the same offsets for free from
    // the start-up burst (tile i of an SM arrives ~0.8 us after tile i-1), there the delay only costs ramp time.
    p->p.stagger_cycles = mode == 2 ? 3600 : 0;
}

void fc_chain_plan_destroy(FcChainPlan *p) {
    if (!p) return;
    if (p->d_w_image) cudaFree(p->d_w_image);
    if (p->h_err) {
        if (*p->h_err) fprintf(stderr, "bitnetmcu_b200: fused FC kernel: bounded wait %d timed out (device trap)\n", *p->h_err);
        cudaFreeHost(p->h_err);
    }
    delete p;
}

static const CUtensorMap *plan_tensor_map(FcChainPlan *plan, const int8_t *in, size_t n) {
    for (auto &t : plan->tmaps)
        if (t.ptr == in && t.n == n) return &t.map;
    FcChainPlan::TmapSlot &t = plan->tmaps[plan->tmap_next++ % 4];
    memset(&t.map, 0, sizeof(t.map));
    cuuint64_t gdim[2] = {(cuuint64_t)plan->in_bytes, (cuuint64_t)n};
    cuuint64_t gstride[1] = {(cuuint64_t)plan->in_bytes};
    cuuint32_t box[2] = {128, (cuuint32_t)kTileM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = get_encode_fn()(&t.map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t *>(in), gdim, gstride, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { t.ptr = nullptr; t.n = 0; return nullptr; }
    t.ptr = in;
    t.n = n;
    return &t.map;
}

int fc_chain_launch(FcChainPlan *plan, const int8_t *in, size_t n, int32_t *logits, uint32_t *labels, const GatherDst *gather,
                    cudaStream_t st, const FcTaps *taps) {
    if (n == 0) return 0;
    if (n > 0x7fffff00ull) return -2;
    if (taps && gather) return -7;
    ChainParams p = plan->p;
    if (taps)
        for (int l = 0; l + 1 < p.n_layers; l++) p.tap[l] = taps->act[l];
    p.logits = logits;
    p.labels = labels;
    p.n = n;
    p.n_lab_dst = p.n_log_dst = 0;
    p.row0 = 0;
    p.lab_u8 = 0;
    if (gather) {
        if (gather->n_labels_dst > (uint32_t)kMaxGatherDst || gather->n_logits_dst > (uint32_t)kMaxGatherDst) return -5;
        p.n_lab_dst = gather->n_labels_dst;
        p.n_log_dst = gather->n_logits_dst;
        p.row0 = gather->row_offset;
        p.lab_u8 = gather->labels_u8 && p.n_classes <= 255;
        if (gather->labels_u8 && !p.lab_u8) return -5;
        for (uint32_t d = 0; d < p.n_lab_dst; d++) p.lab_dst[d] = gather->labels_dst[d];
        for (uint32_t d = 0; d < p.n_log_dst; d++) p.log_dst[d] = gather->logits_dst[d];
    }
    size_t smem_bytes = plan->smem_bytes;
    p.off_gstage = 0;
    if (p.n_log_dst && plan->g_smem_bytes && (p.row0 * p.n_classes) % 4 == 0) {   // 16-byte aligned destination rows: staged bulk stores
        bool aligned = true;
        for (uint32_t d = 0; d < p.n_log_dst; d++) aligned = aligned && ((uintptr_t)p.log_dst[d] & 15) == 0;
        if (aligned) {
            p.n_stages = plan->g_n_stages;
            p.off_w = plan->g_off_w;
            p.off_gstage = plan->g_off_gstage;
            smem_bytes = plan->g_smem_bytes;
        }
    }
    p.n_tiles = (uint32_t)((n + kTileM - 1) / kTileM);
    const CUtensorMap *tmap_p = plan_tensor_map(plan, in, n);
    if (!tmap_p) return -3;
    const CUtensorMap &tmap = *tmap_p;
    unsigned grid = (unsigned)std::min<uint32_t>(p.n_tiles, (uint32_t)plan->sm_count);
    long long *d_trace = nullptr;
    const char *trace_path = (plan->trace_path.empty() || gather || taps || plan->p.n_classes > 16 || p.n_wg > (uint32_t)kMaxWG2) ? nullptr : plan->trace_path.c_str();   // diagnostics build path
    if (trace_path) { cudaMalloc(&d_trace, 2048 * sizeof(long long)); cudaMemset(d_trace, 0, 2048 * sizeof(long long)); }
    p.trace = d_trace;
    // Mode 2 drops the grid-dependency wait, i.e. EVERY ordering against the work enqueued before this launch on the stream
    // (the previous bnm launch and any producer kernel of `images` alike).  The library keeps the wait whenever it can see the
    // promise being broken: first launch on this plan / another stream / a buffer of the previous launch reused.
    // A taps launch is a plain launch whatever the overlap mode (its rows are a debugging aid, not a throughput path), and the
    // launch after it is not declared independent of it.
    const int overlap = taps ? 0 : plan->overlap;
    bool independent = overlap == 2 && plan->prev_valid && plan->prev_stream == st && in != plan->prev_in &&
                       logits != plan->prev_logits && (labels == nullptr || labels != plan->prev_labels);
    p.wait_prior_grid = !independent;
    p.early_trigger = overlap != 0 && grid == (unsigned)plan->sm_count;
    if (taps) p.stagger_cycles = 0;
    if (plan->stagger_override >= 0) p.stagger_cycles = (uint32_t)plan->stagger_override;
    plan->prev_in = in; plan->prev_logits = logits; plan->prev_labels = labels; plan->prev_stream = st; plan->prev_valid = !taps;
    if (trace_path) {
        if (p.n_slots == 1) fc_chain_kernel<1, true, false, false><<<grid, plan->threads, plan->smem_bytes, st>>>(tmap, p);
        else fc_chain_kernel<2, true, false, false><<<grid, plan->threads, plan->smem_bytes, st>>>(tmap, p);
    } else {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3((unsigned)plan->threads);
        cfg.dynamicSmemBytes = smem_bytes;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = overlap ? 1 : 0;
        const bool g = p.n_lab_dst || p.n_log_dst;
        const bool many = p.n_classes > 16;
        const bool smem_a = !g && !many && plan->sa_smem_bytes != 0;
        if (smem_a) {
            p.n_wg = plan->sa_n_wg; p.n_slots = 1;
            p.tmem_wg_cols = plan->sa_tmem_wg_cols;
            p.n_stages = plan->sa_n_stages; p.off_w = plan->sa_off_w; p.off_a = plan->sa_off_a; p.a_slot_bytes = plan->sa_a_slot_bytes;
            cfg.blockDim = dim3(p.n_wg * 160);
            cfg.dynamicSmemBytes = plan->sa_smem_bytes;
        }
        cudaError_t e;
#define BNM_LAUNCH(S, G, M) e = cudaLaunchKernelEx(&cfg, fc_chain_kernel<S, false, G, M>, tmap, p)
#define BNM_LAUNCH4(G, M) e = cudaLaunchKernelEx(&cfg, fc_chain_kernel<1, false, G, M, false, true>, tmap, p)
#define BNM_LAUNCH_T(S, M, W4) e = cudaLaunchKernelEx(&cfg, fc_chain_kernel<S, false, false, M, false, W4, false, true>, tmap, p)
        if (taps) {
            if (smem_a) e = cudaLaunchKernelEx(&cfg, fc_chain_kernel<1, false, false, false, false, false, true, true>, tmap, p);
            else if (p.n_wg > (uint32_t)kMaxWG2) { if (many) BNM_LAUNCH_T(1, true, true); else BNM_LAUNCH_T(1, false, true); }
            else if (p.n_slots == 1) { if (many) BNM_LAUNCH_T(1, true, false); else BNM_LAUNCH_T(1, false, false); }
            else { if (many) BNM_LAUNCH_T(2, true, false); else BNM_LAUNCH_T(2, false, false); }
        } else if (smem_a) e = cudaLaunchKernelEx(&cfg, fc_chain_kernel<1, false, false, false, false, false, true>, tmap, p);
        else if (p.n_wg > (uint32_t)kMaxWG2) { if (g) { if (many) BNM_LAUNCH4(true, true); else BNM_LAUNCH4(true, false); } else { if (many) BNM_LAUNCH4(false, true); else BNM_LAUNCH4(false, false); } }
        else if (p.n_slots == 1) { if (g) { if (many) BNM_LAUNCH(1, true, true); else BNM_LAUNCH(1, true, false); } else { if (many) BNM_LAUNCH(1, false, true); else BNM_LAUNCH(1, false, false); } }
        else { if (g) { if (many) BNM_LAUNCH(2, true, true); else BNM_LAUNCH(2, true, false); } else { if (many) BNM_LAUNCH(2, false, true); else BNM_LAUNCH(2, false, false); } }
#undef BNM_LAUNCH
#undef BNM_LAUNCH4
#undef BNM_LAUNCH_T
        if (e != cudaSuccess) return -4;
    }
    if (trace_path) {   // diagnostics only: synchronous dump of the phase clocks
        std::vector<long long> h(2048);
        cudaStreamSynchronize(st);
        cudaMemcpy(h.data(), d_trace, 2048 * sizeof(long long), cudaMemcpyDeviceToHost);
        cudaFree(d_trace);
        if (FILE *f = fopen(trace_path, "w")) {
            for (int i = 0; i < 1000 && h[i]; i++) fprintf(f, "%lld\n", h[i]);
            fprintf(f, "# entry %lld prologue_done %lld exit %lld\n", h[1020], h[1021], h[1022]);
            {   // per-CTA lifetime from %globaltimer (ns): spread of entry and exit times over the grid
                long long e0 = h[1024], e1 = h[1024], x0 = h[1025], x1 = h[1025];
                for (unsigned b = 0; b < grid && b < 500; b++) {
                    e0 = std::min(e0, h[1024 + 2 * b]); e1 = std::max(e1, h[1024 + 2 * b]);
                    x0 = std::min(x0, h[1025 + 2 * b]); x1 = std::max(x1, h[1025 + 2 * b]);
                }
                for (unsigned b = 0; b < grid && b < 500; b++) fprintf(f, "### cta %u lifetime_ns %lld smid %lld\n", b, h[1025 + 2 * b] - h[1024 + 2 * b], h[1400 + b]);
                fprintf(f, "## globaltimer ns: CTA entry spread %lld, first entry -> first exit %lld, first entry -> last exit %lld\n", e1 - e0, x0 - e0, x1 - e0);
            }
            fprintf(f, "## since entry: barriers %lld, loads issued %lld, tmem alloc %lld\n", h[1016] - h[1020], h[1017] - h[1020], h[1018] - h[1020]);
            fclose(f);
        }
    }
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

bool fc_chain_float_input_supported(const FcChainPlan *plan) {
    return plan && plan->f_smem_bytes != 0 && plan->in_bytes % 16 == 0;
}

// float32 images [n][in_bytes elements] -> logits / labels, the input scaling fused into the load stage (kFloatIn)
int fc_chain_launch_f32(FcChainPlan *plan, const float *in, size_t n, int32_t *logits, uint32_t *labels, cudaStream_t st) {
    if (n == 0) return 0;
    if (n > 0x7fffff00ull) return -2;
    if (!fc_chain_float_input_supported(plan)) return -6;
    ChainParams p = plan->p;
    p.logits = logits;
    p.labels = labels;
    p.n = n;
    p.n_lab_dst = p.n_log_dst = 0;
    p.row0 = 0;
    p.lab_u8 = 0;
    p.off_gstage = 0;
    p.fimages = in;
    p.in_elems = plan->in_bytes;
    if (p.n_wg > kFloatWG) {   // two epilogue warpgroups next to the quantiser warps, two slots each when TMEM allows
        p.n_wg = kFloatWG;
        p.n_slots = std::min<uint32_t>(kMaxSlots, (512 / p.tmem_wg_cols) / kFloatWG);
    }
    p.n_stages = plan->f_n_stages;
    p.off_w = plan->f_off_w;
    p.off_fring = plan->f_off_fring;
    p.n_tiles = (uint32_t)((n + kTileM - 1) / kTileM);
    p.trace = nullptr;
    p.wait_prior_grid = 1;
    p.early_trigger = 0;
    CUtensorMap tmap;   // not used by the float-input kernel (no TMA image loads)
    memset(&tmap, 0, sizeof(tmap));
    const unsigned grid = (unsigned)std::min<uint32_t>(p.n_tiles, (uint32_t)plan->sm_count);
    const unsigned threads = p.n_wg * 160 + 32 * kFloatQuantWarps;   // epilogue + issuer warps + the quantiser warps
    if (p.n_slots == 1) fc_chain_kernel<1, false, false, false, true><<<grid, threads, plan->f_smem_bytes, st>>>(tmap, p);
    else fc_chain_kernel<2, false, false, false, true><<<grid, threads, plan->f_smem_bytes, st>>>(tmap, p);
    plan->prev_valid = false;
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

}  // namespace bnm
