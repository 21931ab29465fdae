// bf16 tensor-core fused Conv1d stack for sm_100a: implicit GEMM on tcgen05
// with accumulators in TMEM and activations resident in shared memory across
// all layers.
//
// Replaces input_layer + frame_encoder (emphases/model/core.py:92-94,
// emphases/model/layers/convolution.py:13-37), i.e. the 7 frame-resolution
// Conv1d(80 -> 80, k, 'same') layers that hold 99 % of the model FLOPs, and
// the word decoder; kernel sizes 1, 3 (the default), 5 and 7 (the reference's
// hyper-parameter sweep) at 80 channels.
//
// GEMM view of one layer on a tile of 128 packed rows:
//     D[128 rows][80 out] = sum_{tap} A_tap[128 rows][80 in] * W_tap[80 in][80 out]
// A lives in smem as bf16 in the no-swizzle K-major "interleaved" UMMA layout
// [k-group of 8 channels][row][8 channels] with all rows of a k-group
// contiguous (SBO = 128 B), so the row shift of tap t is just a 16-byte
// multiple added to the descriptor start address: the same buffer feeds all
// k taps.  Each k-group carries (k - 1) / 2 zero pad rows at each end (one at
// k = 1), so the shifted reads stay inside it.  B (weights) uses the same
// layout per tap, streamed per layer from L2 into a 2- or 3-stage smem ring
// with cp.async.bulk + mbarrier.  D is a 128-lane x 80-column fp32
// accumulator in TMEM.
//
// The CTAs run in clusters of two (a CTA pair on one TPC).  Every MMA is a
// cta_group::2 M=256 instruction issued by rank 0: each CTA supplies the 128
// rows of its own tile as A and holds half of the weights (40 output columns)
// as B, and each CTA's TMEM receives its own 128 x 80 accumulator.  Per SM that
// is the same math as an M=128 MMA with half of the B bytes to fetch from
// shared memory; one such pair MMA costs 47 clk against 102 clk for each of
// the two cta_group::1 MMAs it replaces (profiles/r06_umma_2cta_microbench.md).
// Pair tile p is tiles 2p (rank 0) and 2p + 1 (rank 1).
//
// Warp roles (persistent CTA, one per SM, kSlots tiles in flight):
//   warps 4s .. 4s+3 : epilogue group of tile slot s (TMEM lane quadrant =
//                      warp % 4): tcgen05.ld -> +bias -> activation ->
//                      separator-row zeroing -> bf16 -> back into the slot's
//                      A buffer (next layer's operand), fp32 to HBM after the
//                      last layer
//   warp 4*kSlots    : rank 0: MMA issuer for the pair (one elected lane
//                      issues tcgen05.mma); rank 1: tells rank 0 when its
//                      half of a ring stage has landed
//   warp 4*kSlots+1  : weight producer (cp.async.bulk of this CTA's half)
// While the tensor core works on slot s, the epilogue groups of the other
// slots drain their accumulators, so MMA and epilogue overlap.
#include <cuda_bf16.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"

namespace emph {

namespace tc {

#ifdef EXP_TRACE
// timeline of CTA 0 (tuning builds only): [event][index] clock64 values;
// events 8 + s: the epilogue group of slot s sees mma_done[s]; 12 .. 16
// (slot 0, index = round): tile boundary, see tools/conv_trace.py
constexpr int kTraceEvents = 17;
__device__ long long g_trace[kTraceEvents][512];
#define TRACE(ev, idx) do { if (blockIdx.x == 0 && (idx) < 512) g_trace[ev][idx] = clock64(); } while (0)
#else
#define TRACE(ev, idx) do {} while (0)
#endif

constexpr int C = 80;                 // channels (in = out)
constexpr int KG = C / 8;             // k-groups of 8 channels
constexpr int M = 128;                // rows per tile = UMMA M
constexpr int kStages = 3;            // weight ring
constexpr int kMaxLayers = 16;
constexpr int kSmemLimit = 232448;    // dynamic shared memory one block may opt in to
// Operand buffer of one slot and part, per kernel size: the tile's M rows
// with pad_rows(k) zero rows at each end of every k-group, so that tap t of
// row r reads buffer row r + t + pad_rows(k) - (k - 1) / 2 and never leaves
// the k-group.  k = 1 keeps one pad row each side, as k = 3 does.
__host__ __device__ constexpr int pad_rows(int ks) { return ks > 3 ? (ks - 1) / 2 : 1; }
__host__ __device__ constexpr int buffer_rows(int ks) { return M + 2 * pad_rows(ks); }  // 130 / 132 / 134
__host__ __device__ constexpr int act_bytes(int ks) { return KG * buffer_rows(ks) * 16; }  // 20,800 at k = 3
// parts of a slot lie this far apart: act_bytes rounded up to 128-B alignment
__host__ __device__ constexpr int act_stride(int ks) { return (act_bytes(ks) + 127) / 128 * 128; }
constexpr int CH = C / 2;             // output columns of the weight half one CTA holds
constexpr int W_TAP_BYTES = KG * C * 16;          // 12,800 (both halves)
constexpr int W_HALF_TAP_BYTES = KG * CH * 16;    // 6,400
constexpr int W_BIAS_BYTES = 2 * C * 16;          // bias chunk: 2 k-groups, 2,560
// per kernel size (3, 5, 7: the conv stacks; 1: the per-row linear maps of
// the Transformer variant): bytes of one blob entry, and of the half of its taps
// that one CTA of a pair loads into a ring stage
__host__ __device__ constexpr int conv_bytes(int ks) { return ks * W_TAP_BYTES; }                  // 38,400 at k = 3
__host__ __device__ constexpr int half_bytes(int ks) { return ks * W_HALF_TAP_BYTES; }             // 19,200 at k = 3
__host__ __device__ constexpr int layer_bytes(int ks) { return conv_bytes(ks) + W_BIAS_BYTES; }    // 40,960 at k = 3
constexpr int kTmemCols = 512;

// PARTS = 1: plain bf16 operands (2e-3 mode), 4 tile slots.
// PARTS = 2: "bf16x3" -- activations and weights are each split into a bf16 hi
//   and lo part and every product is formed as hi*hi + lo*hi + hi*lo (three
//   MMAs into the same fp32 accumulator, the lo*lo term ~2^-16 is dropped):
//   16 mantissa bits per operand from the bf16 tensor pipe, ~1e-5-class
//   results.  Two operand buffers per slot (2 slots fit); a layer's weights
//   arrive as two ring entries (W_hi + bias chunk, W_lo).
// PARTS = 3: "bf16x6" -- hi + mid + lo (24 mantissa bits, i.e. all of fp32) and
//   the six products whose weight is above 2^-24: hh, mh, lh, hm, mm, hl.
//   fp32-grade results (the tensor-core form of the exact mode); three operand
//   buffers per slot, three ring entries per layer, a two-stage ring.
// In general ring entry e (weight part e) multiplies activation parts 0 ..
// PARTS-1-e.
template <int PARTS>
struct Config {
    static constexpr int kSlots = PARTS == 1 ? 4 : 2;
    static constexpr int kParts = PARTS;
    static constexpr int kThreads = 128 * kSlots + 64;
    static constexpr int kEntriesPerLayer = PARTS;
    static constexpr int kRing = PARTS == 3 ? 2 : kStages;     // weight ring stages
    // The tensor core accumulates with truncation, so every MMA costs ~2^-24 of
    // the ACCUMULATOR's magnitude: products of the same order (hi*hi | mid*hi,
    // hi*mid | ...) therefore go to their own accumulator ("class" = weight
    // part + activation part) and the epilogue adds the classes in fp32.
    static constexpr int kClasses = PARTS;
    static constexpr int kClassStride = PARTS == 3 ? 80 : 128;   // TMEM columns
    static constexpr int kSlotStride = PARTS == 1 ? 128 : 256;
};

template <int PARTS, int KSIZE>
struct __align__(128) Smem {
    static constexpr int kSlots = Config<PARTS>::kSlots;
    uint8_t act[kSlots][Config<PARTS>::kParts][act_stride(KSIZE)];
    uint8_t w[Config<PARTS>::kRing][half_bytes(KSIZE)];   // this CTA's weight half
    float bias[kMaxLayers][C];                // fp32 bias, added by the epilogue
    uint64_t w_full[kStages];                 // this CTA's half landed
    uint64_t peer_full[kStages];              // rank 0 only: rank 1's half landed
    uint64_t w_empty[kStages];                // the pair's MMAs are done with the stage
    uint64_t act_ready[kSlots];               // rank 0 only: both tiles' operands stored
    uint64_t mma_done[kSlots];
    uint32_t tmem_base;
};

struct Acts {
    int act[kMaxLayers];
};

// Word pooling fused into the last layer's epilogue (emphases/model/core.py:
// 96-101: downsample at the 'intermediate' location).  row_word[g] is the word
// row that packed frame row g belongs to, or -1.  A row of the tile is a TMEM
// lane, 32 consecutive rows are a warp, and the rows of a word are consecutive,
// so a warp reduces its (one to three) word runs itself: the 16 columns of an
// epilogue chunk are transposed through a warp-private piece of the slot's idle
// operand buffer (lane = row writes, lane = (row parity, column) reads), every
// lane adds the consecutive rows of its column and parity and flushes one value
// per run end:
//   kPoolSum    pieces of <= 16 rows are summed in fp32 in row order, converted
//               to 64-bit fixed point (2^-28 units) and added to the word with
//               an integer atomic: integer addition is associative, so the
//               result does not depend on the order the atomics land (bit-
//               identical run to run).  (The first version summed every element
//               in fixed point with a segmented shuffle scan -- 800 shuffles per
//               warp and tile, 1.68 ms against 1.27 + 0.24 unfused; a variant
//               with redux.sync over the segment's lanes measured 3.2 ms.)
//   kPoolMax    maximum of non-negative values (ReLU output) as an integer
//               atomic max on the float's bit pattern; the buffer starts at 0
//   kPoolCenter row_word marks only the centre row of each word: a plain store
enum { kPoolNone = 0, kPoolSum = 1, kPoolMax = 2, kPoolCenter = 3 };
constexpr float kPoolFixedScale = 268435456.f;         // 2^28
constexpr float kPoolFixedClamp = 524288.f;            // 2^19: 2^16 rows of it fit int64
struct PoolArgs {
    const int32_t* row_word;     // [total_rows]
    long long* fixed;            // kPoolSum: [word rows][C] fixed-point sums (zeroed)
    float* out;                  // kPoolMax / kPoolCenter: [word rows][C] (zeroed)
    int mode;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile(
        "{\n\t.reg .b64 state;\n\t"
        "mbarrier.arrive.expect_tx.shared::cta.b64 state, [%0], %1;\n\t}"
        ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    const uint32_t addr = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    } while (!done);
}
// wait with acquire at cluster scope: the barrier's arrivals come from the
// peer CTA too
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    const uint32_t addr = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    } while (!done);
}
// arrive on the barrier at the same offset in CTA 0 of the cluster.
// This knowingly departs from the PTX memory model: the arrive uses the
// default .release.cta semantics, and a cta-scope release in rank 1 is not
// morally strong with rank 0's cluster-scope acquire.  The hand-off of rank
// 1's operand stores to the MMA that rank 0 issues therefore rests on the
// hardware's causality order, the same as the remote arrives of CUTLASS's
// cluster pipelines (ClusterBarrier::arrive(cta_id)).  The .release.cluster
// form is the one the model covers; it made every epilogue hand-off slower
// (frame stack 1.37 against 1.27 ms on one B200, 1000 W).
__device__ __forceinline__ void mbar_arrive_rank0(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .b32 remote;\n\t"
        "mapa.shared::cluster.u32 remote, %0, 0;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [remote];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    return rank;
}
// every thread of both CTAs
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\t"
                 "barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// TMEM of a CTA pair: one warp of each CTA allocates (the same columns in both)
__device__ __forceinline__ void tmem_alloc(uint32_t* dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(dst)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// arrive on the barrier at this offset in both CTAs once the pair's MMAs issued
// so far are complete
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, M = 256 over the pair
__device__ __forceinline__ void umma_bf16(
    uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// No-swizzle K-major smem matrix descriptor (cute::UMMA::SmemDescriptor):
// start address [0,14), leading (K-chunk) byte offset [16,30), stride (8-row
// group) byte offset [32,46), descriptor version 1 at [46,48), layout type 0.
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]),
          "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait();
// 16 columns of each of CLASSES accumulators (STRIDE columns apart), added in
// fp32 from the smallest-magnitude class up
template <int CLASSES, int STRIDE>
__device__ __forceinline__ void tmem_ld16_sum(uint32_t taddr, uint32_t (&r)[16]);
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
template <int CLASSES, int STRIDE>
__device__ __forceinline__ void tmem_ld16_sum(uint32_t taddr, uint32_t (&r)[16]) {
    if constexpr (CLASSES == 1) {
        tmem_ld16(taddr, r);
        tmem_ld_wait();
    } else {
        uint32_t part[CLASSES][16];
#pragma unroll
        for (int c = 0; c < CLASSES; ++c) tmem_ld16(taddr + c * STRIDE, part[c]);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            float v = __uint_as_float(part[CLASSES - 1][j]);
#pragma unroll
            for (int c = CLASSES - 2; c >= 0; --c) v += __uint_as_float(part[c][j]);
            r[j] = __float_as_uint(v);
        }
    }
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
// relu fused into the conversion: max(x, 0) -> bf16x2
__device__ __forceinline__ uint32_t pack_bf16_relu(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__device__ __forceinline__ float4 ld_stream4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ bool elect_one() {
    uint32_t elected;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(elected));
    return elected != 0;
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32 [4,6) = 1,
// A bf16 [7,10) = 1, B bf16 [10,13) = 1, A and B K-major, N >> 3 at [17,23),
// M >> 4 at [24,29); M = 256 rows over the CTA pair
constexpr uint32_t kInstrDesc =
    (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(C >> 3) << 17) | ((uint32_t)(2 * M >> 4) << 24);

// two values -> PARTS bf16x2 words: hi, then the bf16 of what is left, ...
template <int PARTS>
__device__ __forceinline__ void split_pack(float lo_v, float hi_v, uint32_t (&words)[PARTS]) {
#pragma unroll
    for (int p = 0; p < PARTS; ++p) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(lo_v, hi_v);
        words[p] = *reinterpret_cast<const uint32_t*>(&h);
        if (p + 1 < PARTS) {
            const float2 back = __bfloat1622float2(h);
            lo_v -= back.x;
            hi_v -= back.y;
        }
    }
}

// Store 8 consecutive channels of one row into the slot's A-operand buffer(s)
template <int PARTS, int KSIZE>
__device__ __forceinline__ void store_kgroup(uint8_t* act_hi, int kg, int buffer_row, const float (&v)[8]) {
    uint32_t words[4][PARTS];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_pack<PARTS>(v[2 * j], v[2 * j + 1], words[j]);
#pragma unroll
    for (int p = 0; p < PARTS; ++p)
        *reinterpret_cast<uint4*>(act_hi + p * act_stride(KSIZE) +
                                  (kg * buffer_rows(KSIZE) + buffer_row) * 16) =
            make_uint4(words[0][p], words[1][p], words[2][p], words[3][p]);
}

// Rare path: activations other than ReLU / identity.  Out of line so the hot
// loop stays small in the instruction cache.
template <int PARTS, int KSIZE>
__device__ __noinline__ void epilogue_generic(
    uint32_t taddr, uint8_t* act, int row, int a, bool valid, bool last, bool store,
    float* yrow, const float* bias) {
#pragma unroll 1
    for (int c0 = 0; c0 < C; c0 += 16) {
        uint32_t raw[16];
        tmem_ld16_sum<Config<PARTS>::kClasses, Config<PARTS>::kClassStride>(taddr + c0, raw);
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
            v[j] = valid ? apply_activation(__uint_as_float(raw[j]) + bias[c0 + j], a) : 0.f;
        if (!last) {
            const float (&first)[8] = *reinterpret_cast<const float(*)[8]>(&v[0]);
            const float (&second)[8] = *reinterpret_cast<const float(*)[8]>(&v[8]);
            store_kgroup<PARTS, KSIZE>(act, c0 >> 3, row + pad_rows(KSIZE), first);
            store_kgroup<PARTS, KSIZE>(act, (c0 >> 3) + 1, row + pad_rows(KSIZE), second);
        } else if (store) {
            float4* dst = reinterpret_cast<float4*>(yrow + c0);
            dst[0] = make_float4(v[0], v[1], v[2], v[3]);
            dst[1] = make_float4(v[4], v[5], v[6], v[7]);
            dst[2] = make_float4(v[8], v[9], v[10], v[11]);
            dst[3] = make_float4(v[12], v[13], v[14], v[15]);
        }
    }
}

template <int PARTS, int KSIZE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Config<PARTS>::kThreads, 1)
conv_stack_tc_kernel(
    const float* __restrict__ x, const int32_t* __restrict__ row_seq, int total_rows,
    const uint8_t* __restrict__ weights,   // blob entries: [half][tap][kg][40 n][8] bf16 + bias chunk
    Acts acts, int n_layers, int tile_rows, int n_tiles, float* __restrict__ y,
    PoolArgs pool) {
    constexpr int kSlots = Config<PARTS>::kSlots;
    constexpr int kParts = Config<PARTS>::kParts;
    constexpr int kThreads = Config<PARTS>::kThreads;
    constexpr int kEntries = Config<PARTS>::kEntriesPerLayer;
    constexpr int kRing = Config<PARTS>::kRing;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    Smem<PARTS, KSIZE>& sm = *reinterpret_cast<Smem<PARTS, KSIZE>*>(smem_raw);
    constexpr int W_CONV_BYTES = conv_bytes(KSIZE);
    constexpr int W_HALF_BYTES = half_bytes(KSIZE);
    constexpr int W_LAYER_BYTES = layer_bytes(KSIZE);
    constexpr int HALF = (KSIZE - 1) / 2;
    constexpr int PAD = pad_rows(KSIZE);       // tile row r lives in buffer row r + PAD
    constexpr int RB = buffer_rows(KSIZE);
    constexpr int ACT_STRIDE = act_stride(KSIZE);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int halo = n_layers * HALF;
    const int rank = (int)cluster_rank();
    const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    // pair tile p = tiles 2p and 2p + 1; a pair whose second tile is past the
    // end still runs both CTAs: rank 1 may load a few real rows into its halo,
    // but every row it would store lies at or past total_rows, so it stores
    // nothing
    const int n_pairs = (n_tiles + 1) >> 1;
    const int rounds = (n_pairs + n_clusters * kSlots - 1) / (n_clusters * kSlots);

    // ---- one-time setup ----
    // pad rows (buffer rows 0 .. PAD-1 and RB-PAD .. RB-1) of every k-group
    // stay zero forever
    for (int i = tid; i < kSlots * kParts * KG * PAD * 2 * 4; i += kThreads) {
        const int buffer = i / (KG * PAD * 8), rem = i % (KG * PAD * 8);
        const int kg = rem / (PAD * 8), pad = (rem / 8) % PAD, edge = (rem / 4) & 1, word = rem & 3;
        reinterpret_cast<uint32_t*>(
            sm.act[buffer / kParts][buffer % kParts] + (kg * RB + (edge ? RB - 1 - pad : pad)) * 16)[word] = 0u;
    }
    // fp32 bias of every layer, rebuilt exactly from the three bf16 parts the
    // packed blob carries after each layer's taps; the epilogue adds it
    for (int i = tid; i < n_layers * C; i += kThreads) {
        const int layer = i / C, n = i % C;
        const __nv_bfloat16* chunk = reinterpret_cast<const __nv_bfloat16*>(
            weights + (size_t)layer * kEntries * W_LAYER_BYTES + W_CONV_BYTES);
        sm.bias[layer][n] = __bfloat162float(chunk[n * 8]) + __bfloat162float(chunk[n * 8 + 1]) +
                            __bfloat162float(chunk[n * 8 + 2]);
    }
    if (tid == 0) {
        for (int i = 0; i < kRing; ++i) {
            mbar_init(&sm.w_full[i], 1);
            mbar_init(&sm.w_empty[i], 1);
            mbar_init(&sm.peer_full[i], 1);
        }
        for (int s = 0; s < kSlots; ++s) {
            mbar_init(&sm.act_ready[s], 8);     // one elected lane per epilogue warp of the pair
            mbar_init(&sm.mma_done[s], 1);
        }
        fence_barrier_init();
    }
    if (warp == kSlots * 4) tmem_alloc(&sm.tmem_base, kTmemCols);
    fence_proxy_async();
    tc_fence_before();
    cluster_sync();     // no arrive from the peer may meet an uninitialized barrier
    tc_fence_after();
    const uint32_t tmem_base = sm.tmem_base;

    if (warp < kSlots * 4) {
        // =========================== epilogue group ===========================
        const int slot = warp >> 2;
        const int quad = warp & 3;                  // TMEM lane quadrant of this warp
        const int row = quad * 32 + lane;           // tile-local row == TMEM lane
        const int gtid = tid & 127;                 // thread within the group
        uint8_t* act = sm.act[slot][0];             // hi part; lo part follows it
        const uint32_t taddr =
            tmem_base + ((uint32_t)(quad * 32) << 16) + slot * Config<PARTS>::kSlotStride;
        uint32_t done_parity = 0;

        // One tile = M * C / 4 = 2560 float4 = 20 per thread, coalesced.  The
        // first tile is fetched up front; every later one is requested while the
        // tensor core still works on the previous tile's last layer, so its
        // latency never reaches the MMA warp.  The rows wait in registers already
        // converted to bf16 (40 registers per part; with three parts the 80
        // registers of the raw fp32 values are kept instead and split on store).
        constexpr bool kKeepRaw = PARTS == 3;
        uint2 pk[kKeepRaw ? 1 : PARTS][kKeepRaw ? 1 : 20];
        float4 raw_rows[kKeepRaw ? 20 : 1];
        auto fetch_tile = [&](int tile) {
            const int row0 = tile * tile_rows - halo;
            // two batches of 10 loads in flight (the registers for 20 are not there)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float4 v[10];
#pragma unroll
                for (int k = 0; k < 10; ++k) {
                    const int i = gtid + 128 * (10 * half + k);
                    const int gr = row0 + i / (C / 4);
                    v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (gr >= 0 && gr < total_rows)
                        v[k] = ld_stream4(x + (size_t)gr * C + 4 * (i % (C / 4)));
                }
#pragma unroll
                for (int k = 0; k < 10; ++k) {
                    if constexpr (kKeepRaw) {
                        raw_rows[10 * half + k] = v[k];
                    } else {
                        uint32_t a[PARTS], b[PARTS];
                        split_pack<PARTS>(v[k].x, v[k].y, a);
                        split_pack<PARTS>(v[k].z, v[k].w, b);
#pragma unroll
                        for (int p = 0; p < PARTS; ++p) pk[p][10 * half + k] = make_uint2(a[p], b[p]);
                    }
                }
            }
        };
        {
            const int first = cluster * kSlots + slot;
            if (first < n_pairs) fetch_tile(2 * first + rank);
        }

        for (int round = 0; round < rounds; ++round) {
            const int pair = (round * n_clusters + cluster) * kSlots + slot;
            if (pair >= n_pairs) break;
            const int tile = 2 * pair + rank;
            const int next_tile = tile + 2 * n_clusters * kSlots;
            const int row0 = tile * tile_rows - halo;   // global row of local row 0
            const int g = row0 + row;
            const bool in_range = g >= 0 && g < total_rows;
            const bool valid = in_range && __ldg(row_seq + g) >= 0;

            // bf16 rows -> the slot's A operand buffer(s)
#pragma unroll
            for (int it = 0; it < 20; ++it) {
                const int i = gtid + 128 * it;
                const int r = i / (C / 4), c4 = i % (C / 4);
                uint8_t* dst = act + ((c4 >> 1) * RB + r + PAD) * 16 + (c4 & 1) * 8;
                if constexpr (kKeepRaw) {
                    uint32_t a[PARTS], b[PARTS];
                    split_pack<PARTS>(raw_rows[it].x, raw_rows[it].y, a);
                    split_pack<PARTS>(raw_rows[it].z, raw_rows[it].w, b);
#pragma unroll
                    for (int p = 0; p < PARTS; ++p)
                        *reinterpret_cast<uint2*>(dst + p * ACT_STRIDE) = make_uint2(a[p], b[p]);
                } else {
#pragma unroll
                    for (int p = 0; p < PARTS; ++p)
                        *reinterpret_cast<uint2*>(dst + p * ACT_STRIDE) = pk[p][it];
                }
            }
            if (tid == 0) TRACE(13, round);
            fence_proxy_async();        // generic-proxy writes -> visible to the tensor core
            tc_fence_before();          // orders the previous round's TMEM reads too
            __syncwarp();
            if (lane == 0) mbar_arrive_rank0(&sm.act_ready[slot]);
            if (tid == 0) TRACE(16, round);

            // pull the next round's tile of this slot into L2 while this one computes
            if (next_tile < n_tiles) {
                const long lo = (long)max(next_tile * tile_rows - halo, 0) * C * 4;
                const long hi = (long)min(next_tile * tile_rows - halo + M, total_rows) * C * 4;
                const char* base = reinterpret_cast<const char*>(x);
                for (long off = lo + 128 * gtid; off < hi; off += 128 * 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
            }

            // a warp whose 32 rows are all real frames (97 % of warps) skips
            // the separator masking
            const bool zero = !__all_sync(0xffffffffu, valid) && !valid;

            // ---- layers 0 .. n-2: accumulator -> next layer's A operand ----
            for (int layer = 0; layer + 1 < n_layers; ++layer) {
                const int a = acts.act[layer];
                const bool simple = a == EMPH_ACT_RELU || a == EMPH_ACT_NONE;
                const bool relu = a == EMPH_ACT_RELU;
                if (tid == 0) TRACE(0, round * n_layers + layer);
                mbar_wait(&sm.mma_done[slot], done_parity);
                if (tid == 0) TRACE(1, round * n_layers + layer);
                if (gtid == 0) TRACE(8 + slot, round * n_layers + layer);
                done_parity ^= 1;
                tc_fence_after();
                if (simple) {
                    // whole accumulator row, then the fp32 bias: 5 x 16 columns, one wait
                    uint32_t raw[C];
                    if constexpr (PARTS == 1) {
#pragma unroll
                        for (int c0 = 0; c0 < C; c0 += 16)
                            tmem_ld16(taddr + c0, *reinterpret_cast<uint32_t(*)[16]>(&raw[c0]));
                        tmem_ld_wait();
                    } else {
#pragma unroll
                        for (int c0 = 0; c0 < C; c0 += 16)
                            tmem_ld16_sum<Config<PARTS>::kClasses, Config<PARTS>::kClassStride>(
                                taddr + c0, *reinterpret_cast<uint32_t(*)[16]>(&raw[c0]));
                    }
                    {
                        const float4* b4 = reinterpret_cast<const float4*>(sm.bias[layer]);
#pragma unroll
                        for (int c4 = 0; c4 < C / 4; ++c4) {
                            const float4 b = b4[c4];
                            raw[4 * c4 + 0] = __float_as_uint(__uint_as_float(raw[4 * c4 + 0]) + b.x);
                            raw[4 * c4 + 1] = __float_as_uint(__uint_as_float(raw[4 * c4 + 1]) + b.y);
                            raw[4 * c4 + 2] = __float_as_uint(__uint_as_float(raw[4 * c4 + 2]) + b.z);
                            raw[4 * c4 + 3] = __float_as_uint(__uint_as_float(raw[4 * c4 + 3]) + b.w);
                        }
                    }
                    if constexpr (PARTS == 1) {
                        uint8_t* dst = act + (row + PAD) * 16;
#pragma unroll
                        for (int kg = 0; kg < KG; ++kg) {
                            uint32_t p[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float lo = __uint_as_float(raw[8 * kg + 2 * j]);
                                const float hi = __uint_as_float(raw[8 * kg + 2 * j + 1]);
                                p[j] = relu ? pack_bf16_relu(lo, hi) : pack_bf16(lo, hi);
                            }
                            if (zero) p[0] = p[1] = p[2] = p[3] = 0u;
                            *reinterpret_cast<uint4*>(dst + kg * RB * 16) =
                                make_uint4(p[0], p[1], p[2], p[3]);
                        }
                    } else {
#pragma unroll
                        for (int kg = 0; kg < KG; ++kg) {
                            float w[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                w[j] = __uint_as_float(raw[8 * kg + j]);
                                if (relu) w[j] = fmaxf(w[j], 0.f);
                                if (zero) w[j] = 0.f;
                            }
                            store_kgroup<PARTS, KSIZE>(act, kg, row + PAD, w);
                        }
                    }
                } else {
                    epilogue_generic<PARTS, KSIZE>(
                        taddr, act, row, a, valid, false, false, y, sm.bias[layer]);
                }
                if (tid == 0) TRACE(2, round * n_layers + layer);
                fence_proxy_async();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_rank0(&sm.act_ready[slot]);
                if (tid == 0) TRACE(3, round * n_layers + layer);
            }

            // ---- last layer: fp32 rows to HBM ----
            {
                const int layer = n_layers - 1;
                const int a = acts.act[layer];
                const bool simple = a == EMPH_ACT_RELU || a == EMPH_ACT_NONE;
                const bool relu = a == EMPH_ACT_RELU;
                // the next tile's rows travel while this tile's last MMAs run, so
                // their latency never reaches the MMA warp
                // (not across the out-of-line generic epilogue: its call would
                // spill all of them)
                // (unconditional -- rows past the end load nothing -- so the
                // registers are provably dead during the earlier layers)
                if (simple) fetch_tile(next_tile);
                if (tid == 0) TRACE(12, round);
                mbar_wait(&sm.mma_done[slot], done_parity);
                if (gtid == 0) TRACE(8 + slot, round * n_layers + layer);
                done_parity ^= 1;
                tc_fence_after();
                if (simple) {
                    // 16 columns at a time (the next tile's 20 float4 are live in
                    // registers here)
                    const bool store = in_range && row >= halo && row < M - halo;
                    float4* dst = reinterpret_cast<float4*>(y + (size_t)(in_range ? g : 0) * C);
                    // fused word pooling: the run structure of this warp's rows.  Each
                    // half-warp reduces the rows of one parity (half h: rows h, h + 2,
                    // ...), so bit r of `starts` / `ends` says that row r opens / closes
                    // a run of equal words in ITS parity sequence
                    int wid = -1;
                    uint32_t starts = 0, ends = 0;
                    if (pool.mode != kPoolNone) {
                        if (store) wid = __ldg(pool.row_word + g);
                        const int before = __shfl_up_sync(0xffffffffu, wid, 2);
                        const int after = __shfl_down_sync(0xffffffffu, wid, 2);
                        starts = __ballot_sync(0xffffffffu, lane < 2 || before != wid);
                        ends = __ballot_sync(0xffffffffu, lane >= 30 || after != wid);
                    }
                    // scratch of this warp: the interior (rows PAD .. PAD + 127) of
                    // k-group `quad` of the slot's operand buffer = 2048 contiguous
                    // bytes = [32 rows][16 floats]; the last layer's MMAs are done with
                    // it, and the slot's warps meet at a barrier before the next tile is
                    // stored
                    float* scratch = reinterpret_cast<float*>(act + (quad * RB + PAD) * 16);
                    const size_t word_base = (size_t)(wid >= 0 ? wid : 0) * C;
#pragma unroll 1
                    for (int c0 = 0; c0 < C; c0 += 16) {
                        uint32_t raw[16];
                        tmem_ld16_sum<Config<PARTS>::kClasses, Config<PARTS>::kClassStride>(
                            taddr + c0, raw);
                        const float4* b4 = reinterpret_cast<const float4*>(sm.bias[layer] + c0);
                        float w[16];
#pragma unroll
                        for (int c4 = 0; c4 < 4; ++c4) {
                            const float4 b = b4[c4];
                            w[4 * c4 + 0] = __uint_as_float(raw[4 * c4 + 0]) + b.x;
                            w[4 * c4 + 1] = __uint_as_float(raw[4 * c4 + 1]) + b.y;
                            w[4 * c4 + 2] = __uint_as_float(raw[4 * c4 + 2]) + b.z;
                            w[4 * c4 + 3] = __uint_as_float(raw[4 * c4 + 3]) + b.w;
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            if (relu) w[j] = fmaxf(w[j], 0.f);
                            if (zero) w[j] = 0.f;
                        }
                        if (y != nullptr && store) {
#pragma unroll
                            for (int c4 = 0; c4 < 4; ++c4)
                                dst[(c0 >> 2) + c4] =
                                    make_float4(w[4 * c4], w[4 * c4 + 1], w[4 * c4 + 2], w[4 * c4 + 3]);
                        }
                        if (pool.mode == kPoolSum || pool.mode == kPoolMax) {
                            // transpose through shared memory: lane = row writes its 16
                            // values (float4 slot q of row r at q ^ ((r & 7) >> 1):
                            // conflict-free both ways), then lane = (parity, column)
                            // walks its 16 rows and keeps one running value per run
                            __syncwarp();
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                *reinterpret_cast<float4*>(
                                    scratch + lane * 16 + 4 * (q ^ ((lane & 7) >> 1))) =
                                    make_float4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
                            __syncwarp();
                            if constexpr (PARTS == 1) {
                                const int parity = lane >> 4, column = lane & 15;
                                // this lane's 16 values first, so that the run below is
                                // a chain of adds rather than of shared-memory loads (row
                                // r = 2k + parity, (r & 7) >> 1 = k & 3)
                                float v[16];
#pragma unroll
                                for (int k = 0; k < 16; ++k)
                                    v[k] = scratch[(2 * k + parity) * 16 + 4 * ((column >> 2) ^ (k & 3)) +
                                                   (column & 3)];
                                const uint32_t my_starts = starts >> parity, my_ends = ends >> parity;
                                // the loop once per pooling mode: all 16 rows unrolled with
                                // compile-time bit tests.  This epilogue runs in all four
                                // slots at once at every tile boundary, while the tensor
                                // pipe waits for slot 0's next operands, so its
                                // instruction count is the boundary's length
                                auto reduce = [&](auto sum_mode) {
                                    constexpr bool kSum = decltype(sum_mode)::value;
                                    float run = 0.f;
#pragma unroll
                                    for (int k = 0; k < 16; ++k) {
                                        const bool opens = (my_starts >> (2 * k)) & 1u;
                                        run = kSum ? (opens ? v[k] : run + v[k])
                                                   : (opens ? fmaxf(v[k], 0.f) : fmaxf(run, v[k]));
                                        if ((ends >> (2 * k)) & 3u) {          // warp-uniform
                                            const int word = __shfl_sync(0xffffffffu, wid, 2 * k + parity);
                                            if (((my_ends >> (2 * k)) & 1u) && word >= 0) {
                                                const size_t at = (size_t)word * C + c0 + column;
                                                if constexpr (kSum) {
                                                    // <= 16 rows per piece: 2^23 * 2^28 = 2^51,
                                                    // and 2^12 pieces of it fit int64
                                                    const float clamped = fminf(
                                                        fmaxf(run, -16.f * kPoolFixedClamp),
                                                        16.f * kPoolFixedClamp);
                                                    atomicAdd(
                                                        reinterpret_cast<unsigned long long*>(pool.fixed + at),
                                                        (unsigned long long)__float2ll_rn(
                                                            clamped * kPoolFixedScale));
                                                } else {
                                                    atomicMax(reinterpret_cast<int*>(pool.out + at),
                                                              __float_as_int(run));
                                                }
                                            }
                                        }
                                    }
                                };
                                if (pool.mode == kPoolSum) reduce(std::true_type{});
                                else reduce(std::false_type{});
                            } else {
                                // the split modes fuse the pooling only on request
                                // (DESIGN 4.2) and keep the compact loop: the unrolled
                                // one made their kernels' code larger and the bf16x6
                                // step slower
                                const bool is_sum = pool.mode == kPoolSum;
                                const int parity = lane >> 4, column = lane & 15;
                                float run = 0.f;
#pragma unroll 4
                                for (int k = 0; k < 16; ++k) {
                                    const int r = 2 * k + parity;
                                    const float v = scratch[r * 16 + 4 * ((column >> 2) ^ ((r & 7) >> 1)) +
                                                            (column & 3)];
                                    const bool opens = (starts >> r) & 1u;
                                    run = is_sum ? (opens ? v : run + v)
                                                 : (opens ? fmaxf(v, 0.f) : fmaxf(run, v));
                                    if ((ends >> (2 * k)) & 3u) {          // warp-uniform
                                        const int word = __shfl_sync(0xffffffffu, wid, r);
                                        if (((ends >> r) & 1u) && word >= 0) {
                                            const size_t at = (size_t)word * C + c0 + column;
                                            if (is_sum) {
                                                // <= 16 rows per piece: 2^23 * 2^28 = 2^51, and
                                                // 2^12 pieces of it fit int64
                                                const float clamped = fminf(
                                                    fmaxf(run, -16.f * kPoolFixedClamp),
                                                    16.f * kPoolFixedClamp);
                                                atomicAdd(
                                                    reinterpret_cast<unsigned long long*>(pool.fixed + at),
                                                    (unsigned long long)__float2ll_rn(
                                                        clamped * kPoolFixedScale));
                                            } else {
                                                atomicMax(reinterpret_cast<int*>(pool.out + at),
                                                          __float_as_int(run));
                                            }
                                        }
                                    }
                                }
                            }
                        } else if (pool.mode == kPoolCenter) {
                            if (wid >= 0) {
                                float4* out4 = reinterpret_cast<float4*>(pool.out + word_base + c0);
#pragma unroll
                                for (int c4 = 0; c4 < 4; ++c4)
                                    out4[c4] =
                                        make_float4(w[4 * c4], w[4 * c4 + 1], w[4 * c4 + 2], w[4 * c4 + 3]);
                            }
                        }
                    }
                    // the scratch lives in the operand buffer the slot's four warps
                    // fill together for the next tile: nobody stores before all are done
                    if (tid == 0) TRACE(14, round);
                    if (pool.mode == kPoolSum || pool.mode == kPoolMax)
                        asm volatile("bar.sync %0, 128;" ::"r"(slot + 1) : "memory");
                    if (tid == 0) TRACE(15, round);
                } else {
                    epilogue_generic<PARTS, KSIZE>(
                        taddr, act, row, a, valid, true,
                        in_range && row >= halo && row < M - halo,
                        y + (size_t)(in_range ? g : 0) * C, sm.bias[layer]);
                    fetch_tile(next_tile);
                }
            }
        }
    } else if (warp == kSlots * 4 && rank == 1) {
        // ===================== rank 1: ring stage relay ======================
        // rank 0 issues the pair's MMAs only once this CTA's weight half is in
        if (lane == 0) {
            int stage = 0;
            uint32_t full_parity = 0;
            for (int round = 0; round < rounds; ++round) {
                if ((round * n_clusters + cluster) * kSlots >= n_pairs) break;
                for (int entry = 0; entry < n_layers * kEntries; ++entry) {
                    mbar_wait(&sm.w_full[stage], full_parity);
                    mbar_arrive_rank0(&sm.peer_full[stage]);
                    if (++stage == kRing) { stage = 0; full_parity ^= 1; }
                }
            }
        }
    } else if (warp == kSlots * 4) {
        // ====================== rank 0: MMA issuer ======================
        // The whole warp runs this loop (warp-uniform control flow keeps the
        // descriptors in uniform registers); one elected lane issues.  A
        // measured pair tcgen05.mma of this shape costs ~47 clk, so every
        // instruction saved in the issue path counts.
        uint32_t ready_parity = 0;                   // bit s = parity of slot s
        int stage = 0;
        uint32_t full_parity = 0;
        uint64_t d_act[kSlots];
#pragma unroll
        for (int s = 0; s < kSlots; ++s) d_act[s] = make_desc(smem_u32(sm.act[s][0]), RB * 16, 128);
        constexpr uint64_t kLoPart = ACT_STRIDE >> 4;            // hi -> lo operand buffer
        for (int round = 0; round < rounds; ++round) {
            const int pair0 = (round * n_clusters + cluster) * kSlots;
            if (pair0 >= n_pairs) break;
            const int active = min(kSlots, n_pairs - pair0);
            for (int layer = 0; layer < n_layers; ++layer) {
#pragma unroll
                for (int entry = 0; entry < kEntries; ++entry) {
                    // entry e: weight part e, both halves
                    mbar_wait(&sm.w_full[stage], full_parity);
                    mbar_wait_cluster(&sm.peer_full[stage], full_parity);
                    const uint64_t d_w = make_desc(smem_u32(sm.w[stage]), CH * 16, 128);
#pragma unroll
                    for (int s = 0; s < kSlots; ++s) {
                        if (s < active) {
                            if (entry == 0) {
                                if (s == 0 && lane == 0) TRACE(4, round * n_layers + layer);
                                mbar_wait_cluster(&sm.act_ready[s], (ready_parity >> s) & 1);
                                if (s == 0 && lane == 0) TRACE(5, round * n_layers + layer);
                                ready_parity ^= 1u << s;
                                tc_fence_after();
                            }
                            if (elect_one()) {
                                const uint32_t d0 = tmem_base + s * Config<PARTS>::kSlotStride;
                                // weight part e x activation parts 0 .. kParts-1-e
                                const int parts = kParts - entry;
#pragma unroll
                                for (int part = 0; part < kParts; ++part) {
                                    if (part < parts) {
#pragma unroll
                                        for (int tap = 0; tap < KSIZE; ++tap) {
#pragma unroll
                                            for (int kk = 0; kk < C / 16; ++kk) {
                                                umma_bf16(
                                                    d0 + (entry + part) * Config<PARTS>::kClassStride,
                                                    d_act[s] + part * kLoPart +
                                                        // tap t reads buffer row r + t + PAD - HALF
                                                        // (r + t for k >= 3)
                                                        (uint64_t)(((2 * kk) * RB * 16 + (tap + PAD - HALF) * 16) >> 4),
                                                    d_w + (uint64_t)((tap * W_HALF_TAP_BYTES + (2 * kk) * CH * 16) >> 4),
                                                    kInstrDesc,
                                                    // a class is opened by its entry-0 MMA
                                                    (entry | tap | kk) != 0);
                                            }
                                        }
                                    }
                                }
                                if (entry == kEntries - 1) umma_commit_pair(&sm.mma_done[s]);
                            }
                            __syncwarp();
                            if (s == 0 && lane == 0) TRACE(6, round * n_layers + layer);
                            if (s == kSlots - 1 && lane == 0) TRACE(7, round * n_layers + layer);
                        }
                    }
                    if (elect_one()) umma_commit_pair(&sm.w_empty[stage]);   // ring stage consumed
                    __syncwarp();
                    if (++stage == kRing) { stage = 0; full_parity ^= 1; }
                }
            }
        }
    } else {
        // ========================== weight producer ==========================
        if (lane == 0) {
            int stage = 0;
            uint32_t empty_parity = 1;       // first pass over the ring never waits
            for (int round = 0; round < rounds; ++round) {
                if ((round * n_clusters + cluster) * kSlots >= n_pairs) break;
                for (int entry = 0; entry < n_layers * kEntries; ++entry) {
                    mbar_wait(&sm.w_empty[stage], empty_parity);
                    mbar_arrive_expect_tx(&sm.w_full[stage], W_HALF_BYTES);
                    bulk_load(sm.w[stage], weights + (size_t)entry * W_LAYER_BYTES + rank * W_HALF_BYTES,
                              W_HALF_BYTES, &sm.w_full[stage]);
                    if (++stage == kRing) { stage = 0; empty_parity ^= 1; }
                }
            }
            // producer tail: wait until the pair's MMAs release every stage, so
            // that the last w_empty commits (multicast to both CTAs) have landed
            // before this CTA passes the teardown barrier.  A stage never loaded
            // passes at once (parity 1 of a fresh barrier).
            for (int i = 0; i < kRing; ++i) {
                mbar_wait(&sm.w_empty[stage], empty_parity);
                if (++stage == kRing) { stage = 0; empty_parity ^= 1; }
            }
        }
    }

    // ---- teardown ----
    tc_fence_before();
    cluster_sync();     // neither CTA leaves while the pair's MMAs or arrivals can reach it
    if (warp == kSlots * 4) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

// fp32 weights [L][tap][in][out] + bias [L][out] -> blob entries of
// W_LAYER_BYTES: bf16 [half][tap][kg][40 out][8 in] (half h = output columns
// 40h .. 40h+39, the ring stage of CTA h of a pair) followed by the bias chunk
// bf16 [2][out][8] (k-group 0 holds the fp32 bias as three bf16 parts (hi,
// mid, lo, 0, ...), k-group 1 is zero; the kernel reads it once at setup).
// parts = 2 / 3: that many entries per layer -- (W_hi, bias chunk), (W_mid, zeros)
// (, (W_lo, zeros)) with W_hi = bf16(W), W_mid = bf16(W - W_hi), W_lo = bf16 of
// what is still left.
// source: 0 = the packed fp32 layout [L][tap][in][out]; 1 = ONE Conv1d weight
// (out, in, k) as the module holds it; 2 = the adjoint convolution of that
// Conv1d weight (channel matrix transposed, taps flipped: the input-gradient
// pass of the training step)
__device__ __forceinline__ void pack_weights_tc_body(
    const float* __restrict__ w, const float* __restrict__ bias, int n_layers, int parts,
    int ks, int source, __nv_bfloat16* __restrict__ out) {
    const int per_entry = layer_bytes(ks) / 2;
    const int conv = conv_bytes(ks) / 2;
    const int entries = parts;
    const int total = n_layers * entries * per_entry;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int entry = i / per_entry, local = i % per_entry;
        const int layer = entry / entries, part = entry % entries;
        float v = 0.f;
        if (local < conv) {
            const int e = local & 7;
            int rest = local >> 3;
            const int nh = rest % CH; rest /= CH;
            const int kg = rest % KG; rest /= KG;
            const int tap = rest % ks;
            const int n = (rest / ks) * CH + nh;
            const int ci = kg * 8 + e;
            const float value =
                source == 0 ? w[((size_t)(layer * ks + tap) * C + ci) * C + n]
                : source == 1 ? w[((size_t)n * C + ci) * ks + tap]
                : w[((size_t)ci * C + n) * ks + (ks - 1 - tap)];
            v = value;                               // part p: rounded below after
            for (int q = 0; q < part; ++q)           // removing the earlier parts
                v -= __bfloat162float(__float2bfloat16_rn(v));
        } else if (part == 0) {
            const int rem = local - conv;
            const int e = rem & 7, n = (rem >> 3) % C, kg = (rem >> 3) / C;
            if (kg == 0 && e < 3) {                  // bias as three bf16 parts: exact fp32
                v = bias[layer * C + n];
                for (int q = 0; q < e; ++q)
                    v -= __bfloat162float(__float2bfloat16_rn(v));
            }
        }
        out[i] = __float2bfloat16_rn(v);
    }
}

__global__ void pack_weights_tc_kernel(
    const float* __restrict__ w, const float* __restrict__ bias, int n_layers, int parts,
    int ks, int source, __nv_bfloat16* __restrict__ out) {
    pack_weights_tc_body(w, bias, n_layers, parts, ks, source, out);
}

// the Conv1d weights of up to 32 layers, each into its own blob (blockIdx.y =
// layer): the training step packs a whole direction in one launch
struct PackBatch {
    const float* weight[32];
    const float* bias[32];
};
__global__ void pack_conv1d_batch_kernel(
    PackBatch batch, int parts, int ks, int source, size_t blob_elements,
    __nv_bfloat16* __restrict__ out) {
    pack_weights_tc_body(batch.weight[blockIdx.y], batch.bias[blockIdx.y], 1, parts, ks, source,
                         out + blockIdx.y * blob_elements);
}

}  // namespace tc

template <int PARTS, int KSIZE>
static int launch_tc(
    const float* x, const int32_t* row_seq, int32_t total_rows, const float* weights,
    const int32_t* acts_host, int32_t n_layers, float* y, cudaStream_t stream,
    tc::PoolArgs pool = tc::PoolArgs{nullptr, nullptr, nullptr, tc::kPoolNone}) {
    static_assert(sizeof(tc::Smem<PARTS, KSIZE>) + 128 <= tc::kSmemLimit,
                  "conv_tc: the slots and the weight ring do not fit shared memory");
    EMPH_REQUIRE(n_layers <= tc::kMaxLayers, "emph_conv_stack(tc): too many layers");
    const int halo = n_layers * ((KSIZE - 1) / 2);
    const int tile_rows = tc::M - 2 * halo;
    EMPH_REQUIRE(tile_rows >= 32, "emph_conv_stack(tc): %d layers leave no tile", n_layers);
    tc::Acts acts;
    for (int i = 0; i < tc::kMaxLayers; ++i) acts.act[i] = i < n_layers ? acts_host[i] : 0;
    constexpr int kSlots = tc::Config<PARTS>::kSlots;
    const size_t smem = sizeof(tc::Smem<PARTS, KSIZE>) + 128;
    int s = check_cuda(
        cudaFuncSetAttribute(tc::conv_stack_tc_kernel<PARTS, KSIZE>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
        "conv_tc smem attribute");
    if (s != EMPH_OK) return s;
    // CTA pairs the device can keep resident (a pair needs two SMs of one TPC
    // with room for this CTA): the persistent grid never exceeds it.  Cached
    // per device; callers on several threads at once store the same value.
    constexpr int kMaxDevices = 64;
    static int max_clusters_of[kMaxDevices] = {};
    int device = 0;
    s = check_cuda(cudaGetDevice(&device), "conv_tc device");
    if (s != EMPH_OK) return s;
    EMPH_REQUIRE(device < kMaxDevices, "emph_conv_stack(tc): device %d out of range", device);
    int max_clusters = max_clusters_of[device];
    if (max_clusters == 0) {
        cudaLaunchConfig_t config = {};
        config.gridDim = dim3(2 * sm_count());
        config.blockDim = dim3(tc::Config<PARTS>::kThreads);
        config.dynamicSmemBytes = smem;
        s = check_cuda(cudaOccupancyMaxActiveClusters(
                           &max_clusters, (void*)tc::conv_stack_tc_kernel<PARTS, KSIZE>, &config),
                       "conv_tc cluster occupancy");
        if (s != EMPH_OK) return s;
        EMPH_REQUIRE(max_clusters > 0, "emph_conv_stack(tc): no CTA pair fits on the device");
        max_clusters_of[device] = max_clusters;
    }
    const int n_tiles = (total_rows + tile_rows - 1) / tile_rows;
    const int want = ((n_tiles + 1) / 2 + kSlots - 1) / kSlots;
    const int grid = 2 * (want < max_clusters ? want : max_clusters);
    tc::conv_stack_tc_kernel<PARTS, KSIZE><<<grid, tc::Config<PARTS>::kThreads, smem, stream>>>(
        x, row_seq, total_rows, reinterpret_cast<const uint8_t*>(weights), acts,
        n_layers, tile_rows, n_tiles, y, pool);
    EMPH_CHECK_LAUNCH(PARTS == 1 ? "emph_conv_stack(bf16 tc)"
                      : PARTS == 2 ? "emph_conv_stack(bf16x3 tc)" : "emph_conv_stack(bf16x6 tc)");
    return EMPH_OK;
}

// kernel sizes the tensor-core stack is compiled for (at 80 channels)
static bool tc_kernel_size(int kernel_size) {
    return kernel_size == 1 || kernel_size == 3 || kernel_size == 5 || kernel_size == 7;
}

template <int PARTS>
static int launch_tc_ks(
    const float* x, const int32_t* row_seq, int32_t total_rows, const float* weights,
    const int32_t* acts_host, int32_t n_layers, int32_t kernel_size, float* y, cudaStream_t stream,
    tc::PoolArgs pool = tc::PoolArgs{nullptr, nullptr, nullptr, tc::kPoolNone}) {
    switch (kernel_size) {
        case 1: return launch_tc<PARTS, 1>(x, row_seq, total_rows, weights, acts_host, n_layers, y, stream, pool);
        case 3: return launch_tc<PARTS, 3>(x, row_seq, total_rows, weights, acts_host, n_layers, y, stream, pool);
        case 5: return launch_tc<PARTS, 5>(x, row_seq, total_rows, weights, acts_host, n_layers, y, stream, pool);
        case 7: return launch_tc<PARTS, 7>(x, row_seq, total_rows, weights, acts_host, n_layers, y, stream, pool);
    }
    set_error("emph_conv_stack(tc): kernel_size=%d not compiled in", kernel_size);
    return EMPH_ENOSYS;
}

int conv_stack_bf16_tc(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    const float* weights, const float* bias, const int32_t* acts_host,
    int32_t n_layers, int32_t channels, int32_t kernel_size, float* y,
    cudaStream_t stream) {
    if (channels != tc::C || !tc_kernel_size(kernel_size)) {
        set_error("emph_conv_stack(bf16 tc): channels=%d kernel_size=%d not compiled in",
                  channels, kernel_size);
        return EMPH_ENOSYS;
    }
    return launch_tc_ks<1>(x, row_seq, total_rows, weights, acts_host, n_layers, kernel_size, y, stream);
}

int conv_stack_bf16x3_tc(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    const float* weights, const int32_t* acts_host,
    int32_t n_layers, int32_t channels, int32_t kernel_size, float* y,
    cudaStream_t stream) {
    if (channels != tc::C || !tc_kernel_size(kernel_size)) {
        set_error("emph_conv_stack(bf16x3 tc): channels=%d kernel_size=%d not compiled in",
                  channels, kernel_size);
        return EMPH_ENOSYS;
    }
    return launch_tc_ks<2>(x, row_seq, total_rows, weights, acts_host, n_layers, kernel_size, y, stream);
}

int conv_stack_bf16x6_tc(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    const float* weights, const int32_t* acts_host,
    int32_t n_layers, int32_t channels, int32_t kernel_size, float* y,
    cudaStream_t stream) {
    if (channels != tc::C || !tc_kernel_size(kernel_size)) {
        set_error("emph_conv_stack(bf16x6 tc): channels=%d kernel_size=%d not compiled in",
                  channels, kernel_size);
        return EMPH_ENOSYS;
    }
    return launch_tc_ks<3>(x, row_seq, total_rows, weights, acts_host, n_layers, kernel_size, y, stream);
}

// The tensor-core stack of kernel size 3, 5 or 7 with word pooling fused into
// the last layer's epilogue (see tc::PoolArgs); y may be null (frame rows are
// then not written)
int conv_stack_tc_pool(
    const float* x, const int32_t* row_seq, int32_t total_rows,
    const float* weights, const int32_t* acts_host, int32_t n_layers, int32_t channels,
    int32_t kernel_size, int32_t precision, const int32_t* row_word, int32_t pool_mode,
    long long* fixed, float* out, float* y, cudaStream_t stream) {
    if (channels != tc::C || (kernel_size != 3 && kernel_size != 5 && kernel_size != 7)) {
        set_error("emph_conv_stack_pool: channels=%d kernel_size=%d not compiled in",
                  channels, kernel_size);
        return EMPH_ENOSYS;
    }
    const int last = acts_host[n_layers - 1];
    if (last != EMPH_ACT_RELU && !(last == EMPH_ACT_NONE && pool_mode != tc::kPoolMax)) {
        set_error("emph_conv_stack_pool: last activation %d is not fused", last);
        return EMPH_ENOSYS;
    }
    const tc::PoolArgs pool{row_word, fixed, out, pool_mode};
    if (precision == EMPH_PREC_BF16_TC)
        return launch_tc_ks<1>(x, row_seq, total_rows, weights, acts_host, n_layers, kernel_size, y,
                               stream, pool);
    if (precision == EMPH_PREC_BF16X3_TC)
        return launch_tc_ks<2>(x, row_seq, total_rows, weights, acts_host, n_layers, kernel_size, y,
                               stream, pool);
    if (precision == EMPH_PREC_BF16X6_TC)
        return launch_tc_ks<3>(x, row_seq, total_rows, weights, acts_host, n_layers, kernel_size, y,
                               stream, pool);
    set_error("emph_conv_stack_pool: precision %d has no tensor-core kernel", precision);
    return EMPH_ENOSYS;
}

}  // namespace emph

#ifdef EXP_TRACE
extern "C" int emph_conv_trace_read(long long* host) {
    return (int)cudaMemcpyFromSymbol(host, emph::tc::g_trace, sizeof(emph::tc::g_trace));
}
#endif

extern "C" int emph_conv_weights_tc_bytes(
    int32_t n_layers, int32_t channels, int32_t kernel_size, int32_t precision) {
    if (channels != emph::tc::C || !emph::tc_kernel_size(kernel_size) || n_layers <= 0) return 0;
    const int entry = emph::tc::layer_bytes(kernel_size);
    if (precision == EMPH_PREC_BF16X3_TC) return 2 * n_layers * entry;
    if (precision == EMPH_PREC_BF16X6_TC) return 3 * n_layers * entry;
    if (precision != EMPH_PREC_BF16_TC) return 0;
    return n_layers * entry;
}

extern "C" int emph_pack_conv_weights_tc(
    const float* weights, const float* bias, int32_t n_layers, int32_t channels,
    int32_t kernel_size, int32_t precision, void* packed, void* stream) {
    if (channels != emph::tc::C || !emph::tc_kernel_size(kernel_size)) {
        emph::set_error("emph_pack_conv_weights_tc: channels=%d kernel_size=%d not compiled in",
                        channels, kernel_size);
        return EMPH_ENOSYS;
    }
    EMPH_REQUIRE(n_layers > 0, "emph_pack_conv_weights_tc: no layers");
    EMPH_REQUIRE(precision == EMPH_PREC_BF16_TC || precision == EMPH_PREC_BF16X3_TC ||
                     precision == EMPH_PREC_BF16X6_TC,
                 "emph_pack_conv_weights_tc: precision %d has no tensor-core layout", precision);
    const int parts = precision == EMPH_PREC_BF16X6_TC ? 3 : precision == EMPH_PREC_BF16X3_TC ? 2 : 1;
    emph::tc::pack_weights_tc_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(
        weights, bias, n_layers, parts, kernel_size, 0, reinterpret_cast<__nv_bfloat16*>(packed));
    EMPH_CHECK_LAUNCH("emph_pack_conv_weights_tc");
    return EMPH_OK;
}

// One Conv1d (out, in, k) weight (or its adjoint) straight into the operand
// blob of a one-layer stack: what the training step needs every step
namespace emph {
int pack_conv1d_weights_tc(
    const float* conv_weight, const float* bias, int kernel_size, int precision, int adjoint,
    void* packed, cudaStream_t stream) {
    const int parts = precision == EMPH_PREC_BF16X6_TC ? 3 : precision == EMPH_PREC_BF16X3_TC ? 2 : 1;
    tc::pack_weights_tc_kernel<<<64, 256, 0, stream>>>(
        conv_weight, bias, 1, parts, kernel_size, adjoint ? 2 : 1,
        reinterpret_cast<__nv_bfloat16*>(packed));
    EMPH_CHECK_LAUNCH("pack_conv1d_weights_tc");
    return EMPH_OK;
}

// bytes of one layer's operand blob in the given tensor-core precision
size_t conv1d_blob_bytes(int kernel_size, int precision) {
    const int parts = precision == EMPH_PREC_BF16X6_TC ? 3 : precision == EMPH_PREC_BF16X3_TC ? 2 : 1;
    return (size_t)parts * tc::layer_bytes(kernel_size);
}

// n Conv1d weights -> n blobs `stride` bytes apart, one launch
int pack_conv1d_weights_tc_batch(
    const float* const* conv_weights, const float* const* biases, int n, int kernel_size,
    int precision, int adjoint, void* packed, size_t stride, cudaStream_t stream) {
    EMPH_REQUIRE(n >= 0 && n <= 32 && stride % 2 == 0, "pack_conv1d_weights_tc_batch: bad batch");
    if (n == 0) return EMPH_OK;
    const int parts = precision == EMPH_PREC_BF16X6_TC ? 3 : precision == EMPH_PREC_BF16X3_TC ? 2 : 1;
    tc::PackBatch batch;
    for (int i = 0; i < n; ++i) {
        batch.weight[i] = conv_weights[i];
        batch.bias[i] = biases[i];
    }
    tc::pack_conv1d_batch_kernel<<<dim3(16, n), 256, 0, stream>>>(
        batch, parts, kernel_size, adjoint ? 2 : 1, stride / 2,
        reinterpret_cast<__nv_bfloat16*>(packed));
    EMPH_CHECK_LAUNCH("pack_conv1d_weights_tc_batch");
    return EMPH_OK;
}
}  // namespace emph
