// frontend_b200.cu -- fused observation front end of the agent Q-network (SURVEY 8f row f2), sm_100a.
//
// Replaces, for rollouts, HomophilyAgent.rgb_preprocess = conv_to_fc (src/modules/agents/homophily_agent.py:19-27, called
// from src/controllers/homophily_controller.py:132-136):
//     u8 obs (env's padded plane layout)  ->  /256  ->  Conv2d(3, 6, k=3, s=1) + LeakyReLU  ->  Flatten
//                                         ->  Linear(6 (N-2)^2, 32) + LeakyReLU              ->  f32 [rows][32]
// so the fp32 observation (3.4x the bytes the env kernel just wrote) never exists.
//
// One persistent CTA per SM works on tiles of 128 agent views (GEMM rows):
//   * warps 0-7  PRODUCERS: conv3x3 + LeakyReLU on the CUDA cores, straight from the u8 planes (a rolling window of 3 rows x
//                3 planes x 3 aligned 32-bit words = a 3x3x10 byte patch, one new row per chunk; 6 output channels x 8 pixels
//                = 1296 FMAs per patch, issued as 648 packed fp32-pair FMAs -- fma.rn.f32x2, SASS FFMA2, new on sm_100 -- on
//                two output channels at a time: pixel as broadcast scalar, weight pair in a uniform register pair).  The
//                activations are the A operand of the FC contraction: each thread writes its 8 values of an output channel,
//                split as tf32 hi + lo, into the K-major core-matrix layout the tensor core reads (no swizzle: 8 rows x 16 B
//                cores, LBO 128 B, SBO 1536 B);
//   * warp 9     TMA: the FC weight tile of the stage ([32 x 48] hi + lo, pre-packed on the host in the same core-matrix
//                layout) arrives with one cp.async.bulk.tensor.2d (SASS UTMALDG) on the stage's full-barrier;
//   * warps 8,10 MMA: one elected lane each issues tcgen05.mma.kind::tf32 (M=128, N=32, K=8) for every other K step of a
//                stage into its own 8 of the 16 TMEM accumulators (512 columns) -- with MMAs this small the issue rate of one
//                lane, not the tensor core, was the limit;
//   * warps 0-3  EPILOGUE after the last stage of a segment: tcgen05.ld (SASS LDTM) -> + bias -> LeakyReLU -> 128-bit stores.
// Work division: the (tile, chunk) units form one sequence that is dealt out in equal contiguous shares, one per CTA; a tile
// cut by a share boundary is combined, in CTA order, by whichever of its CTAs stores its partial sums last (one launch, result
// independent of timing).
// A chunk is one (16-pixel column block xb, pixel row y) of the conv output, all 6 channels; a stage is half a chunk (3 output
// channels): A 128 x 48 (hi, lo: 48 KB) + B 32 x 48 (hi, lo: 12 KB).  The activations go through a ring of 2 slots (one chunk),
// the weight tiles through their own ring of 4 (the TMA runs two chunks ahead), so the conv of the next chunk overlaps the
// contraction of the previous one and no stage waits for an L2 round trip.  (Stages of one channel in a ring of 6 cost a
// hand-off per channel: 321 us instead of 255 us at V=15, profiles/r2_notes.md.)
//
// Precision: the reference computes in fp32.  tf32 operands keep 10 mantissa bits, so both operands are split a = hi + lo
// with hi = rn_tf32(a) and lo = rn_tf32(a - hi) (a - hi is exact in fp32, |lo| <= 2^-11 |a|), and the contraction is
// hi*hi + lo*hi + hi*lo accumulated in fp32 in TMEM; the dropped lo*lo term and the rounding of lo are below 2^-21 relative
// per product.  What dominates instead is the tensor core's own accumulation: adding a K=8 product sum to the running fp32
// accumulator truncates, and the error grows linearly with the number of MMAs chained on one accumulator (measured: 4e-6
// relative at 468 chained MMAs, 1.5e-5 at 2088).  Hence 16 accumulators: each issuer rotates its hi*hi steps over up to 7, its
// lo terms get their own, and the epilogue adds the partial sums in fp32.  tests/test_gpu_frontend.py states the tolerance against
// torch fp32 and fp64.
//
// K is permuted (we own the packed weight format): k' = ((xb * P + y) * 6 + oc) * 16 + px  <->  reference flatten index
// k = oc * P^2 + y * P + 16 xb + px  (P = N - 2; pixels beyond P are padding: zero weights, zero activations).
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <vector>

#include "ssd_b200.h"

namespace {

constexpr int kOC = 6;                       // conv_out   (config/default.yaml: conv_out 6, conv_kernel 3, conv_stride 1)
constexpr int kFeat = 32;                    // obs_dim_net
constexpr int kTileM = 128;                  // agent views per tile
#ifndef FE_OC_PER_STAGE
#define FE_OC_PER_STAGE 3
#endif
#ifndef FE_STAGES
#define FE_STAGES 2
#endif
#ifndef FE_TMA_SLEEP
#define FE_TMA_SLEEP 64
#endif
#ifndef FE_BSTAGES
#define FE_BSTAGES 4
#endif
constexpr int kG = FE_OC_PER_STAGE;          // output channels per pipeline stage (1, 2, 3 or 6)
constexpr int kStageK = 16 * kG;             // k' per stage: kG output channels x 16 pixels
constexpr int kStagesPerChunk = kOC / kG;
constexpr int kStages = FE_STAGES;                       // A ring: activations written by the producers
constexpr int kBStages = FE_BSTAGES;                     // B ring: FC weight tiles fetched by TMA, deep enough to run ~2 chunks ahead
constexpr int kABytes = kTileM * kStageK * 4;          // 8 KB x kG (one of hi / lo)
constexpr int kBBytes = kFeat * kStageK * 4;           // 2 KB x kG (one of hi / lo)
constexpr int kASbo = 512 * kG, kBSbo = 512 * kG;      // bytes between 8-row groups: 4 kG cores of 128 B
constexpr int kAStageBytes = 2 * kABytes;
constexpr int kBStageBytes = 2 * kBBytes;
constexpr int kSmemBytes = kStages * kAStageBytes + kBStages * kBStageBytes;
static_assert(kOC % kG == 0, "stage must hold whole output channels");
static_assert(kSmemBytes + 1024 <= 227 * 1024, "rings exceed shared memory");
constexpr int kProducerThreads = 256;
constexpr int kIssuers = 2;                              // MMA-issuing warps (8 and 10): the issue rate of one lane was the limit
constexpr int kThreads = kProducerThreads + 96;        // + MMA warp + TMA warp + second MMA warp
constexpr int kAccs = 16;                                // independent fp32 accumulators in TMEM (see `Precision`)
constexpr uint32_t kTmemCols = kAccs * kFeat;          // 512 columns: the whole TMEM of the SM (one CTA per SM)

struct EpilogueParams {                      // what segment_epilogue needs, passed to it by value
    long long rows;
    long long units;                         // n_tiles * n_chunks (< 2^31); CTA i of G works on units [i units / G, (i + 1) units / G)
    float* out;
    float* scratch;                          // [2 G][128][32] partial sums of the tiles a CTA shares with its neighbours
    int* tile_arrivals;                      // [n_tiles] zero between launches: partial segments stored so far
    const float* fc_b;                       // [32] in device memory
    int n_chunks;
    float slope;
};

struct FrontParams {
    unsigned long long conv_w2[kOC / 2][27]; // [oc pair][ch][dy][dx] = (w[2 op], w[2 op + 1]) as packed fp32, pre-scaled by 1/256
                                             // (exact): the conv sees raw bytes
    float conv_b[kOC];
    float slope;
    int N, P, RP, PS, AS, XB, n_chunks;      // obs geometry; chunks per tile = P * XB
    int n_tiles;
    const uint8_t* obs;
    EpilogueParams epi;
    uint32_t pal[3][4];                      // index4 only: byte i of plane c = color_lut[i][c]; behind everything else, so the RGB
                                             // kernel's parameter offsets (the tensor map's included) stay where they were
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" :: "r"(bar), "r"(parity) : "memory");
}
template <int kSleepNs = 64>
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {   // single-lane roles: poll, sleep, poll ...
    for (;;) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return;
        __nanosleep(kSleepNs);               // leave the issue slots to the producer warps
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// K-major, no swizzle: 8-row x 16-byte core matrices; LBO = distance between the two cores of one K=8 step,
// SBO = distance between 8-row groups (cute/arch/mma_sm100_desc.hpp SmemDescriptor, version 1 = Blackwell).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// The MMA warp runs its loop warp-uniformly and only the issue instructions are predicated on the elected lane: descriptors and
// addresses then live in uniform registers, which is what UTCHMMA reads (inside an `if (lane == 0)` block they are computed in
// vector registers and moved over with ~15 R2UR per K step -- and the issue rate of this lane is on the critical path).
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate,
                                          uint32_t elected) {
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
                 "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(elected) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar, uint32_t elected) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
                 "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" :: "r"(bar), "r"(elected) : "memory");
}

__device__ __forceinline__ float leaky(float v, float slope) { return v > 0.f ? v : v * slope; }
__device__ __forceinline__ uint32_t to_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}

__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {   // two IEEE fp32 FMAs
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

// u8 -> f32 on the full-rate pipes: 0x4B0000bb is the float 8388608 + bb (one PRMT), minus 8388608 (one FADD); I2F is a
// quarter-rate conversion-pipe instruction and 90 of them per 1296 FFMAs showed up in the profile
__device__ __forceinline__ float byte_to_float(uint32_t word, int b) {
    uint32_t v;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(v) : "r"(word), "r"(0x4B000000u), "r"(0x7540u + (uint32_t)b));
    return __uint_as_float(v) - 8388608.0f;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t v;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(v) : "r"(a), "r"(b), "r"(sel));
    return v;
}

// Four colour indices -> four channel bytes of one plane through its 16-byte palette `pal`.  A PRMT selector nibble picks one
// of 8 bytes by its low 3 bits (bit 3 would replicate the byte's sign), so `sel` holds the indices & 7, one lookup reads
// entries 0-7, one entries 8-15, and `m` (0xff in the bytes whose index has bit 3 set) picks between them.
__device__ __forceinline__ uint32_t palette4(const uint32_t (&pal)[4], uint32_t sel, uint32_t m) {
    return (prmt(pal[2], pal[3], sel) & m) | (prmt(pal[0], pal[1], sel) & ~m);
}

// hi*hi accumulators each issuer rotates over in a segment of `stages` stages: chains of at most ~24 MMAs each (see `Precision`),
// at most 7 (+ 1 for the lo terms) of the 8 accumulators an issuer owns
__device__ __forceinline__ int rotation(int stages) {
    const int steps = stages * (kStageK / 8) / kIssuers;
    return min(kAccs / kIssuers - 1, (steps + 23) / 24);
}

// Epilogue of one segment, by warps 0-3 (TMEM lane = GEMM row = r).  Kept out of line so that its 32 + 32 live registers do not
// weigh on the register allocation of the convolution loop.  One copy per kernel (IDX is otherwise unused): with a single
// caller the compiler addresses that kernel's `arrivals_s` directly instead of through the pointer argument.
template <bool IDX>
__device__ __noinline__ void segment_epilogue(const EpilogueParams p, uint32_t tmem_base, uint32_t bar_tmem_full, uint32_t bar_tmem_empty,
                                          int* arrivals_s, uint32_t parity, int stages_here, int tile, bool whole_tile,
                                          bool first_segment) {
    const int tid = threadIdx.x, warp = tid >> 5, r = tid & 127;
    const long long row = (long long)tile * kTileM + r;
    mbar_wait(bar_tmem_full, parity);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    float sum[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) sum[j] = 0.f;
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
    // the partial sums are added smallest first (accumulator 0 holds the lo terms), in fp32 round-to-nearest
    const int n_acc = 1 + rotation(stages_here);                   // per issuer; short segments use fewer than 8
    for (int ai = 0; ai < kIssuers * n_acc; ++ai) {
        const int a = (ai % kIssuers) * (kAccs / kIssuers) + ai / kIssuers;   // 0, 8 (the lo terms), 1, 9, 2, 10, ...
        uint32_t v[32];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                     "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                     "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                       "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                       "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                       "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                     : "r"(taddr + (uint32_t)(a * kFeat)) : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 32; ++j) sum[j] += __uint_as_float(v[j]);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    mbar_arrive(bar_tmem_empty);                                   // the accumulator may be overwritten by the next tile
    if (!whole_tile) {
        // A tile shared with neighbouring CTAs: raw partial sums go to this CTA's scratch slot (2 i for the tile it
        // starts in, 2 i + 1 for the tile it ends in); the CTA that stores the tile's LAST part adds all parts in CTA
        // order -- so the result does not depend on which CTA that is -- and writes the output.
        const int slot = 2 * blockIdx.x + (first_segment ? 0 : 1);
        float4* dst = reinterpret_cast<float4*>(p.scratch + ((long long)slot * kTileM + r) * kFeat);
#pragma unroll
        for (int j = 0; j < 8; ++j) __stcg(dst + j, make_float4(sum[4 * j], sum[4 * j + 1], sum[4 * j + 2], sum[4 * j + 3]));
        // CTA that holds unit X: ceil((X + 1) G / U) - 1, because CTA i starts at floor(i U / G)
        const long long x0 = (long long)tile * p.n_chunks, x1 = x0 + p.n_chunks - 1, G = gridDim.x;
        const int i0 = (int)(((x0 + 1) * G + p.units - 1) / p.units) - 1, i1 = (int)(((x1 + 1) * G + p.units - 1) / p.units) - 1;
        __threadfence();                                            // this thread's part is visible device-wide ...
        asm volatile("bar.sync 1, 128;" ::: "memory");              // ... and so is every epilogue thread's
        if (tid == 0) *arrivals_s = atomicAdd(p.tile_arrivals + tile, 1);
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (*arrivals_s == i1 - i0) {                                // the other i1 - i0 parts were stored before this one
            __threadfence();
            if (tid == 0) p.tile_arrivals[tile] = 0;                // ready for the next launch
#pragma unroll
            for (int j = 0; j < 32; ++j) sum[j] = 0.f;
            for (int i = i0; i <= i1; ++i) {
                const int b = (int)((long long)i * p.units / G);
                const int sl = 2 * i + (b >= x0 ? 0 : 1);           // b_i <= x1 for every CTA of this tile
                const float4* src = reinterpret_cast<const float4*>(p.scratch + ((long long)sl * kTileM + r) * kFeat);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 v = __ldcg(src + j);
                    sum[4 * j] += v.x; sum[4 * j + 1] += v.y; sum[4 * j + 2] += v.z; sum[4 * j + 3] += v.w;
                }
            }
            if (row < p.rows) {
                float4* o4 = reinterpret_cast<float4*>(p.out + row * kFeat);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.fc_b) + j);
                    float4 o;
                    o.x = leaky(sum[4 * j + 0] + b4.x, p.slope);
                    o.y = leaky(sum[4 * j + 1] + b4.y, p.slope);
                    o.z = leaky(sum[4 * j + 2] + b4.z, p.slope);
                    o.w = leaky(sum[4 * j + 3] + b4.w, p.slope);
                    o4[j] = o;
                }
            }
        }
    } else if (row < p.rows) {
        float4* dst = reinterpret_cast<float4*>(p.out + row * kFeat);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.fc_b) + j);
            float4 o;
            o.x = leaky(sum[4 * j + 0] + b4.x, p.slope);
            o.y = leaky(sum[4 * j + 1] + b4.y, p.slope);
            o.z = leaky(sum[4 * j + 2] + b4.z, p.slope);
            o.w = leaky(sum[4 * j + 3] + b4.w, p.slope);
            dst[j] = o;
        }
    }
}

// IDX: the views are SSD_OBS_INDEX4 rows (pixel x = nibble x of the row, p.RP bytes apart, p.PS unused) instead of RGB planes.
// Only what a window row is loaded from differs: two nibble words instead of nine byte words, expanded through p.pal into
// the same 3 planes x 3 words of channel bytes, so everything from byte_to_float on is the same code and the same arithmetic.
template <bool IDX>
__global__ void __launch_bounds__(kThreads, 1)
obs_frontend_kernel(const __grid_constant__ FrontParams p, const __grid_constant__ CUtensorMap wmap) {
    extern __shared__ __align__(1024) uint8_t smem[];
    // Two rings with their own barriers: the weight tile of a stage comes from L2 with ~1-2 us of TMA latency, so it must
    // not wait for the activation slot of the same stage to be released (first version: one ring, 0.6 us per stage even
    // with the convolution removed).
    __shared__ __align__(8) uint64_t bar_full[kStages], bar_empty[kStages], bar_bfull[kBStages], bar_bempty[kBStages],
                                     bar_tmem_full, bar_tmem_empty;
    __shared__ uint32_t tmem_base_s;
    __shared__ int arrivals_s;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(smem_u32(&bar_full[s]), kProducerThreads / 32); mbar_init(smem_u32(&bar_empty[s]), kIssuers); }
        for (int s = 0; s < kBStages; ++s) { mbar_init(smem_u32(&bar_bfull[s]), 1); mbar_init(smem_u32(&bar_bempty[s]), kIssuers); }
        mbar_init(smem_u32(&bar_tmem_full), kIssuers);
        mbar_init(smem_u32(&bar_tmem_empty), 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {                                           // one warp allocates the accumulator columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "n"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    const uint32_t smem_base = smem_u32(smem);
    // Work division ("stream-K"): all (tile, chunk) units in one sequence, an equal contiguous share per CTA.  A share is cut at
    // tile boundaries into segments; a segment that covers a whole tile stores the finished output, a partial one stores raw
    // partial sums, and the last of a tile's CTAs to do so adds them up.  Every role walks the same segments.
    const int u_begin = (int)((long long)blockIdx.x * p.epi.units / gridDim.x), u_end = (int)((long long)(blockIdx.x + 1) * p.epi.units / gridDim.x);

    if (warp < 8) {
        // ------------------------------------------------------------------ producers (+ epilogue on warps 0-3)
        const int r = tid & 127, strip = tid >> 7;             // GEMM row within the tile; 8-pixel half of the 16-pixel block
        uint32_t it = 0, item_n = 0;
        unsigned long long bias2[kOC / 2];
#pragma unroll
        for (int op = 0; op < kOC / 2; ++op) bias2[op] = pack2(p.conv_b[2 * op], p.conv_b[2 * op + 1]);
        for (int u = u_begin; u < u_end; ++item_n) {
            const int tile = u / p.n_chunks, c_begin = u - tile * p.n_chunks;
            const int c_end = min(p.n_chunks, c_begin + (u_end - u));
            const bool first_segment = u == u_begin;
            u += c_end - c_begin;
            const int stages_here = (c_end - c_begin) * kStagesPerChunk;
            const long long row = (long long)tile * kTileM + r;
            // Chunks run down a 16-pixel column (c = xb * P + y), so consecutive chunks share two of their three patch rows: the
            // thread keeps a 3-row window of raw words (3 planes x 3 words per row) and loads ONE new row per chunk -- requested
            // before the current chunk is convolved, so its L2 latency hides behind the FMAs.  (A shared-memory row window filled
            // with coalesced loads was measured and dropped: the per-row CTA barrier cost more than the sectors it saved --
            // V=15: 515 us instead of 397 us, profiles/r2_notes.md.)
            const long long row_ld = row < p.epi.rows ? row : p.epi.rows - 1;          // partial last tile: compute on a valid row, never store
            const uint8_t* view = p.obs + row_ld * p.AS;
            uint32_t win[3][9], nxt[9];
            // src points at (row yy, pixel x0) of plane 0; the three guards depend on the column only
            auto load_row = [&](uint32_t (&dst)[9], const uint8_t* src, bool g0, bool g1, bool g2) {
                if constexpr (IDX) {                                           // raw nibble words: pixels x0..x0+7, x0+8..x0+15
                    dst[0] = g0 ? __ldg(reinterpret_cast<const uint32_t*>(src)) : 0u;
                    dst[1] = g2 ? __ldg(reinterpret_cast<const uint32_t*>(src + 4)) : 0u;   // only x0+8, x0+9 < N are used
                } else {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch, src += p.PS) {
#ifdef FE_DIAG_NOLOAD                                                  // diagnostic build: one load per row instead of 9
                    if (ch == 0) dst[0] = __ldg(reinterpret_cast<const uint32_t*>(src));
                    dst[ch * 3] = dst[0] + ch; dst[ch * 3 + 1] = dst[0] ^ ch; dst[ch * 3 + 2] = dst[0] + 3 * ch;
#else
                    dst[ch * 3] = g0 ? __ldg(reinterpret_cast<const uint32_t*>(src)) : 0u;
                    dst[ch * 3 + 1] = g1 ? __ldg(reinterpret_cast<const uint32_t*>(src + 4)) : 0u;
                    dst[ch * 3 + 2] = g2 ? __ldg(reinterpret_cast<const uint32_t*>(src + 8)) : 0u;   // only pixels x0+8, x0+9 < N are used
#endif
                }
                }
            };
            // index4: the two nibble words of a row (raw[0], raw[1]) -> the RGB window row (in place when dst is raw)
            auto expand_row = [&](uint32_t (&dst)[9], const uint32_t (&raw)[9]) {
                const uint32_t w = raw[0], w1 = raw[1];
                const uint32_t s = w & 0x77777777u, s1 = w1 & 0x77u;
                // byte masks from bit 3 of each index: a PRMT selector nibble >= 8 replicates the chosen byte's top bit, which is
                // bit 3 of the odd pixel of that byte of w, or of the even pixel in w << 4
                const uint32_t m0 = prmt(w << 4, w, 0xD9C8u), m1 = prmt(w << 4, w, 0xFBEAu), m2 = prmt(w1 << 4, w1, 0xD9C8u);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    dst[ch * 3] = palette4(p.pal[ch], s, m0);
                    dst[ch * 3 + 1] = palette4(p.pal[ch], s >> 16, m1);
                    dst[ch * 3 + 2] = palette4(p.pal[ch], s1, m2);
                }
            };
            int xb = c_begin / p.P, y = c_begin - xb * p.P;                    // kept incrementally: no division per chunk
            const uint8_t* next_row = view;                                    // row y + 3 of the current column, at pixel x0
            bool g0 = false, g1 = false, g2 = false;
            for (int c = c_begin; c < c_end; ++c) {
                if (c == c_begin || y == 0) {                                  // first chunk of the item or of a column: whole window
                    const int x0 = xb * 16 + strip * 8;
                    // index4: x0 is a multiple of 8, so a nibble word at byte x0 / 2 < ceil(N / 2) <= RP (a multiple of 4) ends
                    // inside the row stride
                    g0 = x0 < (IDX ? p.N : p.RP); g1 = x0 + 4 < p.RP; g2 = x0 + 8 < p.N;
                    const uint8_t* src = view + y * p.RP + (IDX ? x0 >> 1 : x0);
                    load_row(win[0], src, g0, g1, g2);
                    load_row(win[1], src + p.RP, g0, g1, g2);
                    load_row(nxt, src + 2 * p.RP, g0, g1, g2);
                    next_row = src + 3 * p.RP;
                    if constexpr (IDX) { expand_row(win[0], win[0]); expand_row(win[1], win[1]); }
                }
                if constexpr (IDX) {
                    expand_row(win[2], nxt);                                   // nxt stays raw: its loads landed during the last chunk
                } else {
#pragma unroll
                    for (int k = 0; k < 9; ++k) win[2][k] = nxt[k];
                }
                if (c + 1 < c_end && y + 1 < p.P) load_row(nxt, next_row, g0, g1, g2);   // the row the next chunk adds
                next_row += p.RP;
                if (++y == p.P) { y = 0; ++xb; }
                uint32_t cur[27];
#pragma unroll
                for (int ch = 0; ch < 3; ++ch)
#pragma unroll
                    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                        for (int w = 0; w < 3; ++w) cur[(ch * 3 + dy) * 3 + w] = win[dy][ch * 3 + w];
#pragma unroll
                for (int k = 0; k < 9; ++k) { win[0][k] = win[1][k]; win[1][k] = win[2][k]; }
                // The conv runs on packed fp32 pairs (fma.rn.f32x2 -> SASS FFMA2, new on sm_100): one instruction updates the same
                // output pixel of TWO output channels -- the input pixel is the broadcast scalar operand (R.F32), the two conv
                // weights a packed uniform-register pair (UR.F32x2) read straight from the kernel parameters, so no register
                // pairs have to be assembled (pairing neighbouring pixels instead cost 380 MOVs per 648 FFMA2).
                // acc2[op][px] = channels (2 op, 2 op + 1) of pixel px.  Raw bytes go in (the 1/256 lives in the conv weights);
                // pixels beyond the image row are finite garbage that only meets zero FC weights.
                unsigned long long acc2[kOC / 2][8];
#pragma unroll
                for (int op = 0; op < kOC / 2; ++op)
#pragma unroll
                    for (int px = 0; px < 8; ++px) acc2[op][px] = bias2[op];
#ifdef FE_DIAG_NOCONV
#pragma unroll
                for (int k = 0; k < 27; ++k) acc2[k % 3][k & 7] ^= cur[k];
#else
#pragma unroll
                for (int ch = 0; ch < 3; ++ch)
#pragma unroll
                    for (int dy = 0; dy < 3; ++dy) {
                        const int k = (ch * 3 + dy) * 3;
                        float e[10];
#pragma unroll
                        for (int b = 0; b < 4; ++b) { e[b] = byte_to_float(cur[k], b); e[4 + b] = byte_to_float(cur[k + 1], b); }
                        e[8] = byte_to_float(cur[k + 2], 0);
                        e[9] = byte_to_float(cur[k + 2], 1);
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
                            for (int op = 0; op < kOC / 2; ++op) {
                                const unsigned long long w2 = p.conv_w2[op][ch * 9 + dy * 3 + dx];
#pragma unroll
                                for (int px = 0; px < 8; ++px) acc2[op][px] = fma2(pack2(e[px + dx], e[px + dx]), w2, acc2[op][px]);
                            }
                        }
                    }
#endif
#pragma unroll
                for (int g = 0; g < kStagesPerChunk; ++g, ++it) {
                    uint32_t hi[kG][8], lo[kG][8];
#pragma unroll
                    for (int og = 0; og < kG; ++og) {
                        const int oc = g * kG + og;
                        float acc[8];
#pragma unroll
                        for (int px = 0; px < 8; ++px) {
                            float c0, c1;
                            unpack2(acc2[oc >> 1][px], c0, c1);
                            acc[px] = (oc & 1) ? c1 : c0;
                        }
#pragma unroll
                        for (int px = 0; px < 8; ++px) {                       // (padding pixels meet zero weights: no masking)
                            const float a = fmaxf(acc[px], acc[px] * p.slope); // LeakyReLU for 0 <= slope <= 1 (checked at create)
                            hi[og][px] = to_tf32(a);                           // round-to-nearest tf32: exactly what the tensor core will read
                            lo[og][px] = __float_as_uint(a - __uint_as_float(hi[og][px]));   // exact in fp32, |lo| <= 2^-11 |a|; the tensor core keeps its top 10 bits
                        }
                    }
                    const uint32_t s = it % kStages, ph = (it / kStages) & 1u;
                    mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1u);               // the MMAs that read this slot have completed
                    uint8_t* a_hi = smem + s * kAStageBytes + (r >> 3) * kASbo + (r & 7) * 16 + strip * 256;
                    uint8_t* a_lo = a_hi + kABytes;
#pragma unroll
                    for (int og = 0; og < kG; ++og) {                          // k' = og * 16 + strip * 8 + px -> core (k' / 4), 128 B apart
                        *reinterpret_cast<uint4*>(a_hi + og * 512) = make_uint4(hi[og][0], hi[og][1], hi[og][2], hi[og][3]);
                        *reinterpret_cast<uint4*>(a_hi + og * 512 + 128) = make_uint4(hi[og][4], hi[og][5], hi[og][6], hi[og][7]);
                        *reinterpret_cast<uint4*>(a_lo + og * 512) = make_uint4(lo[og][0], lo[og][1], lo[og][2], lo[og][3]);
                        *reinterpret_cast<uint4*>(a_lo + og * 512 + 128) = make_uint4(lo[og][4], lo[og][5], lo[og][6], lo[og][7]);
                    }
#ifndef FE_DIAG_NOFENCE
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // generic-proxy writes -> tensor-core reads
#endif
                    __syncwarp();                                               // every lane's writes + fence precede the warp's one arrival
                    if (lane == 0) mbar_arrive(smem_u32(&bar_full[s]));
                }
            }
            if (warp < 4)
                segment_epilogue<IDX>(p.epi, tmem_base, smem_u32(&bar_tmem_full), smem_u32(&bar_tmem_empty), &arrivals_s, item_n & 1u, stages_here,
                                 tile, c_end - c_begin == p.n_chunks, first_segment);
        }
    } else if (warp != 9) {
        // ---------------------------------------------------------------------- MMA issuers (warps 8 and 10, one elected lane each)
        // Issuer w takes the K steps ks = w, w + 2, w + 4 of every stage and owns accumulators 8 w .. 8 w + 7.
        const uint32_t w = warp == 8 ? 0u : 1u;
        // instruction descriptor: D = f32, A = B = tf32, both K-major, N = 32, M = 128 (cute/arch/mma_sm100_desc.hpp InstrDescriptor)
        constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kFeat >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
        const uint32_t elected = elect_one();
        uint32_t it = 0, item_n = 0;
        for (int u = u_begin; u < u_end; ++item_n) {
            const int c_begin = u % p.n_chunks;
            const int c_end = min(p.n_chunks, c_begin + (u_end - u));
            u += c_end - c_begin;
            const int stages_here = (c_end - c_begin) * kStagesPerChunk;
            if (item_n > 0) mbar_wait_relaxed(smem_u32(&bar_tmem_empty), (item_n - 1) & 1u);   // the epilogue has drained the previous item
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t used = 0;                                                 // accumulators already written in this item
            // the tensor core truncates when it aligns a product sum with the running accumulator, so the error grows with the
            // number of MMAs chained on one accumulator: the hi*hi steps rotate over up to 15 accumulators, the (2^-11 smaller)
            // lo terms have their own; the epilogue adds the partial sums
            const uint32_t n_rot = (uint32_t)rotation(stages_here);
            const uint32_t acc_lo = w * (kAccs / kIssuers);
            uint32_t acc = acc_lo + 1;
            for (int st = 0; st < stages_here; ++st, ++it) {
                const uint32_t s = it % kStages, ph = (it / kStages) & 1u;
                const uint32_t sb = it % kBStages, phb = (it / kBStages) & 1u;
                mbar_wait(smem_u32(&bar_bfull[sb]), phb);                      // weight tile landed (TMA, issued well ahead)
                mbar_wait(smem_u32(&bar_full[s]), ph);                         // activations written by the 256 producers
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_hi = smem_base + s * kAStageBytes, b_hi = smem_base + kStages * kAStageBytes + sb * kBStageBytes;
                uint64_t dah = umma_desc(a_hi + w * 256, 128, kASbo), dal = umma_desc(a_hi + kABytes + w * 256, 128, kASbo);
                uint64_t dbh = umma_desc(b_hi + w * 256, 128, kBSbo), dbl = umma_desc(b_hi + kBBytes + w * 256, 128, kBSbo);
#pragma unroll
                for (int kk = 0; kk < kStageK / 8 / kIssuers; ++kk) {          // one K=8 step = two 16-byte cores, 256 B further on
#ifndef FE_DIAG_NOMMA
                    umma_tf32(tmem_base + acc * kFeat, dah, dbh, idesc, (used >> acc) & 1u, elected);
#endif
#if !defined(FE_DIAG_HIONLY) && !defined(FE_DIAG_NOMMA)                        // diagnostic build: one MMA per K step instead of three
                    umma_tf32(tmem_base + acc_lo * kFeat, dal, dbh, idesc, (used >> acc_lo) & 1u, elected);
                    umma_tf32(tmem_base + acc_lo * kFeat, dah, dbl, idesc, 1u, elected);
#endif
                    used |= (1u << acc_lo) | (1u << acc);
                    acc = acc == acc_lo + n_rot ? acc_lo + 1u : acc + 1u;
                    dah += kIssuers * 256 >> 4; dal += kIssuers * 256 >> 4;    // the address field counts 16-byte units
                    dbh += kIssuers * 256 >> 4; dbl += kIssuers * 256 >> 4;
                }
                umma_commit(smem_u32(&bar_empty[s]), elected);                 // frees both slots when these MMAs have read them
                umma_commit(smem_u32(&bar_bempty[sb]), elected);
                if (st == stages_here - 1) umma_commit(smem_u32(&bar_tmem_full), elected);
            }
        }
    } else {
        // ---------------------------------------------------------------------- TMA: FC weight tile of every stage
        if (lane == 0) {
            uint32_t it = 0;
            for (int u = u_begin; u < u_end;) {
                const int c_begin = u % p.n_chunks;
                const int c_end = min(p.n_chunks, c_begin + (u_end - u));
                u += c_end - c_begin;
                const int st_begin = c_begin * kStagesPerChunk, st_end = c_end * kStagesPerChunk;
                for (int st = st_begin; st < st_end; ++st, ++it) {
                    const uint32_t sb = it % kBStages, phb = (it / kBStages) & 1u;
                    mbar_wait_relaxed<FE_TMA_SLEEP>(smem_u32(&bar_bempty[sb]), phb ^ 1u);
                    const uint32_t full = smem_u32(&bar_bfull[sb]);
                    mbar_arrive_expect_tx(full, kBStageBytes);
                    tma_load_2d(smem_base + kStages * kAStageBytes + sb * kBStageBytes, &wmap, full, 0, st * 4 * kG);   // 4 kG rows of 256 floats = hi + lo
                }
            }
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "n"(kTmemCols) : "memory");
}

thread_local int g_front_cuda_error = 0;

inline float host_tf32(float v) {                              // cvt.rna.tf32.f32: nearest, ties away from zero (finite inputs)
    uint32_t bits; memcpy(&bits, &v, 4);
    bits = (bits + 0x1000u) & 0xffffe000u;
    float r; memcpy(&r, &bits, 4);
    return r;
}

}  // namespace

struct ssd_frontend {
    FrontParams fp;
    CUtensorMap wmap;
    float* d_w;                                                // packed FC weights: [stages][hi | lo] tiles, then the 32 bias floats
    float* d_scratch;                                          // partial sums of shared tiles: [2 sms][128][32]
    int* d_arrivals;                                           // [arrivals_len] per-tile counters, zero between launches
    size_t arrivals_len;
    int device, view, sms;
    size_t smem_bytes;
};

// Launch of either format: `p` is the handle's parameters with the obs strides (and, for index4, the palette) filled in.
static int frontend_launch(ssd_frontend* f, FrontParams& p, bool index4, const uint8_t* obs, int64_t rows, float* out, void* stream) {
    if ((rows + kTileM - 1) / kTileM * p.n_chunks >= (1ll << 31)) return SSD_ERR_INVALID;   // the kernel counts units in 32 bits
    p.epi.rows = rows; p.n_tiles = (int)((rows + kTileM - 1) / kTileM);
    p.obs = obs; p.epi.out = out;
    // Load balance: 160 tiles on 148 persistent CTAs would leave a second, almost empty round, so the (tile, chunk) units are
    // dealt out as one sequence in equal contiguous shares (see the kernel).  Tiles cut by a share boundary are combined in CTA
    // order by whichever CTA stores its part last, so the result does not depend on timing.  The scratch slots and arrival
    // counters belong to the handle: one forward at a time per handle (stream order is enough; concurrent streams need one
    // handle each).
    const long long units = p.epi.units = (long long)p.n_tiles * p.n_chunks;
    // Grid: all SMs with equal shares, or -- few tiles -- s CTAs per tile (shares aligned with the tiles, one segment per CTA);
    // whichever has the cheaper busiest CTA at ~1.5 chunks of pipeline fill + accumulator drain per segment.
    int grid = units < f->sms ? (int)units : f->sms;
    {
        const double share = (double)units / grid;
        double best = share + 1.5 * (share < p.n_chunks ? 2.0 : (double)((long long)(share / p.n_chunks) + 2));
        for (int s_ = 1; s_ <= p.n_chunks && (long long)p.n_tiles * s_ <= f->sms; ++s_) {
            const double cost = (double)((p.n_chunks + s_ - 1) / s_) + 1.5;
            if (cost < best - 1e-9) { best = cost; grid = p.n_tiles * s_; }
        }
    }
    { const char* e_ = getenv("SSD_B200_FRONTEND_GRID"); if (e_ && atoi(e_) >= 1 && atoi(e_) <= grid) grid = atoi(e_); }   // tuning
    int prev = -1;
    cudaError_t e = cudaGetDevice(&prev);
    if (e == cudaSuccess && prev != f->device) e = cudaSetDevice(f->device);
    if (e == cudaSuccess && !f->d_scratch)                     // first call (not capturable): two partial tiles per CTA
        e = cudaMalloc(&f->d_scratch, (size_t)2 * f->sms * kTileM * kFeat * sizeof(float));
    if (e == cudaSuccess && (size_t)p.n_tiles > f->arrivals_len) {             // first call / larger batch (not capturable)
        if (f->d_arrivals) cudaFree(f->d_arrivals);
        f->d_arrivals = nullptr; f->arrivals_len = 0;
        const size_t len = ((size_t)p.n_tiles + 1023) / 1024 * 1024;
        e = cudaMalloc(&f->d_arrivals, len * sizeof(int));
        if (e == cudaSuccess) e = cudaMemsetAsync(f->d_arrivals, 0, len * sizeof(int), (cudaStream_t)stream);
        if (e == cudaSuccess) f->arrivals_len = len;
    }
    p.epi.scratch = f->d_scratch;
    p.epi.tile_arrivals = f->d_arrivals;
    if (e == cudaSuccess) {
        if (index4)
            obs_frontend_kernel<true><<<grid, kThreads, f->smem_bytes, (cudaStream_t)stream>>>(p, f->wmap);
        else
            obs_frontend_kernel<false><<<grid, kThreads, f->smem_bytes, (cudaStream_t)stream>>>(p, f->wmap);
        e = cudaGetLastError();
    }
    if (prev >= 0 && prev != f->device) cudaSetDevice(prev);
    if (e != cudaSuccess) { g_front_cuda_error = (int)e; return SSD_ERR_CUDA; }
    return SSD_OK;
}

extern "C" {

int ssd_frontend_create(int32_t view, const float* conv_w, const float* conv_b, const float* fc_w, const float* fc_b,
                        float negative_slope, int32_t device, ssd_frontend** out) {
    if (!out) return SSD_ERR_INVALID;
    *out = nullptr;
    if (!conv_w || !conv_b || !fc_w || !fc_b || view < 1 || view > 31) return SSD_ERR_INVALID;
    if (!(negative_slope >= 0.0f && negative_slope <= 1.0f)) return SSD_ERR_INVALID;              // LeakyReLU as max(x, slope x)
    const int N = 2 * view + 1, P = N - 2, XB = (P + 15) / 16, n_chunks = P * XB, stages = n_chunks * kStagesPerChunk;
    ssd_frontend* f = new (std::nothrow) ssd_frontend;
    if (!f) return SSD_ERR_INVALID;
    memset(f, 0, sizeof(*f));
    FrontParams& p = f->fp;
    for (int op = 0; op < kOC / 2; ++op)
        for (int t = 0; t < 27; ++t) {                                                // exact scaling: get_obs() = u8 / 256 (map_env.py:943)
            const float w0 = conv_w[(2 * op) * 27 + t] * (1.0f / 256.0f), w1 = conv_w[(2 * op + 1) * 27 + t] * (1.0f / 256.0f);
            uint32_t b0, b1;
            memcpy(&b0, &w0, 4); memcpy(&b1, &w1, 4);
            p.conv_w2[op][t] = (unsigned long long)b0 | ((unsigned long long)b1 << 32);
        }
    for (int i = 0; i < kOC; ++i) p.conv_b[i] = conv_b[i];
    p.slope = p.epi.slope = negative_slope; p.epi.n_chunks = n_chunks; p.N = N; p.P = P; p.XB = XB; p.n_chunks = n_chunks;
    f->view = view; f->device = device;

    // FC weights, permuted to k' and laid out per stage exactly as the shared-memory image the tensor core reads:
    // element (n, kk) of a [32 x 16 kG] tile at float offset (n/8)*128 kG + (kk/4)*32 + (n%8)*4 + kk%4 ; hi image then lo image.
    const size_t stage_floats = 1024 * (size_t)kG, lo_off = 512 * (size_t)kG;
    std::vector<float> packed((size_t)stages * stage_floats, 0.f);
    for (int st = 0; st < stages; ++st) {
        const int c = st / kStagesPerChunk, g = st % kStagesPerChunk, xb = c / P, y = c % P;   // chunks run down a column
        for (int n = 0; n < kFeat; ++n)
            for (int kk = 0; kk < kStageK; ++kk) {
                const int oc = g * kG + kk / 16, x = xb * 16 + kk % 16;
                if (x >= P) continue;
                const float w = fc_w[(size_t)n * (kOC * P * P) + (size_t)oc * P * P + y * P + x];   // nn.Linear.weight [32][6 P^2], Flatten order (oc, y, x)
                const float hi = host_tf32(w);
                const size_t off = (size_t)st * stage_floats + (n / 8) * 128 * kG + (kk / 4) * 32 + (n % 8) * 4 + kk % 4;
                packed[off] = hi;
                packed[off + lo_off] = host_tf32(w - hi);
            }
    }
    int prev = -1;
    cudaError_t e = cudaGetDevice(&prev);
    if (e == cudaSuccess && prev != device) e = cudaSetDevice(device);
    const size_t w_floats = packed.size();
    packed.insert(packed.end(), fc_b, fc_b + kFeat);           // the FC bias rides behind the weight tiles
    if (e == cudaSuccess) e = cudaMalloc(&f->d_w, packed.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(f->d_w, packed.data(), packed.size() * sizeof(float), cudaMemcpyHostToDevice);
    p.epi.fc_b = f->d_w + w_floats;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&f->sms, cudaDevAttrMultiProcessorCount, device);
    int rc = SSD_OK;
    if (e == cudaSuccess) {
        // rank-2 tensor map over the packed weights viewed as [stages * 4][256] f32; box = 4 rows x 256 = one stage (4 KB)
        typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                     const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e == cudaSuccess && (!fn || qres != cudaDriverEntryPointSuccess)) rc = SSD_ERR_CUDA;
        if (e == cudaSuccess && rc == SSD_OK) {
            const cuuint64_t dims[2] = { 256, (cuuint64_t)stages * 4 * kG };
            const cuuint64_t strides[1] = { 1024 };
            const cuuint32_t box[2] = { 256, 4 * kG };
            const cuuint32_t estr[2] = { 1, 1 };
            const CUresult cr = reinterpret_cast<EncodeFn>(fn)(&f->wmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, f->d_w, dims, strides, box, estr,
                                                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (cr != CUDA_SUCCESS) { g_front_cuda_error = (int)cr; rc = SSD_ERR_CUDA; }
        }
    }
    f->smem_bytes = (size_t)kSmemBytes + 1024;
    if (e == cudaSuccess && rc == SSD_OK)
        e = cudaFuncSetAttribute(obs_frontend_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f->smem_bytes);
    if (e == cudaSuccess && rc == SSD_OK)
        e = cudaFuncSetAttribute(obs_frontend_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f->smem_bytes);
    if (prev >= 0 && prev != device) cudaSetDevice(prev);
    if (e != cudaSuccess || rc != SSD_OK) {
        if (e != cudaSuccess) g_front_cuda_error = (int)e;
        if (f->d_w) cudaFree(f->d_w);
        delete f;
        return SSD_ERR_CUDA;
    }
    *out = f;
    return SSD_OK;
}
int ssd_frontend_forward(ssd_frontend* f, const uint8_t* obs, int64_t rows, int32_t obs_agent_stride, int32_t obs_plane_stride,
                         int32_t obs_row_stride, float* out, void* stream) {
    if (!f || !obs || !out || rows < 0) return SSD_ERR_INVALID;
    if (rows == 0) return SSD_OK;
    FrontParams p = f->fp;
    if (obs_row_stride < p.N || (obs_row_stride & 3) || obs_plane_stride < p.N * obs_row_stride || (obs_plane_stride & 3) ||
        obs_agent_stride < 3 * obs_plane_stride || (obs_agent_stride & 3) || (reinterpret_cast<uintptr_t>(obs) & 3) ||
        (reinterpret_cast<uintptr_t>(out) & 15))
        return SSD_ERR_INVALID;
    p.RP = obs_row_stride; p.PS = obs_plane_stride; p.AS = obs_agent_stride;
    return frontend_launch(f, p, false, obs, rows, out, stream);
}

int ssd_frontend_forward_index4(ssd_frontend* f, const uint8_t* obs, int64_t rows, int32_t obs_agent_stride,
                                int32_t obs_row_stride, const uint8_t (*color_lut)[4], float* out, void* stream) {
    if (!f || !obs || !out || !color_lut || rows < 0) return SSD_ERR_INVALID;
    FrontParams p = f->fp;
    if (obs_row_stride < (p.N + 1) / 2 || (obs_row_stride & 3) || obs_agent_stride < p.N * obs_row_stride || (obs_agent_stride & 3) ||
        (reinterpret_cast<uintptr_t>(obs) & 3) || (reinterpret_cast<uintptr_t>(out) & 15))
        return SSD_ERR_INVALID;
    if (rows == 0) return SSD_OK;
    p.RP = obs_row_stride; p.PS = 0; p.AS = obs_agent_stride;
    for (int ch = 0; ch < 3; ++ch)
        for (int j = 0; j < 4; ++j)
            p.pal[ch][j] = (uint32_t)color_lut[4 * j][ch] | (uint32_t)color_lut[4 * j + 1][ch] << 8 |
                           (uint32_t)color_lut[4 * j + 2][ch] << 16 | (uint32_t)color_lut[4 * j + 3][ch] << 24;
    return frontend_launch(f, p, true, obs, rows, out, stream);
}

int ssd_frontend_destroy(ssd_frontend* f) {
    if (!f) return SSD_ERR_INVALID;
    int prev = -1;
    cudaGetDevice(&prev);
    if (prev != f->device) cudaSetDevice(f->device);
    cudaFree(f->d_w);
    if (f->d_scratch) cudaFree(f->d_scratch);
    if (f->d_arrivals) cudaFree(f->d_arrivals);
    if (prev >= 0 && prev != f->device) cudaSetDevice(prev);
    delete f;
    return SSD_OK;
}

int ssd_frontend_last_cuda_error(void) { return g_front_cuda_error; }

}  // extern "C"
