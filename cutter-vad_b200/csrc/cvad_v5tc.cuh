// cvad_v5tc.cuh -- Silero VAD v5 (16 kHz branch) on the 5th-gen tensor cores (tcgen05 + TMEM),
// FP32-accurate through a three-way BF16 operand split.
//
// Same pipeline and same hand-off as cvad_v5.cuh (the reference's per-frame session.run,
// /root/reference/src/real_time_vad/core/silero_model.py:433; graph = SURVEY.md 8a "S5"), but every
// GEMM-shaped stage runs as tcgen05.mma.kind::f16 with FP32 accumulation in TMEM:
//
//   x = x0 + x1 + x2,  w = w0 + w1 + w2   (x0 = bf16(x), x1 = bf16(x - x0), x2 = bf16(x - x0 - x1): 24 bits)
//   w.x ~= w0.x0  +  (w0.x1 + w1.x0)  +  (w0.x2 + w1.x1 + w2.x0)          dropped terms <= 2^-24 relative
//
// A single BF16 pass misses the 1e-4 parity bar by two orders of magnitude and the usual 3-pass split
// (16 bits) leaves 5e-5; the 6-product form is indistinguishable from an FP32 GEMM (tools/tc_probe_accuracy.py,
// measured on B200: 3.2e-7 vs 4.1e-7 relative for cuBLAS-style FP32).
//
// GEMM orientation: A = WEIGHTS (M = 128 or 64 output channels, K-major, streamed from L2 through a
// shared-memory ring by cp.async.bulk, already in the SWIZZLE_128B operand layout), B = ACTIVATIONS
// (N = items x time columns, K-major), D[channel][item] in TMEM.  With the weights as the M side a tile can
// be as small as 32 items, which is what a 4,096-stream frame step needs to fill 128 SMs.  An MMA whose
// operands both come from shared memory costs max(N/2, (M+N)/4, ~41) cycles on B200 (tools/tc_mma_rate.py),
// so time columns are batched into N (N = 96 for the STFT and encoder.0) and the recurrent kernel
// concatenates the three activation parts along N.
//
// The default build (FUSED, H16: one-frame steps, FP16 two-way split with per-stream scaling, three products per MAC) keeps
// the frame loader's operand K-major and writes every operand an EPILOGUE produces MN-major SWIZZLE_64B, so that a thread's
// one channel x eight streams is one 16-byte store (store_row8_mn); DESIGN.md section 3a.
//
// Warp roles (576 threads): warps 0-15 = loader + epilogue (TMEM -> registers -> activation -> next B operand;
// warp w reads TMEM lanes 32 (w % 4).. and column group w / 4), warp 16 = weight producer (one lane),
// warp 17 = MMA issuer (one elected lane).  Layers of one tile are
// strictly sequential, so ONE activation region is reused in place from layer to layer.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "cvad_tc.cuh"
#include "cvad_v5.cuh"

namespace cvad {
namespace tc5 {

constexpr int kEpiWarps = 16;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kProducerWarp = 16;
constexpr int kMmaWarp = 17;
constexpr int kThreadsTC = 576;
constexpr uint32_t kSlotBytes = 16384;       // one 128-row x 64-K BF16 weight tile
constexpr uint32_t kColMain = 0;             // TMEM column of the w0.x0 accumulator
constexpr uint32_t kColCorr = 192;           // TMEM column of the five correction products (columns 384.. hold the fused kernel's gates)

// ---------------------------------------------------------------- front-end weight stream
// Period = 69 tiles, in consumption order (each tile: rows x 64 K-elements, SW128 K-major, BF16 part p):
//   stft : blk 0..1 (0: re bins 0..127; 1: row 0 = re bin 128, rows 1..127 = im bins 1..127) x kb 0..3 x p 0..2   24 x 16 KB
//   enc0 : kb 0..1 x tap {1,0,2} x p   (channel 128, the Nyquist bin, is applied in the epilogue in FP32)           18 x 16 KB
//   enc1 : kb 0..1 x tap {1,2,0} x p   (64 rows)                                                                    18 x  8 KB
//   enc2 : tap {1,2} x p               (64 rows; tap 0 only ever meets the zero pad)                                 6 x  8 KB
//   enc3 : centre tap x p                                                                                            3 x 16 KB
constexpr int kFeSlotsPerTile = 69;
constexpr size_t kFeStreamBytes = 42 * 16384 + 24 * 8192 + 3 * 16384;
__host__ __device__ __forceinline__ void fe_slot(int s, uint32_t &off, uint32_t &bytes) {
    if (s < 42) { off = (uint32_t)s * 16384u; bytes = 16384u; }
    else if (s < 66) { off = 42u * 16384u + (uint32_t)(s - 42) * 8192u; bytes = 8192u; }
    else { off = 42u * 16384u + 24u * 8192u + (uint32_t)(s - 66) * 16384u; bytes = 16384u; }
}
// Recurrent weight stream: gate blk 0..3 (i,f,g,o) x kb 0..3 (K = [x 128 | h 128]) x p 0..2, 16 KB each.
constexpr int kRecSlotsPerFrame = 48;
constexpr size_t kRecStreamBytes = (size_t)kRecSlotsPerFrame * 16384;

// ---------------------------------------------------------------- shared memory plans
// front end: ACT (96 KB) | ring | nyq[96] f32 | barriers | tmem slot | tile meta
constexpr int kFeRing = 7;
constexpr uint32_t kActBytes = 98304;
constexpr uint32_t kActBytesH = 65536;       // FP16 build: two parts (AUD 2 x 32 KB is the largest tenant)
constexpr uint32_t kAudPart = 32768;         // AUD: part stride; K block stride 16384; row = seg*32 + item (128 rows)
constexpr uint32_t kMagPart = 24576;         // MAG/E0: 96 rows x 128 K; K block stride 12288
constexpr uint32_t kMagKb = 12288;
constexpr uint32_t kE1Part = 8192;           // E1: 64 rows x 64 K
constexpr uint32_t kE2Part = 4096;           // E2: 32 rows x 64 K
constexpr size_t kFeSmemTC = 1024 + kActBytes + (size_t)kFeRing * kSlotBytes + 96 * 4 + (2 * kFeRing + 2) * 8 + 16 +
                             3 * kTile * 4 + 64;
constexpr size_t kFeSmemTCH = kFeSmemTC + 2048;   // FP16-split build: + the per-stream maxima
// bytes [kFeatScaleOff, +128) of a feature tile (row 64 of K block 0: the unused third part) carry, in the FP16-split
// build, the 32 streams' joint maxima max(|x|max, 1) as float bit patterns: the scale of this frame's [x | h] operand
constexpr uint32_t kFeatScaleOff = 8192;
// fused single-frame kernel (max_frames == 1): the front end plus the LSTM step of the same 32 streams in one CTA.
// ACT | H operand (24 KB) | ring (6 slots) | nyq | decoder partials | barriers | meta.  Weight stream per tile:
// 24 W_hh tiles (issued while the loader runs), the 69 front-end tiles, 24 W_ih tiles.
constexpr int kPrefetchCtas = 16;            // chained steps: CTAs 0..15, when scheduled early, prefetch the step's audio into L2
constexpr int kFusedRing = 6;
constexpr int kFusedSlotsPerTile = 24 + kFeSlotsPerTile + 24;
constexpr uint32_t kColGate = 384;           // TMEM columns 384 + 32 g: gate g (i,f,g,o), one accumulator per gate
constexpr size_t kFusedSmemTC = 1024 + kActBytes + 24576 + (size_t)kFusedRing * kSlotBytes + 96 * 4 + 128 * 4 +
                                (2 * kFusedRing + 3 + 4) * 8 + 16 + 2 * kTile * 4 + kTile * 16 + 7 * kTile * 4 + kTile * 8 + 5 * kTile * 4 + 16 + 128;
// feature hand-off (front end -> recurrent), per (frame, stream tile): the x half of the recurrent B operand,
// byte for byte: [kb 0..1][row = part*32 + item (96 rows)][128 B], SW128
constexpr uint32_t kFeatTileBytes = 2 * 12288;
// recurrent: X[2] (2 x 24 KB) | H (24 KB) | ring | sbuf f32 [128][33] | dec partials [4][32] | barriers | meta
constexpr int kRecRing = 7;
constexpr uint32_t kXhKb = 12288;
constexpr size_t kRecSmemTC = 1024 + 3 * (size_t)kFeatTileBytes + (size_t)kRecRing * kSlotBytes + 128 * 33 * 4 + 4 * 32 * 4 +
                              (2 * kRecRing + 4) * 8 + 16 + kTile * (2 * 8 + 2 * 4) + 64;

// ---------------------------------------------------------------- small device helpers
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
// programmatic dependent launch, secondary side: blocks until the preceding grid of the stream has completed and its
// writes are visible (returns at once when the kernel was launched without the attribute)
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Gate nonlinearities of the LSTM cell on the SFU (MUFU.EX2 + MUFU.RCP): absolute error 2e-7 .. 4e-7 on values in
// (-1, 1).  Round 2 measured what that costs: a variant at float32-level accuracy (Newton step on the reciprocal, tanh as
// an odd polynomial below |x| = 1: 8e-8) changed NOTHING on 512,000 stateful frames (max |dp| 1.32e-4 vs 1.37e-4 on the
// same frame) and cost 1.7 % of the step -- the deviation of the tensor-core builds at ill-conditioned frames comes from
// tcgen05's truncating FP32 accumulation in TMEM (DESIGN.md "Accuracy at scale"), not from here.
__device__ __forceinline__ float sfu_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float sfu_tanh(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

// MUFU.SQRT: one instruction, <= 1 ulp (the IEEE sqrtf sequence is ~10 instructions per magnitude bin)
__device__ __forceinline__ float sfu_sqrt(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// 16-byte read-once global load that stays where it is written (volatile: issued right behind the state fetch that
// precedes it in program order, so that both latencies overlap), not allocated in L1
__device__ __forceinline__ float4 ldg_stream4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// 4-byte read-only global load as a volatile asm: keeps its program order relative to ldg_stream4 (state before audio)
__device__ __forceinline__ float ldg_ordered(const float *p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// x -> three BF16 parts (bit patterns)
__device__ __forceinline__ void split3(float x, unsigned short &p0, unsigned short &p1, unsigned short &p2) {
    const __nv_bfloat16 b0 = __float2bfloat16_rn(x);
    const float r1 = x - __bfloat162float(b0);
    const __nv_bfloat16 b1 = __float2bfloat16_rn(r1);
    const float r2 = r1 - __bfloat162float(b1);
    const __nv_bfloat16 b2 = __float2bfloat16_rn(r2);
    p0 = __bfloat16_as_ushort(b0);
    p1 = __bfloat16_as_ushort(b1);
    p2 = __bfloat16_as_ushort(b2);
}
// two values at once: word j holds part j of a (low half) and of b (high half); one F2FP per part
__device__ __forceinline__ void split3x2(float a, float b, uint32_t &w0, uint32_t &w1, uint32_t &w2) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w0) : "f"(b), "f"(a));
    const float ra = a - __uint_as_float(w0 << 16), rb = b - __uint_as_float(w0 & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w1) : "f"(rb), "f"(ra));
    const float sa = ra - __uint_as_float(w1 << 16), sb = rb - __uint_as_float(w1 & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w2) : "f"(sb), "f"(sa));
}
// store the parts of values a (row) and b (row + 1) at column k of a B operand with R rows (part stride ps);
// rows row and row + 1 lie in the same 8-row swizzle atom (row even)
__device__ __forceinline__ void store_parts2(unsigned char *base, uint32_t ps, uint32_t row, uint32_t k, uint32_t R, float a, float b) {
    uint32_t w0, w1, w2;
    split3x2(a, b, w0, w1, w2);
    unsigned char *da = base + tc::sw128_offset(row, k, R);
    unsigned char *db = base + tc::sw128_offset(row + 1, k, R);
    *reinterpret_cast<unsigned short *>(da) = (unsigned short)w0;
    *reinterpret_cast<unsigned short *>(da + ps) = (unsigned short)w1;
    *reinterpret_cast<unsigned short *>(da + 2 * ps) = (unsigned short)w2;
    *reinterpret_cast<unsigned short *>(db) = (unsigned short)(w0 >> 16);
    *reinterpret_cast<unsigned short *>(db + ps) = (unsigned short)(w1 >> 16);
    *reinterpret_cast<unsigned short *>(db + 2 * ps) = (unsigned short)(w2 >> 16);
}
// store the three parts of v at element (row, k) of a B operand with R rows (part stride ps)
__device__ __forceinline__ void store_parts(unsigned char *base, uint32_t ps, uint32_t row, uint32_t k, uint32_t R, float v) {
    unsigned short p0, p1, p2;
    split3(v, p0, p1, p2);
    unsigned char *d = base + tc::sw128_offset(row, k, R);
    *reinterpret_cast<unsigned short *>(d) = p0;
    *reinterpret_cast<unsigned short *>(d + ps) = p1;
    *reinterpret_cast<unsigned short *>(d + 2 * ps) = p2;
}

// warp-uniform: does tile (frame, stream tile) hold at least one live (stream, frame) item?
__device__ __forceinline__ bool tile_live(const V5Step &p, int frame, int st, int lane, int *slot_out, int *valid_out) {
    const int i = st * kTile + lane;
    int valid = 0, slot = -1;
    if (i < p.n_streams) {
        slot = p.slots ? p.slots[i] : i;
        const int nf = p.n_frames ? p.n_frames[i] : p.max_frames;
        valid = frame < nf;
    }
    if (slot_out) *slot_out = slot;
    if (valid_out) *valid_out = valid;
    return __any_sync(0xffffffffu, valid);
}

// MMAs of one weight tile (part wp of the A operand) for one 64-element K block: four K steps against the
// activation parts that pair with wp.  b0 = address of activation part 0 for this K block, parts are ps apart.
// w0.x0 accumulates in d_main, everything else in d_corr.
__device__ __forceinline__ void issue_split(int wp, uint32_t a_addr, uint32_t b0, uint32_t ps, uint32_t d_main,
                                            uint32_t d_corr, uint32_t idesc, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr);
    const uint64_t bd0 = tc::smem_desc_sw128(b0), bd1 = tc::smem_desc_sw128(b0 + ps), bd2 = tc::smem_desc_sw128(b0 + 2 * ps);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        const uint32_t fresh = (first && ks == 0) ? 0u : 1u;
        if (wp == 0) {
            tc::mma_bf16(d_corr, ad + ks * 2, bd2 + ks * 2, idesc, fresh);
            tc::mma_bf16(d_corr, ad + ks * 2, bd1 + ks * 2, idesc, 1u);
            tc::mma_bf16(d_main, ad + ks * 2, bd0 + ks * 2, idesc, fresh);
        } else if (wp == 1) {
            tc::mma_bf16(d_corr, ad + ks * 2, bd1 + ks * 2, idesc, 1u);
            tc::mma_bf16(d_corr, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        } else {
            tc::mma_bf16(d_corr, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        }
    }
}

__device__ __forceinline__ long long gtime_ns() {
    long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// The MMA issuer runs every line of its code once per tile, and the kernel's 170 KB of SASS do not stay in the
// instruction caches from launch to launch: with its outer loops rolled all but the first trip of a layer are fetched
// from the cache instead of L2 (tile 59.6 k -> 58.4 k cycles).  The inner loops stay unrolled -- the MMA operands must be
// compile-time offsets in uniform registers: one shared, non-inlined routine for all slots ran at 74 k cycles per tile.
#ifndef CVAD_ROLL_ISSUE
#define CVAD_ROLL_ISSUE 1
#endif
#if CVAD_ROLL_ISSUE
#define CVAD_ISSUE_ROLL _Pragma("unroll 1")
#else
#define CVAD_ISSUE_ROLL
#endif
// The marks compile away in the kernel build that runs when no profile was asked for (PROF = false: the ~45 tests of
// p.prof, each a parameter-bank read and a branch on the epilogue warps' path, were ~3 % of the kernel's stall samples).
#define CVAD_PROF_NS(k) do { if (PROF && p.prof && blockIdx.x == 0 && threadIdx.x == 0) p.prof[(k)] = gtime_ns(); } while (0)
// chained steps under cvad_set_profile: global-timer marks of CTAs 0, 64 and the last one, kept for the last 8 steps
// (prof[128 + 64 (step_seq % 8) + 8 b + k], k: 0 entry, 1 prologue done, 2 grid dependency resolved, 3 tile start, 4 tile end, 5 exit)
#define CVAD_CHAIN_NS(k) do { if (PROF && FUSED && p.prof && p.step_ctr && threadIdx.x == 0) {                                       \
        const int b_ = blockIdx.x == 0 ? 0 : (blockIdx.x == 64 ? 1 : (blockIdx.x == gridDim.x - 1 ? 2 : -1));                \
        if (b_ >= 0) p.prof[128 + 64 * (p.step_seq & 7) + 8 * b_ + (k)] = gtime_ns(); } } while (0)
#define CVAD_PROF(k) do { if (PROF && p.prof && blockIdx.x == 0 && first_tile) p.prof[(k)] = clock64(); } while (0)

// LSTM gate products of one weight tile (part wp) in the fused kernel: all six products of a MAC go to ONE
// accumulator (TMEM has no room for column groups next to the front end's); b0 = activation part 0, parts 4096 B apart
__device__ __forceinline__ void issue_gate(int wp, uint32_t a_addr, uint32_t b0, uint32_t d, uint32_t idesc, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr);
    const uint64_t bd0 = tc::smem_desc_sw128(b0), bd1 = tc::smem_desc_sw128(b0 + 4096u), bd2 = tc::smem_desc_sw128(b0 + 8192u);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        if (wp == 0) {
            tc::mma_bf16(d, ad + ks * 2, bd2 + ks * 2, idesc, (first && ks == 0) ? 0u : 1u);
            tc::mma_bf16(d, ad + ks * 2, bd1 + ks * 2, idesc, 1u);
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        } else if (wp == 1) {
            tc::mma_bf16(d, ad + ks * 2, bd1 + ks * 2, idesc, 1u);
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        } else {
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        }
    }
}

// ---------------------------------------------------------------- FP16 two-way split (CVAD_MATH_TC16, fused kernel only)
// x = x0 + x1 with x0 = fp16(s x), x1 = fp16(s x - x0): 22 significant bits once the operand is scaled by a power
// of two s that brings its largest element to [2^14, 2^15) -- per STREAM for activations (so that a stream's
// result does not depend on its neighbours in the batch), per layer for weights (host, pack_v5_tc16).  Three
// products per MAC (w0.x0 + w0.x1 + w1.x0; the dropped w1.x1 is 2^-22 relative) instead of the BF16 split's six:
// same FP32-level accuracy (tools/tc_split_sim.py: fp16x3 1e-6 vs bf16x6 5e-7 vs plain FP32 1.3e-6 on the
// probability), half the tensor-pipe and shared-memory-port time.  Elements far below the row maximum fall into
// FP16's subnormal range and keep an ABSOLUTE error of 2^-25 of the scaled unit, i.e. 2^-39 of the maximum.
struct Scale { float s, inv; };
// scale for an operand whose largest magnitude has the float bit pattern `max_bits` (non-negative): the power of two that
// brings it to [2^14, 2^15), capped at 2^125.  An all-zero (or subnormal) operand gets the cap: zeros stay zeros and the
// products are unscaled by 2^-125 again -- no special case (these few integer operations run ~90 times per thread and
// tile; with a branch for E == 0 and one load per value they were 9 % of the kernel's stall samples).
__device__ __forceinline__ Scale scale_from_max(uint32_t max_bits) {
    const uint32_t se = min(268u - (max_bits >> 23), 252u);    // 2^(14 - (E - 127)), biased
    Scale r;
    r.s = __uint_as_float(se << 23);
    r.inv = __uint_as_float((254u - se) << 23);
    return r;
}
// the same for eight consecutive streams (a 32-byte aligned stretch of the per-stream maxima): two 16-byte loads
__device__ __forceinline__ void amax_load8(const uint32_t *a, uint32_t (&m)[8]) {
    const uint4 lo = *reinterpret_cast<const uint4 *>(a), hi = *reinterpret_cast<const uint4 *>(a + 4);
    m[0] = lo.x; m[1] = lo.y; m[2] = lo.z; m[3] = lo.w; m[4] = hi.x; m[5] = hi.y; m[6] = hi.z; m[7] = hi.w;
}
__device__ __forceinline__ void scales8(const uint32_t *a, float (&s8)[8]) {
    uint32_t m[8];
    amax_load8(a, m);
#pragma unroll
    for (int e = 0; e < 8; ++e) s8[e] = scale_from_max(m[e]).s;
}
__device__ __forceinline__ void inv_scales8(const uint32_t *a, float mul, float (&i8)[8]) {
    uint32_t m[8];
    amax_load8(a, m);
#pragma unroll
    for (int e = 0; e < 8; ++e) i8[e] = scale_from_max(m[e]).inv * mul;
}
constexpr float kHScale = 16384.f, kHInv = 1.f / 16384.f;     // |h| < 1: static scale of the recurrent operand
// two values at once: word j holds part j of a (low half) and of b (high half)
__device__ __forceinline__ void split2x2_h(float a, float b, uint32_t &w0, uint32_t &w1) {
    const __half2 h0 = __floats2half2_rn(a, b);
    const float2 f0 = __half22float2(h0);
    const __half2 h1 = __floats2half2_rn(a - f0.x, b - f0.y);
    w0 = *reinterpret_cast<const uint32_t *>(&h0);
    w1 = *reinterpret_cast<const uint32_t *>(&h1);
}
// store the two parts of (already scaled) values a (row) and b (row + 1) at column k of a B operand with R rows
__device__ __forceinline__ void store_parts2_h(unsigned char *base, uint32_t ps, uint32_t row, uint32_t k, uint32_t R, float a, float b) {
    uint32_t w0, w1;
    split2x2_h(a, b, w0, w1);
    unsigned char *da = base + tc::sw128_offset(row, k, R);
    unsigned char *db = base + tc::sw128_offset(row + 1, k, R);
    *reinterpret_cast<unsigned short *>(da) = (unsigned short)w0;
    *reinterpret_cast<unsigned short *>(da + ps) = (unsigned short)w1;
    *reinterpret_cast<unsigned short *>(db) = (unsigned short)(w0 >> 16);
    *reinterpret_cast<unsigned short *>(db + ps) = (unsigned short)(w1 >> 16);
}
// ---- B operands MN-major SWIZZLE_64B (fused FP16 build, every operand an epilogue writes: MAG, E0, E1, E2, X, H)
// An epilogue thread owns ONE channel (its TMEM lane = the next layer's k) and EIGHT consecutive streams: with N as the
// contiguous dimension those are one 16-byte chunk per part and time column -- 2 STS.128 where the K-major layout took
// 16 two-byte stores with their address arithmetic (the store pass of the STFT epilogue: 2.0 k cycles of a 59 k tile).
// N atom g (32 streams) = time column or part, 512 B apart; K groups `sbo` apart (tc::mn64_offset).  A quarter warp
// (8 lanes = one K group, same chunk column) touches 8 distinct 16-byte bank groups: conflict-free.
__device__ __forceinline__ void store_row8_mn(unsigned char *dst, uint32_t ps, const float (&v)[8]) {
    uint32_t w0[4], w1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split2x2_h(v[2 * j], v[2 * j + 1], w0[j], w1[j]);
    *reinterpret_cast<uint4 *>(dst) = make_uint4(w0[0], w0[1], w0[2], w0[3]);
    *reinterpret_cast<uint4 *>(dst + ps) = make_uint4(w1[0], w1[1], w1[2], w1[3]);
}
// MMAs of one weight tile (part wp) for one 64-element K block against an MN-major operand: K step = two K groups
__device__ __forceinline__ void issue_split_mn(int wp, uint32_t a_addr, uint32_t b0, uint32_t ps, uint32_t sbo, uint32_t d_main,
                                               uint32_t d_corr, uint32_t idesc, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr);
    const uint64_t bd0 = tc::smem_desc_mn64(b0, 512u, sbo), bd1 = tc::smem_desc_mn64(b0 + ps, 512u, sbo);
    const uint64_t kst = (uint64_t)((2u * sbo) >> 4);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        const uint32_t fresh = (first && ks == 0) ? 0u : 1u;
        if (wp == 0) {
            tc::mma_bf16(d_corr, ad + ks * 2, bd1 + ks * kst, idesc, fresh);
            tc::mma_bf16(d_main, ad + ks * 2, bd0 + ks * kst, idesc, fresh);
        } else {
            tc::mma_bf16(d_corr, ad + ks * 2, bd0 + ks * kst, idesc, 1u);
        }
    }
}
// W_hh . h: the two parts are N atoms 0 and 1 of the H operand (K groups 1,024 B apart), all products to one accumulator
__device__ __forceinline__ void issue_gate_mn(int wp, uint32_t a_addr, uint32_t b0, uint32_t d, uint32_t idesc, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr);
    const uint64_t bd0 = tc::smem_desc_mn64(b0, 512u, 1024u), bd1 = tc::smem_desc_mn64(b0 + 512u, 512u, 1024u);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        if (wp == 0) {
            tc::mma_bf16(d, ad + ks * 2, bd1 + ks * 128, idesc, (first && ks == 0) ? 0u : 1u);
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 128, idesc, 1u);
        } else {
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 128, idesc, 1u);
        }
    }
}
// W_ih . x with [x0 | x1] = N atoms 0 and 1 (issue_gate_h_cat's products)
__device__ __forceinline__ void issue_gate_cat_mn(int wp, uint32_t a_addr, uint32_t b0, uint32_t d, uint32_t idesc64,
                                                  uint32_t idesc32, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr), bd = tc::smem_desc_mn64(b0, 512u, 1024u);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        if (wp == 0) tc::mma_bf16(d, ad + ks * 2, bd + ks * 128, idesc64, (first && ks == 0) ? 0u : 1u);
        else tc::mma_bf16(d + 32u, ad + ks * 2, bd + ks * 128, idesc32, 1u);
    }
}

// N (<= 8) per-stream maxima at once, values one per lane, streams slot[0], slot[stride], ...: the N warp reductions are
// independent and pipeline, then lanes 0..N-1 issue ONE shared atomic each.  (Eight dependent redux -> branch -> atomic
// round trips cost an epilogue ~730 cycles per layer; tools/tc_phase_profile.py marks 17 / 18.)
template <int N>
__device__ __forceinline__ void amax_push_n(uint32_t *slot, int stride, const float (&v)[N], int lane) {
    uint32_t m[N];
#pragma unroll
    for (int e = 0; e < N; ++e) m[e] = __reduce_max_sync(0xffffffffu, __float_as_uint(v[e]) & 0x7fffffffu);   // (a ReLU may hand over -0.0)
    uint32_t mine = m[0];
#pragma unroll
    for (int e = 1; e < N; ++e) mine = lane == e ? m[e] : mine;
    if (lane < N && mine != 0u) atomicMax(slot + lane * stride, mine);
}
// instruction descriptor, kind::f16: D = F32, A = B = FP16
__host__ __device__ constexpr uint32_t idesc_f16_f32(uint32_t M, uint32_t N) {
    return (1u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// front-end weight stream of the FP16 build: the BF16 stream's order with two parts per tile group (46 tiles)
constexpr int kFeSlotsPerTileH = 46;
constexpr size_t kFeStreamBytesH = 28 * 16384 + 16 * 8192 + 2 * 16384;
__host__ __device__ __forceinline__ void fe_slot_h(int s, uint32_t &off, uint32_t &bytes) {
    if (s < 28) { off = (uint32_t)s * 16384u; bytes = 16384u; }
    else if (s < 44) { off = 28u * 16384u + (uint32_t)(s - 28) * 8192u; bytes = 8192u; }
    else { off = 28u * 16384u + 16u * 8192u + (uint32_t)(s - 44) * 16384u; bytes = 16384u; }
}
constexpr size_t kRecStreamBytesH = (size_t)32 * 16384;       // gate x kb 0..3 x part 0..1
constexpr int kFusedSlotsPerTileH = 16 + kFeSlotsPerTileH + 16;
constexpr uint32_t kColIh = 0;                                // TMEM columns of the W_ih . x accumulators (64 per gate; free after encoder.3)
// MMAs of one weight tile (part wp) for one 64-element K block, FP16 split: w0.x0 -> d_main, w0.x1 and w1.x0 -> d_corr
__device__ __forceinline__ void issue_split_h(int wp, uint32_t a_addr, uint32_t b0, uint32_t ps, uint32_t d_main,
                                              uint32_t d_corr, uint32_t idesc, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr);
    const uint64_t bd0 = tc::smem_desc_sw128(b0), bd1 = tc::smem_desc_sw128(b0 + ps);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        const uint32_t fresh = (first && ks == 0) ? 0u : 1u;
        if (wp == 0) {
            tc::mma_bf16(d_corr, ad + ks * 2, bd1 + ks * 2, idesc, fresh);
            tc::mma_bf16(d_main, ad + ks * 2, bd0 + ks * 2, idesc, fresh);
        } else {
            tc::mma_bf16(d_corr, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        }
    }
}
// LSTM gate products, FP16 split: all three products of a MAC go to one accumulator; parts 4096 B apart
__device__ __forceinline__ void issue_gate_h(int wp, uint32_t a_addr, uint32_t b0, uint32_t d, uint32_t idesc, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr);
    const uint64_t bd0 = tc::smem_desc_sw128(b0), bd1 = tc::smem_desc_sw128(b0 + 4096u);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        if (wp == 0) {
            tc::mma_bf16(d, ad + ks * 2, bd1 + ks * 2, idesc, (first && ks == 0) ? 0u : 1u);
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        } else {
            tc::mma_bf16(d, ad + ks * 2, bd0 + ks * 2, idesc, 1u);
        }
    }
}

// W_ih . x of the fused FP16 kernel with the two activation parts concatenated along N (rows 0..63 of the operand are
// [x0 | x1]): part 0 of a weight tile in ONE N = 64 MMA (columns [d, d+32) collect w0.x0, [d+32, d+64) w0.x1), part 1
// against x0 alone into [d+32, d+64): two MMAs per K step instead of three
__device__ __forceinline__ void issue_gate_h_cat(int wp, uint32_t a_addr, uint32_t b0, uint32_t d, uint32_t idesc64,
                                                 uint32_t idesc32, bool first) {
    const uint64_t ad = tc::smem_desc_sw128(a_addr), bd = tc::smem_desc_sw128(b0);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        if (wp == 0) tc::mma_bf16(d, ad + ks * 2, bd + ks * 2, idesc64, (first && ks == 0) ? 0u : 1u);
        else tc::mma_bf16(d + 32u, ad + ks * 2, bd + ks * 2, idesc32, 1u);
    }
}

struct Ring {
    uint32_t buf;        // shared address of slot 0
    uint64_t *full;      // [n]
    uint64_t *empty;     // [n]
};

// =====================================================================================
// Front end: frame loader -> STFT -> magnitude -> encoder.0..3 -> feat (BF16x3 operand for the recurrent kernel)
// =====================================================================================
// FUSED (max_frames == 1): the same CTA also runs the LSTM step, decoder and state machine of its 32 streams
// (the W_hh.h products are issued while the frame loader runs, the W_ih.x products after encoder.3).
// H16 (CVAD_MATH_TC16, FUSED only): FP16 two-way operand split with per-stream dynamic scaling, three products per MAC.
template <bool DBG, bool FUSED, bool H16 = false, bool PROF = true>
__global__ void __launch_bounds__(kThreadsTC, 1) v5tc_frontend_kernel(const V5Step p) {
    static_assert(!H16 || !DBG, "the debug dump runs the BF16-split build");
    // the FP16 build's activation region holds two parts instead of three: the 32 KB go to two more ring slots (the weight
    // supply of a phase is bound by the L2 -> shared latency of the tiles in flight, not by bandwidth)
    constexpr uint32_t ACT = H16 ? kActBytesH : kActBytes;
    constexpr int RING = (FUSED ? kFusedRing : kFeRing) + (H16 ? 2 : 0);
    constexpr int NP = H16 ? 2 : 3;                   // operand parts
    // fused FP16 build: every B operand an epilogue writes is MN-major SWIZZLE_64B (store_row8_mn); the frame loader's
    // AUD operand (a thread holds 8 consecutive samples = k) stays K-major
    constexpr bool BMN = FUSED && H16;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
    unsigned char *act = base;
    unsigned char *hbuf = act + ACT;                                         // FUSED: [2 K blocks][96 rows][128 B]
    unsigned char *ring_buf = hbuf + (FUSED ? 24576 : 0);
    float *nyq = reinterpret_cast<float *>(ring_buf + RING * kSlotBytes);    // [96] |X[128]| per (t, item)
    float *dpart = nyq + 96;                                                 // FUSED: [4][32] decoder partial sums
    uint64_t *bars = reinterpret_cast<uint64_t *>(dpart + (FUSED ? 128 : 0));
    uint64_t *full = bars, *empty = bars + RING, *act_ready = bars + 2 * RING, *acc_ready = act_ready + 1,
             *h_ready = acc_ready + 1, *gate_ready = h_ready + 1;          // FUSED: gate_ready[4], one per LSTM gate
    // (an odd number of barriers is padded by one: the words behind them -- the per-stream maxima above all -- are read
    // with 16-byte loads)
    constexpr int kBars = 2 * RING + 3 + (FUSED ? 4 : 0);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + kBars + (kBars & 1));
    int *s_slot = reinterpret_cast<int *>(tmem_slot + 4);
    int *s_valid = s_slot + kTile;
    double *s_thr = reinterpret_cast<double *>(s_valid + kTile);             // FUSED: start_p[32], end_p[32]
    uint32_t *amax = reinterpret_cast<uint32_t *>(s_thr + 2 * kTile);        // H16: [6][32] per-stream maxima (bit patterns) of AUD, MAG, E0, E1, E2, X
    int *s_dn = FUSED ? reinterpret_cast<int *>(amax + 6 * kTile) : s_valid + kTile;   // [32] per-stream denoise flag (fetched with the slot ids)
    long long *s_f0 = reinterpret_cast<long long *>(s_dn + kTile);           // FUSED: [32] frames_done
    int *s_sm = reinterpret_cast<int *>(s_f0 + kTile);                       // FUSED: [5][32] is_voice_active, start / end counters, N_s, N_e
    int *s_grp = s_sm + 5 * kTile;                                           // FUSED: [4] first slot of stream group g when its 8 slots are consecutive from a multiple of 8, else -1

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    CVAD_PROF_NS(120);
    CVAD_CHAIN_NS(0);

    if (tid == 0) {
        for (int i = 0; i < RING; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(act_ready, 1);
        mbar_init(acc_ready, 1);
        mbar_init(h_ready, 1);
        if (FUSED)
            for (int i = 0; i < 4; ++i) mbar_init(&gate_ready[i], 1);
        mbar_fence_init();
    }
    if (warp == kProducerWarp) tc::tmem_alloc(tmem_slot, 512);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (*tmem_slot != 0u) __trap();   // sole CTA on the SM and all 512 columns: TMEM base is lane 0 / column 0
    CVAD_PROF_NS(121);
    CVAD_CHAIN_NS(1);
    // programmatic dependent launch: the recurrent kernel may be scheduled now; it runs its own prologue (state
    // load, weight prefetch) and blocks in griddepcontrol.wait until this grid has completed
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const int n_tiles = p.max_frames * p.n_stiles;
    const uint32_t act_s = smem_u32(act), ring_s = smem_u32(ring_buf), h_s = smem_u32(hbuf);

    if (warp == kProducerWarp) {
        // ------------------------------------------------------------ weight producer
        constexpr int S_TILE = H16 ? (FUSED ? kFusedSlotsPerTileH : kFeSlotsPerTileH) : FUSED ? kFusedSlotsPerTile : kFeSlotsPerTile;
        // weight tile s of a tile's stream -> ring slot g % RING
        auto feed = [&](const int s, const uint32_t g) {
            const uint32_t slot = g % RING;
            mbar_wait(&empty[slot], ((g / RING) & 1u) ^ 1u);
            uint32_t off, bytes;
            const unsigned char *src;
            if (H16 && !FUSED) {
                fe_slot_h(s, off, bytes);
                mbar_arrive_expect_tx(&full[slot], bytes);
                bulk_g2s(ring_buf + slot * kSlotBytes, p.w_fe_h + off, bytes, &full[slot]);
                return;
            }
            if (H16) {
                // same order with two parts: hh gate g = 4 tiles | STFT 16 | enc0 12 | enc1 12 | enc2 + enc3 6 | W_ih 16
                int fe_idx = s, gate = -1, kb = 0, part = 0;
                if (s < 4) { gate = 0; kb = 2 + s / 2; part = s % 2; }
                else if (s < 20) fe_idx = s - 4;
                else if (s < 24) { gate = 1; kb = 2 + (s - 20) / 2; part = (s - 20) % 2; }
                else if (s < 36) fe_idx = s - 24 + 16;
                else if (s < 40) { gate = 2; kb = 2 + (s - 36) / 2; part = (s - 36) % 2; }
                else if (s < 52) fe_idx = s - 40 + 28;
                else if (s < 56) { gate = 3; kb = 2 + (s - 52) / 2; part = (s - 52) % 2; }
                else if (s < 62) fe_idx = s - 56 + 40;
                else { const int r = s - 62; gate = r / 4; kb = (r / 2) % 2; part = r % 2; }
                if (gate >= 0) {
                    src = p.w_rec_h + (size_t)((gate * 4 + kb) * 2 + part) * kSlotBytes;
                    bytes = kSlotBytes;
                } else {
                    fe_slot_h(fe_idx, off, bytes);
                    src = p.w_fe_h + off;
                }
                mbar_arrive_expect_tx(&full[slot], bytes);
                bulk_g2s(ring_buf + slot * kSlotBytes, src, bytes, &full[slot]);
                return;
            }
            // FUSED order: hh gate 0 | STFT (24) | hh gate 1 | enc0 (18) | hh gate 2 | enc1 (18) | hh gate 3 |
            //              enc2 + enc3 (9) | W_ih of the four gates (24).  hh gate g = 6 tiles (K blocks 2,3 x part)
            int fe_idx = s, gate = -1, kb = 0, part = 0;
            if (FUSED) {
                if (s < 6) { gate = 0; kb = 2 + s / 3; part = s % 3; }
                else if (s < 30) fe_idx = s - 6;
                else if (s < 36) { gate = 1; kb = 2 + (s - 30) / 3; part = (s - 30) % 3; }
                else if (s < 54) fe_idx = s - 36 + 24;
                else if (s < 60) { gate = 2; kb = 2 + (s - 54) / 3; part = (s - 54) % 3; }
                else if (s < 78) fe_idx = s - 60 + 42;
                else if (s < 84) { gate = 3; kb = 2 + (s - 78) / 3; part = (s - 78) % 3; }
                else if (s < 93) fe_idx = s - 84 + 60;
                else { const int r = s - 93; gate = r / 6; kb = (r / 3) % 2; part = r % 3; }
            }
            if (gate >= 0) {
                src = p.w_rec_tc + (size_t)((gate * 4 + kb) * 3 + part) * kSlotBytes;
                bytes = kSlotBytes;
            } else {
                fe_slot(fe_idx, off, bytes);
                src = p.w_fe_tc + off;
            }
            mbar_arrive_expect_tx(&full[slot], bytes);
            bulk_g2s(ring_buf + slot * kSlotBytes, src, bytes, &full[slot]);
        };
        uint32_t g = 0;
        int pre = 0;                                   // weight tiles of the NEXT live tile that are already in flight
        if (FUSED) {
            // chained one-frame steps (programmatic dependent launch): the first RING weight tiles do not depend on
            // the previous step's grid, so they are fetched while it is still finishing
            if (lane == 0)
                for (; pre < RING; ++pre, ++g) feed(pre, g);
            pre = __shfl_sync(0xffffffffu, pre, 0);
            griddep_wait();
        }
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int frame = tile / p.n_stiles, st = tile - frame * p.n_stiles;
            if (!tile_live(p, frame, st, lane, nullptr, nullptr)) continue;
            if (lane == 0)
                for (int s = pre; s < S_TILE; ++s, ++g) feed(s, g);
            pre = 0;
            __syncwarp();
        }
        // no live tile at all: the prefetched copies must land before the CTA may exit
        if (FUSED && pre && lane == 0)
            for (int s = 0; s < pre; ++s) mbar_wait(&full[s], 0u);
    } else if (warp == kMmaWarp) {
        // ------------------------------------------------------------ MMA issuer
        if (FUSED && p.step_ctr && blockIdx.x < kPrefetchCtas) {
            // Chained steps: ~20 CTAs of a 128-tile step are scheduled on idle SMs while the previous step still runs and
            // would only wait.  A CTA that finds the completed-steps counter behind its own sequence number is one of
            // them: it pulls the audio of every 16th tile into L2 (this warp has nothing to do until h_ready), so that
            // the step's loaders -- all 128 start at once -- read from L2 instead of sharing one HBM burst.  Hints only:
            // the addresses are the ones the loaders read, no data is consumed ahead of griddepcontrol.wait.
            const int done = *reinterpret_cast<volatile const int *>(p.step_ctr);
            if (done - p.step_seq < 0) {
                const size_t es = p.pcm == 0 ? 4 : 2;
                const int flen = p.frame_len < 512 ? p.frame_len : 512;
                const int lines = (int)((flen * es + 127) / 128);
                for (int t = blockIdx.x; t < p.n_stiles; t += kPrefetchCtas) {
                    const int rows = min(kTile, p.n_streams - t * kTile);
                    for (int l = lane; l < rows * lines; l += 32) {
                        const int s = l / lines, c = l - s * lines;
                        const unsigned char *a = reinterpret_cast<const unsigned char *>(p.audio) +
                                                 (size_t)((long long)(t * kTile + s) * p.stride) * es + (size_t)c * 128;
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
                    }
                }
            }
        }
        if (FUSED) griddep_wait();
        uint32_t g = 0, act_phase = 0, h_phase = 0;
        const uint32_t i128_96 = H16 ? idesc_f16_f32(128, 96) : tc::idesc_bf16_f32(128, 96),
                       i128_64 = H16 ? idesc_f16_f32(128, 64) : tc::idesc_bf16_f32(128, 64),
                       i128_32 = H16 ? idesc_f16_f32(128, 32) : tc::idesc_bf16_f32(128, 32),
                       i64_64 = H16 ? idesc_f16_f32(64, 64) : tc::idesc_bf16_f32(64, 64),
                       i64_32 = H16 ? idesc_f16_f32(64, 32) : tc::idesc_bf16_f32(64, 32);
        constexpr uint32_t MN = BMN ? tc::kIdescBMajorMN : 0u;     // operands written by an epilogue
        // one weight tile of part WP against the activation parts that pair with it (BF16: 3 / 2 / 1 products, FP16: 2 / 1)
#define CVAD_SPLIT(WP, B0, PS, DM, DC, IDESC, FIRST)                                   \
    do {                                                                               \
        if (H16) issue_split_h(WP, a_addr, B0, PS, DM, DC, IDESC, FIRST);              \
        else issue_split(WP, a_addr, B0, PS, DM, DC, IDESC, FIRST);                    \
    } while (0)
        // the same against an operand an epilogue wrote: MN-major in the fused FP16 build (K groups SBO apart; row offsets
        // of the K-major form are N-atom offsets, 512 B per 32 rows), else K-major at B0
#define CVAD_SPLIT_E(WP, B0, B0MN, PS, SBO, DM, DC, IDESC, FIRST)                      \
    do {                                                                               \
        if (BMN) issue_split_mn(WP, a_addr, B0MN, PS, SBO, DM, DC, (IDESC) | MN, FIRST); \
        else CVAD_SPLIT(WP, B0, PS, DM, DC, IDESC, FIRST);                             \
    } while (0)
#define CVAD_GATE(WP, B0, D, IDESC, FIRST)                                             \
    do {                                                                               \
        if (H16) issue_gate_h(WP, a_addr, B0, D, IDESC, FIRST);                        \
        else issue_gate(WP, a_addr, B0, D, IDESC, FIRST);                              \
    } while (0)
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int frame = tile / p.n_stiles, st = tile - frame * p.n_stiles;
            if (!tile_live(p, frame, st, lane, nullptr, nullptr)) continue;
            const bool first_tile = tile == (int)blockIdx.x && lane == 0;
#define CVAD_TC_SLOT(BODY)                                                   \
    {                                                                        \
        const uint32_t slot = g % RING;                                      \
        mbar_wait(&full[slot], (g / RING) & 1u);                             \
        tc::fence_after_sync();                                              \
        const uint32_t a_addr = ring_s + slot * kSlotBytes;                  \
        if (tc::elect_one()) {                                               \
            BODY;                                                            \
            tc::mma_commit(&empty[slot]);                                    \
        }                                                                    \
        __syncwarp();                                                        \
        ++g;                                                                 \
    }
            // FUSED: W_hh . h of gate G needs only the resident state; the four gates are issued where the tensor pipe
            // would otherwise idle: under the frame loader and under the epilogues of the STFT, encoder.0 and encoder.1
#define CVAD_TC_HH(G)                                                                                              \
    if (FUSED) {                                                                                                   \
        CVAD_ISSUE_ROLL                                                                                            \
        for (int kb = 0; kb < 2; ++kb)                                                                             \
            for (int wp = 0; wp < NP; ++wp)                                                                         \
            {                                                                                                  \
                if (BMN) CVAD_TC_SLOT(issue_gate_mn(wp, a_addr, h_s + kb * 8192u, kColGate + 32 * (G), i128_32 | MN, kb == 0 && wp == 0)) \
                else CVAD_TC_SLOT(CVAD_GATE(wp, h_s + kb * kXhKb, kColGate + 32 * (G), i128_32, kb == 0 && wp == 0)) \
            }                                                                                                  \
    }
            if (FUSED) {
                mbar_wait(h_ready, h_phase); h_phase ^= 1u;
                tc::fence_after_sync();
            }
            CVAD_TC_HH(0)
            CVAD_PROF(42);
            // ---- STFT: D[blk][bin][(t, item)] = sum_k W[bin][k] x[128 t + k]; K block kb uses segment rows t + kb/2
            mbar_wait(act_ready, act_phase); act_phase ^= 1u;
            CVAD_PROF(32);
            tc::fence_after_sync();
            CVAD_ISSUE_ROLL
            for (int blk = 0; blk < 2; ++blk)
                CVAD_ISSUE_ROLL
                for (int kb = 0; kb < 4; ++kb)
                    for (int wp = 0; wp < NP; ++wp)
                        CVAD_TC_SLOT(CVAD_SPLIT(wp, act_s + (kb & 1) * 16384u + (kb >> 1) * 4096u, kAudPart,
                                                 kColMain + blk * 96, kColCorr + blk * 96, i128_96, kb == 0 && wp == 0))
            if (tc::elect_one()) tc::mma_commit(acc_ready);
            CVAD_TC_HH(1)
            CVAD_PROF(33);
            __syncwarp();
            // ---- encoder.0 (k3 s1 p1): tap 1: out t <- in t (N 96); tap 0: out 1,2 <- in 0,1; tap 2: out 0,1 <- in 1,2
            mbar_wait(act_ready, act_phase); act_phase ^= 1u;
            CVAD_PROF(34);
            tc::fence_after_sync();
            CVAD_ISSUE_ROLL
            for (int kb = 0; kb < 2; ++kb) {
                CVAD_ISSUE_ROLL
                for (int tap = 0; tap < 3; ++tap) {       // centre (N 96), tap 0 (D columns 32..), tap 2 (rows 32..)
                    const uint32_t b0 = act_s + kb * kMagKb + (tap == 2 ? 32u * 128u : 0u), dsh = tap == 1 ? 32u : 0u;
                    const uint32_t b0mn = act_s + kb * kMagKb + (tap == 2 ? 512u : 0u);
                    const uint32_t idesc = tap == 0 ? i128_96 : i128_64;
                    for (int wp = 0; wp < NP; ++wp)
                        CVAD_TC_SLOT(CVAD_SPLIT_E(wp, b0, b0mn, kMagPart, 1536u, kColMain + dsh, kColCorr + dsh, idesc,
                                                   kb == 0 && tap == 0 && wp == 0))
                }
            }
            if (tc::elect_one()) tc::mma_commit(acc_ready);
            CVAD_TC_HH(2)
            CVAD_PROF(35);
            __syncwarp();
            // ---- encoder.1 (k3 s2 p1, 64 out): E0 row blocks are stored in time order {0, 2, 1}
            //      tap 1: out 0,1 <- in 0,2 (rows 0..63); tap 2: out 0 <- in 1 (rows 64..95); tap 0: out 1 <- in 1
            mbar_wait(act_ready, act_phase); act_phase ^= 1u;
            CVAD_PROF(36);
            tc::fence_after_sync();
            CVAD_ISSUE_ROLL
            for (int kb = 0; kb < 2; ++kb) {
                CVAD_ISSUE_ROLL
                for (int tap = 0; tap < 3; ++tap) {       // tap 1 (rows 0..63, N 64), tap 2 (rows 64.., out 0), tap 0 (rows 64.., out 1)
                    const uint32_t b0 = act_s + kb * kMagKb + (tap == 0 ? 0u : 64u * 128u), dsh = tap == 2 ? 32u : 0u;
                    const uint32_t b0mn = act_s + kb * kMagKb + (tap == 0 ? 0u : 1024u);
                    const uint32_t idesc = tap == 0 ? i64_64 : i64_32;
                    for (int wp = 0; wp < NP; ++wp)
                        CVAD_TC_SLOT(CVAD_SPLIT_E(wp, b0, b0mn, kMagPart, 1536u, kColMain + dsh, kColCorr + dsh, idesc,
                                                   kb == 0 && tap == 0 && wp == 0))
                }
            }
            if (tc::elect_one()) tc::mma_commit(acc_ready);
            CVAD_TC_HH(3)
            CVAD_PROF(37);
            __syncwarp();
            // ---- encoder.2 (k3 s2 p1, 64 out, T 2 -> 1): tap 1 <- in 0 (rows 0..31), tap 2 <- in 1 (rows 32..63)
            mbar_wait(act_ready, act_phase); act_phase ^= 1u;
            CVAD_PROF(38);
            tc::fence_after_sync();
            for (int wp = 0; wp < NP; ++wp)
                CVAD_TC_SLOT(CVAD_SPLIT_E(wp, act_s, act_s, kE1Part, 1024u, kColMain, kColCorr, i64_32, wp == 0))
            for (int wp = 0; wp < NP; ++wp)
                CVAD_TC_SLOT(CVAD_SPLIT_E(wp, act_s + 32 * 128, act_s + 512u, kE1Part, 1024u, kColMain, kColCorr, i64_32, false))
            if (tc::elect_one()) tc::mma_commit(acc_ready);
            CVAD_PROF(39);
            __syncwarp();
            // ---- encoder.3 (centre tap, 128 out)
            mbar_wait(act_ready, act_phase); act_phase ^= 1u;
            CVAD_PROF(40);
            tc::fence_after_sync();
            for (int wp = 0; wp < NP; ++wp)
                CVAD_TC_SLOT(CVAD_SPLIT_E(wp, act_s, act_s, kE2Part, 512u, kColMain, kColCorr, i128_32, wp == 0))
            if (tc::elect_one()) tc::mma_commit(acc_ready);
            CVAD_PROF(41);
            __syncwarp();
            if (FUSED) {
                // ---- W_ih . x: x = encoder.3 output, written into ACT as a 96-row operand by the epilogue
                mbar_wait(act_ready, act_phase); act_phase ^= 1u;
                tc::fence_after_sync();
                CVAD_PROF(43);
                CVAD_ISSUE_ROLL
                for (int gate = 0; gate < 4; ++gate) {
                    CVAD_ISSUE_ROLL
                    for (int kb = 0; kb < 2; ++kb)
                        for (int wp = 0; wp < NP; ++wp)
                        {
                            if (BMN) CVAD_TC_SLOT(issue_gate_cat_mn(wp, a_addr, act_s + kb * 8192u, kColIh + 64 * gate, i128_64 | MN, i128_32 | MN,
                                                                    kb == 0 && wp == 0))
                            else if (H16) CVAD_TC_SLOT(issue_gate_h_cat(wp, a_addr, act_s + kb * kXhKb, kColIh + 64 * gate, i128_64, i128_32,
                                                                   kb == 0 && wp == 0))
                            else CVAD_TC_SLOT(CVAD_GATE(wp, act_s + kb * kXhKb, kColGate + 32 * gate, i128_32, false))
                        }
                    // the cell consumes the gates one by one (i, f, g, o), each under the next gate's products: every gate
                    // has its own barrier (one phase per tile), so a commit can never run two phases ahead of its reader
                    if (BMN && tc::elect_one()) tc::mma_commit(&gate_ready[gate]);
                }
                if (!BMN && tc::elect_one()) tc::mma_commit(acc_ready);
                CVAD_PROF(44);
                __syncwarp();
            }
#undef CVAD_TC_HH
#undef CVAD_TC_SLOT
#undef CVAD_SPLIT
#undef CVAD_SPLIT_E
#undef CVAD_GATE
        }
    } else {
        // ------------------------------------------------------------ loader + epilogue warps
        const int q = warp & 3, cg = warp >> 2;          // TMEM lane quadrant, column group 0..3
        const uint32_t lane_addr = (uint32_t)(32 * q) << 16;
        uint32_t acc_phase = 0, gate_phase = 0;
        const int flen = p.frame_len < 512 ? p.frame_len : 512;
        // (Measured and dropped: a rehearsal trip of the tile's first code -- tile_live, the slot data of warp 0 -- ahead of
        // griddepcontrol.wait, to take its instruction and parameter-bank misses off the 1.1 us between the resolved
        // dependency and the tile's start: the CTAs that matter are scheduled only 0.9 us before the dependency resolves
        // and the rehearsal itself took longer than that; tools/dev/chain_timeline.py.)
        // Streams in slot order with no per-stream frame counts (the device-pointer steps of a service that owns its slots):
        // which of the tile's streams are live, their slots and the per-stream maxima's reset need nothing but kernel
        // parameters -- the first tile's are set up AHEAD of griddepcontrol.wait (0.7 us of cold code and parameter-bank
        // reads that sat between the resolved dependency and the tile's first barrier, tools/dev/chain_timeline.py).
        const bool ident = FUSED && p.slots == nullptr && p.n_frames == nullptr;
        int pre_slot = -1, pre_valid = 0;
        bool pre_live = false;
        auto stream_groups = [&](int slot, int valid) {
            // stream group g = streams 8g .. 8g+7 (one epilogue thread's share): are its slots one aligned row of the state?
            const int base = __shfl_sync(0xffffffffu, slot, lane & ~7);
            const unsigned okm = __ballot_sync(0xffffffffu, valid && (base & 7) == 0 && slot == base + (lane & 7));
            const int gbase = __shfl_sync(0xffffffffu, base, (lane & 3) * 8);
            if (lane < 4) s_grp[lane] = ((okm >> (8 * lane)) & 0xffu) == 0xffu ? gbase : -1;
        };
        if (ident && (int)blockIdx.x < n_tiles) {
            const int frame = (int)blockIdx.x / p.n_stiles, st = (int)blockIdx.x - frame * p.n_stiles;
            pre_live = tile_live(p, frame, st, lane, &pre_slot, &pre_valid);
            if (warp == 0) {
                s_slot[lane] = pre_slot;
                s_valid[lane] = pre_valid;
                stream_groups(pre_slot, pre_valid);
            }
            if (H16 && warp >= 1 && warp <= 6) amax[(warp - 1) * kTile + lane] = 0u;
        }
        if (FUSED) {
            griddep_wait();
            CVAD_CHAIN_NS(2);
        }
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int frame = tile / p.n_stiles, st = tile - frame * p.n_stiles;
            const bool pre = ident && tile == (int)blockIdx.x;          // set up above
            int my_slot = pre_slot, my_valid = pre_valid;
            const bool live = pre ? pre_live : tile_live(p, frame, st, lane, &my_slot, &my_valid);
            CVAD_CHAIN_NS(6);
            // chained steps arrive without a memset in front of them: the tile clears its streams' status words itself
            // (one tile per stream when max_frames == 1), ordered before the loader's atomicOr by the barrier below
            if (FUSED && p.status_zero && warp == 0 && st * kTile + lane < p.n_streams) p.status[st * kTile + lane] = 0u;
            if (!live) continue;
            // thresholds, denoise flag and state-machine words of the tile's streams are fetched in one batch with the slot
            // data (their latency would otherwise sit at the very end of the tile).  FUSED: the loads are only ISSUED
            // ahead of the barrier -- the values reach shared memory once the audio and state loads are in flight as well,
            // so that no warp waits for this round trip before it starts its own (first readers: the loader's second
            // half, two barriers further down)
            double sp = 0.0, ep = 0.0;
            int a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0, dn = 0;
            long long f0 = 0;
            if (warp == 0) {
                if (!pre) {
                    s_slot[lane] = my_slot;
                    s_valid[lane] = my_valid;
                    if (FUSED) stream_groups(my_slot, my_valid);
                }
                if (my_slot >= 0) dn = (int)p.denoise[my_slot];
                if (!FUSED) s_dn[lane] = dn;
                if (FUSED && my_slot >= 0) {
                    sp = p.start_p[my_slot]; ep = p.end_p[my_slot];
                    a0 = p.sm_active[my_slot]; a1 = p.sm_scount[my_slot]; a2 = p.sm_ecount[my_slot];
                    a3 = p.n_start[my_slot]; a4 = p.n_end[my_slot];
                    f0 = p.frames_done[my_slot];
                }
            }
            if (H16 && !pre && warp >= 1 && warp <= 6) amax[(warp - 1) * kTile + lane] = 0u;
            CVAD_CHAIN_NS(7);
            epi_bar();
            const bool dbg = DBG && tile == 0;
            const bool first_tile = tile == (int)blockIdx.x && tid == 0;
            CVAD_PROF(0);
            CVAD_PROF_NS(126);
            CVAD_CHAIN_NS(3);
            // ---- frame loader (audio.py:164-190 split, :104-121 gate, silero_model.py:449-474 pad/truncate):
            //      8 samples per work unit -> 3 x 16-byte BF16 chunks of the AUD operand, row = segment*32 + item.
            //      All global loads of the thread's 4 units are issued before the first use -- and, in the fused
            //      kernel, before the resident state is fetched, so that both latencies overlap.
            float creg[8], hreg[8];
            const int u_own = 32 * q + lane, i_own = 8 * cg;   // this thread's hidden unit (TMEM lane) and 8 streams
                // vector loads whenever a frame is a whole number of 8-sample units (512, or the websocket service's 480:
                // units past the frame's end are the zero padding of _prepare_audio_input, silero_model.py:449-474)
                const bool fast = p.vec_ok && (flen & 7) == 0;
                float v[4][8];
                bool ok[4];
#pragma unroll
                for (int u4 = 0; u4 < 4; ++u4) {
                    const int unit = u4 * kEpiThreads + tid;
                    const int s = unit >> 6, c8 = unit & 63;
                    ok[u4] = s_valid[s] != 0;
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[u4][e] = 0.f;
                    if (ok[u4]) {
                        const long long b0 = (long long)(st * kTile + s) * p.stride + (long long)frame * p.hop + 8 * c8;
                        if (fast && 8 * c8 >= flen) {
                            // zero padding
                        } else if (fast && p.pcm == 0) {
                            const float4 *src = reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(p.audio) + b0);
                            const float4 t0 = ldg_stream4(src), t1 = ldg_stream4(src + 1);
                            v[u4][0] = t0.x; v[u4][1] = t0.y; v[u4][2] = t0.z; v[u4][3] = t0.w;
                            v[u4][4] = t1.x; v[u4][5] = t1.y; v[u4][6] = t1.z; v[u4][7] = t1.w;
                        } else if (fast) {
                            const short4 *src = reinterpret_cast<const short4 *>(reinterpret_cast<const short *>(p.audio) + b0);
                            const short4 t0 = __ldg(src), t1 = __ldg(src + 1);
                            v[u4][0] = (float)t0.x; v[u4][1] = (float)t0.y; v[u4][2] = (float)t0.z; v[u4][3] = (float)t0.w;
                            v[u4][4] = (float)t1.x; v[u4][5] = (float)t1.y; v[u4][6] = (float)t1.z; v[u4][7] = (float)t1.w;
                        } else {
#pragma unroll
                            for (int e = 0; e < 8; ++e)
                                if (8 * c8 + e < flen)
                                    v[u4][e] = p.pcm == 0 ? __ldg(reinterpret_cast<const float *>(p.audio) + b0 + e)
                                                          : (float)__ldg(reinterpret_cast<const short *>(p.audio) + b0 + e);
                        }
                    }
                }
            // FUSED: resident state of the tile's streams: h -> rows of the H operand, c -> registers.  The state is laid out
            // [slot / 8][unit][slot % 8] (state_at): the 8 streams of this thread are one 32-byte row when their slots are
            // consecutive from a multiple of 8 (s_grp), read with two 16-byte loads straight into the registers that own
            // them -- a warp's 32 units are 1 KB contiguous; any other slot list is gathered element by element.
            if (FUSED) {
                const int gb = s_grp[cg];
                if (gb >= 0) {
                    const float4 *ph = reinterpret_cast<const float4 *>(p.h_state + state_at(u_own, gb));
                    const float4 *pc = reinterpret_cast<const float4 *>(p.c_state + state_at(u_own, gb));
                    const float4 h0 = __ldg(ph), h1 = __ldg(ph + 1), c0 = __ldg(pc), c1 = __ldg(pc + 1);
                    hreg[0] = h0.x; hreg[1] = h0.y; hreg[2] = h0.z; hreg[3] = h0.w;
                    hreg[4] = h1.x; hreg[5] = h1.y; hreg[6] = h1.z; hreg[7] = h1.w;
                    creg[0] = c0.x; creg[1] = c0.y; creg[2] = c0.z; creg[3] = c0.w;
                    creg[4] = c1.x; creg[5] = c1.y; creg[6] = c1.z; creg[7] = c1.w;
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int slot = s_valid[i_own + e] ? s_slot[i_own + e] : -1;
                        hreg[e] = slot >= 0 ? __ldg(p.h_state + state_at(u_own, slot)) : 0.f;
                        creg[e] = slot >= 0 ? __ldg(p.c_state + state_at(u_own, slot)) : 0.f;
                    }
                }
                if (warp == 0) {
                    // the slot data fetched at tile start (by now every global load of this warp is in flight)
                    s_dn[lane] = dn;
                    if (my_slot >= 0) {
                        s_thr[lane] = sp; s_thr[kTile + lane] = ep;
                        s_sm[lane] = a0; s_sm[kTile + lane] = a1; s_sm[2 * kTile + lane] = a2;
                        s_sm[3 * kTile + lane] = a3; s_sm[4 * kTile + lane] = a4;
                        s_f0[lane] = f0;
                    }
                }
                if constexpr (BMN) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) hreg[e] *= kHScale;
                    store_row8_mn(hbuf + tc::mn64_offset((uint32_t)i_own, (uint32_t)u_own, 512u, 1024u), 512u, hreg);
                } else {
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        if (H16) store_parts2_h(hbuf, 32 * 128, (uint32_t)(i_own + e), (uint32_t)u_own, 96u, hreg[e] * kHScale, hreg[e + 1] * kHScale);
                        else store_parts2(hbuf, 32 * 128, (uint32_t)(i_own + e), (uint32_t)u_own, 96u, hreg[e], hreg[e + 1]);
                    }
                }
                tc::fence_async_smem();
                epi_bar();
                if (tid == 0) mbar_arrive(h_ready);
                CVAD_PROF(12);
            }

            // ---- frame loader, second half: convert, gate, split, store
            {
#pragma unroll
                for (int u4 = 0; u4 < 4; ++u4) {
                    const int unit = u4 * kEpiThreads + tid;
                    const int s = unit >> 6, c8 = unit & 63;
                    if (ok[u4]) {
                        const bool dn = s_dn[s] != 0;
                        // int16 PCM is scaled first (one uniform branch per unit, not per sample); the non-finite test is
                        // one integer maximum over the unit: exponent all ones <=> NaN or Inf (audio.py:227-228)
                        if (p.pcm == 1) {
#pragma unroll
                            for (int e = 0; e < 8; ++e) v[u4][e] = __fdiv_rn(v[u4][e], 32767.0f);
                        } else if (p.pcm == 2) {
#pragma unroll
                            for (int e = 0; e < 8; ++e) v[u4][e] = v[u4][e] * (1.0f / 32768.0f);
                        }
                        uint32_t amx = 0u;
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const float x = v[u4][e];
                            amx = max(amx, __float_as_uint(x) & 0x7fffffffu);
                            v[u4][e] = (dn && !(fabsf(x) > 0.01f)) ? 0.0f : x;
                        }
                        if (amx >= 0x7f800000u && p.status) atomicOr(&p.status[st * kTile + s], 1u);
                    }
                    if constexpr (!H16) {
                        uint32_t w[3][4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) split3x2(v[u4][2 * e], v[u4][2 * e + 1], w[0][e], w[1][e], w[2][e]);
                        const uint32_t seg = (uint32_t)c8 >> 4, kk = ((uint32_t)c8 & 15u) * 8u;   // k inside the 128-sample segment
                        const uint32_t off = tc::sw128_offset(seg * 32u + (uint32_t)s, kk, 128u);
#pragma unroll
                        for (int part = 0; part < 3; ++part)
                            *reinterpret_cast<uint4 *>(act + part * kAudPart + off) = make_uint4(w[part][0], w[part][1], w[part][2], w[part][3]);
                    }
                }
                if (H16) {
                    CVAD_PROF(20);
                    // per-stream maximum of the gated frame (a unit's stream is warp-uniform: s = 8 u4 + tid / 64) ...
                    float m4[4];
#pragma unroll
                    for (int u4 = 0; u4 < 4; ++u4) {
                        float m = 0.f;
#pragma unroll
                        for (int e = 0; e < 8; ++e) m = fmaxf(m, fabsf(v[u4][e]));
                        m4[u4] = m;
                    }
                    amax_push_n<4>(&amax[tid >> 6], 8, m4, lane);
                    CVAD_PROF(15);
                    epi_bar();
                    CVAD_PROF(16);
                    // ... then scale, split into two FP16 parts, store
#pragma unroll
                    for (int u4 = 0; u4 < 4; ++u4) {
                        const int unit = u4 * kEpiThreads + tid;
                        const int s = unit >> 6, c8 = unit & 63;
                        const float sc = scale_from_max(amax[s]).s;
                        uint32_t w[2][4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) split2x2_h(v[u4][2 * e] * sc, v[u4][2 * e + 1] * sc, w[0][e], w[1][e]);
                        const uint32_t seg = (uint32_t)c8 >> 4, kk = ((uint32_t)c8 & 15u) * 8u;
                        const uint32_t off = tc::sw128_offset(seg * 32u + (uint32_t)s, kk, 128u);
#pragma unroll
                        for (int part = 0; part < 2; ++part)
                            *reinterpret_cast<uint4 *>(act + part * kAudPart + off) = make_uint4(w[part][0], w[part][1], w[part][2], w[part][3]);
                    }
                }
            }
            tc::fence_async_smem();
            epi_bar();
            if (tid == 0) mbar_arrive(act_ready);
            CVAD_PROF(1);

            // ---- STFT epilogue: magnitude = sqrt(re^2 + im^2), squares rounded separately (ONNX Pow, Pow, Add, Sqrt)
            mbar_wait(acc_ready, acc_phase); acc_phase ^= 1u;
            CVAD_PROF(2);
            tc::fence_after_sync();
            if (H16) {
                // a thread owns bin b of streams 8 cg .. 8 cg + 7 at all three time columns: one scale per stream
                const int b = 32 * q + lane, i0 = 8 * cg;
                const float iw = p.tc16_inv_w[0];
                float inv[8], mag[3][8], mx[8];
                inv_scales8(amax + i0, iw, inv);
#pragma unroll
                for (int e = 0; e < 8; ++e) mx[e] = 0.f;
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const int c0 = t * 32 + i0;
                    float mr[8], mi[8], cr[8], ci[8];
                    tmem_ld8(lane_addr + kColMain + c0, mr);
                    tmem_ld8(lane_addr + kColMain + 96 + c0, mi);
                    tmem_ld8(lane_addr + kColCorr + c0, cr);
                    tmem_ld8(lane_addr + kColCorr + 96 + c0, ci);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float re = (mr[e] + cr[e]) * inv[e];
                        float im = (mi[e] + ci[e]) * inv[e];
                        if (b == 0) {
                            nyq[c0 + e] = fabsf(im);           // sqrt(x*x + 0*0)
                            im = 0.f;
                        }
                        mag[t][e] = sfu_sqrt(__fadd_rn(__fmul_rn(re, re), __fmul_rn(im, im)));
                        mx[e] = fmaxf(mx[e], mag[t][e]);
                    }
                }
                CVAD_PROF(17);
                amax_push_n<8>(&amax[kTile + i0], 1, mx, lane);
                CVAD_PROF(18);
                epi_bar();
                CVAD_PROF(19);
                scales8(amax + kTile + i0, inv);
                if constexpr (BMN) {
                    unsigned char *dst = act + tc::mn64_offset((uint32_t)i0, (uint32_t)b, 512u, 1536u);
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) mag[t][e] *= inv[e];
                        store_row8_mn(dst + t * 512, kMagPart, mag[t]);
                    }
                } else {
#pragma unroll
                    for (int t = 0; t < 3; ++t)
#pragma unroll
                        for (int e = 0; e < 8; e += 2)
                            store_parts2_h(act, kMagPart, (uint32_t)(t * 32 + i0 + e), (uint32_t)b, 96u, mag[t][e] * inv[e], mag[t][e + 1] * inv[e + 1]);
                }
            } else {
                const int b = 32 * q + lane;   // bin; TMEM lane b of block 1 holds im[b] (b >= 1) or re[128] (b == 0)
#pragma unroll 1
                for (int ch = 0; ch < 3; ++ch) {
                    const int c0 = cg * 24 + ch * 8;
                    float mr[8], mi[8], cr[8], ci[8];
                    tmem_ld8(lane_addr + kColMain + c0, mr);
                    tmem_ld8(lane_addr + kColMain + 96 + c0, mi);
                    tmem_ld8(lane_addr + kColCorr + c0, cr);
                    tmem_ld8(lane_addr + kColCorr + 96 + c0, ci);
                    tmem_wait_ld();
                    float mag[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float re = mr[e] + cr[e];
                        float im = mi[e] + ci[e];
                        if (b == 0) {
                            const float m128 = fabsf(im);      // sqrt(x*x + 0*0)
                            nyq[c0 + e] = m128;
                            if (dbg) p.dbg[(128 * 3 + ((c0 + e) >> 5)) * 32 + ((c0 + e) & 31)] = m128;
                            im = 0.f;
                        }
                        mag[e] = sfu_sqrt(__fadd_rn(__fmul_rn(re, re), __fmul_rn(im, im)));
                        if (dbg) p.dbg[(b * 3 + ((c0 + e) >> 5)) * 32 + ((c0 + e) & 31)] = mag[e];
                    }
#pragma unroll
                    for (int e = 0; e < 8; e += 2) store_parts2(act, kMagPart, (uint32_t)(c0 + e), (uint32_t)b, 96u, mag[e], mag[e + 1]);
                }
            }
            tc::fence_async_smem();
            tc::fence_before_sync();
            epi_bar();
            if (tid == 0) mbar_arrive(act_ready);
            CVAD_PROF(3);

            // ---- encoder.0 epilogue: + bias + Nyquist channel (FP32) -> ReLU -> E0 (row blocks in time order 0,2,1)
            mbar_wait(acc_ready, acc_phase); acc_phase ^= 1u;
            CVAD_PROF(4);
            tc::fence_after_sync();
            if (H16) {
                const int o = 32 * q + lane, i0 = 8 * cg;
                const float bias = __ldg(p.b_fe + o), iw = p.tc16_inv_w[1];
                const float wn0 = __ldg(p.nyq_w + 4 * o), wn1 = __ldg(p.nyq_w + 4 * o + 1), wn2 = __ldg(p.nyq_w + 4 * o + 2);
                float sc[8], v[3][8], mx[8];
                inv_scales8(amax + kTile + i0, iw, sc);
#pragma unroll
                for (int e = 0; e < 8; ++e) mx[e] = 0.f;
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const int c0 = t * 32 + i0;
                    float m[8], cr[8];
                    tmem_ld8(lane_addr + kColMain + c0, m);
                    tmem_ld8(lane_addr + kColCorr + c0, cr);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int i = i0 + e;
                        float a = (m[e] + cr[e]) * sc[e];
                        if (t > 0) a = fmaf(wn0, nyq[(t - 1) * 32 + i], a);
                        a = fmaf(wn1, nyq[t * 32 + i], a);
                        if (t < 2) a = fmaf(wn2, nyq[(t + 1) * 32 + i], a);
                        v[t][e] = fmaxf(a + bias, 0.f);
                        mx[e] = fmaxf(mx[e], v[t][e]);
                    }
                }
                amax_push_n<8>(&amax[2 * kTile + i0], 1, mx, lane);
                epi_bar();
                scales8(amax + 2 * kTile + i0, sc);
                if constexpr (BMN) {
                    unsigned char *dst = act + tc::mn64_offset((uint32_t)i0, (uint32_t)o, 512u, 1536u);
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) v[t][e] *= sc[e];
                        store_row8_mn(dst + (t == 0 ? 0 : (t == 1 ? 1024 : 512)), kMagPart, v[t]);   // N atoms in time order 0, 2, 1
                    }
                } else {
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
                        const uint32_t rb = t == 0 ? 0u : (t == 1 ? 64u : 32u);
#pragma unroll
                        for (int e = 0; e < 8; e += 2)
                            store_parts2_h(act, kMagPart, rb + (uint32_t)(i0 + e), (uint32_t)o, 96u, v[t][e] * sc[e], v[t][e + 1] * sc[e + 1]);
                    }
                }
            } else {
                const int o = 32 * q + lane;
                const float bias = __ldg(p.b_fe + o);
                const float wn0 = __ldg(p.nyq_w + 4 * o), wn1 = __ldg(p.nyq_w + 4 * o + 1), wn2 = __ldg(p.nyq_w + 4 * o + 2);
#pragma unroll 1
                for (int ch = 0; ch < 3; ++ch) {
                    const int c0 = cg * 24 + ch * 8;
                    const int t = c0 >> 5, i0 = c0 & 31;
                    const uint32_t rb = t == 0 ? 0u : (t == 1 ? 64u : 32u);
                    float m[8], cr[8], v[8];
                    tmem_ld8(lane_addr + kColMain + c0, m);
                    tmem_ld8(lane_addr + kColCorr + c0, cr);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int i = i0 + e;
                        float a = m[e] + cr[e];
                        if (t > 0) a = fmaf(wn0, nyq[(t - 1) * 32 + i], a);
                        a = fmaf(wn1, nyq[t * 32 + i], a);
                        if (t < 2) a = fmaf(wn2, nyq[(t + 1) * 32 + i], a);
                        v[e] = fmaxf(a + bias, 0.f);
                        if (dbg) p.dbg[kDbgMag + (o * 3 + t) * 32 + i] = v[e];
                    }
#pragma unroll
                    for (int e = 0; e < 8; e += 2) store_parts2(act, kMagPart, rb + (uint32_t)(i0 + e), (uint32_t)o, 96u, v[e], v[e + 1]);
                }
            }
            tc::fence_async_smem();
            tc::fence_before_sync();
            epi_bar();
            if (tid == 0) mbar_arrive(act_ready);
            CVAD_PROF(5);

            // ---- encoder.1 epilogue (M = 64: channel 16q + lane lives in TMEM lane 32q + lane, lanes >= 16 idle)
            mbar_wait(acc_ready, acc_phase); acc_phase ^= 1u;
            CVAD_PROF(6);
            tc::fence_after_sync();
            if (H16) {
                const int o = 16 * q + (lane & 15), i0 = 8 * cg;
                const float bias = __ldg(p.b_fe + 128 + o), iw = p.tc16_inv_w[2];
                float sc[8], v[2][8], mx[8];
                inv_scales8(amax + 2 * kTile + i0, iw, sc);
#pragma unroll
                for (int e = 0; e < 8; ++e) mx[e] = 0.f;
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int c0 = t * 32 + i0;
                    float m[8], cr[8];
                    tmem_ld8(lane_addr + kColMain + c0, m);
                    tmem_ld8(lane_addr + kColCorr + c0, cr);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float a = fmaxf((m[e] + cr[e]) * sc[e] + bias, 0.f);
                        v[t][e] = lane < 16 ? a : 0.f;
                        mx[e] = fmaxf(mx[e], v[t][e]);
                    }
                }
                amax_push_n<8>(&amax[3 * kTile + i0], 1, mx, lane);
                epi_bar();
                if (lane < 16) {
                    scales8(amax + 3 * kTile + i0, sc);
                    if constexpr (BMN) {
                        unsigned char *dst = act + tc::mn64_offset((uint32_t)i0, (uint32_t)o, 512u, 1024u);
#pragma unroll
                        for (int t = 0; t < 2; ++t) {
#pragma unroll
                            for (int e = 0; e < 8; ++e) v[t][e] *= sc[e];
                            store_row8_mn(dst + t * 512, kE1Part, v[t]);
                        }
                    } else {
#pragma unroll
                        for (int t = 0; t < 2; ++t)
#pragma unroll
                            for (int e = 0; e < 8; e += 2)
                                store_parts2_h(act, kE1Part, (uint32_t)(t * 32 + i0 + e), (uint32_t)o, 64u, v[t][e] * sc[e], v[t][e + 1] * sc[e + 1]);
                    }
                }
            } else {
                const int o = 16 * q + (lane & 15);
                const float bias = __ldg(p.b_fe + 128 + o);
#pragma unroll 1
                for (int ch = 0; ch < 2; ++ch) {
                    const int c0 = cg * 16 + ch * 8;
                    float m[8], cr[8], v[8];
                    tmem_ld8(lane_addr + kColMain + c0, m);
                    tmem_ld8(lane_addr + kColCorr + c0, cr);
                    tmem_wait_ld();
                    if (lane < 16) {
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            v[e] = fmaxf(m[e] + cr[e] + bias, 0.f);
                            if (dbg) p.dbg[kDbgMag + kDbgE0 + (o * 2 + ((c0 + e) >> 5)) * 32 + ((c0 + e) & 31)] = v[e];
                        }
#pragma unroll
                        for (int e = 0; e < 8; e += 2) store_parts2(act, kE1Part, (uint32_t)(c0 + e), (uint32_t)o, 64u, v[e], v[e + 1]);
                    }
                }
            }
            tc::fence_async_smem();
            tc::fence_before_sync();
            epi_bar();
            if (tid == 0) mbar_arrive(act_ready);
            CVAD_PROF(7);

            // ---- encoder.2 epilogue (M = 64, 32 columns)
            mbar_wait(acc_ready, acc_phase); acc_phase ^= 1u;
            CVAD_PROF(8);
            tc::fence_after_sync();
            if (H16) {
                const int o = 16 * q + (lane & 15);
                const float bias = __ldg(p.b_fe + 192 + o), iw = p.tc16_inv_w[3];
                const int c0 = cg * 8;
                float m[8], cr[8], v[8];
                tmem_ld8(lane_addr + kColMain + c0, m);
                tmem_ld8(lane_addr + kColCorr + c0, cr);
                tmem_wait_ld();
                float si[8];
                inv_scales8(amax + 3 * kTile + c0, iw, si);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float a = fmaxf((m[e] + cr[e]) * si[e] + bias, 0.f);
                    v[e] = lane < 16 ? a : 0.f;
                }
                amax_push_n<8>(&amax[4 * kTile + c0], 1, v, lane);
                epi_bar();
                if (lane < 16) {
                    if constexpr (BMN) {
                        scales8(amax + 4 * kTile + c0, si);
#pragma unroll
                        for (int e = 0; e < 8; ++e) v[e] *= si[e];
                        store_row8_mn(act + tc::mn64_offset((uint32_t)c0, (uint32_t)o, 512u, 512u), kE2Part, v);
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; e += 2)
                            store_parts2_h(act, kE2Part, (uint32_t)(c0 + e), (uint32_t)o, 32u, v[e] * scale_from_max(amax[4 * kTile + c0 + e]).s,
                                           v[e + 1] * scale_from_max(amax[4 * kTile + c0 + e + 1]).s);
                    }
                }
            } else {
                const int o = 16 * q + (lane & 15);
                const float bias = __ldg(p.b_fe + 192 + o);
                const int c0 = cg * 8;
                float m[8], cr[8], v[8];
                tmem_ld8(lane_addr + kColMain + c0, m);
                tmem_ld8(lane_addr + kColCorr + c0, cr);
                tmem_wait_ld();
                if (lane < 16) {
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        v[e] = fmaxf(m[e] + cr[e] + bias, 0.f);
                        if (dbg) p.dbg[kDbgMag + kDbgE0 + kDbgE1 + o * 32 + c0 + e] = v[e];
                    }
#pragma unroll
                    for (int e = 0; e < 8; e += 2) store_parts2(act, kE2Part, (uint32_t)(c0 + e), (uint32_t)o, 32u, v[e], v[e + 1]);
                }
            }
            tc::fence_async_smem();
            tc::fence_before_sync();
            epi_bar();
            if (tid == 0) mbar_arrive(act_ready);
            CVAD_PROF(9);

            // ---- encoder.3 epilogue -> feat tile in HBM, already in the recurrent kernel's B-operand bytes
            mbar_wait(acc_ready, acc_phase); acc_phase ^= 1u;
            CVAD_PROF(10);
            tc::fence_after_sync();
            if (H16) {
                const int o = 32 * q + lane;
                const float bias = __ldg(p.b_fe + 256 + o), iw = p.tc16_inv_w[4];
                const int c0 = cg * 8;
                float m[8], cr[8], v[8];
                tmem_ld8(lane_addr + kColMain + c0, m);
                tmem_ld8(lane_addr + kColCorr + c0, cr);
                tmem_wait_ld();
                float si[8];
                inv_scales8(amax + 4 * kTile + c0, iw, si);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = fmaxf((m[e] + cr[e]) * si[e] + bias, 0.f);
                amax_push_n<8>(&amax[5 * kTile + c0], 1, v, lane);
                tc::fence_before_sync();   // the W_ih accumulators reuse these TMEM columns
                epi_bar();
                if constexpr (FUSED) {
                    // [x0 | x1] = N atoms 0 and 1, K groups 1,024 B apart
                    scales8(amax + 5 * kTile + c0, si);
#pragma unroll
                    for (int e = 0; e < 8; ++e) v[e] *= si[e];
                    store_row8_mn(act + tc::mn64_offset((uint32_t)c0, (uint32_t)o, 512u, 1024u), 512u, v);
                } else {
                    // two-kernel form: x goes to HBM as the recurrent kernel's operand, scaled like the h it will sit
                    // next to in K: by the stream's joint maximum max(|x|max, 1) (|h| < 1), handed over in the tile
                    unsigned char *fout = p.feat_tc + (size_t)tile * kFeatTileBytes;
                    uint32_t jm[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) jm[e] = max(amax[5 * kTile + c0 + e], 0x3f800000u);
#pragma unroll
                    for (int e = 0; e < 8; e += 2)
                        store_parts2_h(fout, 32 * 128, (uint32_t)(c0 + e), (uint32_t)o, 96u, v[e] * scale_from_max(jm[e]).s,
                                       v[e + 1] * scale_from_max(jm[e + 1]).s);
                    if (q == 0 && lane < 8)
                        *reinterpret_cast<uint32_t *>(fout + kFeatScaleOff + 4 * (c0 + lane)) = max(amax[5 * kTile + c0 + lane], 0x3f800000u);
                }
            } else {
                const int o = 32 * q + lane;
                const float bias = __ldg(p.b_fe + 256 + o);
                const int c0 = cg * 8;
                float m[8], cr[8], v[8];
                tmem_ld8(lane_addr + kColMain + c0, m);
                tmem_ld8(lane_addr + kColCorr + c0, cr);
                tmem_wait_ld();
                unsigned char *fout = FUSED ? act : p.feat_tc + (size_t)tile * kFeatTileBytes;
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    v[e] = fmaxf(m[e] + cr[e] + bias, 0.f);
                    if (dbg) p.dbg[kDbgMag + kDbgE0 + kDbgE1 + kDbgE2 + o * 32 + c0 + e] = v[e];
                }
#pragma unroll
                for (int e = 0; e < 8; e += 2) store_parts2(fout, 32 * 128, (uint32_t)(c0 + e), (uint32_t)o, 96u, v[e], v[e + 1]);
            }
            if (FUSED) tc::fence_async_smem();
            tc::fence_before_sync();   // TMEM reads of this tile are ordered before the next tile's act_ready arrive
            epi_bar();
            CVAD_PROF(11);
            if (FUSED) {
                if (tid == 0) mbar_arrive(act_ready);          // x operand is in ACT: the W_ih products may start
                // ---- LSTM cell, decoder, state machine (same arithmetic as v5tc_recurrent_kernel, one frame)
                const int u = u_own, i0 = i_own;
                const float b_i = __ldg(p.b_rec_tc + u), b_f = __ldg(p.b_rec_tc + 128 + u),
                            b_g = __ldg(p.b_rec_tc + 256 + u), b_o = __ldg(p.b_rec_tc + 384 + u);
                const float wd = __ldg(p.w_dec + u), dec_b = __ldg(p.w_dec + 128);
                // NaN/Inf streams were flagged by this CTA's own loader (atomicOr at L2): the reference raises
                // before any frame runs, so such a stream keeps its state and reports nothing
                if (warp == 0) {
                    const int i = st * kTile + lane;
                    if (s_valid[lane] && p.status && __ldcg(p.status + i) != 0u) s_valid[lane] = 0;
                }
                epi_bar();
                float dv[8], hn[8];
                if constexpr (BMN) {
                    // gate by gate as the W_ih products complete: sigmoid(i), sigmoid(f), then g -> c' -> tanh(c') run under the
                    // products of the following gates; only sigmoid(o) and h' are left when the last product lands.  Same
                    // operations in the same order per element as the all-at-once form below (bit-identical).
                    const float ih_w = p.tc16_inv_w[5], hh = kHInv * p.tc16_inv_w[6];
                    float ix[8], ga[2][8];
                    inv_scales8(amax + 5 * kTile + i0, ih_w, ix);
#pragma unroll
                    for (int gi = 0; gi < 4; ++gi) {
                        mbar_wait(&gate_ready[gi], gate_phase);
                        tc::fence_after_sync();
                        if (gi == 0) CVAD_PROF(13);
                        float gh[8], gx[8], gy[8];
                        tmem_ld8(lane_addr + kColGate + 32 * gi + i0, gh);
                        tmem_ld8(lane_addr + kColIh + 64 * gi + i0, gx);
                        tmem_ld8(lane_addr + kColIh + 64 * gi + 32 + i0, gy);
                        tmem_wait_ld();
                        const float bias = gi == 0 ? b_i : (gi == 1 ? b_f : (gi == 2 ? b_g : b_o));
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const float z = fmaf(gx[e] + gy[e], ix[e], gh[e] * hh) + bias;
                            if (gi < 2) {
                                ga[gi][e] = sfu_sigmoid(z);
                            } else if (gi == 2) {
                                const float cn = __fadd_rn(__fmul_rn(ga[1][e], creg[e]), __fmul_rn(ga[0][e], sfu_tanh(z)));
                                creg[e] = cn;
                                ga[0][e] = sfu_tanh(cn);
                            } else {
                                hn[e] = sfu_sigmoid(z) * ga[0][e];
                                dv[e] = wd * fmaxf(hn[e], 0.f);
                            }
                        }
                        if (gi == 2) CVAD_PROF(21);
                    }
                    gate_phase ^= 1u;
                } else {
                mbar_wait(acc_ready, acc_phase); acc_phase ^= 1u;
                tc::fence_after_sync();
                CVAD_PROF(13);
                float gate[4][8];
#pragma unroll
                for (int gi = 0; gi < 4; ++gi) tmem_ld8(lane_addr + kColGate + 32 * gi + i0, gate[gi]);
                tmem_wait_ld();
                if (H16) {
                    // gate = W_hh.h (static scale) + W_ih.x (the stream's own scale), each in its own accumulator
                    float gx[4][8], gy[4][8];
#pragma unroll
                    for (int gi = 0; gi < 4; ++gi) {
                        tmem_ld8(lane_addr + kColIh + 64 * gi + i0, gx[gi]);
                        tmem_ld8(lane_addr + kColIh + 64 * gi + 32 + i0, gy[gi]);
                    }
                    tmem_wait_ld();
#pragma unroll
                    for (int gi = 0; gi < 4; ++gi)
#pragma unroll
                        for (int e = 0; e < 8; ++e) gx[gi][e] += gy[gi][e];
                    const float ih_w = p.tc16_inv_w[5], hh = kHInv * p.tc16_inv_w[6];
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const float ix = scale_from_max(amax[5 * kTile + i0 + e]).inv * ih_w;
#pragma unroll
                        for (int gi = 0; gi < 4; ++gi) gate[gi][e] = fmaf(gx[gi][e], ix, gate[gi][e] * hh);
                    }
                }
                CVAD_PROF(21);
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float ig = sfu_sigmoid(gate[0][e] + b_i);
                    const float fg = sfu_sigmoid(gate[1][e] + b_f);
                    const float gg = sfu_tanh(gate[2][e] + b_g);
                    const float og = sfu_sigmoid(gate[3][e] + b_o);
                    const float cn = __fadd_rn(__fmul_rn(fg, creg[e]), __fmul_rn(ig, gg));
                    hn[e] = og * sfu_tanh(cn);
                    creg[e] = cn;
                    dv[e] = wd * fmaxf(hn[e], 0.f);
                }
                }
                CVAD_PROF(22);
#pragma unroll
                for (int w = 4; w >= 1; w >>= 1) {
                    const bool upper = (lane & w) != 0;
#pragma unroll
                    for (int e = 0; e < w; ++e) {
                        const float send = upper ? dv[e] : dv[e + w];
                        const float keep = upper ? dv[e + w] : dv[e];
                        dv[e] = keep + __shfl_xor_sync(0xffffffffu, send, w);
                    }
                }
                dv[0] += __shfl_xor_sync(0xffffffffu, dv[0], 8);
                dv[0] += __shfl_xor_sync(0xffffffffu, dv[0], 16);
                if (lane < 8) dpart[q * 32 + i0 + lane] = dv[0];
                // new state back to HBM: one 32-byte row per thread when the group's slots are a row of the state (s_grp) and
                // none of its streams was flagged non-finite (such a stream keeps its old state), else element by element
                if (p.commit) {
                    bool all8 = true;
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {          // (s_valid is 8-byte aligned)
                        const int2 v2 = *reinterpret_cast<const int2 *>(s_valid + i0 + e);
                        all8 = all8 && v2.x && v2.y;
                    }
                    const int gb = s_grp[cg];
                    if (gb >= 0 && all8) {
                        float4 *ph = reinterpret_cast<float4 *>(p.h_state + state_at(u, gb));
                        float4 *pc = reinterpret_cast<float4 *>(p.c_state + state_at(u, gb));
                        ph[0] = make_float4(hn[0], hn[1], hn[2], hn[3]);
                        ph[1] = make_float4(hn[4], hn[5], hn[6], hn[7]);
                        pc[0] = make_float4(creg[0], creg[1], creg[2], creg[3]);
                        pc[1] = make_float4(creg[4], creg[5], creg[6], creg[7]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 8; ++e)
                            if (s_valid[i0 + e]) {
                                const size_t at = state_at(u, s_slot[i0 + e]);
                                p.h_state[at] = hn[e];
                                p.c_state[at] = creg[e];
                            }
                    }
                }
                epi_bar();   // dpart
                CVAD_PROF(23);
                CVAD_PROF(24);
                // sigmoid(w . relu(h') + b), then the start/end state machine (silero_model.py:790-923)
                if (warp == 0 && s_valid[lane]) {
                    const int slot = s_slot[lane];
                    int sm_active = s_sm[lane], sm_sc = s_sm[kTile + lane], sm_ec = s_sm[2 * kTile + lane];
                    const int sm_ns = s_sm[3 * kTile + lane], sm_ne = s_sm[4 * kTile + lane];
                    const long long sm_f0 = s_f0[lane];
                    const float a = (dpart[lane] + dpart[32 + lane]) + (dpart[64 + lane] + dpart[96 + lane]);
                    const float prob = sigmoid_f(a + dec_b);
                    const double pd = (double)prob;
                    unsigned int fl = 0u;
                    if (!sm_active) {
                        if (pd >= s_thr[lane]) {
                            ++sm_sc;
                            if (sm_sc >= sm_ns && sm_ns <= 20) {  // deque(maxlen=20), silero_model.py:620-623
                                sm_active = 1; sm_sc = 0; sm_ec = 0; fl |= 1u;
                            }
                        } else {
                            sm_sc = 0;
                        }
                    } else {
                        fl |= 4u;
                        if (pd < s_thr[kTile + lane]) {
                            ++sm_ec;
                            if (sm_ec >= sm_ne && sm_ne <= 100) {  // deque(maxlen=100), :625-628
                                sm_active = 0; sm_ec = 0; fl |= 2u;
                            }
                        } else {
                            sm_ec = 0;
                        }
                    }
                    const int i = st * kTile + lane;
                    if (p.probs) p.probs[(size_t)i * p.max_frames] = prob;
                    if (p.flags) p.flags[(size_t)i * p.max_frames] = (unsigned char)fl;
                    if ((fl & 3u) && p.n_events) {
                        EventRec *ev = reinterpret_cast<EventRec *>(p.events);
                        for (unsigned int kind = 1u; kind <= 2u; kind <<= 1) {
                            if (fl & kind) {
                                const int at = atomicAdd(p.ev_ctr ? p.ev_ctr : p.n_events, 1);
                                if (ev && at < p.max_events) {
                                    ev[at].stream = i; ev[at].slot = slot; ev[at].frame = 0;
                                    ev[at].kind = (int)kind; ev[at].stream_frame = sm_f0;
                                }
                            }
                        }
                    }
                    if (p.commit) {
                        p.sm_active[slot] = sm_active;
                        p.sm_scount[slot] = sm_sc;
                        p.sm_ecount[slot] = sm_ec;
                        p.frames_done[slot] = sm_f0 + 1;
                    }
                }
                epi_bar();   // ACT, dpart and s_valid are rewritten by the next tile
                CVAD_PROF(14);
                CVAD_PROF_NS(127);
                CVAD_CHAIN_NS(4);
            }
        }
        if (FUSED && (p.ev_ctr || p.step_ctr) && tid == 0) {
            // chained steps: events were counted in the engine's own counter (ev_ctr[0]); the last CTA to take a ticket
            // publishes the total, leaves counter and ticket at zero for the next step -- no memset between the kernels --
            // and counts the step as completed (read by the next step's early CTAs, above).  ONE ticket for both: the
            // atomic's round trip (~0.4 us with 128 CTAs on one address) sits between the tile and the CTA's exit.
            // No fence: every event atomicAdd of this CTA returned its index to warp 0 before the barrier above, i.e.
            // it has been performed at L2, where the ticket and the exchange below are performed too.
            // (Measured and dropped: taking the ticket inside the last tile, right behind the state machine, with the state
            // stores moved behind it so that the round trip runs under them -- 4.149 M against 4.156 M audio-s/s: the tail
            // of the tile grew by what the exit saved.)
            int *ticket = p.ev_ctr ? p.ev_ctr + 1 : p.step_ctr + 1;
            if (atomicAdd(ticket, 1) == (int)gridDim.x - 1) {
                if (p.ev_ctr) {
                    const int total = atomicExch(p.ev_ctr, 0);
                    if (p.n_events) *p.n_events = total;
                }
                *ticket = 0;
                if (p.step_ctr) atomicAdd(p.step_ctr, 1);
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == kProducerWarp) tc::tmem_dealloc(0u, 512);
    CVAD_PROF_NS(122);
    CVAD_CHAIN_NS(5);
}

// =====================================================================================
// Recurrent part: LSTMCell(128) gates on the tensor cores, cell + decoder + state machine on the CUDA cores
// =====================================================================================
// B operand XH: rows = part*32 + item (96 rows), K = [x 128 | h 128] = 4 K blocks.  One weight tile of part wp
// multiplies the first (3 - wp) activation parts in ONE MMA (N = 96 / 64 / 32) whose output lands at TMEM column
// 32*wp of the gate block, so that columns [0,32) collect w0.x0, [32,64) w0.x1 + w1.x0 and [64,96) the three
// smallest products.
// H16 (CVAD_MATH_TC16): two FP16 parts; the [x | h] operand of a stream carries ONE scale per frame, the power of two
// that brings max(|x|max, 1) to [2^14, 2^15) (the front end scales x with it and hands its bit pattern over in the feature
// tile, the cell epilogue scales the h it writes for the next frame with that frame's).  Part wp of a weight tile
// multiplies the first (2 - wp) activation parts in one MMA (N = 64 / 32): columns [0,32) collect w0.x0, [32,64)
// w0.x1 + w1.x0.  W_ih and W_hh share one weight scale (pack_v5_tc16).
template <bool H16>
__global__ void __launch_bounds__(kThreadsTC, 1) v5tc_recurrent_kernel(const V5Step p) {
    constexpr bool PROF = true;
    constexpr int NP = H16 ? 2 : 3;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
    unsigned char *xbuf = base;                               // [2][kFeatTileBytes]
    unsigned char *hbuf = xbuf + 2 * kFeatTileBytes;          // [kFeatTileBytes]: K blocks 2,3
    unsigned char *ring_buf = hbuf + kFeatTileBytes;
    float *sbuf = reinterpret_cast<float *>(ring_buf + kRecRing * kSlotBytes);   // [128][33]
    float *dpart = sbuf + 128 * 33;                                              // [4][32]
    uint64_t *bars = reinterpret_cast<uint64_t *>(dpart + 128);
    uint64_t *full = bars, *empty = bars + kRecRing, *xfull = bars + 2 * kRecRing, *h_ready = xfull + 2,
             *acc_ready = h_ready + 1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_ready + 1);
    double *s_startp = reinterpret_cast<double *>(tmem_slot + 4);
    double *s_endp = s_startp + kTile;
    int *s_slot = reinterpret_cast<int *>(s_endp + kTile);
    int *s_nfr = s_slot + kTile;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int st = blockIdx.x;
    CVAD_PROF_NS(123);

    if (tid < kTile) {
        const int i = st * kTile + tid;
        int slot = -1, nf = 0;
        if (i < p.n_streams) {
            slot = p.slots ? p.slots[i] : i;
            nf = p.n_frames ? p.n_frames[i] : p.max_frames;   // loop bound; the NaN/Inf status is applied after the grid dependency
            s_startp[tid] = p.start_p[slot];
            s_endp[tid] = p.end_p[slot];
        }
        s_slot[tid] = slot;
        s_nfr[tid] = nf;
    }
    if (tid == 0) {
        for (int i = 0; i < kRecRing; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(&xfull[0], 1);
        mbar_init(&xfull[1], 1);
        mbar_init(h_ready, 1);
        mbar_init(acc_ready, 1);
        mbar_fence_init();
    }
    if (warp == kProducerWarp) tc::tmem_alloc(tmem_slot, 512);
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    if (*tmem_slot != 0u) __trap();
    CVAD_PROF_NS(124);
    int tmax = 0;
    {
        int v = s_nfr[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
        tmax = v;
    }
    const uint32_t ring_s = smem_u32(ring_buf), x_s = smem_u32(xbuf), h_s = smem_u32(hbuf);

    if (tmax > 0) {
        if (warp == kProducerWarp) {
            if (lane == 0) {
                uint32_t g = 0;
                const unsigned char *wsrc = H16 ? p.w_rec_h : p.w_rec_tc;
                for (int j = 0; j < tmax; ++j)
                    for (int s = 0; s < 16 * NP; ++s, ++g) {
                        const uint32_t slot = g % kRecRing;
                        mbar_wait(&empty[slot], ((g / kRecRing) & 1u) ^ 1u);
                        mbar_arrive_expect_tx(&full[slot], kSlotBytes);
                        bulk_g2s(ring_buf + slot * kSlotBytes, wsrc + (size_t)s * kSlotBytes, kSlotBytes, &full[slot]);
                    }
            }
            __syncwarp();
        } else if (warp == kMmaWarp) {
            uint32_t g = 0;
            const uint32_t idesc[3] = {H16 ? idesc_f16_f32(128, 64) : tc::idesc_bf16_f32(128, 96),
                                       H16 ? idesc_f16_f32(128, 32) : tc::idesc_bf16_f32(128, 64), tc::idesc_bf16_f32(128, 32)};
            for (int j = 0; j < tmax; ++j) {
                const bool first_tile = lane == 0 && j < 8;
                mbar_wait(&xfull[j & 1], (uint32_t)(j >> 1) & 1u);
                CVAD_PROF(96 + 3 * j);
                mbar_wait(h_ready, (uint32_t)j & 1u);
                tc::fence_after_sync();
                CVAD_PROF(97 + 3 * j);
                for (int blk = 0; blk < 4; ++blk)
                    for (int kb = 0; kb < 4; ++kb) {
                        const uint32_t b_addr = kb < 2 ? x_s + (j & 1) * kFeatTileBytes + kb * kXhKb : h_s + (kb - 2) * kXhKb;
                        for (int wp = 0; wp < NP; ++wp, ++g) {
                            const uint32_t slot = g % kRecRing;
                            mbar_wait(&full[slot], (g / kRecRing) & 1u);
                            tc::fence_after_sync();
                            if (tc::elect_one()) {
                                const uint64_t ad = tc::smem_desc_sw128(ring_s + slot * kSlotBytes);
                                const uint64_t bd = tc::smem_desc_sw128(b_addr);
#pragma unroll
                                for (int ks = 0; ks < 4; ++ks)
                                    tc::mma_bf16(blk * 96 + wp * 32, ad + ks * 2, bd + ks * 2, idesc[wp],
                                                 (kb == 0 && wp == 0 && ks == 0) ? 0u : 1u);
                                tc::mma_commit(&empty[slot]);
                            }
                            __syncwarp();
                        }
                    }
                if (tc::elect_one()) tc::mma_commit(acc_ready);
                __syncwarp();
                CVAD_PROF(98 + 3 * j);
            }
        } else {
            // -------------------------------------------------------- state + epilogue warps
            const int q = warp & 3, cg = warp >> 2;
            const uint32_t lane_addr = (uint32_t)(32 * q) << 16;
            const int u = 32 * q + lane;          // hidden unit owned by this thread (TMEM lane)
            const int i0 = 8 * cg;                // its 8 streams
            bool first_tile = tid == 0;
            CVAD_PROF(64);
            // resident state: h -> BF16x3 rows of the B operand, c -> registers (coalesced through sbuf;
            // both global reads are in flight before the first barrier)
            float hreg[8], creg[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int idx = e * kEpiThreads + tid;
                const int slot = s_slot[idx & 31];
                hreg[e] = slot >= 0 ? __ldg(p.h_state + state_at(idx >> 5, slot)) : 0.f;
                creg[e] = slot >= 0 ? __ldg(p.c_state + state_at(idx >> 5, slot)) : 0.f;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int idx = e * kEpiThreads + tid;
                sbuf[(idx >> 5) * 33 + (idx & 31)] = hreg[e];
            }
            epi_bar();
#pragma unroll
            for (int e = 0; e < 8; ++e) hreg[e] = sbuf[u * 33 + i0 + e];
            if (!H16) {
#pragma unroll
                for (int e = 0; e < 8; e += 2) store_parts2(hbuf, 32 * 128, (uint32_t)(i0 + e), (uint32_t)u, 96u, hreg[e], hreg[e + 1]);
            }
            epi_bar();
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int idx = e * kEpiThreads + tid;
                sbuf[(idx >> 5) * 33 + (idx & 31)] = creg[e];
            }
            epi_bar();
#pragma unroll
            for (int e = 0; e < 8; ++e) creg[e] = sbuf[u * 33 + i0 + e];
            if (!H16) {
                tc::fence_async_smem();
                epi_bar();
                if (tid == 0) mbar_arrive(h_ready);
            }
            CVAD_PROF(65);
            // ---- everything above only touched state owned by this kernel; the front end's outputs (status, feat)
            //      are read after the grid dependency resolves
            asm volatile("griddepcontrol.wait;" ::: "memory");
            if (warp == 0) {
                const int i = st * kTile + lane;
                if (i < p.n_streams && p.status && p.status[i] != 0u) s_nfr[lane] = 0;  // NaN/Inf: the reference raises before any frame runs
            }
            epi_bar();
            if (tid == 0)
                for (int j = 0; j < 2 && j < tmax; ++j) {
                    mbar_arrive_expect_tx(&xfull[j], kFeatTileBytes);
                    bulk_g2s(xbuf + j * kFeatTileBytes, p.feat_tc + ((size_t)j * p.n_stiles + st) * kFeatTileBytes,
                             kFeatTileBytes, &xfull[j]);
                }

            // state machine words (warp 0, one lane per stream)
            int sm_active = 0, sm_sc = 0, sm_ec = 0, sm_ns = 1, sm_ne = 1;
            long long sm_f0 = 0;
            if (warp == 0 && s_slot[lane] >= 0) {
                const int slot = s_slot[lane];
                sm_active = p.sm_active[slot];
                sm_sc = p.sm_scount[slot];
                sm_ec = p.sm_ecount[slot];
                sm_ns = p.n_start[slot];
                sm_ne = p.n_end[slot];
                sm_f0 = p.frames_done[slot];
            }
            const float b_i = __ldg(p.b_rec_tc + u), b_f = __ldg(p.b_rec_tc + 128 + u), b_g = __ldg(p.b_rec_tc + 256 + u),
                        b_o = __ldg(p.b_rec_tc + 384 + u);
            const float wd = __ldg(p.w_dec + u), dec_b = __ldg(p.w_dec + 128);
            int nfr[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) nfr[e] = s_nfr[i0 + e];
            // H16: scale of frame 0's operand from its feature tile, then h (resident state) into the operand with it
            float g_inv[8];                                   // 1 / (this frame's operand scale x weight scale)
            if (H16) {
                mbar_wait(&xfull[0], 0u);
                float s_h[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const Scale S = scale_from_max(*reinterpret_cast<const uint32_t *>(xbuf + kFeatScaleOff + 4 * (i0 + e)));
                    s_h[e] = S.s;
                    g_inv[e] = S.inv * p.tc16_inv_w[5];
                }
#pragma unroll
                for (int e = 0; e < 8; e += 2)
                    store_parts2_h(hbuf, 32 * 128, (uint32_t)(i0 + e), (uint32_t)u, 96u, hreg[e] * s_h[e], hreg[e + 1] * s_h[e + 1]);
                tc::fence_async_smem();
                epi_bar();
                if (tid == 0) mbar_arrive(h_ready);
            }

            for (int j = 0; j < tmax; ++j) {
                first_tile = tid == 0 && j < 8;
                mbar_wait(acc_ready, (uint32_t)j & 1u);
                tc::fence_after_sync();
                CVAD_PROF(66 + 3 * j);
                // frame j's MMAs are complete: its x buffer is free for frame j + 2
                if (tid == 0 && j + 2 < tmax) {
                    mbar_arrive_expect_tx(&xfull[j & 1], kFeatTileBytes);
                    bulk_g2s(xbuf + (j & 1) * kFeatTileBytes, p.feat_tc + ((size_t)(j + 2) * p.n_stiles + st) * kFeatTileBytes,
                             kFeatTileBytes, &xfull[j & 1]);
                }
                float gate[4][8];
#pragma unroll
                for (int blk = 0; blk < 4; ++blk) {
                    float g0[8], g1[8], g2[8];
                    tmem_ld8(lane_addr + blk * 96 + i0, g0);
                    tmem_ld8(lane_addr + blk * 96 + 32 + i0, g1);
                    if (!H16) tmem_ld8(lane_addr + blk * 96 + 64 + i0, g2);
                    tmem_wait_ld();
#pragma unroll
                    for (int e = 0; e < 8; ++e) gate[blk][e] = H16 ? (g0[e] + g1[e]) * g_inv[e] : g0[e] + (g1[e] + g2[e]);
                }
                float dv[8], hn[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float ig = sfu_sigmoid(gate[0][e] + b_i);
                    const float fg = sfu_sigmoid(gate[1][e] + b_f);
                    const float gg = sfu_tanh(gate[2][e] + b_g);
                    const float og = sfu_sigmoid(gate[3][e] + b_o);
                    const float cn = __fadd_rn(__fmul_rn(fg, creg[e]), __fmul_rn(ig, gg));
                    const float hv = og * sfu_tanh(cn);
                    const bool live = j < nfr[e];
                    creg[e] = live ? cn : creg[e];
                    hreg[e] = live ? hv : hreg[e];
                    hn[e] = hreg[e];                  // a finished stream keeps its last h in the operand
                    dv[e] = wd * fmaxf(hv, 0.f);
                }
                if (H16) {
                    if (j + 1 < tmax) {
                        // the next frame's operand scale (its tile was requested two frames ago) -> h with it
                        mbar_wait(&xfull[(j + 1) & 1], (uint32_t)((j + 1) >> 1) & 1u);
                        const unsigned char *xt = xbuf + ((j + 1) & 1) * kFeatTileBytes + kFeatScaleOff;
                        float s_h[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const Scale S = scale_from_max(*reinterpret_cast<const uint32_t *>(xt + 4 * (i0 + e)));
                            s_h[e] = S.s;
                            g_inv[e] = S.inv * p.tc16_inv_w[5];
                        }
#pragma unroll
                        for (int e = 0; e < 8; e += 2)
                            store_parts2_h(hbuf, 32 * 128, (uint32_t)(i0 + e), (uint32_t)u, 96u, hn[e] * s_h[e], hn[e + 1] * s_h[e + 1]);
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 8; e += 2) store_parts2(hbuf, 32 * 128, (uint32_t)(i0 + e), (uint32_t)u, 96u, hn[e], hn[e + 1]);
                }
                // decoder dot over the 128 units: 8 values x 32 lanes -> every lane ends with item (lane & 7)
#pragma unroll
                for (int w = 4; w >= 1; w >>= 1) {
                    const bool upper = (lane & w) != 0;
#pragma unroll
                    for (int e = 0; e < w; ++e) {
                        const float send = upper ? dv[e] : dv[e + w];
                        const float keep = upper ? dv[e + w] : dv[e];
                        dv[e] = keep + __shfl_xor_sync(0xffffffffu, send, w);
                    }
                }
                dv[0] += __shfl_xor_sync(0xffffffffu, dv[0], 8);
                dv[0] += __shfl_xor_sync(0xffffffffu, dv[0], 16);
                if (lane < 8) dpart[q * 32 + i0 + lane] = dv[0];
                tc::fence_async_smem();
                tc::fence_before_sync();
                epi_bar();
                if (tid == 0) mbar_arrive(h_ready);
                CVAD_PROF(67 + 3 * j);
                // sigmoid(w . relu(h') + b), then the start/end state machine (silero_model.py:790-923)
                if (warp == 0 && j < s_nfr[lane]) {
                    const float a = (dpart[lane] + dpart[32 + lane]) + (dpart[64 + lane] + dpart[96 + lane]);
                    const float prob = sigmoid_f(a + dec_b);
                    const double pd = (double)prob;
                    unsigned int fl = 0u;
                    if (!sm_active) {
                        if (pd >= s_startp[lane]) {
                            ++sm_sc;
                            if (sm_sc >= sm_ns && sm_ns <= 20) {  // deque(maxlen=20), silero_model.py:620-623
                                sm_active = 1; sm_sc = 0; sm_ec = 0; fl |= 1u;
                            }
                        } else {
                            sm_sc = 0;
                        }
                    } else {
                        fl |= 4u;
                        if (pd < s_endp[lane]) {
                            ++sm_ec;
                            if (sm_ec >= sm_ne && sm_ne <= 100) {  // deque(maxlen=100), :625-628
                                sm_active = 0; sm_ec = 0; fl |= 2u;
                            }
                        } else {
                            sm_ec = 0;
                        }
                    }
                    const int i = st * kTile + lane;
                    if (p.probs) p.probs[(size_t)i * p.max_frames + j] = prob;
                    if (p.flags) p.flags[(size_t)i * p.max_frames + j] = (unsigned char)fl;
                    if ((fl & 3u) && p.n_events) {
                        EventRec *ev = reinterpret_cast<EventRec *>(p.events);
                        for (unsigned int kind = 1u; kind <= 2u; kind <<= 1) {
                            if (fl & kind) {
                                const int at = atomicAdd(p.n_events, 1);
                                if (ev && at < p.max_events) {
                                    ev[at].stream = i; ev[at].slot = s_slot[lane]; ev[at].frame = j;
                                    ev[at].kind = (int)kind; ev[at].stream_frame = sm_f0 + j;
                                }
                            }
                        }
                    }
                }
                epi_bar();   // dpart is rewritten by the next frame
                CVAD_PROF(68 + 3 * j);
            }

            // ---- write the resident state back (coalesced through sbuf)
            if (p.commit) {
#pragma unroll
                for (int e = 0; e < 8; ++e) sbuf[u * 33 + i0 + e] = hreg[e];
                epi_bar();
                for (int idx = tid; idx < 4096; idx += kEpiThreads) {
                    const int s = idx & 31, uu = idx >> 5;
                    const int slot = s_slot[s];
                    if (slot >= 0 && s_nfr[s] > 0) p.h_state[state_at(uu, slot)] = sbuf[uu * 33 + s];
                }
                epi_bar();
#pragma unroll
                for (int e = 0; e < 8; ++e) sbuf[u * 33 + i0 + e] = creg[e];
                epi_bar();
                for (int idx = tid; idx < 4096; idx += kEpiThreads) {
                    const int s = idx & 31, uu = idx >> 5;
                    const int slot = s_slot[s];
                    if (slot >= 0 && s_nfr[s] > 0) p.c_state[state_at(uu, slot)] = sbuf[uu * 33 + s];
                }
                if (warp == 0 && s_slot[lane] >= 0 && s_nfr[lane] > 0) {
                    const int slot = s_slot[lane];
                    p.sm_active[slot] = sm_active;
                    p.sm_scount[slot] = sm_sc;
                    p.sm_ecount[slot] = sm_ec;
                    p.frames_done[slot] = sm_f0 + s_nfr[lane];
                }
            }
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == kProducerWarp) tc::tmem_dealloc(0u, 512);
    CVAD_PROF_NS(125);
}

}  // namespace tc5
}  // namespace cvad
