// cvad_capi.cu -- host side of the C ABI declared in include/cutter_vad_b200.h.
//
// Owns: the engine object (one GPU, one stream), weight repacking into the kernels'
// streaming layout, the per-slot state arena in HBM, per-step scratch buffers and the
// pinned staging used by the host-buffer entry point.  There is no CPU fallback: if no
// sm_100 device is present every compute entry point fails with CVAD_E_NOGPU.
#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/cutter_vad_b200.h"
#include <cmath>

#include "cvad_resample.cuh"
#include "cvad_tc.cuh"
#include "cvad_v4.cuh"
#include "cvad_v4tc.cuh"
#include "cvad_fftk.cuh"
#include "cvad_v5tc.cuh"

namespace {

thread_local std::string g_create_error;

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

}  // namespace

constexpr int kLanes = 4;   // host-buffer steps in flight (cvad_step_submit)

struct cvad_engine {
    int device = 0;
    int version = 0;
    int max_streams = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int64_t launches = 0;

    // weights
    float *w_fe = nullptr, *b_fe = nullptr, *w_rec = nullptr, *b_rec = nullptr, *w_dec = nullptr;
    // tensor-core path (v5 only): BF16x3 tile streams + the FP32 side tables
    int math = CVAD_MATH_FP32;
    bool v4_t2 = false;                // CVAD_MODEL_V4_8K: two LSTM time steps per frame
    bool fuse_single_frame = true;     // CVAD_FUSE=0 keeps the two-kernel form for one-frame steps (measurement)
    bool chain_steps = true;           // CVAD_CHAIN=0: device-pointer steps are not chained (memsets + event record per step; measurement)
    unsigned char *w_fe_tc = nullptr, *w_rec_tc = nullptr;
    unsigned char *w_fe_h = nullptr, *w_rec_h = nullptr;   // CVAD_MATH_TC16: two FP16 parts, per-layer scale
    float tc16_inv_w[8] = {0};
    float *nyq_w = nullptr, *b_rec_tc = nullptr;
    DevBuf d_feat_tc;
    DevBuf d_v4_mag;                   // v4 tensor-core path: |STFT| tiles between the two front-end kernels
    // double-precision FFT path (cvad_fftk.cuh): the resampler of every model, and v4's STFT (CVAD_MATH_FFT)
    double2 *fft_T = nullptr;          // master twiddle table exp(-2 pi i j / 1536)
    int resampler = CVAD_RESAMPLE_FFT;
    unsigned char *w_v4_corr = nullptr;// v4: (file basis - exact Hann x DFT basis) * 2^24 as 8 single-part BF16 tiles
    bool v4_fft_ok = false;            // the blob's basis IS Hann x DFT-256 up to float32 rounding (else CVAD_MATH_FFT is refused)
    DevBuf d_v4_fft;                   // exact-basis STFT tiles between v4_stft_fft_kernel and v4tc_stft_kernel<true>
    long long *d_prof = nullptr;       // 128 clock64 marks of CTA 0 (cvad_set_profile)
    // per-slot state
    float *h_state = nullptr, *c_state = nullptr;
    int *sm_active = nullptr, *sm_scount = nullptr, *sm_ecount = nullptr;
    long long *frames_done = nullptr;
    double *start_p = nullptr, *end_p = nullptr;
    int *n_start = nullptr, *n_end = nullptr;
    unsigned char *denoise = nullptr;
    // scratch shared by every step (kernels of consecutive steps are serialised by `last_done`)
    DevBuf d_status_dev, d_feat, d_dbg, d_cfg_slots;
    cudaEvent_t last_done = nullptr;   // recorded after the kernels of the most recent step
    // chained device-pointer steps (cvad_step_device, fused one-frame kernel): consecutive steps are launched with
    // programmatic stream serialization and NOTHING between the kernels -- no memset (the kernel clears its status words
    // and counts events in `d_evctr`), no event record (`last_done` is recorded lazily, when another stream needs it)
    int *d_evctr = nullptr;            // {event count of the step in flight, CTA ticket}; zero between steps
    // chained steps: [2] = chained steps completed (the last CTA of each counts), [3] = its CTA ticket; chain_seq = chained
    // steps launched.  A CTA that finds [2] behind its own sequence number was scheduled while the previous step still runs
    int chain_seq = 0;
    bool chain_pending = false;        // the tail of `chain_stream` is a chained kernel without a `last_done` record
    cudaStream_t chain_stream = nullptr;
    float *rs_rt[3] = {nullptr, nullptr, nullptr};  // R^T for 8 / 24 / 48 kHz, built on first use
    unsigned char *rs_tc[3] = {nullptr, nullptr, nullptr};  // the same operators as BF16x3 tiles for resample_tc_kernel
    unsigned char *rs_h[3] = {nullptr, nullptr, nullptr};   // ... and as two scaled FP16 parts (CVAD_MATH_TC16)
    float rs_h_inv[3] = {1.f, 1.f, 1.f};
    DevBuf d_mono;                     // interleaved multi-channel input averaged to mono (cvad_step_args::channels > 1)
    DevBuf d_res;                      // resampled 16 kHz audio of the step being launched
    DevBuf d_rate_lists;               // mixed-rate steps: [4][n] stream lists + 4 counters
    DevBuf d_state_blk, h_state_blk;   // cvad_get_state / cvad_export_states / cvad_import_states: records (device scratch, pinned host)
    uint64_t fingerprint = 0;          // cvad_model_fingerprint
    // host-buffer steps run on kLanes lanes so that later steps' H2D copies overlap earlier steps' kernels and D2H
    struct Lane {
        cudaStream_t stream = nullptr;
        DevBuf d_audio, d_slots, d_nframes, d_probs, d_flags, d_status, d_events, d_rates;
        int *d_nevents = nullptr;
        DevBuf h_in, h_out;             // pinned staging
        bool busy = false;
        cvad_step_args args{};          // caller's (host) argument block of the step in flight
        std::vector<int32_t> nfr_copy;  // n_frames as submitted (caller may reuse its array)
    } lanes[kLanes];
    int next_lane = 0;
    // optional per-kernel timing (bench): event triples (before FE, between, after REC)
    bool timing = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
};

namespace {

int fail(cvad_engine *e, int code, const std::string &msg) {
    if (e) e->err = msg; else g_create_error = msg;
    return code;
}

#define CU_TRY(e, call)                                                                        \
    do {                                                                                       \
        cudaError_t _st = (call);                                                              \
        if (_st != cudaSuccess)                                                                \
            return fail((e), CVAD_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_st)); \
    } while (0)

int grow(cvad_engine *e, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap) return CVAD_OK;
    if (b.p) CU_TRY(e, cudaFree(b.p));
    b.p = nullptr; b.cap = 0;
    size_t cap = bytes + bytes / 4 + 256;
    CU_TRY(e, cudaMalloc(&b.p, cap));
    b.cap = cap;
    return CVAD_OK;
}

int grow_host(cvad_engine *e, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap) return CVAD_OK;
    if (b.p) CU_TRY(e, cudaFreeHost(b.p));
    b.p = nullptr; b.cap = 0;
    size_t cap = bytes + bytes / 4 + 256;
    CU_TRY(e, cudaMallocHost(&b.p, cap));
    b.cap = cap;
    return CVAD_OK;
}

bool is_host_pinned_or_device(const void *p, bool want_device) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (want_device) return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
    return at.type == cudaMemoryTypeHost;
}

// ---- v5 weight repack (canonical blob order: see include/ and oracle/silero_ref.c)
struct V5Packed {
    std::vector<float> w_fe, b_fe, w_rec, b_rec, w_dec;
};

V5Packed pack_v5(const float *blob) {
    const float *basis = blob;                       // [258][256]
    const float *e0w = basis + 258 * 256;            // [128][129][3]
    const float *e0b = e0w + 128 * 129 * 3;
    const float *e1w = e0b + 128;                    // [64][128][3]
    const float *e1b = e1w + 64 * 128 * 3;
    const float *e2w = e1b + 64;                     // [64][64][3]
    const float *e2b = e2w + 64 * 64 * 3;
    const float *e3w = e2b + 64;                     // [128][64][3]
    const float *e3b = e3w + 128 * 64 * 3;
    const float *wih = e3b + 128;                    // [512][128]
    const float *whh = wih + 512 * 128;
    const float *bih = whh + 512 * 128;
    const float *bhh = bih + 512;
    const float *decw = bhh + 512;                   // [128]
    const float *decb = decw + 128;

    V5Packed P;
    P.w_fe.assign(cvad::kFeStreamFloats, 0.f);
    float *o = P.w_fe.data();
    for (int k = 0; k < 256; ++k)
        for (int n = 0; n < 256; ++n) {
            int row;
            if (n == 0) row = 0;
            else if (n == 1) row = 128;
            else row = (n & 1) ? 129 + (n >> 1) : (n >> 1);
            o[k * 256 + n] = basis[row * 256 + k];
        }
    o += 65536;
    for (int c = 0; c < 129; ++c)
        for (int t = 0; t < 3; ++t)
            for (int oc = 0; oc < 128; ++oc) o[(c * 3 + t) * 128 + oc] = e0w[(oc * 129 + c) * 3 + t];
    o += 129 * 384;
    for (int c = 0; c < 128; ++c)
        for (int t = 0; t < 3; ++t)
            for (int oc = 0; oc < 64; ++oc) o[(c * 3 + t) * 64 + oc] = e1w[(oc * 128 + c) * 3 + t];
    o += 128 * 192;
    for (int c = 0; c < 64; ++c)
        for (int t = 0; t < 2; ++t)
            for (int oc = 0; oc < 64; ++oc) o[(c * 2 + t) * 64 + oc] = e2w[(oc * 64 + c) * 3 + (t + 1)];
    o += 64 * 128;
    for (int c = 0; c < 64; ++c)
        for (int oc = 0; oc < 128; ++oc) o[c * 128 + oc] = e3w[(oc * 64 + c) * 3 + 1];

    P.b_fe.resize(cvad::kFeBiasFloats);
    std::memcpy(P.b_fe.data(), e0b, 128 * 4);
    std::memcpy(P.b_fe.data() + 128, e1b, 64 * 4);
    std::memcpy(P.b_fe.data() + 192, e2b, 64 * 4);
    std::memcpy(P.b_fe.data() + 256, e3b, 128 * 4);

    P.w_rec.resize(cvad::kRecStreamFloats);
    P.b_rec.resize(512);
    for (int n = 0; n < 512; ++n) {
        const int unit = n >> 2, gate = n & 3;
        const int row = gate * 128 + unit;
        for (int k = 0; k < 128; ++k) {
            P.w_rec[k * 512 + n] = wih[row * 128 + k];
            P.w_rec[(128 + k) * 512 + n] = whh[row * 128 + k];
        }
        P.b_rec[n] = bih[row] + bhh[row];
    }
    P.w_dec.resize(129);
    std::memcpy(P.w_dec.data(), decw, 128 * 4);
    P.w_dec[128] = decb[0];
    return P;
}


// ---- v5 tensor-core repack: every GEMM weight as three BF16 parts (w = w0 + w1 + w2 to 24 bits), cut into
// (rows x 64 K) tiles in the SWIZZLE_128B K-major operand layout, in the order cvad_v5tc.cuh consumes them.
struct V5TcPacked {
    std::vector<unsigned char> w_fe, w_rec;
    std::vector<float> nyq_w, b_rec;
};

uint16_t bf16_rn_bits(float x) {
    uint32_t u;
    std::memcpy(&u, &x, 4);
    const uint32_t r = ((u >> 16) & 1u) + 0x7FFFu;
    return (uint16_t)((u + r) >> 16);
}
float bf16_val(uint16_t b) {
    const uint32_t u = (uint32_t)b << 16;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}

// append the three part tiles of W(row, k), rows x [k0, k0 + 64)
template <typename F>
void emit_tiles(std::vector<unsigned char> &out, int rows, int k0, F W) {
    const size_t tile = (size_t)rows * 128;
    const size_t at = out.size();
    out.resize(at + 3 * tile, 0);
    for (int r = 0; r < rows; ++r)
        for (int kk = 0; kk < 64; ++kk) {
            float x = W(r, k0 + kk);
            const size_t off = (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 + (size_t)((((kk >> 3) ^ r) & 7) << 4) + (size_t)(kk & 7) * 2;
            for (int part = 0; part < 3; ++part) {
                const uint16_t b = bf16_rn_bits(x);
                std::memcpy(&out[at + part * tile + off], &b, 2);
                x -= bf16_val(b);
            }
        }
}

V5TcPacked pack_v5_tc(const float *blob) {
    const float *basis = blob;                       // [258][256]
    const float *e0w = basis + 258 * 256;            // [128][129][3]
    const float *e0b = e0w + 128 * 129 * 3;
    const float *e1w = e0b + 128;                    // [64][128][3]
    const float *e1b = e1w + 64 * 128 * 3;
    const float *e2w = e1b + 64;                     // [64][64][3]
    const float *e2b = e2w + 64 * 64 * 3;
    const float *e3w = e2b + 64;                     // [128][64][3]
    const float *e3b = e3w + 128 * 64 * 3;
    const float *wih = e3b + 128;                    // [512][128]
    const float *whh = wih + 512 * 128;
    const float *bih = whh + 512 * 128;
    const float *bhh = bih + 512;

    V5TcPacked P;
    P.w_fe.reserve(cvad::tc5::kFeStreamBytes);
    for (int blk = 0; blk < 2; ++blk)
        for (int kb = 0; kb < 4; ++kb)
            emit_tiles(P.w_fe, 128, kb * 64, [&](int m, int k) {
                const int row = blk == 0 ? m : (m == 0 ? 128 : 129 + m);
                return basis[row * 256 + k];
            });
    static const int taps0[3] = {1, 0, 2}, taps1[3] = {1, 2, 0};
    for (int kb = 0; kb < 2; ++kb)
        for (int ti = 0; ti < 3; ++ti)
            emit_tiles(P.w_fe, 128, kb * 64, [&](int o, int c) { return e0w[(o * 129 + c) * 3 + taps0[ti]]; });
    for (int kb = 0; kb < 2; ++kb)
        for (int ti = 0; ti < 3; ++ti)
            emit_tiles(P.w_fe, 64, kb * 64, [&](int o, int c) { return e1w[(o * 128 + c) * 3 + taps1[ti]]; });
    for (int tap = 1; tap <= 2; ++tap)
        emit_tiles(P.w_fe, 64, 0, [&](int o, int c) { return e2w[(o * 64 + c) * 3 + tap]; });
    emit_tiles(P.w_fe, 128, 0, [&](int o, int c) { return e3w[(o * 64 + c) * 3 + 1]; });

    for (int g = 0; g < 4; ++g)
        for (int kb = 0; kb < 4; ++kb)
            emit_tiles(P.w_rec, 128, kb * 64, [&](int u, int k) {
                const int row = g * 128 + u;
                return k < 128 ? wih[row * 128 + k] : whh[row * 128 + (k - 128)];
            });

    P.nyq_w.assign(128 * 4, 0.f);
    for (int o = 0; o < 128; ++o)
        for (int t = 0; t < 3; ++t) P.nyq_w[o * 4 + t] = e0w[(o * 129 + 128) * 3 + t];
    P.b_rec.resize(512);
    for (int n = 0; n < 512; ++n) P.b_rec[n] = bih[n] + bhh[n];
    return P;
}

// ---- v5 FP16-split repack (CVAD_MATH_TC16): the same tile order with TWO FP16 parts per weight, every layer scaled
// by the power of two that brings its largest weight to [2^14, 2^15) (inverse returned in inv_w: stft, enc0..3, W_ih, W_hh)
struct V5HPacked {
    std::vector<unsigned char> w_fe, w_rec;
    float inv_w[8] = {0};
};

template <typename F>
void emit_tiles_h(std::vector<unsigned char> &out, int rows, int k0, float scale, F W) {
    const size_t tile = (size_t)rows * 128;
    const size_t at = out.size();
    out.resize(at + 2 * tile, 0);
    for (int r = 0; r < rows; ++r)
        for (int kk = 0; kk < 64; ++kk) {
            float x = W(r, k0 + kk) * scale;
            const size_t off = (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 + (size_t)((((kk >> 3) ^ r) & 7) << 4) + (size_t)(kk & 7) * 2;
            for (int part = 0; part < 2; ++part) {
                const __half h = __float2half_rn(x);
                const unsigned short b = __half_as_ushort(h);
                std::memcpy(&out[at + part * tile + off], &b, 2);
                x -= __half2float(h);
            }
        }
}

float pow2_scale_for(float maxabs, float *inv) {
    if (!(maxabs > 0.f)) { *inv = 1.f; return 1.f; }
    int ex;
    std::frexp(maxabs, &ex);                 // maxabs = m * 2^ex, m in [0.5, 1)  ->  maxabs in [2^(ex-1), 2^ex)
    const float s = std::ldexp(1.0f, 15 - ex);
    *inv = std::ldexp(1.0f, ex - 15);
    return s;
}

V5HPacked pack_v5_tc16(const float *blob) {
    const float *basis = blob;                       // [258][256]
    const float *e0w = basis + 258 * 256;            // [128][129][3]
    const float *e0b = e0w + 128 * 129 * 3;
    const float *e1w = e0b + 128;                    // [64][128][3]
    const float *e1b = e1w + 64 * 128 * 3;
    const float *e2w = e1b + 64;                     // [64][64][3]
    const float *e2b = e2w + 64 * 64 * 3;
    const float *e3w = e2b + 64;                     // [128][64][3]
    const float *e3b = e3w + 128 * 64 * 3;
    const float *wih = e3b + 128;                    // [512][128]
    const float *whh = wih + 512 * 128;
    auto maxabs = [](const float *w, size_t n) { float m = 0.f; for (size_t i = 0; i < n; ++i) m = std::max(m, std::fabs(w[i])); return m; };
    V5HPacked P;
    const float s_stft = pow2_scale_for(maxabs(basis, 258 * 256), &P.inv_w[0]);
    const float s_e0 = pow2_scale_for(maxabs(e0w, 128 * 129 * 3), &P.inv_w[1]);
    const float s_e1 = pow2_scale_for(maxabs(e1w, 64 * 128 * 3), &P.inv_w[2]);
    const float s_e2 = pow2_scale_for(maxabs(e2w, 64 * 64 * 3), &P.inv_w[3]);
    const float s_e3 = pow2_scale_for(maxabs(e3w, 128 * 64 * 3), &P.inv_w[4]);
    // one scale for [W_ih | W_hh]: the recurrent kernel accumulates both halves of K in the same TMEM columns
    const float s_ih = pow2_scale_for(std::max(maxabs(wih, 512 * 128), maxabs(whh, 512 * 128)), &P.inv_w[5]);
    const float s_hh = s_ih;
    P.inv_w[6] = P.inv_w[5];
    P.w_fe.reserve(cvad::tc5::kFeStreamBytesH);
    for (int blk = 0; blk < 2; ++blk)
        for (int kb = 0; kb < 4; ++kb)
            emit_tiles_h(P.w_fe, 128, kb * 64, s_stft, [&](int m, int k) {
                const int row = blk == 0 ? m : (m == 0 ? 128 : 129 + m);
                return basis[row * 256 + k];
            });
    static const int taps0[3] = {1, 0, 2}, taps1[3] = {1, 2, 0};
    for (int kb = 0; kb < 2; ++kb)
        for (int ti = 0; ti < 3; ++ti)
            emit_tiles_h(P.w_fe, 128, kb * 64, s_e0, [&](int o, int c) { return e0w[(o * 129 + c) * 3 + taps0[ti]]; });
    for (int kb = 0; kb < 2; ++kb)
        for (int ti = 0; ti < 3; ++ti)
            emit_tiles_h(P.w_fe, 64, kb * 64, s_e1, [&](int o, int c) { return e1w[(o * 128 + c) * 3 + taps1[ti]]; });
    for (int tap = 1; tap <= 2; ++tap)
        emit_tiles_h(P.w_fe, 64, 0, s_e2, [&](int o, int c) { return e2w[(o * 64 + c) * 3 + tap]; });
    emit_tiles_h(P.w_fe, 128, 0, s_e3, [&](int o, int c) { return e3w[(o * 64 + c) * 3 + 1]; });
    for (int g = 0; g < 4; ++g)
        for (int kb = 0; kb < 4; ++kb)
            emit_tiles_h(P.w_rec, 128, kb * 64, kb < 2 ? s_ih : s_hh, [&](int u, int k) {
                const int row = g * 128 + u;
                return k < 128 ? wih[row * 128 + k] : whh[row * 128 + (k - 128)];
            });
    return P;
}

// v4 tensor-core STFT: the basis as 24 BF16x3 tiles (same row packing as v5's STFT block of pack_v5_tc)
std::vector<unsigned char> pack_v4_stft_tc(const float *blob) {
    const float *basis = blob;   // [258][256]
    std::vector<unsigned char> out;
    out.reserve(cvad::tc5::kV4StftStreamBytes);
    for (int blk = 0; blk < 2; ++blk)
        for (int kb = 0; kb < 4; ++kb)
            emit_tiles(out, 128, kb * 64, [&](int m, int k) {
                const int row = blk == 0 ? m : (m == 0 ? 128 : 129 + m);
                return basis[row * 256 + k];
            });
    return out;
}

// v4 FFT path: delta = (the file's float32 STFT basis) - (periodic Hann x DFT-256, evaluated in double) -- what the
// exact-basis FFT lacks.  Scaled by 2^24 it is O(1) and goes to the tensor cores as ONE BF16 part per weight
// (8 tiles, blk x kb, same row packing as pack_v4_stft_tc).  Returns max |delta| (7.7e-8 for the reference's file).
double pack_v4_stft_corr(const float *blob, const double2 *T, std::vector<unsigned char> &out) {
    const float *basis = blob;   // [258][256]: rows 0..128 real part, 129..257 imaginary part (-sin)
    double worst = 0.0;
    std::vector<float> delta(258 * 256);
    for (int row = 0; row < 258; ++row) {
        const int k = row < 129 ? row : row - 129;
        for (int n = 0; n < 256; ++n) {
            const double2 w = T[6 * ((k * n) & 255)];                 // exp(-2 pi i k n / 256)
            const double hann = 0.5 - 0.5 * T[6 * n].x;
            const double exact = hann * (row < 129 ? w.x : w.y);
            const double d = (double)basis[row * 256 + n] - exact;
            worst = std::max(worst, std::fabs(d));
            delta[row * 256 + n] = (float)(d * 16777216.0);
        }
    }
    out.clear();
    out.reserve(cvad::tc5::kV4CorrStreamBytes);
    for (int blk = 0; blk < 2; ++blk)
        for (int kb = 0; kb < 4; ++kb) {
            const size_t tile = 128 * 128, at = out.size();
            out.resize(at + tile, 0);
            for (int r = 0; r < 128; ++r)
                for (int kk = 0; kk < 64; ++kk) {
                    const int row = blk == 0 ? r : (r == 0 ? 128 : 129 + r);
                    const uint16_t b = bf16_rn_bits(delta[row * 256 + kb * 64 + kk]);
                    const size_t off = (size_t)(r >> 3) * 1024 + (size_t)(r & 7) * 128 + (size_t)((((kk >> 3) ^ r) & 7) << 4) + (size_t)(kk & 7) * 2;
                    std::memcpy(&out[at + off], &b, 2);
                }
        }
    return worst;
}

// ---- v4 weight repack (canonical blob order: oracle/silero_ref.c "Silero VAD v4")
V5Packed pack_v4(const float *blob) {
    const float *p = blob;
    auto take = [&](size_t n) { const float *r = p; p += n; return r; };
    const float *basis = take(258 * 256), *nfilt = take(7);
    const float *f_dw = take(258 * 5), *f_dwb = take(258), *f_pw = take(16 * 258), *f_pwb = take(16),
                *f_pj = take(16 * 258), *f_pjb = take(16);
    const float *c1 = take(256), *c1b = take(16);
    const float *e3_dw = take(80), *e3_dwb = take(16), *e3_pw = take(512), *e3_pwb = take(32), *e3_pj = take(512),
                *e3_pjb = take(32);
    const float *c2 = take(1024), *c2b = take(32);
    const float *e7_dw = take(160), *e7_dwb = take(32), *e7_pw = take(1024), *e7_pwb = take(32);
    const float *c3 = take(1024), *c3b = take(32);
    const float *e11_dw = take(160), *e11_dwb = take(32), *e11_pw = take(2048), *e11_pwb = take(64),
                *e11_pj = take(2048), *e11_pjb = take(64);
    const float *c4 = take(4096), *c4b = take(64);
    const float *l1w = take(16384), *l1r = take(16384), *l1b = take(512);
    const float *l2w = take(16384), *l2r = take(16384), *l2b = take(512);
    const float *decw = take(64), *decb = take(1);

    V5Packed P;
    P.w_fe.assign(cvad::kV4FeStreamFloats, 0.f);
    float *o = P.w_fe.data();
    for (int k = 0; k < 256; ++k)
        for (int n = 0; n < 256; ++n) {
            int row;
            if (n == 0) row = 0;
            else if (n == 1) row = 128;
            else row = (n & 1) ? 129 + (n >> 1) : (n >> 1);
            o[k * 256 + n] = basis[row * 256 + k];
        }
    o = P.w_fe.data() + cvad::kV4OffFirst;
    for (int c = 0; c < 258; ++c) {
        float *r = o + c * 40;
        for (int d = 0; d < 5; ++d) r[d] = f_dw[c * 5 + d];
        r[5] = f_dwb[c];
        for (int oc = 0; oc < 16; ++oc) { r[8 + oc] = f_pw[oc * 258 + c]; r[24 + oc] = f_pj[oc * 258 + c]; }
    }
    auto put_T = [](float *dst, const float *w, int cout, int cin) {  // w[co][ci] -> dst[ci][co]
        for (int co = 0; co < cout; ++co)
            for (int ci = 0; ci < cin; ++ci) dst[ci * cout + co] = w[co * cin + ci];
    };
    auto put_dw = [](float *dst, const float *w, int c) {             // w[c][5] -> dst[5][c]
        for (int ch = 0; ch < c; ++ch)
            for (int d = 0; d < 5; ++d) dst[d * c + ch] = w[ch * 5 + d];
    };
    o = P.w_fe.data() + cvad::kV4OffS0;
    put_T(o, c1, 16, 16); std::memcpy(o + 256, c1b, 64);
    put_dw(o + 272, e3_dw, 16); std::memcpy(o + 352, e3_dwb, 64);
    put_T(o + 368, e3_pw, 32, 16); std::memcpy(o + 880, e3_pwb, 128);
    put_T(o + 912, e3_pj, 32, 16); std::memcpy(o + 1424, e3_pjb, 128);
    put_T(o + 1456, c2, 32, 32); std::memcpy(o + 2480, c2b, 128);
    o = P.w_fe.data() + cvad::kV4OffS1;
    put_dw(o, e7_dw, 32); std::memcpy(o + 160, e7_dwb, 128);
    put_T(o + 192, e7_pw, 32, 32); std::memcpy(o + 1216, e7_pwb, 128);
    put_T(o + 1248, c3, 32, 32); std::memcpy(o + 2272, c3b, 128);
    o = P.w_fe.data() + cvad::kV4OffS2;
    put_dw(o, e11_dw, 32); std::memcpy(o + 160, e11_dwb, 128);
    put_T(o + 192, e11_pw, 64, 32); std::memcpy(o + 2240, e11_pwb, 256);
    o = P.w_fe.data() + cvad::kV4OffS3;
    put_T(o, e11_pj, 64, 32); std::memcpy(o + 2048, e11_pjb, 256); std::memcpy(o + 2112, c4b, 256);
    o = P.w_fe.data() + cvad::kV4OffS4;
    put_T(o, c4, 64, 64);
    o = P.w_fe.data() + cvad::kV4OffMisc;
    for (int oc = 0; oc < 16; ++oc) o[oc] = f_pwb[oc] + f_pjb[oc];
    for (int d = 0; d < 7; ++d) o[16 + d] = nfilt[d];
    P.b_fe.assign(4, 0.f);  // unused for v4

    P.w_rec.assign(cvad::kV4RecStreamFloats, 0.f);
    P.b_rec.assign(512, 0.f);
    const float *W[2] = {l1w, l2w}, *R[2] = {l1r, l2r}, *B[2] = {l1b, l2b};
    for (int l = 0; l < 2; ++l)
        for (int n = 0; n < 256; ++n) {
            const int unit = n >> 2, gate = n & 3;
            const int row = gate * 64 + unit;  // ONNX order i,o,f,c
            for (int k = 0; k < 64; ++k) {
                P.w_rec[(size_t)l * 32768 + k * 256 + n] = W[l][row * 64 + k];
                P.w_rec[(size_t)l * 32768 + (64 + k) * 256 + n] = R[l][row * 64 + k];
            }
            P.b_rec[l * 256 + n] = B[l][row] + B[l][256 + row];
        }
    P.w_dec.resize(65);
    std::memcpy(P.w_dec.data(), decw, 64 * 4);
    P.w_dec[64] = decb[0];
    return P;
}

template <typename T>
int upload(cvad_engine *e, T **dst, const std::vector<T> &src) {
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(dst), src.size() * sizeof(T)));
    CU_TRY(e, cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return CVAD_OK;
}

template <typename T>
int alloc_fill(cvad_engine *e, T **dst, size_t n, T value) {
    std::vector<T> tmp(n, value);
    return upload(e, dst, tmp);
}

size_t elem_size(int pcm) { return pcm == CVAD_PCM_F32 ? 4 : 2; }

int rate_index(int src_rate) { return src_rate == 8000 ? 0 : src_rate == 24000 ? 1 : src_rate == 48000 ? 2 : -1; }
int rate_n_in(int src_rate) { return (int)((long long)src_rate * 512 / 16000); }

int validate_args(cvad_engine *e, const cvad_step_args *a) {
    if (!e) return CVAD_E_INVALID;
    if (!a) return fail(e, CVAD_E_INVALID, "step args are NULL");
    if (a->n_streams < 0 || a->n_streams > e->max_streams)
        return fail(e, CVAD_E_CAPACITY, "n_streams outside [0, max_streams]");
    if (a->n_streams > 0 && !a->audio) return fail(e, CVAD_E_INVALID, "Audio data is empty");
    if (a->pcm_format < 0 || a->pcm_format > 2) return fail(e, CVAD_E_INVALID, "unknown pcm_format");
    if (a->max_frames < 0) return fail(e, CVAD_E_INVALID, "max_frames < 0");
    if (a->max_events < 0) return fail(e, CVAD_E_INVALID, "max_events < 0");
    if (a->channels < 0 || a->channels > 8) return fail(e, CVAD_E_INVALID, "channels outside [0, 8]");
    if (a->channels > 1 && a->stream_stride % a->channels != 0)
        return fail(e, CVAD_E_INVALID, "stream_stride must be a multiple of channels");
    if (a->src_rates) return CVAD_OK;   // per-stream rates: frame_len / hop / src_rate are not used
    if (a->frame_len < 1 || a->frame_len > 2048) return fail(e, CVAD_E_INVALID, "frame_len outside [1, 2048]");
    if (a->hop < 1) return fail(e, CVAD_E_INVALID, "hop < 1");
    if (a->src_rate != 0 && a->src_rate != 16000) {
        if (rate_index(a->src_rate) < 0) return fail(e, CVAD_E_INVALID, "src_rate must be 8000, 16000, 24000 or 48000");
        const int n_in = rate_n_in(a->src_rate);
        if (a->frame_len != n_in || a->hop != n_in)
            return fail(e, CVAD_E_INVALID,
                        "resampled streams: frame_len and hop must equal 512*src_rate/16000 source samples");
    }
    if (a->max_events < 0) return fail(e, CVAD_E_INVALID, "max_events < 0");
    return CVAD_OK;
}

// R^T[m][n] of scipy.signal.resample(x[N_in] -> 512), float64 closed form rounded to float32
// (formula and the two Nyquist rules: cvad_resample.cuh header).
void build_resample_rt(int n_in, std::vector<float> &rt) {
    const int num = 512;
    const double PI = 3.14159265358979323846;
    const int K = std::min(num, n_in) / 2;
    rt.assign((size_t)n_in * num, 0.f);
    for (int m = 0; m < n_in; ++m)
        for (int n = 0; n < num; ++n) {
            // theta/2 = pi (n/num - m/n_in), reduced with exact integer arithmetic
            const long long L = (long long)num * n_in;
            long long r = ((long long)n * n_in - (long long)m * num) % L;
            if (r < 0) r += L;
            const double half = PI * (double)r / (double)L;  // in [0, pi)
            double dk;
            if (r == 0) dk = 2.0 * K - 1.0;
            else dk = std::sin((2.0 * K - 1.0) * half) / std::sin(half);
            double nyq;
            if (n_in > num) nyq = 2.0 * std::cos(PI * (double)(((long long)num * m) % (2LL * n_in)) / (double)n_in) *
                                  ((n & 1) ? -1.0 : 1.0);
            else nyq = std::cos(2.0 * K * half);
            rt[(size_t)m * num + n] = (float)((dk + nyq) / (double)n_in);
        }
}

// Enqueue the two kernels.  Every pointer in `a` is a DEVICE pointer here.
int ensure_rt(cvad_engine *e, int src_rate, cudaStream_t stream) {
    const int ri = rate_index(src_rate), n_in = rate_n_in(src_rate);
    if (e->rs_rt[ri]) return CVAD_OK;
    std::vector<float> rt;
    build_resample_rt(n_in, rt);
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->rs_rt[ri]), rt.size() * sizeof(float)));
    CU_TRY(e, cudaMemcpyAsync(e->rs_rt[ri], rt.data(), rt.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    CU_TRY(e, cudaStreamSynchronize(stream));
    return CVAD_OK;
}

// R as BF16x3 tiles for resample_tc_kernel: K block kb-major, then output block (128 samples), then part
int ensure_rt_tc(cvad_engine *e, int src_rate, cudaStream_t stream) {
    const int ri = rate_index(src_rate), n_in = rate_n_in(src_rate);
    if (e->rs_tc[ri]) return CVAD_OK;
    std::vector<float> rt;
    build_resample_rt(n_in, rt);            // R^T [n_in][512]
    std::vector<unsigned char> tiles;
    tiles.reserve((size_t)512 * n_in * 6);
    for (int kb = 0; kb < n_in / 64; ++kb)
        for (int blk = 0; blk < 4; ++blk)
            emit_tiles(tiles, 128, kb * 64, [&](int r, int m) { return rt[(size_t)m * 512 + blk * 128 + r]; });
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->rs_tc[ri]), tiles.size()));
    CU_TRY(e, cudaMemcpyAsync(e->rs_tc[ri], tiles.data(), tiles.size(), cudaMemcpyHostToDevice, stream));
    // the FP16 two-part form of the same operator, scaled so that its largest entry lies in [2^14, 2^15)
    float mx = 0.f;
    for (float v : rt) mx = std::max(mx, std::fabs(v));
    const float sw = pow2_scale_for(mx, &e->rs_h_inv[ri]);
    std::vector<unsigned char> th;
    th.reserve((size_t)512 * n_in * 4);
    for (int kb = 0; kb < n_in / 64; ++kb)
        for (int blk = 0; blk < 4; ++blk)
            emit_tiles_h(th, 128, kb * 64, sw, [&](int r, int m) { return rt[(size_t)m * 512 + blk * 128 + r]; });
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->rs_h[ri]), th.size()));
    CU_TRY(e, cudaMemcpyAsync(e->rs_h[ri], th.data(), th.size(), cudaMemcpyHostToDevice, stream));
    CU_TRY(e, cudaStreamSynchronize(stream));
    return CVAD_OK;
}

// `rates_mask`: which of the rate slots {8000, 24000, 48000, 16000} may occur in a->src_rates (bit r); callers
// that cannot look at the array (device-pointer steps) pass 0xF
// Does the model part of this step run as ONE fused kernel (the form cvad_step_device chains)?
bool fused_single_frame(const cvad_engine *e, const cvad_step_args *a) {
    return e->chain_steps && e->version == CVAD_MODEL_V5 && e->math != CVAD_MATH_FP32 && a->max_frames == 1 && e->fuse_single_frame &&
           a->channels <= 1;
}

// a chained kernel sits at the tail of its stream without a `last_done` record: place the record now
int flush_chain(cvad_engine *e) {
    if (e->chain_pending) {
        e->chain_pending = false;
        CU_TRY(e, cudaEventRecord(e->last_done, e->chain_stream));
    }
    return CVAD_OK;
}

// AudioUtils.convert_to_mono (audio.py:193-208) on the device: out[i][k] = float32 mean over the C interleaved channels
// of sample frame k of stream i -- the channels added in order, the sum divided by C, as np.mean does for float32 input.
// PCM samples are converted to float first (the reference converts before it reaches the wrapper).  Per-stream rates:
// stream i holds max_frames * 512 * src_rates[i] / 16000 sample frames.
__global__ void downmix_kernel(const void *audio, int pcm, long long stride, int C, int n_streams, long long frames,
                               const int *src_rates, int max_frames, float *out) {
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long long)n_streams * frames;
         idx += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / frames);
        const long long k = idx - (long long)i * frames;
        if (src_rates && k >= (long long)max_frames * (512LL * src_rates[i] / 16000)) continue;
        const long long base = (long long)i * stride + k * C;
        float acc = 0.f;
        for (int c = 0; c < C; ++c) {
            float x;
            if (pcm == 0) x = __ldg(reinterpret_cast<const float *>(audio) + base + c);
            else {
                x = (float)__ldg(reinterpret_cast<const short *>(audio) + base + c);
                x = pcm == 1 ? __fdiv_rn(x, 32767.0f) : x * (1.0f / 32768.0f);
            }
            acc = c == 0 ? x : __fadd_rn(acc, x);
        }
        out[(size_t)i * frames + k] = __fdiv_rn(acc, (float)C);
    }
}

// `chain` (cvad_step_device on a fused one-frame step): the caller enqueued no memset; see cvad_engine::d_evctr.
// `input_out` != nullptr (cvad_debug_input): run the input stages only, their output buffer filled with NaN first, and
// return the device address of the mono 16 kHz samples the model kernels would read in *input_out.
int launch_step(cvad_engine *e, const cvad_step_args *a, unsigned int *d_status, int commit, float *d_dbg,
                cudaStream_t stream, unsigned rates_mask = 0xFu, bool chain = false, const float **input_out = nullptr) {
    if (a->n_streams == 0 || a->max_frames == 0) return CVAD_OK;
    cvad_step_args a_mono;
    if (a->channels > 1) {
        // stage -1: interleaved channels -> mono float32 in HBM; everything downstream sees a mono float stream
        if (chain) return fail(e, CVAD_E_INVALID, "internal: chained step with multi-channel input");
        int rcf = flush_chain(e);
        if (rcf) return rcf;
        CU_TRY(e, cudaStreamWaitEvent(stream, e->last_done, 0));     // d_mono is shared by consecutive steps
        const long long frames = a->src_rates ? std::min<long long>((long long)a->max_frames * 1536, a->stream_stride / a->channels)
                                              : (long long)(a->max_frames - 1) * a->hop + a->frame_len;
        int rcg = grow(e, e->d_mono, (size_t)a->n_streams * (size_t)frames * sizeof(float));
        if (rcg) return rcg;
        if (input_out) CU_TRY(e, cudaMemsetAsync(e->d_mono.p, 0xFF, (size_t)a->n_streams * (size_t)frames * sizeof(float), stream));
        const long long total = (long long)a->n_streams * frames;
        const int grid = (int)std::min<long long>((total + 255) / 256, (long long)e->num_sms * 16);
        downmix_kernel<<<grid, 256, 0, stream>>>(a->audio, a->pcm_format, a->stream_stride, a->channels, a->n_streams, frames,
                                                 a->src_rates, a->max_frames, static_cast<float *>(e->d_mono.p));
        CU_TRY(e, cudaGetLastError());
        e->launches++;
        a_mono = *a;
        a_mono.audio = e->d_mono.p;
        a_mono.pcm_format = CVAD_PCM_F32;
        a_mono.stream_stride = frames;
        a_mono.channels = 1;
        a = &a_mono;
    }
    // state and `feat` are shared: kernels of consecutive steps never overlap, whatever stream they use.  A chained
    // step behind a chained step on the same stream is ordered by the stream itself.
    if (!(chain && e->chain_pending && e->chain_stream == stream)) {
        int rcf = flush_chain(e);
        if (rcf) return rcf;
        CU_TRY(e, cudaStreamWaitEvent(stream, e->last_done, 0));
    }
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    const bool timed = e->timing && !d_dbg && !input_out;
    if (timed) {
        while (e->ev_pool.size() < e->ev_used + 3) {
            cudaEvent_t x;
            CU_TRY(e, cudaEventCreate(&x));
            e->ev_pool.push_back(x);
        }
        for (int i = 0; i < 3; ++i) ev[i] = e->ev_pool[e->ev_used + i];
        e->ev_used += 3;
        CU_TRY(e, cudaEventRecord(ev[0], stream));
    }
    const int n_stiles = (a->n_streams + cvad::kTile - 1) / cvad::kTile;
    const size_t feat_bytes = (size_t)a->max_frames * n_stiles * 128 * cvad::kTile * sizeof(float);   // v4: 64 x (1 or 2 time steps)
    int rc = grow(e, e->d_feat, feat_bytes);
    if (rc) return rc;

    cvad::V5Step p{};
    p.audio = a->audio;
    p.pcm = a->pcm_format;
    p.stride = a->stream_stride;
    p.frame_len = a->frame_len;
    p.hop = a->hop;
    const bool mixed = a->src_rates != nullptr;
    const bool resampled = mixed || (a->src_rate != 0 && a->src_rate != 16000);
    if (resampled) {
        // stage 0: source-rate chunks -> 16 kHz float frames in HBM; the model kernels then see native input
        if ((rc = grow(e, e->d_res, (size_t)a->n_streams * a->max_frames * 512 * sizeof(float)))) return rc;
        if (input_out) CU_TRY(e, cudaMemsetAsync(e->d_res.p, 0xFF, (size_t)a->n_streams * a->max_frames * 512 * sizeof(float), stream));
        cvad::ResampleStep r{};
        r.audio = a->audio; r.pcm = a->pcm_format; r.stride = a->stream_stride;
        r.n_streams = a->n_streams; r.n_stiles = n_stiles; r.max_frames = a->max_frames; r.n_frames = a->n_frames;
        r.out = static_cast<float *>(e->d_res.p);
        const int grid_rs = std::min(a->max_frames * n_stiles, e->num_sms);
        const bool rs_tc = e->math != CVAD_MATH_FP32;
        // fewer 64-stream tiles than SMs: share a tile's four output blocks among 2 or 4 CTAs
        const int rs_tiles = a->max_frames * ((a->n_streams + cvad::tc5::kRsTcTile - 1) / cvad::tc5::kRsTcTile);
        // (mixed-rate steps launch once per rate over that rate's share of the streams: assume an even share)
        const int n_rates = mixed ? std::max(1, __builtin_popcount(rates_mask & 7u)) : 1;
        const int rs_share = (rs_tiles + n_rates - 1) / n_rates;
        r.osplit = 4 * rs_share <= e->num_sms ? 4 : (2 * rs_share <= e->num_sms ? 2 : 1);
        const int grid_rs_tc = std::min(rs_tiles * r.osplit, e->num_sms);
        const bool rs_fft = e->resampler == CVAD_RESAMPLE_FFT;
        auto launch_rs_fft = [&](int n_in) {
            // one warp per two frames; 1 CTA per SM (shared memory), grid = enough CTAs for the launch's upper bound of units
            const long long units = (long long)a->max_frames * ((a->n_streams + 1) / 2);
            const double2 *T = e->fft_T;
            if (n_in == 256) {
                const int g = (int)std::min<long long>((units + cvad::RsFft<1>::WPC - 1) / cvad::RsFft<1>::WPC, e->num_sms);
                cvad::resample_fft_kernel<1><<<g, cvad::RsFft<1>::WPC * 32, cvad::RsFft<1>::kSmem, stream>>>(r, T);
            } else if (n_in == 768) {
                const int g = (int)std::min<long long>((units + cvad::RsFft<3>::WPC - 1) / cvad::RsFft<3>::WPC, e->num_sms);
                cvad::resample_fft_kernel<3><<<g, cvad::RsFft<3>::WPC * 32, cvad::RsFft<3>::kSmem, stream>>>(r, T);
            } else {
                const int g = (int)std::min<long long>((units + cvad::RsFft<6>::WPC - 1) / cvad::RsFft<6>::WPC, e->num_sms);
                cvad::resample_fft_kernel<6><<<g, cvad::RsFft<6>::WPC * 32, cvad::RsFft<6>::kSmem, stream>>>(r, T);
            }
        };
        if (!mixed) {
            r.n_in = rate_n_in(a->src_rate);
            if (rs_fft) {
                launch_rs_fft(r.n_in);
            } else if (rs_tc) {
                if ((rc = ensure_rt_tc(e, a->src_rate, stream))) return rc;
                const int ri = rate_index(a->src_rate);
                if (e->math == CVAD_MATH_TC16)
                    cvad::tc5::resample_tc_kernel<true><<<grid_rs_tc, cvad::tc5::kThreadsTC, cvad::tc5::kRsTcSmem, stream>>>(
                        r, e->rs_h[ri], e->rs_h_inv[ri]);
                else
                    cvad::tc5::resample_tc_kernel<false><<<grid_rs_tc, cvad::tc5::kThreadsTC, cvad::tc5::kRsTcSmem, stream>>>(
                        r, e->rs_tc[ri], 1.f);
            } else {
                if ((rc = ensure_rt(e, a->src_rate, stream))) return rc;
                r.rt = e->rs_rt[rate_index(a->src_rate)];
                cvad::resample_kernel<<<grid_rs, cvad::kThreads, cvad::kRsSmemBytes, stream>>>(r);
            }
            CU_TRY(e, cudaGetLastError());
            e->launches++;
        } else {
            // one launch per source rate over that rate's stream list (built on the device: no host round trip)
            const size_t n = (size_t)a->n_streams;
            if ((rc = grow(e, e->d_rate_lists, (4 * n + 4) * sizeof(int)))) return rc;
            int *lists = static_cast<int *>(e->d_rate_lists.p);
            int *counts = lists + 4 * n;
            CU_TRY(e, cudaMemsetAsync(counts, 0, 4 * sizeof(int), stream));
            cvad::rate_lists_kernel<<<(a->n_streams + 255) / 256, 256, 0, stream>>>(a->src_rates, a->n_streams, lists, counts,
                                                                                  d_status, chain ? 1 : 0);
            CU_TRY(e, cudaGetLastError());
            e->launches++;
            static const int kRates[3] = {8000, 24000, 48000};
            for (int ri = 0; ri < 3; ++ri) {
                if (!(rates_mask & (1u << ri))) continue;
                r.n_in = rate_n_in(kRates[ri]);
                r.list = lists + (size_t)ri * n;
                r.count = counts + ri;
                if (rs_fft) {
                    launch_rs_fft(r.n_in);
                } else if (rs_tc) {
                    if ((rc = ensure_rt_tc(e, kRates[ri], stream))) return rc;
                    if (e->math == CVAD_MATH_TC16)
                        cvad::tc5::resample_tc_kernel<true><<<grid_rs_tc, cvad::tc5::kThreadsTC, cvad::tc5::kRsTcSmem, stream>>>(
                            r, e->rs_h[ri], e->rs_h_inv[ri]);
                    else
                        cvad::tc5::resample_tc_kernel<false><<<grid_rs_tc, cvad::tc5::kThreadsTC, cvad::tc5::kRsTcSmem, stream>>>(
                            r, e->rs_tc[ri], 1.f);
                } else {
                    if ((rc = ensure_rt(e, kRates[ri], stream))) return rc;
                    r.rt = e->rs_rt[ri];
                    cvad::resample_kernel<<<grid_rs, cvad::kThreads, cvad::kRsSmemBytes, stream>>>(r);
                }
                CU_TRY(e, cudaGetLastError());
                e->launches++;
            }
            if (rates_mask & 8u) {
                r.n_in = 512;
                r.list = lists + 3 * n;
                r.count = counts + 3;
                cvad::passthrough_kernel<<<std::min(4 * e->num_sms, (a->n_streams * a->max_frames * 2) + 1), 256, 0, stream>>>(r);
                CU_TRY(e, cudaGetLastError());
                e->launches++;
            }
        }
        p.audio = e->d_res.p;
        p.pcm = CVAD_PCM_F32;
        p.stride = (long long)a->max_frames * 512;
        p.frame_len = 512;
        p.hop = 512;
    }
    if (input_out) {
        *input_out = static_cast<const float *>(p.audio);
        return CVAD_OK;
    }
    const size_t es = elem_size(p.pcm);
    const uintptr_t addr = reinterpret_cast<uintptr_t>(p.audio);
    p.vec_ok = (addr % (4 * es) == 0) && (p.stride % 4 == 0) && (p.hop % 4 == 0);
    p.n_streams = a->n_streams;
    p.n_stiles = n_stiles;
    p.max_frames = a->max_frames;
    p.max_streams = e->max_streams;
    p.slots = a->slots;
    p.n_frames = a->n_frames;
    p.denoise = e->denoise;
    p.status = d_status;
    p.feat = static_cast<float *>(e->d_feat.p);
    p.w_fe = e->w_fe; p.b_fe = e->b_fe; p.w_rec = e->w_rec; p.b_rec = e->b_rec; p.w_dec = e->w_dec;
    p.h_state = e->h_state; p.c_state = e->c_state;
    p.sm_active = e->sm_active; p.sm_scount = e->sm_scount; p.sm_ecount = e->sm_ecount;
    p.frames_done = e->frames_done;
    p.start_p = e->start_p; p.end_p = e->end_p; p.n_start = e->n_start; p.n_end = e->n_end;
    p.probs = a->probs_out;
    p.flags = a->flags_out;
    p.events = a->events_out;
    p.max_events = a->max_events;
    p.n_events = a->n_events_out;
    p.commit = commit;
    p.dbg = d_dbg;
    p.v4_t2 = e->v4_t2 ? 1 : 0;

    if (e->version == CVAD_MODEL_V5 && e->math != CVAD_MATH_FP32) {
        if ((rc = grow(e, e->d_feat_tc, (size_t)a->max_frames * n_stiles * cvad::tc5::kFeatTileBytes))) return rc;
        p.w_fe_tc = e->w_fe_tc; p.w_rec_tc = e->w_rec_tc; p.nyq_w = e->nyq_w; p.b_rec_tc = e->b_rec_tc;
        p.feat_tc = static_cast<unsigned char *>(e->d_feat_tc.p);
        p.prof = e->d_prof;
        const int grid = std::min(a->max_frames * n_stiles, e->num_sms);
        if (a->max_frames == 1 && !d_dbg && e->fuse_single_frame) {
            // one frame per stream: front end + LSTM step + state machine in ONE kernel (no hand-off, no second launch)
            if (chain) {
                p.status_zero = mixed ? 0 : 1;      // mixed rates: rate_lists_kernel has written every status word
                p.ev_ctr = a->n_events_out ? e->d_evctr : nullptr;
            }
            // chained steps: the grid may be scheduled while the previous step's kernel is still running (its CTAs set up
            // barriers and TMEM and prefetch weight tiles, then block in griddepcontrol.wait); not when timing events
            // sit between the kernels
            const bool overlap = chain && !timed;
            if (overlap && p.audio == a->audio) {        // (not when a kernel of this step produced the 16 kHz frames)
                // the CTAs that are scheduled early prefetch the step's audio into L2 while they wait (v5tc_frontend_kernel)
                p.step_ctr = e->d_evctr + 2;
                p.step_seq = e->chain_seq++;
            }
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3((unsigned)grid);
            cfg.blockDim = dim3((unsigned)cvad::tc5::kThreadsTC);
            cfg.dynamicSmemBytes = cvad::tc5::kFusedSmemTC;
            cfg.stream = stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = overlap ? 1 : 0;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            if (e->math == CVAD_MATH_TC16) {
                p.w_fe_h = e->w_fe_h; p.w_rec_h = e->w_rec_h;
                std::memcpy(p.tc16_inv_w, e->tc16_inv_w, sizeof(p.tc16_inv_w));
                if (p.prof) CU_TRY(e, cudaLaunchKernelEx(&cfg, cvad::tc5::v5tc_frontend_kernel<false, true, true, true>, p));
                else CU_TRY(e, cudaLaunchKernelEx(&cfg, cvad::tc5::v5tc_frontend_kernel<false, true, true, false>, p));
            } else {
                CU_TRY(e, cudaLaunchKernelEx(&cfg, cvad::tc5::v5tc_frontend_kernel<false, true, false>, p));
            }
            CU_TRY(e, cudaGetLastError());
            e->launches++;
            if (timed) {   // the whole step is the "front-end" interval, the "recurrent" interval is empty
                CU_TRY(e, cudaEventRecord(ev[1], stream));
                CU_TRY(e, cudaEventRecord(ev[2], stream));
            }
            if (overlap) {
                e->chain_pending = true;
                e->chain_stream = stream;
            } else {
                CU_TRY(e, cudaEventRecord(e->last_done, stream));
            }
            return CVAD_OK;
        }
        if (chain) return fail(e, CVAD_E_INVALID, "internal: chained step outside the fused one-frame path");
        const bool h16 = e->math == CVAD_MATH_TC16 && !d_dbg;
        if (h16) {
            p.w_fe_h = e->w_fe_h; p.w_rec_h = e->w_rec_h;
            std::memcpy(p.tc16_inv_w, e->tc16_inv_w, sizeof(p.tc16_inv_w));
        }
        if (d_dbg) cvad::tc5::v5tc_frontend_kernel<true, false><<<grid, cvad::tc5::kThreadsTC, cvad::tc5::kFeSmemTC, stream>>>(p);
        else if (h16) cvad::tc5::v5tc_frontend_kernel<false, false, true><<<grid, cvad::tc5::kThreadsTC, cvad::tc5::kFeSmemTCH, stream>>>(p);
        else cvad::tc5::v5tc_frontend_kernel<false, false><<<grid, cvad::tc5::kThreadsTC, cvad::tc5::kFeSmemTC, stream>>>(p);
        CU_TRY(e, cudaGetLastError());
        e->launches++;
        if (timed) CU_TRY(e, cudaEventRecord(ev[1], stream));
        if (!d_dbg) {
            // programmatic dependent launch: the recurrent grid is scheduled while the front end still runs and
            // overlaps its prologue with it (not when per-kernel timing events sit between the two launches)
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3((unsigned)n_stiles);
            cfg.blockDim = dim3((unsigned)cvad::tc5::kThreadsTC);
            cfg.dynamicSmemBytes = cvad::tc5::kRecSmemTC;
            cfg.stream = stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = timed ? 0 : 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            if (h16) CU_TRY(e, cudaLaunchKernelEx(&cfg, cvad::tc5::v5tc_recurrent_kernel<true>, p));
            else CU_TRY(e, cudaLaunchKernelEx(&cfg, cvad::tc5::v5tc_recurrent_kernel<false>, p));
            CU_TRY(e, cudaGetLastError());
            e->launches++;
        }
        if (timed) CU_TRY(e, cudaEventRecord(ev[2], stream));
        CU_TRY(e, cudaEventRecord(e->last_done, stream));
        return CVAD_OK;
    }

    const bool v4 = e->version == CVAD_MODEL_V4;
    const int n_tiles = a->max_frames * n_stiles * (v4 ? 2 : 1);
    const int grid_fe = std::min(n_tiles, e->num_sms);
    if (v4 && e->math == CVAD_MATH_FFT) {
        // STFT = double-precision FFT with the exact basis (float32 re / im through HBM) + one BF16 tensor-core product
        // with the basis' float32 rounding; the magnitude tiles then feed the FP32 front end like the TC path's
        if ((rc = grow(e, e->d_v4_fft, (size_t)n_tiles * cvad::kV4FftTile * sizeof(float)))) return rc;
        if ((rc = grow(e, e->d_v4_mag, (size_t)n_tiles * cvad::tc5::kV4MagTile * sizeof(float)))) return rc;
        cvad::v4_stft_fft_kernel<<<grid_fe, 512, cvad::kV4FftSmem, stream>>>(p, e->fft_T, static_cast<float *>(e->d_v4_fft.p));
        CU_TRY(e, cudaGetLastError());
        e->launches++;
        p.w_fe_tc = e->w_v4_corr;
        p.v4_fft = static_cast<const float *>(e->d_v4_fft.p);
        p.v4_mag = static_cast<float *>(e->d_v4_mag.p);
        cvad::tc5::v4tc_stft_kernel<true><<<grid_fe, cvad::tc5::kThreadsTC, cvad::tc5::kV4tcSmem, stream>>>(p);
        CU_TRY(e, cudaGetLastError());
        e->launches++;
    }
    if (v4 && e->math == CVAD_MATH_TC) {
        // the STFT (77 % of v4's MACs) on the tensor cores; |STFT| tiles go through HBM to the FP32 front end
        if ((rc = grow(e, e->d_v4_mag, (size_t)n_tiles * cvad::tc5::kV4MagTile * sizeof(float)))) return rc;
        p.w_fe_tc = e->w_fe_tc;
        p.v4_mag = static_cast<float *>(e->d_v4_mag.p);
        cvad::tc5::v4tc_stft_kernel<false><<<grid_fe, cvad::tc5::kThreadsTC, cvad::tc5::kV4tcSmem, stream>>>(p);
        CU_TRY(e, cudaGetLastError());
        e->launches++;
    }
    if (v4) cvad::v4_frontend_kernel<<<grid_fe, cvad::kThreads, cvad::kV4FeSmemBytes, stream>>>(p);
    else cvad::v5_frontend_kernel<<<grid_fe, cvad::kThreads, cvad::kFeSmemBytes, stream>>>(p);
    CU_TRY(e, cudaGetLastError());
    e->launches++;
    if (timed) CU_TRY(e, cudaEventRecord(ev[1], stream));
    if (!d_dbg) {
        if (v4) cvad::v4_recurrent_kernel<<<n_stiles, cvad::kThreads, cvad::kV4RecSmemBytes, stream>>>(p);
        else cvad::v5_recurrent_kernel<<<n_stiles, cvad::kThreads, cvad::kRecSmemBytes, stream>>>(p);
        CU_TRY(e, cudaGetLastError());
        e->launches++;
    }
    if (timed) CU_TRY(e, cudaEventRecord(ev[2], stream));
    CU_TRY(e, cudaEventRecord(e->last_done, stream));
    return CVAD_OK;
}

}  // namespace

namespace {
template <typename T>
__global__ void fill_slots_kernel(T *dst, const int *slots, int n, int all_n, T value, int ld, int rows) {
    // dst is [rows][ld]; set column slot (or every column when slots == nullptr) to value
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int count = slots ? n : all_n;
    if (idx >= count * rows) return;
    const int r = idx / count, k = idx - r * count;
    const int slot = slots ? slots[k] : k;
    dst[(size_t)r * ld + slot] = value;
}

// the same for the LSTM state (128 rows per slot, laid out by cvad::state_at)
__global__ void fill_state_kernel(float *dst, const int *slots, int n, int all_n, float value) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int count = slots ? n : all_n;
    if (idx >= count * 128) return;
    const int r = idx / count, k = idx - r * count;
    dst[cvad::state_at(r, slots ? slots[k] : k)] = value;
}
int fill_state(cvad_engine *e, float *dst, const int *d_slots, int n, float value) {
    const int count = d_slots ? n : e->max_streams;
    if (count == 0) return CVAD_OK;
    fill_state_kernel<<<(count * 128 + 255) / 256, 256, 0, e->stream>>>(dst, d_slots, n, e->max_streams, value);
    CU_TRY(e, cudaGetLastError());
    return CVAD_OK;
}

template <typename T>
int fill_slots(cvad_engine *e, T *dst, const int *d_slots, int n, T value, int rows) {
    const int count = d_slots ? n : e->max_streams;
    if (count == 0) return CVAD_OK;
    const int total = count * rows;
    fill_slots_kernel<T><<<(total + 255) / 256, 256, 0, e->stream>>>(dst, d_slots, n, e->max_streams, value,
                                                                    e->max_streams, rows);
    CU_TRY(e, cudaGetLastError());
    return CVAD_OK;
}

int stage_slots(cvad_engine *e, int n, const int32_t *slots, const int **d_slots) {
    *d_slots = nullptr;
    if (!slots) return CVAD_OK;
    for (int i = 0; i < n; ++i)
        if (slots[i] < 0 || slots[i] >= e->max_streams) return fail(e, CVAD_E_CAPACITY, "slot id out of range");
    int rc = grow(e, e->d_cfg_slots, (size_t)std::max(n, 1) * sizeof(int));
    if (rc) return rc;
    CU_TRY(e, cudaMemcpyAsync(e->d_cfg_slots.p, slots, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, e->stream));
    CU_TRY(e, cudaStreamSynchronize(e->stream));  // `slots` is pageable caller memory
    *d_slots = static_cast<const int *>(e->d_cfg_slots.p);
    return CVAD_OK;
}
}  // namespace

namespace {

int quiesce(cvad_engine *e) {
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    for (auto &ln : e->lanes) CU_TRY(e, cudaStreamSynchronize(ln.stream));
    return CVAD_OK;
}

// Floats cvad_debug_input writes for the (validated) step `a`: the d_res layout for resampled and mixed-rate steps,
// the d_mono layout for down-mix-only steps; -1 = the step has no input stage (16 kHz mono).
long long input_stage_floats(const cvad_step_args *a) {
    if (a->n_streams == 0 || a->max_frames == 0) return 0;
    if (a->src_rates || (a->src_rate != 0 && a->src_rate != 16000)) return (long long)a->n_streams * a->max_frames * 512;
    if (a->channels > 1) return (long long)a->n_streams * ((long long)(a->max_frames - 1) * a->hop + a->frame_len);
    return -1;
}

// Enqueue one host-buffer step on `ln` (H2D, kernels, D2H) without waiting for it.
// `dbg_out` != nullptr turns it into the debug dump (front end only, no commit); `input_out` != nullptr into
// cvad_debug_input (input stages only, no commit).
int step_submit_impl(cvad_engine *e, cvad_engine::Lane &ln, const cvad_step_args *a, float *dbg_out, size_t dbg_floats,
                     float *input_out, size_t input_floats);

// every failure after the lane was marked busy must release it again, whichever statement it comes from
int step_submit(cvad_engine *e, cvad_engine::Lane &ln, const cvad_step_args *a, float *dbg_out, size_t dbg_floats,
                float *input_out = nullptr, size_t input_floats = 0) {
    const int rc = step_submit_impl(e, ln, a, dbg_out, dbg_floats, input_out, input_floats);
    if (rc != CVAD_OK) ln.busy = false;
    return rc;
}

int step_submit_impl(cvad_engine *e, cvad_engine::Lane &ln, const cvad_step_args *a, float *dbg_out, size_t dbg_floats,
                     float *input_out, size_t input_floats) {
    int rc = validate_args(e, a);
    if (rc) return rc;
    if (input_out) {
        const long long nf = input_stage_floats(a);
        if (nf < 0) return fail(e, CVAD_E_INVALID, "cvad_debug_input: the step has no input stage (16 kHz mono)");
        if (input_floats < (size_t)nf) return fail(e, CVAD_E_CAPACITY, "cvad_debug_input: out too small");
    }
    CU_TRY(e, cudaSetDevice(e->device));
    const int n = a->n_streams, T = a->max_frames;
    ln.args = *a;
    ln.nfr_copy.clear();
    ln.busy = true;
    if (n == 0 || T == 0) return CVAD_OK;
    if (a->slots) {
        for (int i = 0; i < n; ++i)
            if (a->slots[i] < 0 || a->slots[i] >= e->max_streams) {
                ln.busy = false;
                return fail(e, CVAD_E_CAPACITY, "slot id out of range");
            }
    }
    if (a->n_frames) {
        for (int i = 0; i < n; ++i)
            if (a->n_frames[i] < 0 || a->n_frames[i] > T) {
                ln.busy = false;
                return fail(e, CVAD_E_INVALID, "n_frames[i] outside [0, max_frames]");
            }
        ln.nfr_copy.assign(a->n_frames, a->n_frames + n);
    }
    const size_t es = elem_size(a->pcm_format);
    const size_t nch = a->channels > 1 ? (size_t)a->channels : 1;     // rows are counted in ELEMENTS (sample frames x channels)
    size_t row = ((size_t)(T - 1) * a->hop + a->frame_len) * nch;
    size_t last_row = row;
    unsigned rates_mask = 0;
    if (a->src_rates) {
        row = 0;
        for (int i = 0; i < n; ++i) {
            const int r = cvad::rate_slot(a->src_rates[i]);
            if (r < 0) {
                ln.busy = false;
                return fail(e, CVAD_E_INVALID, "src_rates[i] must be 8000, 16000, 24000 or 48000");
            }
            rates_mask |= 1u << r;
            last_row = (size_t)T * (size_t)rate_n_in(a->src_rates[i]) * nch;
            row = std::max(row, last_row);
        }
    }
    // also for a single stream: stream_stride is then the only statement of the buffer's length the caller makes
    if (a->stream_stride < 0 || (size_t)a->stream_stride < row) {
        ln.busy = false;
        return fail(e, CVAD_E_INVALID, "stream_stride shorter than one stream's samples in this step");
    }
    // rows much wider than what this step reads (a caller stepping the first frames of a longer block): only the
    // samples that are read cross PCIe, as a 2-D copy into a dense device block
    const size_t row_al = (row + 7) & ~(size_t)7;
    const bool dense2d = n > 1 && !a->src_rates && nch == 1 && (size_t)a->stream_stride > row_al + row_al / 4;
    const size_t dev_stride = dense2d ? row_al : (size_t)a->stream_stride;
    const size_t audio_elems = dense2d ? (size_t)n * row_al : (size_t)(n - 1) * a->stream_stride + last_row;
    const size_t audio_bytes = audio_elems * es;
    auto bail = [&](int code) { ln.busy = false; return code; };

    // ---- device scratch of this lane
    if ((rc = grow(e, ln.d_audio, audio_bytes + 16)) || (rc = grow(e, ln.d_slots, (size_t)n * 4)) ||
        (rc = grow(e, ln.d_nframes, (size_t)n * 4)) || (rc = grow(e, ln.d_probs, (size_t)n * T * 4)) ||
        (rc = grow(e, ln.d_flags, (size_t)n * T)) || (rc = grow(e, ln.d_status, (size_t)n * 4)) ||
        (rc = grow(e, ln.d_events, (size_t)std::max(a->max_events, 1) * sizeof(cvad_event))) ||
        (a->src_rates && (rc = grow(e, ln.d_rates, (size_t)n * 4))))
        return bail(rc);

    // ---- host -> device (pinned caller memory goes straight; pageable memory is staged)
    const size_t small_in = (size_t)n * 12;
    const bool direct = is_host_pinned_or_device(a->audio, false);
    if ((rc = grow_host(e, ln.h_in, (direct ? 0 : audio_bytes) + small_in + 128))) return bail(rc);
    unsigned char *hin = static_cast<unsigned char *>(ln.h_in.p);
    int *h_slots = reinterpret_cast<int *>(hin);
    int *h_nfr = h_slots + n;
    if (a->slots) std::memcpy(h_slots, a->slots, (size_t)n * 4);
    if (a->n_frames) std::memcpy(h_nfr, a->n_frames, (size_t)n * 4);
    int *h_rates = h_nfr + n;
    if (a->src_rates) std::memcpy(h_rates, a->src_rates, (size_t)n * 4);
    const void *src_audio = a->audio;
    if (!direct) {
        unsigned char *stage = hin + ((small_in + 63) / 64) * 64;
        if (dense2d) {
            for (int i = 0; i < n; ++i)
                std::memcpy(stage + (size_t)i * row_al * es,
                            static_cast<const unsigned char *>(a->audio) + (size_t)i * a->stream_stride * es, row * es);
        } else {
            std::memcpy(stage, a->audio, audio_bytes);
        }
        src_audio = stage;
    }
    cudaStream_t st = ln.stream;
    if (direct && dense2d)
        CU_TRY(e, cudaMemcpy2DAsync(ln.d_audio.p, row_al * es, src_audio, (size_t)a->stream_stride * es, row * es, (size_t)n,
                                    cudaMemcpyHostToDevice, st));
    else
        CU_TRY(e, cudaMemcpyAsync(ln.d_audio.p, src_audio, audio_bytes, cudaMemcpyHostToDevice, st));
    if (a->slots) CU_TRY(e, cudaMemcpyAsync(ln.d_slots.p, h_slots, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    if (a->n_frames) CU_TRY(e, cudaMemcpyAsync(ln.d_nframes.p, h_nfr, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    if (a->src_rates) CU_TRY(e, cudaMemcpyAsync(ln.d_rates.p, h_rates, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU_TRY(e, cudaMemsetAsync(ln.d_status.p, 0, (size_t)n * 4, st));
    CU_TRY(e, cudaMemsetAsync(ln.d_nevents, 0, sizeof(int), st));

    cvad_step_args d = *a;
    d.audio = ln.d_audio.p;
    d.stream_stride = (int64_t)dev_stride;
    d.slots = a->slots ? static_cast<const int32_t *>(ln.d_slots.p) : nullptr;
    d.n_frames = a->n_frames ? static_cast<const int32_t *>(ln.d_nframes.p) : nullptr;
    d.src_rates = a->src_rates ? static_cast<const int32_t *>(ln.d_rates.p) : nullptr;
    d.probs_out = static_cast<float *>(ln.d_probs.p);
    d.flags_out = static_cast<uint8_t *>(ln.d_flags.p);
    d.status_out = nullptr;
    d.events_out = static_cast<cvad_event *>(ln.d_events.p);
    d.n_events_out = ln.d_nevents;

    if (input_out) {
        const float *d_in = nullptr;
        rc = launch_step(e, &d, static_cast<unsigned int *>(ln.d_status.p), 0, nullptr, st, a->src_rates ? rates_mask : 0xFu,
                         false, &d_in);
        if (rc) return bail(rc);
        CU_TRY(e, cudaMemcpyAsync(input_out, d_in, (size_t)input_stage_floats(a) * sizeof(float), cudaMemcpyDeviceToHost, st));
        return CVAD_OK;
    }
    float *d_dbg = nullptr;
    if (dbg_out) {
        const size_t nd = e->version == CVAD_MODEL_V4 ? (size_t)cvad::kV4DbgFloats : (size_t)cvad::kDbgFloats;
        if (dbg_floats < nd) return bail(fail(e, CVAD_E_CAPACITY, "dbg_out too small"));
        if ((rc = grow(e, e->d_dbg, nd * 4))) return bail(rc);
        d_dbg = static_cast<float *>(e->d_dbg.p);
        CU_TRY(e, cudaMemsetAsync(d_dbg, 0, nd * 4, st));
    }
    rc = launch_step(e, &d, static_cast<unsigned int *>(ln.d_status.p), dbg_out ? 0 : 1, d_dbg, st,
                     a->src_rates ? rates_mask : 0xFu);
    if (rc) return bail(rc);
    if (dbg_out) {
        const size_t nd = e->version == CVAD_MODEL_V4 ? (size_t)cvad::kV4DbgFloats : (size_t)cvad::kDbgFloats;
        CU_TRY(e, cudaMemcpyAsync(dbg_out, d_dbg, nd * 4, cudaMemcpyDeviceToHost, st));
        return CVAD_OK;
    }

    // ---- device -> host into this lane's pinned block (unpacked by step_collect)
    const size_t probs_b = (size_t)n * T * 4, flags_b = (size_t)n * T, status_b = (size_t)n * 4;
    const size_t ev_b = (size_t)a->max_events * sizeof(cvad_event);
    const size_t out_total = probs_b + flags_b + status_b + 64 + ev_b + 256;
    if ((rc = grow_host(e, ln.h_out, out_total))) return bail(rc);
    unsigned char *ho = static_cast<unsigned char *>(ln.h_out.p);
    if (a->probs_out) CU_TRY(e, cudaMemcpyAsync(ho, ln.d_probs.p, probs_b, cudaMemcpyDeviceToHost, st));
    CU_TRY(e, cudaMemcpyAsync(ho + probs_b, ln.d_status.p, status_b, cudaMemcpyDeviceToHost, st));
    CU_TRY(e, cudaMemcpyAsync(ho + probs_b + status_b, ln.d_nevents, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (a->flags_out)
        CU_TRY(e, cudaMemcpyAsync(ho + probs_b + status_b + 64 + ((ev_b + 63) / 64) * 64, ln.d_flags.p, flags_b,
                                  cudaMemcpyDeviceToHost, st));
    return CVAD_OK;
}

// Wait for the step in flight on `ln` and unpack its results into the caller's buffers.
int step_collect(cvad_engine *e, cvad_engine::Lane &ln, bool is_dbg) {
    if (!ln.busy) return fail(e, CVAD_E_INVALID, "no step in flight on this ticket");
    ln.busy = false;
    CU_TRY(e, cudaSetDevice(e->device));
    const cvad_step_args *a = &ln.args;
    const int n = a->n_streams, T = a->max_frames;
    if (a->n_events_out) *a->n_events_out = 0;
    if (n == 0 || T == 0) return CVAD_OK;
    CU_TRY(e, cudaStreamSynchronize(ln.stream));
    if (is_dbg) return e->version == CVAD_MODEL_V4 ? cvad::kV4DbgFloats : cvad::kDbgFloats;
    const size_t probs_b = (size_t)n * T * 4, status_b = (size_t)n * 4;
    const size_t ev_b = (size_t)a->max_events * sizeof(cvad_event);
    unsigned char *ho = static_cast<unsigned char *>(ln.h_out.p);
    float *h_probs = reinterpret_cast<float *>(ho);
    unsigned int *h_status = reinterpret_cast<unsigned int *>(ho + probs_b);
    int *h_nev = reinterpret_cast<int *>(ho + probs_b + status_b);
    cvad_event *h_ev = reinterpret_cast<cvad_event *>(ho + probs_b + status_b + 64);
    unsigned char *h_flags = ho + probs_b + status_b + 64 + ((ev_b + 63) / 64) * 64;
    const int nev = *h_nev;
    if (a->n_events_out) *a->n_events_out = nev;
    if (a->events_out && a->max_events > 0 && nev > 0) {
        const int take = std::min(nev, a->max_events);
        CU_TRY(e, cudaMemcpy(h_ev, ln.d_events.p, (size_t)take * sizeof(cvad_event), cudaMemcpyDeviceToHost));
        std::sort(h_ev, h_ev + take, [](const cvad_event &x, const cvad_event &y) {
            if (x.stream != y.stream) return x.stream < y.stream;
            if (x.frame != y.frame) return x.frame < y.frame;
            return x.kind < y.kind;
        });
        std::memcpy(a->events_out, h_ev, (size_t)take * sizeof(cvad_event));
    }
    const bool ragged = !ln.nfr_copy.empty();
    bool any_bad = false;
    for (int i = 0; i < n && !any_bad; ++i) any_bad = h_status[i] != 0u;
    if (!ragged && !any_bad) {
        if (a->probs_out) std::memcpy(a->probs_out, h_probs, probs_b);
        if (a->flags_out) std::memcpy(a->flags_out, h_flags, (size_t)n * T);
    } else {
        // frames that never ran (ragged n_frames, rejected streams) read as 0
        for (int i = 0; i < n; ++i) {
            const int nf = (h_status[i] != 0u) ? 0 : (ragged ? ln.nfr_copy[i] : T);
            if (a->probs_out) {
                std::memcpy(a->probs_out + (size_t)i * T, h_probs + (size_t)i * T, (size_t)nf * 4);
                for (int j = nf; j < T; ++j) a->probs_out[(size_t)i * T + j] = 0.f;
            }
            if (a->flags_out) {
                std::memcpy(a->flags_out + (size_t)i * T, h_flags + (size_t)i * T, (size_t)nf);
                for (int j = nf; j < T; ++j) a->flags_out[(size_t)i * T + j] = 0;
            }
        }
    }
    if (a->status_out)
        for (int i = 0; i < n; ++i) a->status_out[i] = (uint8_t)(h_status[i] & 0xffu);
    return CVAD_OK;
}
}  // namespace

extern "C" {

int cvad_abi_version(void) { return CVAD_ABI_VERSION; }

int cvad_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        cudaDeviceProp pr{};
        if (cudaGetDeviceProperties(&pr, d) == cudaSuccess && pr.major == 10) ++ok;
    }
    return ok;
}

const char *cvad_last_error(const cvad_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int cvad_create(const float *weights, size_t n_weight_floats, int model_version, int max_streams, int device,
                cvad_engine **out) {
    if (!out) return fail(nullptr, CVAD_E_INVALID, "out is NULL");
    *out = nullptr;
    if (!weights) return fail(nullptr, CVAD_E_INVALID, "weights is NULL");
    if (max_streams < 1) return fail(nullptr, CVAD_E_INVALID, "max_streams < 1");
    const bool v4_8k = model_version == CVAD_MODEL_V4_8K;
    if (v4_8k) model_version = CVAD_MODEL_V4;   // same kernels and blob layout, T = 2 at the LSTM
    if (model_version != CVAD_MODEL_V5 && model_version != CVAD_MODEL_V4)
        return fail(nullptr, CVAD_E_INVALID, "model_version must be CVAD_MODEL_V5, CVAD_MODEL_V4 or CVAD_MODEL_V4_8K");
    if (model_version == CVAD_MODEL_V5 && n_weight_floats != CVAD_V5_WEIGHT_FLOATS)
        return fail(nullptr, CVAD_E_WEIGHTS, "v5 weight blob must hold 309633 floats");
    if (model_version == CVAD_MODEL_V4 && n_weight_floats != CVAD_V4_WEIGHT_FLOATS)
        return fail(nullptr, CVAD_E_WEIGHTS, "v4 weight blob must hold 155908 floats");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, CVAD_E_NOGPU, "no CUDA device visible (this engine has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return fail(nullptr, CVAD_E_INVALID, "device index out of range");
    cudaDeviceProp pr{};
    if (cudaGetDeviceProperties(&pr, device) != cudaSuccess || pr.major != 10)
        return fail(nullptr, CVAD_E_NOGPU, "device is not sm_100 (kernels are built for sm_100a only)");

    cvad_engine *e = new cvad_engine();
    e->device = device;
    e->version = model_version;
    e->v4_t2 = v4_8k;
    e->max_streams = max_streams;
    e->num_sms = pr.multiProcessorCount;
    {
        // cvad_model_fingerprint: FNV-1a 64 over the model version (little-endian int32) and the weight blob's bytes
        const int32_t mv = v4_8k ? CVAD_MODEL_V4_8K : model_version;
        uint64_t hsh = 0xcbf29ce484222325ull;
        auto mix = [&hsh](const unsigned char *p, size_t n) {
            for (size_t i = 0; i < n; ++i) { hsh ^= p[i]; hsh *= 0x100000001b3ull; }
        };
        mix(reinterpret_cast<const unsigned char *>(&mv), sizeof(mv));
        mix(reinterpret_cast<const unsigned char *>(weights), n_weight_floats * sizeof(float));
        e->fingerprint = hsh;
    }
    auto bail = [&](int rc) {
        g_create_error = e->err;
        cvad_destroy(e);
        return rc;
    };
#define CR_TRY(call)                                                              \
    do {                                                                          \
        cudaError_t _st = (call);                                                 \
        if (_st != cudaSuccess) {                                                 \
            e->err = std::string(#call) + ": " + cudaGetErrorString(_st);         \
            return bail(CVAD_E_CUDA);                                             \
        }                                                                         \
    } while (0)
    CR_TRY(cudaSetDevice(device));
    CR_TRY(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    e->own_stream = true;
    CR_TRY(cudaFuncSetAttribute(cvad::v5_frontend_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::kFeSmemBytes));
    CR_TRY(cudaFuncSetAttribute(cvad::v5_recurrent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::kRecSmemBytes));
    CR_TRY(cudaFuncSetAttribute(cvad::resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::kRsSmemBytes));
    CR_TRY(cudaFuncSetAttribute(cvad::v4_frontend_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::kV4FeSmemBytes));
    CR_TRY(cudaFuncSetAttribute(cvad::v4_recurrent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::kV4RecSmemBytes));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_frontend_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kFeSmemTC));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_frontend_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kFeSmemTC));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_frontend_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kFusedSmemTC));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_frontend_kernel<false, true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kFusedSmemTC));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_frontend_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kFusedSmemTC));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_frontend_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kFeSmemTCH));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_recurrent_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kRecSmemTC));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v5tc_recurrent_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kRecSmemTC));
    if (model_version == CVAD_MODEL_V5) {
        V5TcPacked T = pack_v5_tc(weights);
        if (T.w_fe.size() != cvad::tc5::kFeStreamBytes || T.w_rec.size() != cvad::tc5::kRecStreamBytes) {
            e->err = "internal: tensor-core weight stream has the wrong size";
            return bail(CVAD_E_WEIGHTS);
        }
        int rc;
        if ((rc = upload(e, &e->w_fe_tc, T.w_fe)) || (rc = upload(e, &e->w_rec_tc, T.w_rec)) ||
            (rc = upload(e, &e->nyq_w, T.nyq_w)) || (rc = upload(e, &e->b_rec_tc, T.b_rec)))
            return bail(rc);
        {
            V5HPacked H = pack_v5_tc16(weights);
            if (H.w_fe.size() != cvad::tc5::kFeStreamBytesH || H.w_rec.size() != cvad::tc5::kRecStreamBytesH) {
                e->err = "internal: FP16 weight stream has the wrong size";
                return bail(CVAD_E_WEIGHTS);
            }
            if ((rc = upload(e, &e->w_fe_h, H.w_fe)) || (rc = upload(e, &e->w_rec_h, H.w_rec))) return bail(rc);
            std::memcpy(e->tc16_inv_w, H.inv_w, sizeof(e->tc16_inv_w));
        }
        const char *m = std::getenv("CVAD_MATH");
        e->math = (m && std::strcmp(m, "fp32") == 0) ? CVAD_MATH_FP32
                  : (m && std::strcmp(m, "tc") == 0) ? CVAD_MATH_TC : CVAD_MATH_TC16;
        const char *fz = std::getenv("CVAD_FUSE");
        e->fuse_single_frame = !(fz && std::strcmp(fz, "0") == 0);
        const char *ch = std::getenv("CVAD_CHAIN");
        e->chain_steps = !(ch && std::strcmp(ch, "0") == 0);
    }
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v4tc_stft_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kV4tcSmem));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::v4tc_stft_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kV4tcSmem));
    CR_TRY(cudaFuncSetAttribute(cvad::v4_stft_fft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cvad::kV4FftSmem));
    CR_TRY(cudaFuncSetAttribute(cvad::resample_fft_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::RsFft<1>::kSmem));
    CR_TRY(cudaFuncSetAttribute(cvad::resample_fft_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::RsFft<3>::kSmem));
    CR_TRY(cudaFuncSetAttribute(cvad::resample_fft_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::RsFft<6>::kSmem));
    std::vector<double2> fftT(cvad::fft::kMaster);
    cvad::fft::build_master(fftT.data());
    {
        int rc;
        if ((rc = upload(e, &e->fft_T, fftT))) return bail(rc);
        const char *rsm = std::getenv("CVAD_RESAMPLE");
        e->resampler = (rsm && std::strcmp(rsm, "gemm") == 0) ? CVAD_RESAMPLE_GEMM : CVAD_RESAMPLE_FFT;
    }
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::resample_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kRsTcSmem));
    CR_TRY(cudaFuncSetAttribute(cvad::tc5::resample_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)cvad::tc5::kRsTcSmem));
    if (model_version == CVAD_MODEL_V4) {
        std::vector<unsigned char> T = pack_v4_stft_tc(weights);
        int rc;
        if ((rc = upload(e, &e->w_fe_tc, T))) return bail(rc);
        // v4 feeds log(1 + 2^20 |STFT|) into the network, which amplifies the tensor cores' (truncating) FP32
        // accumulation on weak bins, so the tensor-core STFT (CVAD_MATH_TC) is opt-in although it is the fastest v4 path.
        // The STFT as a double-precision FFT plus a tensor-core correction for the basis' float32 rounding
        // (CVAD_MATH_FFT) is the closest to the float64 evaluation of the graph of the three; it is the default
        // whenever the blob's basis is Hann x DFT-256 (true for both sub-models of the reference's file)
        std::vector<unsigned char> C;
        const double worst = pack_v4_stft_corr(weights, fftT.data(), C);
        e->v4_fft_ok = worst <= 2.0e-7;
        if (e->v4_fft_ok && (rc = upload(e, &e->w_v4_corr, C))) return bail(rc);
        const char *m = std::getenv("CVAD_MATH");
        e->math = (m && std::strcmp(m, "tc") == 0) ? CVAD_MATH_TC
                  : (m && std::strcmp(m, "fp32") == 0) || !e->v4_fft_ok ? CVAD_MATH_FP32 : CVAD_MATH_FFT;
    }
    {
        V5Packed P = model_version == CVAD_MODEL_V5 ? pack_v5(weights) : pack_v4(weights);
        int rc;
        if ((rc = upload(e, &e->w_fe, P.w_fe)) || (rc = upload(e, &e->b_fe, P.b_fe)) ||
            (rc = upload(e, &e->w_rec, P.w_rec)) || (rc = upload(e, &e->b_rec, P.b_rec)) ||
            (rc = upload(e, &e->w_dec, P.w_dec)))
            return bail(rc);
    }
    {
        const size_t ms = (size_t)max_streams;
        int rc;
        const size_t ms8 = ((size_t)ms + 7) / 8 * 8;       // state rows are grouped by 8 slots (cvad::state_at)
        if ((rc = alloc_fill<float>(e, &e->h_state, 128 * ms8, 0.f)) ||
            (rc = alloc_fill<float>(e, &e->c_state, 128 * ms8, 0.f)) ||
            (rc = alloc_fill<int>(e, &e->sm_active, ms, 0)) || (rc = alloc_fill<int>(e, &e->sm_scount, ms, 0)) ||
            (rc = alloc_fill<int>(e, &e->sm_ecount, ms, 0)) ||
            (rc = alloc_fill<long long>(e, &e->frames_done, ms, 0)) ||
            (rc = alloc_fill<double>(e, &e->start_p, ms, 0.7)) || (rc = alloc_fill<double>(e, &e->end_p, ms, 0.7)) ||
            (rc = alloc_fill<int>(e, &e->n_start, ms, 10)) || (rc = alloc_fill<int>(e, &e->n_end, ms, 50)) ||
            (rc = alloc_fill<unsigned char>(e, &e->denoise, ms, 1)))
            return bail(rc);
    }
    CR_TRY(cudaEventCreateWithFlags(&e->last_done, cudaEventDisableTiming));
    CR_TRY(cudaMalloc(reinterpret_cast<void **>(&e->d_evctr), 4 * sizeof(int)));
    CR_TRY(cudaMemset(e->d_evctr, 0, 4 * sizeof(int)));
    for (auto &ln : e->lanes) {
        CR_TRY(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking));
        CR_TRY(cudaMalloc(reinterpret_cast<void **>(&ln.d_nevents), sizeof(int)));
    }
#undef CR_TRY
    *out = e;
    return CVAD_OK;
}

int cvad_destroy(cvad_engine *e) {
    if (!e) return CVAD_OK;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (auto &ln : e->lanes)
        if (ln.stream) cudaStreamSynchronize(ln.stream);
    void *ptrs[] = {e->w_fe, e->b_fe, e->w_rec, e->b_rec, e->w_dec, e->h_state, e->c_state, e->sm_active,
                    e->sm_scount, e->sm_ecount, e->frames_done, e->start_p, e->end_p, e->n_start, e->n_end,
                    e->denoise, e->d_status_dev.p, e->d_feat.p, e->d_dbg.p, e->d_cfg_slots.p, e->d_res.p,
                    e->rs_rt[0], e->rs_rt[1], e->rs_rt[2], e->rs_h[0], e->rs_h[1], e->rs_h[2], e->w_fe_tc, e->w_rec_tc, e->w_fe_h, e->w_rec_h, e->nyq_w, e->b_rec_tc,
                    e->d_feat_tc.p, e->d_prof, e->d_evctr, e->d_rate_lists.p, e->d_v4_mag.p, e->rs_tc[0], e->rs_tc[1], e->rs_tc[2],
                    e->fft_T, e->w_v4_corr, e->d_v4_fft.p, e->d_mono.p, e->d_state_blk.p};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    if (e->h_state_blk.p) cudaFreeHost(e->h_state_blk.p);
    for (auto &ln : e->lanes) {
        if (ln.stream) cudaStreamSynchronize(ln.stream);
        void *lp[] = {ln.d_audio.p, ln.d_slots.p, ln.d_nframes.p, ln.d_probs.p, ln.d_flags.p, ln.d_status.p,
                      ln.d_events.p, ln.d_nevents, ln.d_rates.p};
        for (void *p : lp)
            if (p) cudaFree(p);
        if (ln.h_in.p) cudaFreeHost(ln.h_in.p);
        if (ln.h_out.p) cudaFreeHost(ln.h_out.p);
        if (ln.stream) cudaStreamDestroy(ln.stream);
    }
    if (e->last_done) cudaEventDestroy(e->last_done);
    for (cudaEvent_t x : e->ev_pool) cudaEventDestroy(x);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return CVAD_OK;
}

int cvad_set_math(cvad_engine *e, int math) {
    if (!e) return CVAD_E_INVALID;
    if (math != CVAD_MATH_FP32 && math != CVAD_MATH_TC && math != CVAD_MATH_TC16 && math != CVAD_MATH_FFT)
        return fail(e, CVAD_E_INVALID, "math must be CVAD_MATH_FP32, CVAD_MATH_TC, CVAD_MATH_TC16 or CVAD_MATH_FFT");
    if (math == CVAD_MATH_TC16 && e->version != CVAD_MODEL_V5)
        return fail(e, CVAD_E_INVALID, "CVAD_MATH_TC16 exists for the v5 model only");
    if (math == CVAD_MATH_FFT && (e->version != CVAD_MODEL_V4 || !e->v4_fft_ok))
        return fail(e, CVAD_E_INVALID, "CVAD_MATH_FFT exists for v4 models whose STFT basis is Hann x DFT-256");
    e->math = math;
    return CVAD_OK;
}

int cvad_set_resampler(cvad_engine *e, int resampler) {
    if (!e) return CVAD_E_INVALID;
    if (resampler != CVAD_RESAMPLE_FFT && resampler != CVAD_RESAMPLE_GEMM)
        return fail(e, CVAD_E_INVALID, "resampler must be CVAD_RESAMPLE_FFT or CVAD_RESAMPLE_GEMM");
    e->resampler = resampler;
    return CVAD_OK;
}

int cvad_get_resampler(const cvad_engine *e) { return e ? e->resampler : CVAD_E_INVALID; }

int cvad_get_math(const cvad_engine *e) { return e ? e->math : CVAD_E_INVALID; }

int cvad_set_profile(cvad_engine *e, int enabled) {
    if (!e) return CVAD_E_INVALID;
    if (enabled && !e->d_prof) {
        CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->d_prof), (128 + 512) * sizeof(long long)));
        CU_TRY(e, cudaMemset(e->d_prof, 0, (128 + 512) * sizeof(long long)));
    } else if (!enabled && e->d_prof) {
        CU_TRY(e, cudaDeviceSynchronize());
        cudaFree(e->d_prof);
        e->d_prof = nullptr;
    }
    return CVAD_OK;
}

int cvad_read_profile_chain(cvad_engine *e, long long *out512) {
    if (!e || !out512 || !e->d_prof) return CVAD_E_INVALID;
    CU_TRY(e, cudaSetDevice(e->device));
    { int rcq = quiesce(e); if (rcq) return rcq; }
    CU_TRY(e, cudaMemcpy(out512, e->d_prof + 128, 512 * sizeof(long long), cudaMemcpyDeviceToHost));
    return CVAD_OK;
}

int cvad_read_profile(cvad_engine *e, long long *out128) {
    if (!e || !out128 || !e->d_prof) return CVAD_E_INVALID;
    CU_TRY(e, cudaDeviceSynchronize());
    CU_TRY(e, cudaMemcpy(out128, e->d_prof, 128 * sizeof(long long), cudaMemcpyDeviceToHost));
    return CVAD_OK;
}

int cvad_set_stream(cvad_engine *e, void *cuda_stream) {
    if (!e) return CVAD_E_INVALID;
    CU_TRY(e, cudaSetDevice(e->device));
    if (e->stream) CU_TRY(e, cudaStreamSynchronize(e->stream));
    { int rcf = flush_chain(e); if (rcf) return rcf; }
    if (cuda_stream == nullptr) {
        if (!e->own_stream) {
            CU_TRY(e, cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
            e->own_stream = true;
        }
        return CVAD_OK;
    }
    if (e->own_stream && e->stream) CU_TRY(e, cudaStreamDestroy(e->stream));
    e->own_stream = false;
    e->stream = static_cast<cudaStream_t>(cuda_stream);
    return CVAD_OK;
}

int cvad_reset(cvad_engine *e, int n, const int32_t *slots) {
    if (!e) return CVAD_E_INVALID;
    if (slots && n < 0) return fail(e, CVAD_E_INVALID, "n < 0");
    CU_TRY(e, cudaSetDevice(e->device));
    const int *ds = nullptr;
    int rc = quiesce(e);
    if (rc) return rc;
    if ((rc = stage_slots(e, n, slots, &ds))) return rc;
    if ((rc = fill_state(e, e->h_state, ds, n, 0.f)) || (rc = fill_state(e, e->c_state, ds, n, 0.f)) ||
        (rc = fill_slots<int>(e, e->sm_active, ds, n, 0, 1)) || (rc = fill_slots<int>(e, e->sm_scount, ds, n, 0, 1)) ||
        (rc = fill_slots<int>(e, e->sm_ecount, ds, n, 0, 1)) ||
        (rc = fill_slots<long long>(e, e->frames_done, ds, n, 0ll, 1)))
        return rc;
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    return CVAD_OK;
}

int cvad_configure(cvad_engine *e, int n, const int32_t *slots, double vad_start_probability,
                   double vad_end_probability, int voice_start_frame_count, int voice_end_frame_count,
                   int enable_denoising) {
    if (!e) return CVAD_E_INVALID;
    if (slots && n < 0) return fail(e, CVAD_E_INVALID, "n < 0");
    if (voice_start_frame_count < 1 || voice_end_frame_count < 1)
        return fail(e, CVAD_E_INVALID, "frame counts must be >= 1");
    if (!(vad_start_probability >= 0.0 && vad_start_probability <= 1.0) ||
        !(vad_end_probability >= 0.0 && vad_end_probability <= 1.0))
        return fail(e, CVAD_E_INVALID, "probabilities must be within [0, 1]");
    CU_TRY(e, cudaSetDevice(e->device));
    const int *ds = nullptr;
    int rc = quiesce(e);
    if (rc) return rc;
    if ((rc = stage_slots(e, n, slots, &ds))) return rc;
    if ((rc = fill_slots<double>(e, e->start_p, ds, n, vad_start_probability, 1)) ||
        (rc = fill_slots<double>(e, e->end_p, ds, n, vad_end_probability, 1)) ||
        (rc = fill_slots<int>(e, e->n_start, ds, n, voice_start_frame_count, 1)) ||
        (rc = fill_slots<int>(e, e->n_end, ds, n, voice_end_frame_count, 1)) ||
        (rc = fill_slots<unsigned char>(e, e->denoise, ds, n, (unsigned char)(enable_denoising ? 1 : 0), 1)))
        return rc;
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    return CVAD_OK;
}

}  // extern "C"

#include "cvad_state.cuh"

extern "C" {

// cvad_get_state is export_states_kernel for one record: one small kernel packs the slot's words, ONE device-to-host copy
// brings them over (the per-call path of the drop-in wrapper reads the state after every call: seven separate synchronous
// copies were 0.1 ms of its 0.4 ms).
int cvad_get_state(cvad_engine *e, int slot, float *h, float *c, int32_t *sm, int64_t *frames_done) {
    if (!e) return CVAD_E_INVALID;
    if (slot < 0 || slot >= e->max_streams) return fail(e, CVAD_E_CAPACITY, "slot id out of range");
    CU_TRY(e, cudaSetDevice(e->device));
    { int rcq = quiesce(e); if (rcq) return rcq; }
    const size_t bytes = sizeof(cvad_stream_state);
    int rc = grow(e, e->d_state_blk, bytes);
    if (rc) return rc;
    if ((rc = grow_host(e, e->h_state_blk, bytes))) return rc;
    export_states_kernel<<<1, 256, 0, e->stream>>>(state_arrays(e), nullptr, slot, 1, static_cast<uint32_t *>(e->d_state_blk.p));
    CU_TRY(e, cudaGetLastError());
    CU_TRY(e, cudaMemcpyAsync(e->h_state_blk.p, e->d_state_blk.p, bytes, cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    const cvad_stream_state *r = static_cast<const cvad_stream_state *>(e->h_state_blk.p);
    if (h) std::memcpy(h, r->h, 128 * sizeof(float));
    if (c) std::memcpy(c, r->c, 128 * sizeof(float));
    if (sm) {
        sm[0] = r->is_voice_active; sm[1] = r->voice_start_frame_count; sm[2] = r->voice_end_frame_count; sm[3] = 0;
    }
    if (frames_done) *frames_done = r->frames_done;
    return CVAD_OK;
}

int cvad_set_state(cvad_engine *e, int slot, const float *h, const float *c, const int32_t *sm) {
    if (!e) return CVAD_E_INVALID;
    if (slot < 0 || slot >= e->max_streams) return fail(e, CVAD_E_CAPACITY, "slot id out of range");
    CU_TRY(e, cudaSetDevice(e->device));
    { int rcq = quiesce(e); if (rcq) return rcq; }
    const size_t pitch = 8 * sizeof(float), at = cvad::state_at(0, slot);
    if (h) CU_TRY(e, cudaMemcpy2D(e->h_state + at, pitch, h, sizeof(float), sizeof(float), 128, cudaMemcpyHostToDevice));
    if (c) CU_TRY(e, cudaMemcpy2D(e->c_state + at, pitch, c, sizeof(float), sizeof(float), 128, cudaMemcpyHostToDevice));
    if (sm) {
        CU_TRY(e, cudaMemcpy(e->sm_active + slot, &sm[0], sizeof(int), cudaMemcpyHostToDevice));
        CU_TRY(e, cudaMemcpy(e->sm_scount + slot, &sm[1], sizeof(int), cudaMemcpyHostToDevice));
        CU_TRY(e, cudaMemcpy(e->sm_ecount + slot, &sm[2], sizeof(int), cudaMemcpyHostToDevice));
    }
    return CVAD_OK;
}

int cvad_sync(cvad_engine *e) {
    if (!e) return CVAD_E_INVALID;
    CU_TRY(e, cudaSetDevice(e->device));
    return quiesce(e);
}

int64_t cvad_launch_count(const cvad_engine *e) { return e ? e->launches : 0; }

int cvad_set_timing(cvad_engine *e, int enabled) {
    if (!e) return CVAD_E_INVALID;
    e->timing = enabled != 0;
    e->ev_used = 0;
    return CVAD_OK;
}

int cvad_read_timing(cvad_engine *e, double *frontend_ms, double *recurrent_ms, int *n_steps) {
    if (!e) return CVAD_E_INVALID;
    CU_TRY(e, cudaSetDevice(e->device));
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    double fe = 0.0, rec = 0.0;
    const size_t n = e->ev_used / 3;
    for (size_t i = 0; i < n; ++i) {
        float a = 0.f, b = 0.f;
        CU_TRY(e, cudaEventElapsedTime(&a, e->ev_pool[3 * i], e->ev_pool[3 * i + 1]));
        CU_TRY(e, cudaEventElapsedTime(&b, e->ev_pool[3 * i + 1], e->ev_pool[3 * i + 2]));
        fe += a; rec += b;
    }
    if (frontend_ms) *frontend_ms = fe;
    if (recurrent_ms) *recurrent_ms = rec;
    if (n_steps) *n_steps = (int)n;
    e->ev_used = 0;
    return CVAD_OK;
}

void *cvad_alloc_pinned(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void cvad_free_pinned(void *p) {
    if (p) cudaFreeHost(p);
}

int cvad_step_device(cvad_engine *e, const cvad_step_args *a) {
    int rc = validate_args(e, a);
    if (rc) return rc;
    CU_TRY(e, cudaSetDevice(e->device));
    if (a->n_streams == 0 || a->max_frames == 0) return CVAD_OK;
    unsigned int *d_status = nullptr;
    if (a->status_out) {
        // status is one byte per stream at the ABI; the kernels use a 32-bit word per stream
        return fail(e, CVAD_E_INVALID, "cvad_step_device: status_out must be NULL (use cvad_step for status)");
    }
    if ((size_t)a->n_streams * sizeof(unsigned int) > e->d_status_dev.cap) {
        // (re)allocation frees the old buffer: nothing of an earlier step may still be using it
        if ((rc = quiesce(e))) return rc;
        if ((rc = grow(e, e->d_status_dev, (size_t)a->n_streams * sizeof(unsigned int)))) return rc;
    }
    d_status = static_cast<unsigned int *>(e->d_status_dev.p);
    // fused one-frame steps are chained kernel to kernel: the kernel (or, with per-stream rates, rate_lists_kernel)
    // clears the status words and events are counted in the engine's counter, so nothing but kernels is enqueued
    const bool chain = fused_single_frame(e, a);
    if (!chain) {
        CU_TRY(e, cudaMemsetAsync(d_status, 0, (size_t)a->n_streams * sizeof(unsigned int), e->stream));
        if (a->n_events_out) CU_TRY(e, cudaMemsetAsync(a->n_events_out, 0, sizeof(int), e->stream));
    }
    return launch_step(e, a, d_status, 1, nullptr, e->stream, 0xFu, chain);
}

int cvad_resample_matrix(int src_rate, float *rt_out, size_t n_floats) {
    if (rate_index(src_rate) < 0 || !rt_out) return CVAD_E_INVALID;
    const int n_in = rate_n_in(src_rate);
    if (n_floats < (size_t)n_in * 512) return CVAD_E_CAPACITY;
    std::vector<float> rt;
    build_resample_rt(n_in, rt);
    std::memcpy(rt_out, rt.data(), rt.size() * sizeof(float));
    return n_in;
}

int cvad_step_submit(cvad_engine *e, const cvad_step_args *a, int *ticket) {
    if (!e) return CVAD_E_INVALID;
    if (!ticket) return fail(e, CVAD_E_INVALID, "ticket is NULL");
    const int lane = e->next_lane;
    if (e->lanes[lane].busy) return fail(e, CVAD_E_CAPACITY, "four steps are already in flight: collect one first");
    int rc = step_submit(e, e->lanes[lane], a, nullptr, 0);
    if (rc) return rc;
    *ticket = lane;
    e->next_lane = (lane + 1) % kLanes;
    return CVAD_OK;
}

int cvad_step_collect(cvad_engine *e, int ticket) {
    if (!e) return CVAD_E_INVALID;
    if (ticket < 0 || ticket >= kLanes) return fail(e, CVAD_E_INVALID, "bad ticket");
    return step_collect(e, e->lanes[ticket], false);
}

int cvad_step(cvad_engine *e, const cvad_step_args *a) {
    int ticket = 0;
    int rc = cvad_step_submit(e, a, &ticket);
    if (rc) return rc;
    return cvad_step_collect(e, ticket);
}

int cvad_debug_dump(cvad_engine *e, const cvad_step_args *a, float *dbg_out, size_t dbg_floats) {
    if (!e) return CVAD_E_INVALID;
    if (!dbg_out) return fail(e, CVAD_E_INVALID, "dbg_out is NULL");
    int rc = quiesce(e);
    if (rc) return rc;
    cvad_engine::Lane &ln = e->lanes[0];
    for (auto &l : e->lanes)
        if (l.busy) return fail(e, CVAD_E_INVALID, "steps in flight");
    rc = step_submit(e, ln, a, dbg_out, dbg_floats);
    if (rc) return rc;
    return step_collect(e, ln, true);
}

int cvad_debug_input(cvad_engine *e, const cvad_step_args *a, float *out, size_t n_floats) {
    if (!e) return CVAD_E_INVALID;
    if (!out) return fail(e, CVAD_E_INVALID, "out is NULL");
    int rc = quiesce(e);
    if (rc) return rc;
    cvad_engine::Lane &ln = e->lanes[0];
    for (auto &l : e->lanes)
        if (l.busy) return fail(e, CVAD_E_INVALID, "steps in flight");
    rc = step_submit(e, ln, a, nullptr, 0, out, n_floats);
    if (rc) return rc;
    rc = step_collect(e, ln, true);
    if (rc < 0) return rc;
    return (int)input_stage_floats(a);
}

}  // extern "C"

#include "cvad_feeder.cuh"
