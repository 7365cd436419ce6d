// cvad_capi.cu -- host side of the C ABI declared in include/cutter_vad_b200.h.
//
// Owns: the engine object (one GPU, one stream), the upload of the weight streams that
// cvad_pack.cuh packs, the per-slot state arena in HBM, per-step scratch buffers and the
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
#include "cvad_pack.cuh"

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

bool is_g711(int pcm) { return pcm == CVAD_PCM_ULAW || pcm == CVAD_PCM_ALAW; }
size_t elem_size(int pcm) { return pcm == CVAD_PCM_F32 ? 4 : is_g711(pcm) ? 1 : 2; }

// ITU-T G.711 expansion of one code to its 16-bit linear value (audioop.ulaw2lin / alaw2lin with width 2): mu-law spans
// +-32124 (codes 0x7F and 0xFF are 0), A-law +-32256.  Integer arithmetic only, so the decoded sample linear / 32768.0f
// is exact and equals AudioUtils.pcm_to_float32 of the linear PCM.  The feeder builds its payload tables from it.
__host__ __device__ inline int g711_linear(int pcm, unsigned code) {
    if (pcm == CVAD_PCM_ULAW) {
        const unsigned u = ~code & 0xFFu;
        const int t = (int)(((u & 0x0Fu) << 3) + 0x84u) << ((u & 0x70u) >> 4);
        return (u & 0x80u) ? 0x84 - t : t - 0x84;
    }
    const unsigned a = (code & 0xFFu) ^ 0x55u;
    const unsigned seg = (a & 0x70u) >> 4;
    const int t = (int)((a & 0x0Fu) << 4);
    const int m = seg == 0 ? t + 8 : (t + 0x108) << (seg - 1);
    return (a & 0x80u) ? m : -m;
}

int rate_index(int src_rate) { return src_rate == 8000 ? 0 : src_rate == 24000 ? 1 : src_rate == 48000 ? 2 : -1; }
int rate_n_in(int src_rate) { return (int)((long long)src_rate * 512 / 16000); }

int validate_args(cvad_engine *e, const cvad_step_args *a) {
    if (!e) return CVAD_E_INVALID;
    if (!a) return fail(e, CVAD_E_INVALID, "step args are NULL");
    if (a->n_streams < 0 || a->n_streams > e->max_streams)
        return fail(e, CVAD_E_CAPACITY, "n_streams outside [0, max_streams]");
    if (a->n_streams > 0 && !a->audio) return fail(e, CVAD_E_INVALID, "Audio data is empty");
    if (a->pcm_format < 0 || a->pcm_format > CVAD_PCM_ALAW) return fail(e, CVAD_E_INVALID, "unknown pcm_format");
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

// A source rate's resampling operator, built and uploaded on its first use: R^T for resample_kernel (FP32 math), both
// tile forms for resample_tc_kernel (TC and TC16 math)
int ensure_rt(cvad_engine *e, int src_rate, cudaStream_t stream) {
    const int ri = rate_index(src_rate);
    if (e->rs_rt[ri]) return CVAD_OK;
    const std::vector<float> rt = build_resample_operator(rate_n_in(src_rate)).rt;
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->rs_rt[ri]), rt.size() * sizeof(float)));
    CU_TRY(e, cudaMemcpyAsync(e->rs_rt[ri], rt.data(), rt.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    CU_TRY(e, cudaStreamSynchronize(stream));
    return CVAD_OK;
}

int ensure_rt_tc(cvad_engine *e, int src_rate, cudaStream_t stream) {
    const int ri = rate_index(src_rate);
    if (e->rs_tc[ri]) return CVAD_OK;
    const ResampleOperator op = build_resample_operator(rate_n_in(src_rate));
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->rs_tc[ri]), op.tc.size()));
    CU_TRY(e, cudaMemcpyAsync(e->rs_tc[ri], op.tc.data(), op.tc.size(), cudaMemcpyHostToDevice, stream));
    CU_TRY(e, cudaMalloc(reinterpret_cast<void **>(&e->rs_h[ri]), op.tc16.size()));
    CU_TRY(e, cudaMemcpyAsync(e->rs_h[ri], op.tc16.data(), op.tc16.size(), cudaMemcpyHostToDevice, stream));
    e->rs_h_inv[ri] = op.inv;
    CU_TRY(e, cudaStreamSynchronize(stream));
    return CVAD_OK;
}

// `rates_mask`: which of the rate slots {8000, 24000, 48000, 16000} may occur in a->src_rates (bit r); callers
// that cannot look at the array (device-pointer steps) pass 0xF
// Does the model part of this step run as ONE fused kernel (the form cvad_step_device chains)?
bool fused_single_frame(const cvad_engine *e, const cvad_step_args *a) {
    return e->chain_steps && e->version == CVAD_MODEL_V5 && e->math != CVAD_MATH_FP32 && a->max_frames == 1 && e->fuse_single_frame &&
           a->channels <= 1 && !is_g711(a->pcm_format);
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
// PCM samples are converted to float first (the reference converts before it reaches the wrapper); G.711 codes are
// decoded to linear / 32768, so with C == 1 this is the G.711 decode alone.  Per-stream rates: stream i holds
// max_frames * 512 * src_rates[i] / 16000 sample frames.
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
            else if (pcm >= CVAD_PCM_ULAW) {
                x = (float)g711_linear(pcm, __ldg(reinterpret_cast<const unsigned char *>(audio) + base + c)) * (1.0f / 32768.0f);
            } else {
                x = (float)__ldg(reinterpret_cast<const short *>(audio) + base + c);
                x = pcm == 1 ? __fdiv_rn(x, 32767.0f) : x * (1.0f / 32768.0f);
            }
            acc = c == 0 ? x : __fadd_rn(acc, x);
        }
        out[(size_t)i * frames + k] = __fdiv_rn(acc, (float)C);
    }
}

// Enqueue the step's kernels.  Every pointer in `a` is a DEVICE pointer here.
// `chain` (cvad_step_device on a fused one-frame step): the caller enqueued no memset; see cvad_engine::d_evctr.
// `input_out` != nullptr (cvad_debug_input): run the input stages only, their output buffer filled with NaN first, and
// return the device address of the mono 16 kHz samples the model kernels would read in *input_out.
int launch_step(cvad_engine *e, const cvad_step_args *a, unsigned int *d_status, int commit, float *d_dbg,
                cudaStream_t stream, unsigned rates_mask = 0xFu, bool chain = false, const float **input_out = nullptr) {
    if (a->n_streams == 0 || a->max_frames == 0) return CVAD_OK;
    cvad_step_args a_mono;
    if (a->channels > 1 || is_g711(a->pcm_format)) {
        // stage -1: interleaved channels and / or G.711 codes -> mono float32 in HBM; everything downstream sees a mono
        // float stream
        if (chain) return fail(e, CVAD_E_INVALID, "internal: chained step with multi-channel or G.711 input");
        int rcf = flush_chain(e);
        if (rcf) return rcf;
        CU_TRY(e, cudaStreamWaitEvent(stream, e->last_done, 0));     // d_mono is shared by consecutive steps
        const int nch = std::max(a->channels, 1);
        const long long frames = a->src_rates ? std::min<long long>((long long)a->max_frames * 1536, a->stream_stride / nch)
                                              : (long long)(a->max_frames - 1) * a->hop + a->frame_len;
        int rcg = grow(e, e->d_mono, (size_t)a->n_streams * (size_t)frames * sizeof(float));
        if (rcg) return rcg;
        if (input_out) CU_TRY(e, cudaMemsetAsync(e->d_mono.p, 0xFF, (size_t)a->n_streams * (size_t)frames * sizeof(float), stream));
        const long long total = (long long)a->n_streams * frames;
        const int grid = (int)std::min<long long>((total + 255) / 256, (long long)e->num_sms * 16);
        downmix_kernel<<<grid, 256, 0, stream>>>(a->audio, a->pcm_format, a->stream_stride, nch, a->n_streams, frames,
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
        // fewer 64-stream tiles than SMs: share a tile's four output blocks among 2 or 4 CTAs
        const int rs_tiles = a->max_frames * ((a->n_streams + cvad::tc5::kRsTcTile - 1) / cvad::tc5::kRsTcTile);
        // (mixed-rate steps launch once per rate over that rate's share of the streams: assume an even share)
        const int n_rates = mixed ? std::max(1, __builtin_popcount(rates_mask & 7u)) : 1;
        const int rs_share = (rs_tiles + n_rates - 1) / n_rates;
        r.osplit = 4 * rs_share <= e->num_sms ? 4 : (2 * rs_share <= e->num_sms ? 2 : 1);
        const int grid_rs_tc = std::min(rs_tiles * r.osplit, e->num_sms);
        // run source rate `src_rate`'s resampler over `r`: every stream of the step, or the streams of r.list
        auto launch_rs = [&](int src_rate) -> int {
            const int ri = rate_index(src_rate);
            r.n_in = rate_n_in(src_rate);
            if (e->resampler == CVAD_RESAMPLE_FFT) {
                // one warp per two frames; 1 CTA per SM (shared memory), grid = enough CTAs for the launch's upper bound of units
                const long long units = (long long)a->max_frames * ((a->n_streams + 1) / 2);
                auto fft = [&](auto kernel, int wpc, int smem) {
                    const int g = (int)std::min<long long>((units + wpc - 1) / wpc, e->num_sms);
                    kernel<<<g, wpc * 32, smem, stream>>>(r, e->fft_T);
                };
                if (r.n_in == 256) fft(cvad::resample_fft_kernel<1>, cvad::RsFft<1>::WPC, cvad::RsFft<1>::kSmem);
                else if (r.n_in == 768) fft(cvad::resample_fft_kernel<3>, cvad::RsFft<3>::WPC, cvad::RsFft<3>::kSmem);
                else fft(cvad::resample_fft_kernel<6>, cvad::RsFft<6>::WPC, cvad::RsFft<6>::kSmem);
            } else if (e->math != CVAD_MATH_FP32) {
                if ((rc = ensure_rt_tc(e, src_rate, stream))) return rc;
                if (e->math == CVAD_MATH_TC16)
                    cvad::tc5::resample_tc_kernel<true><<<grid_rs_tc, cvad::tc5::kThreadsTC, cvad::tc5::kRsTcSmem, stream>>>(
                        r, e->rs_h[ri], e->rs_h_inv[ri]);
                else
                    cvad::tc5::resample_tc_kernel<false><<<grid_rs_tc, cvad::tc5::kThreadsTC, cvad::tc5::kRsTcSmem, stream>>>(
                        r, e->rs_tc[ri], 1.f);
            } else {
                if ((rc = ensure_rt(e, src_rate, stream))) return rc;
                r.rt = e->rs_rt[ri];
                cvad::resample_kernel<<<grid_rs, cvad::kThreads, cvad::kRsSmemBytes, stream>>>(r);
            }
            CU_TRY(e, cudaGetLastError());
            e->launches++;
            return CVAD_OK;
        };
        if (!mixed) {
            if ((rc = launch_rs(a->src_rate))) return rc;
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
                r.list = lists + (size_t)ri * n;
                r.count = counts + ri;
                if ((rc = launch_rs(kRates[ri]))) return rc;
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
// the d_mono layout for 16 kHz steps with a down-mix or G.711 decode; -1 = the step has no input stage (16 kHz mono
// float32 / int16).
long long input_stage_floats(const cvad_step_args *a) {
    if (a->n_streams == 0 || a->max_frames == 0) return 0;
    if (a->src_rates || (a->src_rate != 0 && a->src_rate != 16000)) return (long long)a->n_streams * a->max_frames * 512;
    if (a->channels > 1 || is_g711(a->pcm_format))
        return (long long)a->n_streams * ((long long)(a->max_frames - 1) * a->hop + a->frame_len);
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
        if (nf < 0) return fail(e, CVAD_E_INVALID, "cvad_debug_input: the step has no input stage (16 kHz mono float32 / int16)");
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
        Fp32Packed P = model_version == CVAD_MODEL_V5 ? pack_v5(weights) : pack_v4(weights);
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
    // the rule of cvad_import_states (validate_states_kernel), checked before anything is copied
    if (h)
        for (int j = 0; j < 128; ++j)
            if (!(std::fabs(h[j]) <= 2.f))
                return fail(e, CVAD_E_INVALID, "h[" + std::to_string(j) + "] is not within [-2, 2]; no state was changed");
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
