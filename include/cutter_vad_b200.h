/*
 * cutter_vad_b200.h -- C ABI of the B200-native Silero-VAD stream engine.
 *
 * This is the drop-in boundary for the reference's hot path: every entry point
 * below replaces a piece of Picurit/cutter-vad's per-frame Python/onnxruntime
 * pipeline (paths relative to the reference root):
 *
 *   cvad_create          <- ort.InferenceSession(model_path, ...)         src/real_time_vad/core/silero_model.py:321-325
 *                           + SileroVADModel._reset_states                silero_model.py:384-401
 *   cvad_step            <- the hot loop of VADWrapper._process_audio_frames
 *                           src/real_time_vad/core/vad_wrapper.py:627-644, i.e. per frame:
 *                             AudioUtils.split_into_frames                src/real_time_vad/utils/audio.py:164-190
 *                             AudioUtils.validate_audio_data              audio.py:211-231
 *                             AudioUtils.denoise_audio                    audio.py:104-121
 *                             SileroVADModel._prepare_audio_input         silero_model.py:449-474
 *                             session.run (v5 / v4 16 kHz graph)          silero_model.py:433
 *                             _extract_probability / _update_states       silero_model.py:501-537
 *                             VADProcessor._process_voice_state           silero_model.py:790-923
 *                           and, where the north star adds it,
 *                             AudioUtils.resample_audio                   audio.py:19-55
 *                             AudioUtils.convert_to_mono (channels > 1)   audio.py:193-208
 *   cvad_configure       <- VADConfig thresholds                          src/real_time_vad/core/config.py:54-94
 *                           as applied by VADWrapper.set_thresholds       vad_wrapper.py:367-419
 *   cvad_reset           <- VADProcessor.reset / SileroVADModel.reset     silero_model.py:951-968, :539-546
 *   cvad_get_state/set   <- SileroVADModel.model_state (numpy h/c)        silero_model.py:264-267, :526-537
 *   cvad_last_error      <- the VADError family's messages                src/real_time_vad/core/exceptions.py
 *   cvad_export/import_states, cvad_feeder_export/import: stream snapshots, which the reference has no equivalent of
 *                           (its state lives in per-client Python objects, silero_model.py:264-267, :596-628)
 *
 * Plain pointers and sizes only; no torch / numpy types.  All functions return 0
 * on success and a negative CVAD_E_* code on failure (cvad_last_error gives text).
 * One engine = one GPU = one CUDA stream; call it from one thread at a time.
 * Streams ("slots") are independent: h/c state, the three state-machine words and
 * the per-slot thresholds live in HBM for the engine's lifetime.
 */
#ifndef CUTTER_VAD_B200_H
#define CUTTER_VAD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVAD_ABI_VERSION 4

/* error codes */
#define CVAD_OK 0
#define CVAD_E_INVALID (-1)   /* bad argument */
#define CVAD_E_CUDA (-2)      /* CUDA runtime failure */
#define CVAD_E_NOGPU (-3)     /* no usable sm_100 device: there is no CPU fallback */
#define CVAD_E_WEIGHTS (-4)   /* weight blob has the wrong size for the model version */
#define CVAD_E_CAPACITY (-5)  /* slot id or buffer size out of range */

/* model versions (SileroModelVersion, config.py:23-26) */
#define CVAD_MODEL_V5 5
#define CVAD_MODEL_V4 4
#define CVAD_MODEL_V4_8K 48    /* v4's 8 kHz sub-model (`model_8k.*`): what the reference runs for v4 with sample_rate 8000
                                (silero_model.py:433 feeds sr; the graph's else-branch): 512-sample frames of 8 kHz audio,
                                two LSTM time steps per frame, the two sigmoid outputs averaged */

/* arithmetic of the v5 GEMM stages (cvad_set_math).  All hold the 1e-4 parity bar (observed: <= 4e-5 on every test):
   FP32  = packed FP32 FMA on the CUDA cores;
   TC    = tcgen05 tensor cores, BF16 operands split three ways (6 products, FP32 accumulation in TMEM);
   TC16  = tcgen05 tensor cores, FP16 operands split two ways, every activation operand scaled per stream by a power
           of two (3 products; results do not depend on batch neighbours).  The debug dump runs as TC. */
#define CVAD_MATH_FP32 0
#define CVAD_MATH_TC 1
#define CVAD_MATH_TC16 2   /* v5: FP16 operands split two ways with per-stream power-of-two scaling, 3 products per MAC
                              instead of 6 (fused one-frame kernel, two-kernel multi-frame form and the resampler) */
#define CVAD_MATH_FFT 3    /* v4 (its default): the STFT -- 77 % of v4's MACs, and the stage whose FP32 rounding v4's
                              log(1 + 2^20 |STFT|) amplifies -- as a double-precision FFT with the exact Hann x DFT basis,
                              plus one BF16 tensor-core product with (file basis - exact basis); the other layers FP32.
                              Matches the float64 evaluation of the graph to ~1e-6 where two FP32 executors differ by 1e-3 */

/* resampler implementations (cvad_set_resampler) */
#define CVAD_RESAMPLE_FFT 0   /* default: scipy.signal.resample's FFT method in double, rounded once to float32 */
#define CVAD_RESAMPLE_GEMM 1  /* the dense operator R x (FP32 FMA or split-precision tensor cores, following cvad_set_math) */

/* audio sample formats accepted by cvad_step, cvad_step_device and the stream feeder */
#define CVAD_PCM_F32 0        /* float32 in [-1, 1] */
#define CVAD_PCM_S16_32767 1  /* int16, divided by 32767.0f  (websocket server, vad_websocket_server.py:341) */
#define CVAD_PCM_S16_32768 2  /* int16, divided by 32768.0f  (AudioUtils.pcm_to_float32, audio.py:308) */
#define CVAD_PCM_ULAW 3       /* G.711 mu-law, one byte per sample: the ITU-T G.711 linear value (+-32124) / 32768.0f */
#define CVAD_PCM_ALAW 4       /* G.711 A-law, one byte per sample: the ITU-T G.711 linear value (+-32256) / 32768.0f */

/* per-frame flag bits written to flags_out (ProcessingResult, silero_model.py:99-113) */
#define CVAD_FLAG_STARTED 1u
#define CVAD_FLAG_ENDED 2u
#define CVAD_FLAG_CONTINUING 4u

/* per-stream status bits written to status_out */
#define CVAD_STATUS_NONFINITE 1u /* NaN/Inf in the stream's audio: no frame of it was processed (audio.py:227-228) */

/* number of float32 values in the canonical weight blob, per model version */
#define CVAD_V5_WEIGHT_FLOATS 309633
#define CVAD_V4_WEIGHT_FLOATS 155908

typedef struct cvad_engine cvad_engine;

/* One voice start / end, in stream-then-frame order. */
typedef struct cvad_event {
    int32_t stream;      /* index into this step's slot list */
    int32_t slot;        /* engine slot id */
    int32_t frame;       /* frame index inside this step (0-based) */
    int32_t kind;        /* CVAD_FLAG_STARTED or CVAD_FLAG_ENDED */
    int64_t stream_frame;/* frame index since the slot's last reset */
} cvad_event;

/* Arguments of one batched step: every listed slot advances by n_frames[i] frames. */
typedef struct cvad_step_args {
    int32_t n_streams;        /* number of slots stepped in this call (>= 0) */
    const int32_t *slots;     /* [n_streams] distinct slot ids; NULL = 0..n_streams-1 */
    const void *audio;        /* sample (i, k) at audio[i*stream_stride + k] (elements) */
    int32_t pcm_format;       /* CVAD_PCM_*.  CVAD_PCM_ULAW / CVAD_PCM_ALAW (one byte per sample) are decoded on the GPU by
                                 the input stage before anything else; cvad_step_device runs such steps unchained
                                 (memset + event record per step, like multi-channel steps) */
    int64_t stream_stride;    /* elements between consecutive streams' first samples (bytes for G.711) */
    const int32_t *n_frames;  /* [n_streams] frames per stream (0..max_frames); NULL = max_frames each */
    int32_t max_frames;       /* row length of probs_out / flags_out */
    int32_t frame_len;        /* samples per frame before zero-padding/truncation to 512 (1..2048) */
    int32_t hop;              /* samples between frame starts (>= 1) */
    int32_t src_rate;         /* 16000 or 0: native.  8000/24000/48000: every chunk of 512*src_rate/16000 source
                                 samples (= frame_len = hop) is resampled to one 512-sample frame on the GPU with
                                 scipy.signal.resample's operator (AudioUtils.resample_audio, audio.py:19-55) */
    float *probs_out;         /* [n_streams][max_frames] speech probabilities (may be NULL) */
    uint8_t *flags_out;       /* [n_streams][max_frames] CVAD_FLAG_* (may be NULL) */
    uint8_t *status_out;      /* [n_streams] CVAD_STATUS_* (may be NULL) */
    cvad_event *events_out;   /* [max_events] (may be NULL) */
    int32_t max_events;
    int32_t *n_events_out;    /* total events produced, even if > max_events (may be NULL) */
    const int32_t *src_rates; /* ABI 2. [n_streams] per-stream source rate (8000 / 16000 / 24000 / 48000), or NULL.
                                 When given, src_rate, frame_len and hop are ignored: stream i delivers max_frames
                                 chunks of 512*src_rates[i]/16000 samples back to back from audio[i*stream_stride],
                                 each resampled (or, at 16000, passed through) to one 512-sample model frame. */
    int32_t channels;         /* ABI 4. 0 or 1: mono.  2..8: `audio` holds interleaved sample frames (sample k of stream i,
                                 channel c at audio[i*stream_stride + k*channels + c]; stream_stride still counts ELEMENTS)
                                 and every sample frame is averaged to mono on the GPU before anything else, exactly as
                                 AudioUtils.convert_to_mono does (np.mean over axis 1 in float32, audio.py:193-208;
                                 called from VADWrapper._validate_and_prepare_audio, vad_wrapper.py:603-606) */
} cvad_step_args;

/* Library / device probes. */
int cvad_abi_version(void);
int cvad_device_count(void);              /* number of sm_100 devices visible; 0 = none */
const char *cvad_last_error(const cvad_engine *e); /* e may be NULL: last create() failure */

/*
 * Build an engine on `device`.  `weights` is the canonical float32 blob for the
 * model version (order documented in DESIGN.md and oracle/silero_ref.c); it is
 * repacked into the kernels' streaming layout and copied to HBM once.
 */
int cvad_create(const float *weights, size_t n_weight_floats, int model_version,
                int max_streams, int device, cvad_engine **out);
int cvad_destroy(cvad_engine *e);

/* Select the arithmetic of the model kernels (CVAD_MATH_*).  For v5 every GEMM stage moves to the tensor cores;
   for v4 the STFT (77 % of its MACs) does, the small layers and the two LSTM(64) stay FP32.
   A v5 engine starts in CVAD_MATH_TC16 unless the environment variable CVAD_MATH is "tc" or "fp32"; a v4 engine starts in
   CVAD_MATH_FFT unless CVAD_MATH is "fp32" or "tc" (v4's log(1 + 2^20 |STFT|) amplifies accumulation-order differences). */
int cvad_set_math(cvad_engine *e, int math);
int cvad_get_math(const cvad_engine *e);

/* Select how 8 / 24 / 48 kHz input is resampled (CVAD_RESAMPLE_*).  Engines start with CVAD_RESAMPLE_FFT unless the
   environment variable CVAD_RESAMPLE is "gemm". */
int cvad_set_resampler(cvad_engine *e, int resampler);
int cvad_get_resampler(const cvad_engine *e);

/* Development aid for the tensor-core kernels: when enabled, CTA 0 of each kernel records SM-clock marks at its
   phase boundaries (layout in csrc/cvad_v5tc.cuh, CVAD_PROF); cvad_read_profile copies the 128 marks out. */
int cvad_set_profile(cvad_engine *e, int enabled);
int cvad_read_profile(cvad_engine *e, long long *out128);
/* Chained device steps (cvad_step_device, one frame per step) under cvad_set_profile: global-timer nanoseconds of CTAs
   0, 64 and the last one for the last 8 steps, out512[64 (step % 8) + 8 b + k], k = entry, prologue done, grid dependency
   resolved, tile start, tile end, exit. */
int cvad_read_profile_chain(cvad_engine *e, long long *out512);

/* Use an existing CUDA stream (cudaStream_t passed as void*); NULL = engine's own. */
int cvad_set_stream(cvad_engine *e, void *cuda_stream);

/* Zero h/c, clear the state machine and the frame counter.  slots==NULL: all slots. */
int cvad_reset(cvad_engine *e, int n, const int32_t *slots);

/*
 * Per-slot thresholds and options (VADConfig, config.py:54-100).  Probabilities are
 * compared in double exactly as the reference's Python does (silero_model.py:832,:898).
 * slots==NULL: all slots.  Does NOT reset state (VADWrapper.set_thresholds resets
 * explicitly, vad_wrapper.py:411-413; the host mirror calls cvad_reset).
 */
int cvad_configure(cvad_engine *e, int n, const int32_t *slots, double vad_start_probability,
                   double vad_end_probability, int voice_start_frame_count,
                   int voice_end_frame_count, int enable_denoising);

/* LSTM state of one slot: h[128], c[128] for v5; h[2*64], c[2*64] for v4.
   sm[4] = {is_voice_active, voice_start_frame_count, voice_end_frame_count, reserved}.
   cvad_set_state refuses an h outside [-2, 2] (NaN included) with CVAD_E_INVALID before it writes anything: the FP16-split
   tensor-core kernels hold |h| <= 2 exactly, and an LSTM's own h = o * tanh(c) never leaves [-1, 1]. */
int cvad_get_state(cvad_engine *e, int slot, float *h, float *c, int32_t *sm, int64_t *frames_done);
int cvad_set_state(cvad_engine *e, int slot, const float *h, const float *c, const int32_t *sm);

/*
 * Stream snapshots: everything the engine keeps for one slot, as one fixed-layout record of 1,072 bytes without padding,
 * so that live streams can move between engines, processes and GPUs (restart a service without dropping its streams).
 */
typedef struct cvad_stream_state {
    float   h[128];                 /* v5: h; v4 / v4_8k: layer 0 then layer 1 (cvad_get_state's order) */
    float   c[128];
    int64_t frames_done;            /* frames run since the slot's last reset (cvad_event::stream_frame continues from it) */
    double  vad_start_probability, vad_end_probability;
    int32_t is_voice_active, voice_start_frame_count, voice_end_frame_count;
    int32_t n_start, n_end;         /* configured voice_start/end_frame_count */
    int32_t enable_denoising;
} cvad_stream_state;

/* The model version given to cvad_create, then the FNV-1a 64 hash of its weight blob: FNV-1a over the version as a
   little-endian int32 followed by the blob's bytes.  Records move between engines with equal fingerprints only.  The
   math mode is not part of it: the state is FP32 in every mode. */
int cvad_model_fingerprint(const cvad_engine *e, uint64_t *out);
/* Copy the state of n slots (slots: host memory, distinct ids; NULL = 0..n-1) into out[n] / from in[n].  out / in may be
   host memory (pageable or pinned) or device memory on the engine's device, 8-byte aligned (CVAD_E_INVALID otherwise);
   one copy each way.  Device records are read and written on the engine's stream: whatever the caller wrote into them
   on another stream must be complete before cvad_import_states, and exported records are complete when it returns.
   Both wait for the steps
   in flight first and synchronise before returning, like cvad_reset, so the next step (chained device steps included)
   reads the imported state.  Import is all or nothing: every record is checked on the device first (h within [-2, 2],
   which the FP16-split tensor-core kernels hold exactly and which no LSTM step leaves; c finite; is_voice_active and enable_denoising 0 or 1, counts and frames_done >= 0, probabilities in [0, 1], n_start and
   n_end >= 1); one bad record fails the call with CVAD_E_INVALID, cvad_last_error names its index, and no slot changes.
   CVAD_E_CAPACITY: a slot id out of range; CVAD_E_INVALID: a slot listed twice. */
int cvad_export_states(cvad_engine *e, int n, const int32_t *slots, cvad_stream_state *out);
int cvad_import_states(cvad_engine *e, int n, const int32_t *slots, const cvad_stream_state *in);

/*
 * One batched step with HOST buffers: pinned staging + H2D, kernels, D2H, sync.
 * This is what the reference-facing Python mirror calls.
 */
int cvad_step(cvad_engine *e, const cvad_step_args *a);

/*
 * Pipelined form of cvad_step: submit enqueues H2D, kernels and D2H and returns; collect
 * waits and fills the output buffers named in `a` (which, like `a->audio` when it is
 * pinned memory, must stay valid and untouched until then).  Up to four steps may be in
 * flight; they execute in submission order, and later steps' host-to-device copies
 * overlap earlier steps' kernels and result copies.  cvad_step == submit + collect.
 */
int cvad_step_submit(cvad_engine *e, const cvad_step_args *a, int *ticket);
int cvad_step_collect(cvad_engine *e, int ticket);

/*
 * Same step with every pointer in `a` (audio, slots, n_frames, outputs) already in
 * DEVICE memory; enqueues on the engine's stream and returns without synchronising.
 * events_out/n_events_out (device) are filled by the kernel in arbitrary order; n_events_out
 * holds the step's total once the step has finished (its value in between is unspecified).
 * One-frame steps of the v5 tensor-core builds are chained: consecutive calls enqueue
 * nothing but kernels (no memset, no event record), the model kernel launched with
 * programmatic stream serialization, so a step's grid is scheduled while its predecessor drains (every read of
 * `a`'s buffers still happens after whatever precedes the call on the stream has completed).
 */
int cvad_step_device(cvad_engine *e, const cvad_step_args *a);

/* Block until everything enqueued on the engine's stream has finished. */
int cvad_sync(cvad_engine *e);

/* The resampler's operator for tests and non-GPU hosts: R^T[m][n] (n_in x 512 floats, row-major)
   such that y[n] = sum_m R^T[m][n] x[m] equals scipy.signal.resample(x, 512).  Returns n_in. */
int cvad_resample_matrix(int src_rate, float *rt_out, size_t n_floats);

/* Page-locked host memory for callers that want cvad_step to DMA straight from their
   buffer (pageable buffers are staged through the engine's own pinned area). */
void *cvad_alloc_pinned(size_t bytes);
void cvad_free_pinned(void *p);

/* Number of kernel launches issued by this engine since creation (for bench accounting). */
int64_t cvad_launch_count(const cvad_engine *e);

/*
 * Per-kernel device timing for bench.py: while enabled, every step records CUDA
 * events on the engine's stream around the front-end and the recurrent kernel.
 * cvad_read_timing synchronises, returns the summed durations (ms) and the number of
 * steps they cover, and clears the record.
 */
int cvad_set_timing(cvad_engine *e, int enabled);
int cvad_read_timing(cvad_engine *e, double *frontend_ms, double *recurrent_ms, int *n_steps);

/*
 * Test hook: run the front end + one recurrent step for the first tile (<= 32 streams,
 * frame 0) of `a` WITHOUT touching engine state and copy the intermediate activations
 * to `dbg_out` (host).  Layout in DESIGN.md ("debug dump").  Returns floats written.
 */
int cvad_debug_dump(cvad_engine *e, const cvad_step_args *a, float *dbg_out, size_t dbg_floats);

/*
 * Test hook: run only the input stages of the step `a` describes (the down-mix of interleaved channels or the G.711
 * decode, and the resampler, or the pass-through of 16 kHz streams in a mixed-rate step), staged exactly as cvad_step
 * stages it, and copy to `out` (host) the float32 mono 16 kHz samples the model kernels would read:
 *   resampled or mixed-rate steps:     [n_streams][max_frames * 512];
 *   down-mix or G.711 decode only:     [n_streams][(max_frames - 1) * hop + frame_len].
 * The device buffer is filled with 0xFF bytes (NaN) before the stages run, so a frame beyond a stream's n_frames
 * reads NaN in resampled output.  No model kernel runs and engine state is untouched.  Returns the number of floats
 * written, CVAD_E_CAPACITY if `n_floats` is too small, CVAD_E_INVALID for a step without an input stage (16 kHz mono float32 / int16).
 */
int cvad_debug_input(cvad_engine *e, const cvad_step_args *a, float *out, size_t n_floats);


/* ------------------------------------------------------------------------------------------------------------
 * Stream feeder (ABI 3): the host half of the service mode, in native code.
 *
 * The reference's websocket server keeps one VADWrapper per client and runs one model call per message on the
 * event loop (websocket_service/server/vad_websocket_server.py:248-290, :326-369).  A feeder keeps every
 * client's pending samples in ONE pinned arena (a row per slot); cvad_feeder_push appends a message,
 * cvad_feeder_step frames whatever is complete (AudioUtils.split_into_frames, src/real_time_vad/utils/audio.py:164-190,
 * leftovers carried), runs ONE cvad_step over all of those streams, and replays the callback side of VADProcessor
 * from the device's per-frame flags: the pre-roll buffered since the first above-threshold frame, the voice segment
 * handed to voice_end, the gated frame handed to voice_continue
 * (src/real_time_vad/core/silero_model.py:839-869, :891-895, :925-949; vad_wrapper.py:498-519).
 *
 * Threading: cvad_feeder_push / push_many may be called from any thread, also while a step runs.
 * open / close / clear / step: one thread at a time.  Pointers in cvad_feeder_result stay valid until the next
 * cvad_feeder_step on the same feeder.
 */
typedef struct cvad_feeder cvad_feeder;

/* what a stream wants back besides probabilities and events */
#define CVAD_PAYLOAD_NONE 0      /* nothing: only the voice-active mirror is kept */
#define CVAD_PAYLOAD_EVENTS 1    /* a delivery record on the frames that start / end a voice segment */
#define CVAD_PAYLOAD_SEGMENTS 2  /* + the gated float32 samples of the finished segment on the end record */
#define CVAD_PAYLOAD_FRAMES 3    /* + a record with the gated float32 frame for every frame while voice is active */

typedef struct cvad_delivery {
    int32_t slot;            /* engine slot id */
    int32_t stream;          /* row of this stream in the step (index into slots / counts / probs / raw) */
    int32_t step_frame;      /* frame index inside this step */
    int32_t flags;           /* CVAD_FLAG_* of the frame */
    const float *frame;      /* CVAD_PAYLOAD_FRAMES: the gated 16 kHz frame handed to voice_continue, else NULL */
    const float *segment;    /* on CVAD_FLAG_ENDED with CVAD_PAYLOAD_SEGMENTS/FRAMES: the finished segment, else NULL */
    int64_t segment_len;     /* samples in `segment` */
    int32_t frame_len;       /* samples in `frame` */
    float prob;              /* the frame's speech probability */
    const void *raw;         /* streams whose source rate is not 16 kHz and that want audio: the frame's source-rate
                                samples in the feeder's PCM format (the host resamples its payloads); a record is
                                then produced for EVERY frame and frame / segment stay NULL */
    int64_t raw_len;
} cvad_delivery;

typedef struct cvad_feeder_result {
    int32_t n_streams;                 /* streams that ran at least one frame */
    int32_t max_frames;                /* row length of probs / flags */
    int64_t n_frames_total;
    const int32_t *slots;              /* [n_streams] */
    const int32_t *counts;             /* [n_streams] frames run per stream */
    const float *probs;                /* [n_streams][max_frames]; columns >= counts[k] are 0 */
    const uint8_t *flags;              /* [n_streams][max_frames] */
    int32_t n_events;
    int32_t n_deliveries;
    const cvad_event *events;          /* stream-then-frame order */
    const cvad_delivery *deliveries;   /* stream-then-frame order */
    const void *raw;                   /* the block that was stepped: [n_streams][raw_stride] samples, PCM format of the feeder;
                                          NULL when the step ran frame by frame (2..4 frames per stream: the feeder then gathers
                                          frame-major planes and runs one one-frame step per round) */
    int64_t raw_stride;
    double gather_ms, gpu_ms, deliver_ms;   /* wall time of the three phases of this step (framing, cvad_step, callbacks' side) */
} cvad_feeder_result;

/* e == NULL builds a feeder for the gather / deliver test hooks only (max_streams is then taken from the argument,
   otherwise from the engine).  src_rate 0 = every stream has its own rate (cvad_feeder_open), frame_len / hop are then
   ignored; src_rate 8000 / 24000 / 48000 fixes frame_len = hop = 512*src_rate/16000.  capacity_frames = frames a stream
   runs per step at most (>= 2; a stream further behind catches up over several steps) and the initial row size;
   rows grow when a producer runs ahead of step(). */
int cvad_feeder_create(cvad_engine *e, int max_streams, int pcm_format, int frame_len, int hop, int src_rate,
                       int capacity_frames, cvad_feeder **out);
int cvad_feeder_destroy(cvad_feeder *f);
const char *cvad_feeder_last_error(const cvad_feeder *f);

/* Start / restart buffering for a slot (pending samples and any half-built segment are dropped).  The engine side of a
   stream (cvad_reset, cvad_configure) is the caller's; vad_start_probability and enable_denoising are needed here
   because the pre-roll starts at the first frame whose probability reaches the start threshold and payloads are gated
   like the model input (silero_model.py:832-845, :782-783).  src_rate 0 = the feeder's. */
int cvad_feeder_open(cvad_feeder *f, int slot, int src_rate, int payload, double vad_start_probability,
                     int enable_denoising);
int cvad_feeder_close(cvad_feeder *f, int slot);
int cvad_feeder_clear(cvad_feeder *f, int slot);          /* VADProcessor.reset: drop pending samples and segment */
int cvad_feeder_is_active(cvad_feeder *f, int slot);      /* host mirror of is_voice_active: 1 / 0 */
int64_t cvad_feeder_pending(cvad_feeder *f, int slot);    /* samples buffered */

/* Append samples (feeder's PCM format; bytes for G.711) to a slot.  float32 input containing NaN / Inf is rejected here,
   before any state changes (AudioUtils.validate_audio_data, audio.py:227-228); every G.711 byte is a valid sample.
   Voice-end segments and voice-continue frames of a G.711 feeder hold the decoded, gated float32 audio.  CVAD_E_CAPACITY when the arena cannot grow further. */
int cvad_feeder_push(cvad_feeder *f, int slot, const void *samples, int64_t n_samples);
/* block[i*row_stride .. +n_samples) is appended to slots[i]; all or nothing. */
int cvad_feeder_push_many(cvad_feeder *f, int n, const int32_t *slots, const void *block, int64_t row_stride,
                          int64_t n_samples);

/* Frame, step and deliver (see above). */
int cvad_feeder_step(cvad_feeder *f, cvad_feeder_result *out);

/* Test hooks for hosts without a GPU: the two host phases of cvad_feeder_step on their own.  gather_only frames
   and compacts (probs / flags read as 0); deliver_only replays the callback side for the gathered streams from
   caller-supplied probs / flags [n_streams][max_frames]. */
int cvad_feeder_gather_only(cvad_feeder *f, cvad_feeder_result *out);
int cvad_feeder_deliver_only(cvad_feeder *f, const float *probs, const uint8_t *flags, cvad_feeder_result *out);

/*
 * Row snapshots: the host half of a stream (pending samples, the pre-roll and the half-built segment) as a persistable
 * blob, the companion of cvad_export_states.  Both calls take the feeder's lock, so a snapshot is a consistent cut
 * against concurrent pushes.  Export fails with CVAD_E_INVALID for a slot that is not open; out == NULL only reports
 * *needed, and out_bytes < *needed is CVAD_E_CAPACITY (with *needed set and nothing written).  Import (re)opens the target slots like cvad_feeder_open, after
 * checking the whole blob (magic, version, the feeder's PCM format and framing -- or, on a mixed-rate feeder, per-slot
 * rates of 8000 / 16000 / 24000 / 48000 --, payload modes, lengths against in_bytes); a refused blob changes no slot.
 * A row whose payload mode carries no audio (below CVAD_PAYLOAD_SEGMENTS) is imported without its pre-roll and segment.
 * Rows grow as cvad_feeder_push makes them grow.  Both work on a feeder built with e == NULL.
 *
 * Blob layout, little-endian, no padding:
 *   header (32 bytes): uint32 magic CVAD_FEEDER_SNAPSHOT_MAGIC, uint32 version CVAD_FEEDER_SNAPSHOT_VERSION,
 *                      int32 pcm_format, frame_len, hop, src_rate (0 = mixed), int32 n (rows that follow), int32 0
 *   n rows, in the order of `slots`, each a 64-byte head
 *       int32 rate, n_in (source samples per model frame), payload (CVAD_PAYLOAD_*), enable_denoising (0 / 1),
 *       float64 vad_start_probability, int32 voice active (the host mirror, 0 / 1), int32 0,
 *       int64 skip (hop > frame_len: samples still to drop from the next push), int64 n_pending, n_pre_roll, n_segment
 *   followed by n_pending samples in the feeder's PCM format (4, 2 or, for G.711, 1 byte each), then n_pre_roll and
 *   n_segment float32 samples.
 */
#define CVAD_FEEDER_SNAPSHOT_MAGIC 0x53465643u   /* "CVFS" */
#define CVAD_FEEDER_SNAPSHOT_VERSION 1
int cvad_feeder_export(cvad_feeder *f, int n, const int32_t *slots, void *out, size_t out_bytes, size_t *needed);
int cvad_feeder_import(cvad_feeder *f, int n, const int32_t *slots, const void *in, size_t in_bytes);

#ifdef __cplusplus
}
#endif
#endif /* CUTTER_VAD_B200_H */
