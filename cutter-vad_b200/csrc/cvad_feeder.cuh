// cvad_feeder.cuh -- host half of the service mode: per-slot pending-audio arena in pinned memory,
// native gather / compaction around one cvad_step, and voice-segment assembly from the device's flags.
//
// What it replaces in the reference (one VADWrapper + one onnxruntime session per websocket client):
//   ClientState.process_audio_frame        websocket_service/server/vad_websocket_server.py:326-369   -> cvad_feeder_push
//   VADWrapper._process_audio_frames       src/real_time_vad/core/vad_wrapper.py:610-647               -> cvad_feeder_step
//   VADProcessor voice_buffer / current_voice_data / _finalize_voice_segment
//                                          src/real_time_vad/core/silero_model.py:839-869,:925-949     -> deliver()
// Included by cvad_capi.cu (one translation unit); plain C++17, no device code.
#pragma once

#include <algorithm>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

// A few persistent helper threads for the row copies of push_many and gather (10,000 streams x 30 ms of int16 are
// ~10 MB per tick on each side: one thread's memcpy rate is what bounded both).  run(parts, body) executes body(0..parts-1)
// on the helpers AND the calling thread and returns when all parts are done.
class FeederPool {
public:
    explicit FeederPool(int workers) {
        for (int i = 0; i < workers; ++i) th_.emplace_back([this] { loop(); });
    }
    ~FeederPool() {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    void run(int parts, const std::function<void(int)> &body) {
        if (parts <= 1 || th_.empty()) {
            for (int t = 0; t < parts; ++t) body(t);
            return;
        }
        { std::lock_guard<std::mutex> lk(m_); job_ = &body; total_ = parts; next_ = 0; done_ = 0; ++gen_; }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m_);
        cv_done_.wait(lk, [&] { return done_ == total_; });
        job_ = nullptr;
    }

private:
    void work() {
        for (;;) {
            int t;
            const std::function<void(int)> *job;
            {
                std::lock_guard<std::mutex> lk(m_);
                if (!job_ || next_ >= total_) return;
                t = next_++;
                job = job_;
            }
            (*job)(t);
            {
                std::lock_guard<std::mutex> lk(m_);
                if (++done_ == total_) cv_done_.notify_all();
            }
        }
    }
    void loop() {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || (gen_ != seen && job_ != nullptr); });
                if (stop_) return;
                seen = gen_;
            }
            work();
        }
    }
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_, cv_done_;
    const std::function<void(int)> *job_ = nullptr;
    int total_ = 0, next_ = 0, done_ = 0;
    uint64_t gen_ = 0;
    bool stop_ = false;
};

struct cvad_feeder {
    cvad_engine *eng = nullptr;        // may be NULL: gather / deliver test hooks only
    int max_streams = 0;
    int pcm_format = CVAD_PCM_F32;
    int frame_len = 512, hop = 512;
    int src_rate = 16000;              // 0 = per-slot rates (mixed)
    int max_step_frames = 8;           // frames one stream may run per step (a stream further behind catches up over steps)
    size_t es = 4;                     // bytes per sample
    size_t cap = 0;                    // arena row length (samples)
    unsigned char *arena = nullptr;    // pinned [max_streams][cap]
    std::mutex mu;                     // guards arena + fill + slot table (push vs step)
    std::string err;

    struct Slot {
        int rate = 16000;
        int n_in = 512;                // source samples per model frame (mixed mode)
        bool denoise = true;
        double start_p = 0.7;
        std::vector<float> pre_roll, segment;
    };
    std::vector<Slot> slot;
    std::vector<int64_t> fill;
    // what the per-step loops over ALL streams read, side by side (a Slot is two cache lines: at 10,000 streams the walk
    // over the structs was most of the segment-assembly phase): open flag, CVAD_PAYLOAD_*, host mirror of is_voice_active
    std::vector<uint8_t> opn, pay, act;
    std::vector<int64_t> skp;          // hop > frame_len: samples between frames that had not arrived when their frame ran

    // step scratch (valid until the next step)
    unsigned char *stage[2] = {nullptr, nullptr};   // pinned gather targets, alternating
    size_t stage_cap[2] = {0, 0};
    int cur = 0;
    std::vector<int32_t> ids, counts, rates;
    std::vector<float> probs;
    std::vector<uint8_t> flags, status;
    std::vector<cvad_event> events;
    std::vector<cvad_delivery> deliveries;
    // segment assembly runs on the helper pool over contiguous ranges of the payload-carrying streams; each range keeps
    // its own records and payload storage (the records point into them; merged in stream order, valid until the next step)
    struct DeliverPart {
        std::vector<cvad_delivery> deliv;
        std::vector<float> pool;                     // gated frames handed to voice_continue this step
        std::vector<std::vector<float>> segs;        // segments finished this step
    };
    std::vector<DeliverPart> dparts;
    std::vector<int32_t> dwork;                      // indices k of the streams that carry payloads
    int64_t row = 0;
    int tmax = 0;
    int threads = 1;
    std::unique_ptr<FeederPool> pool;                // threads - 1 helpers, created with the feeder
    std::vector<uint32_t> mark;                      // push_many: per-slot stamp (parallel row copies need distinct slots)
    uint32_t mark_gen = 0;
    // layout of the gathered block: rows ([n][row], frame j of stream k at k*row + j*hop) or, for the frame-by-frame
    // rounds of cvad_feeder_step, planes ([tmax][n][plane_row]: plane r holds everybody's r-th frame, contiguous, so
    // that round 0 is ONE dense host-to-device copy)
    bool planes = false;
    int64_t plane_row = 0;
    // planes r >= 1 are DENSE: they hold only the streams that have an r-th frame, in stream order, so that round r's
    // input is plane r as it stands.  plane_off[r] = first row of plane r, ppos[(r - 1) n + k] = row of stream k inside it
    int64_t plane_off[5] = {0, 0, 0, 0, 0};
    std::vector<int32_t> ppos;
};

namespace {

constexpr size_t kFeederArenaLimit = (size_t)16 << 30;   // pinned bytes the arena may grow to

int ffail(cvad_feeder *f, int code, const std::string &msg) {
    if (f) f->err = msg;
    return code;
}

inline float feeder_sample(const cvad_feeder *f, const unsigned char *p, size_t k) {
    if (f->pcm_format == CVAD_PCM_F32) return reinterpret_cast<const float *>(p)[k];
    const float v = (float)reinterpret_cast<const int16_t *>(p)[k];
    return f->pcm_format == CVAD_PCM_S16_32767 ? v / 32767.0f : v / 32768.0f;
}

// numpy's `np.where(np.abs(f) > 0.01, f, 0.0)` on float32 data (audio.py:117-118): the threshold is float32(0.01)
// One loop per sample format and gate setting, branch-free inside (the compiler vectorises them; the per-sample format
// test of feeder_sample kept the 480-sample loop scalar: ~0.5 us per frame, most of the segment-assembly phase).
template <int FMT, bool GATE>
inline void feeder_gate_loop(const unsigned char *__restrict__ src, int n, float *__restrict__ d) {
    for (int k = 0; k < n; ++k) {
        float v;
        if (FMT == CVAD_PCM_F32) v = reinterpret_cast<const float *>(src)[k];
        else if (FMT == CVAD_PCM_S16_32767) v = (float)reinterpret_cast<const int16_t *>(src)[k] / 32767.0f;
        else v = (float)reinterpret_cast<const int16_t *>(src)[k] / 32768.0f;
        d[k] = (!GATE || std::fabs(v) > 0.01f) ? v : 0.0f;
    }
}
inline void feeder_gate_append(const cvad_feeder *f, const cvad_feeder::Slot &s, const unsigned char *src, int n,
                               std::vector<float> &dst) {
    const size_t o = dst.size();
    dst.resize(o + (size_t)n);
    float *d = dst.data() + o;
    const bool g = s.denoise;
    switch (f->pcm_format) {
        case CVAD_PCM_F32: g ? feeder_gate_loop<CVAD_PCM_F32, true>(src, n, d) : feeder_gate_loop<CVAD_PCM_F32, false>(src, n, d); break;
        case CVAD_PCM_S16_32767:
            g ? feeder_gate_loop<CVAD_PCM_S16_32767, true>(src, n, d) : feeder_gate_loop<CVAD_PCM_S16_32767, false>(src, n, d); break;
        default: g ? feeder_gate_loop<CVAD_PCM_S16_32768, true>(src, n, d) : feeder_gate_loop<CVAD_PCM_S16_32768, false>(src, n, d); break;
    }
}

int feeder_grow_stage(cvad_feeder *f, int which, size_t bytes) {
    if (bytes <= f->stage_cap[which]) return CVAD_OK;
    if (f->stage[which]) {
        if (f->eng) cudaFreeHost(f->stage[which]); else std::free(f->stage[which]);
        f->stage[which] = nullptr;
        f->stage_cap[which] = 0;
    }
    const size_t cap = bytes + bytes / 4 + 4096;
    if (f->eng) {
        void *p = nullptr;
        if (cudaMallocHost(&p, cap) != cudaSuccess) { cudaGetLastError(); return ffail(f, CVAD_E_CUDA, "cudaMallocHost failed"); }
        f->stage[which] = static_cast<unsigned char *>(p);
    } else {
        f->stage[which] = static_cast<unsigned char *>(std::malloc(cap));
        if (!f->stage[which]) return ffail(f, CVAD_E_CAPACITY, "out of host memory");
    }
    f->stage_cap[which] = cap;
    return CVAD_OK;
}

// Phase 1 of a step, under the lock: pick the streams that hold at least one whole frame, copy their
// pending samples into a dense [n][row] block (split_into_frames' input, audio.py:164-190) and drop
// what the step will consume from the arena (leftovers shorter than a hop stay for the next step).
inline const unsigned char *feeder_frame_ptr(const cvad_feeder *f, const unsigned char *stage, int n, int k, int j, int64_t step_len) {
    if (f->planes) {
        const size_t r = j == 0 ? (size_t)k : (size_t)f->plane_off[j] + (size_t)f->ppos[(size_t)(j - 1) * (size_t)n + (size_t)k];
        return stage + r * (size_t)f->plane_row * f->es;
    }
    return stage + ((size_t)k * (size_t)f->row + (size_t)j * (size_t)step_len) * f->es;
}

// Copy into the pinned block the next host-to-device copy reads: streaming (non-temporal) stores.  Measured on the B200
// box: after the helper threads had gathered 8.4 MB with ordinary stores, the lines sat dirty in six cores' private
// caches and the DMA engine read them at 12 GB/s (0.7 ms) instead of the 50 GB/s (0.17 ms) it gets from memory.
inline void feeder_copy_nt(unsigned char *dst, const unsigned char *src, size_t bytes) {
#if defined(__SSE2__)
    if ((((uintptr_t)dst | (uintptr_t)src) & 15u) == 0) {
        size_t i = 0;
        for (; i + 64 <= bytes; i += 64) {
            const __m128i a = _mm_load_si128(reinterpret_cast<const __m128i *>(src + i));
            const __m128i b = _mm_load_si128(reinterpret_cast<const __m128i *>(src + i + 16));
            const __m128i c = _mm_load_si128(reinterpret_cast<const __m128i *>(src + i + 32));
            const __m128i d = _mm_load_si128(reinterpret_cast<const __m128i *>(src + i + 48));
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), a);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 32), c);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 48), d);
        }
        for (; i + 16 <= bytes; i += 16)
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), _mm_load_si128(reinterpret_cast<const __m128i *>(src + i)));
        if (i < bytes) std::memcpy(dst + i, src + i, bytes - i);
        return;
    }
#endif
    std::memcpy(dst, src, bytes);
}
inline void feeder_copy_fence() {
#if defined(__SSE2__)
    _mm_sfence();
#endif
}

int feeder_gather(cvad_feeder *f, bool allow_planes = false) {
    std::lock_guard<std::mutex> lk(f->mu);
    f->cur ^= 1;
    f->ids.clear(); f->counts.clear(); f->rates.clear();
    const bool mixed = f->src_rate == 0;
    int tmax = 0;
    int64_t row = 0;
    for (int s = 0; s < f->max_streams; ++s) {
        if (!f->opn[s]) continue;
        const cvad_feeder::Slot &sl = f->slot[s];
        const int64_t have = f->fill[s];
        int64_t c;
        if (mixed) c = have / sl.n_in;
        else c = have >= f->frame_len ? (have - f->frame_len) / f->hop + 1 : 0;
        if (c <= 0) continue;
        if (c > f->max_step_frames) c = f->max_step_frames;
        f->ids.push_back(s);
        f->counts.push_back((int32_t)c);
        if (mixed) {
            f->rates.push_back(sl.rate);
            row = std::max<int64_t>(row, c * sl.n_in);
        }
        tmax = std::max(tmax, (int)c);
    }
    const int n = (int)f->ids.size();
    f->tmax = tmax;
    if (n == 0) { f->row = 0; return CVAD_OK; }
    if (!mixed) row = (int64_t)(tmax - 1) * f->hop + f->frame_len;
    row += (-row) & 7;                         // rows start 16-byte aligned in either sample format
    f->row = row;
    f->planes = allow_planes && !mixed && tmax >= 2 && tmax <= 4;
    f->plane_row = ((int64_t)f->frame_len + 7) & ~(int64_t)7;
    size_t plane_rows = (size_t)n;
    if (f->planes) {
        f->ppos.assign((size_t)(tmax - 1) * (size_t)n, 0);
        f->plane_off[0] = 0;
        for (int j = 1; j < tmax; ++j) {
            f->plane_off[j] = (int64_t)plane_rows;
            int32_t at = 0;
            for (int k = 0; k < n; ++k)
                if (f->counts[k] > j) f->ppos[(size_t)(j - 1) * (size_t)n + (size_t)k] = at++;
            plane_rows += (size_t)at;
        }
    }
    const size_t stage_bytes = f->planes ? plane_rows * (size_t)f->plane_row * f->es : (size_t)n * (size_t)row * f->es;
    int rc = feeder_grow_stage(f, f->cur, stage_bytes);
    if (rc) return rc;
    unsigned char *stage = f->stage[f->cur];
    auto work = [&](int k0, int k1) {
        for (int k = k0; k < k1; ++k) {
            const int s = f->ids[k];
            const cvad_feeder::Slot &sl = f->slot[s];
            unsigned char *src = f->arena + (size_t)s * f->cap * f->es;
            const int64_t have = f->fill[s];
            const int64_t used = (int64_t)f->counts[k] * (mixed ? sl.n_in : f->hop);
            const int64_t need = mixed ? used : (int64_t)(f->counts[k] - 1) * f->hop + f->frame_len;
            if (f->planes) {
                for (int j = 0; j < f->counts[k]; ++j)
                    feeder_copy_nt(const_cast<unsigned char *>(feeder_frame_ptr(f, stage, n, k, j, f->hop)),
                                   src + (size_t)j * (size_t)f->hop * f->es, (size_t)f->frame_len * f->es);
            } else {
                feeder_copy_nt(stage + (size_t)k * (size_t)row * f->es, src, (size_t)need * f->es);
            }
            const int64_t rem = have - used;
            if (rem > 0) std::memmove(src, src + (size_t)used * f->es, (size_t)rem * f->es);
            f->fill[s] = rem > 0 ? rem : 0;
            if (rem < 0) f->skp[s] = -rem;
        }
        feeder_copy_fence();
    };
    const size_t bytes = (size_t)n * (size_t)row * f->es;
    const int nt = (f->threads > 1 && bytes > (1u << 20)) ? std::min(f->threads, n) : 1;
    if (nt <= 1 || !f->pool) {
        work(0, n);
    } else {
        f->pool->run(nt, [&](int t) { work((int)((int64_t)n * t / nt), (int)((int64_t)n * (t + 1) / nt)); });
    }
    return CVAD_OK;
}

// Phase 3: the callback side of VADProcessor (silero_model.py:818-949) replayed from the device's per-frame
// flags -- host mirror of is_voice_active, pre-roll / segment assembly, delivery records.
void feeder_deliver(cvad_feeder *f) {
    const int n = (int)f->ids.size(), T = f->tmax;
    f->deliveries.clear();
    const unsigned char *stage = f->stage[f->cur];
    const bool mixed = f->src_rate == 0;
    // streams without payloads only update the host mirror of is_voice_active (hot arrays: no Slot is touched)
    f->dwork.clear();
    for (int k = 0; k < n; ++k) {
        const int s = f->ids[k];
        if (f->pay[s] == CVAD_PAYLOAD_NONE) {
            const uint8_t last = f->flags[(size_t)k * T + (size_t)(f->counts[k] - 1)];
            f->act[s] = !(last & CVAD_FLAG_ENDED) && (last & (CVAD_FLAG_STARTED | CVAD_FLAG_CONTINUING));
        } else {
            f->dwork.push_back(k);
        }
    }
    const int m = (int)f->dwork.size();
    const int parts = (f->pool && m >= 128) ? std::min(f->threads, m / 64) : 1;
    if ((int)f->dparts.size() < parts) f->dparts.resize((size_t)parts);
    for (auto &P : f->dparts) { P.deliv.clear(); P.pool.clear(); P.segs.clear(); }
    auto run_part = [&](int part) {
        cvad_feeder::DeliverPart &P = f->dparts[(size_t)part];
        const int i0 = (int)((int64_t)m * part / parts), i1 = (int)((int64_t)m * (part + 1) / parts);
        // how many continue-frames will be pooled (so that the pool never reallocates under the records)
        size_t need = 0;
        for (int i = i0; i < i1; ++i) {
            const int k = f->dwork[(size_t)i], s = f->ids[k];
            if (f->pay[s] == CVAD_PAYLOAD_FRAMES && f->slot[s].rate == 16000) need += (size_t)f->counts[k] * (size_t)f->frame_len;
        }
        P.pool.reserve(need);
        for (int i = i0; i < i1; ++i) {
            const int k = f->dwork[(size_t)i], s = f->ids[k];
            const int c = f->counts[k];
            const uint8_t *fl = f->flags.data() + (size_t)k * T;
            const float *pr = f->probs.data() + (size_t)k * T;
            const int payload = f->pay[s];
            cvad_feeder::Slot &sl = f->slot[s];
            bool active = f->act[s] != 0;
            const bool raw_mode = payload >= CVAD_PAYLOAD_SEGMENTS && sl.rate != 16000;   // host resamples the payloads
            const int64_t step_len = mixed ? sl.n_in : f->hop;
            const int flen = mixed ? sl.n_in : f->frame_len;
            for (int j = 0; j < c; ++j) {
                const uint8_t b = fl[j];
                const unsigned char *fp = feeder_frame_ptr(f, stage, n, k, j, step_len);
                cvad_delivery d{};
                d.slot = s; d.stream = k; d.step_frame = j; d.flags = b;
                d.prob = pr[j];
                if (raw_mode) {
                    // every frame is handed over; the host keeps pre-roll / segment for this stream itself
                    d.raw = fp; d.raw_len = flen;
                    active = !(b & CVAD_FLAG_ENDED) && (b & (CVAD_FLAG_STARTED | CVAD_FLAG_CONTINUING));
                    P.deliv.push_back(d);
                    continue;
                }
                const bool audio = payload >= CVAD_PAYLOAD_SEGMENTS;
                bool emit = false;
                if (!active) {
                    if ((double)pr[j] >= sl.start_p) {
                        if (audio) feeder_gate_append(f, sl, fp, flen, sl.pre_roll);
                        if (b & CVAD_FLAG_STARTED) {
                            sl.segment.swap(sl.pre_roll);
                            sl.pre_roll.clear();
                            active = true;
                            emit = true;
                        }
                    } else {
                        sl.pre_roll.clear();
                    }
                } else {
                    size_t frame_at = 0;
                    if (audio) {
                        frame_at = sl.segment.size();
                        feeder_gate_append(f, sl, fp, flen, sl.segment);
                    }
                    if (payload == CVAD_PAYLOAD_FRAMES) {
                        const size_t o = P.pool.size();
                        P.pool.insert(P.pool.end(), sl.segment.begin() + (ptrdiff_t)frame_at, sl.segment.end());
                        d.frame = P.pool.data() + o;
                        d.frame_len = flen;
                        emit = true;
                    }
                    if (b & CVAD_FLAG_ENDED) {
                        P.segs.emplace_back();
                        P.segs.back().swap(sl.segment);
                        sl.segment.clear();
                        d.segment = P.segs.back().data();
                        d.segment_len = (int64_t)P.segs.back().size();
                        active = false;
                        emit = true;
                    }
                }
                if (emit) P.deliv.push_back(d);
            }
            f->act[s] = active ? 1 : 0;
        }
    };
    if (parts <= 1) run_part(0);
    else f->pool->run(parts, run_part);
    for (int part = 0; part < parts; ++part)
        f->deliveries.insert(f->deliveries.end(), f->dparts[(size_t)part].deliv.begin(), f->dparts[(size_t)part].deliv.end());
}

}  // namespace

extern "C" {

int cvad_feeder_create(cvad_engine *e, int max_streams, int pcm_format, int frame_len, int hop, int src_rate,
                       int capacity_frames, cvad_feeder **out) {
    if (!out) return CVAD_E_INVALID;
    *out = nullptr;
    if (e) max_streams = e->max_streams;
    if (max_streams < 1) return fail(e, CVAD_E_INVALID, "feeder: max_streams < 1");
    if (pcm_format < 0 || pcm_format > 2) return fail(e, CVAD_E_INVALID, "feeder: unknown pcm_format");
    if (src_rate != 0 && src_rate != 16000) {
        if (rate_index(src_rate) < 0) return fail(e, CVAD_E_INVALID, "feeder: src_rate must be 0, 8000, 16000, 24000 or 48000");
        frame_len = hop = rate_n_in(src_rate);
    }
    if (src_rate == 0) frame_len = hop = rate_n_in(48000);      // arena sizing; per-slot chunk sizes in Slot::n_in
    if (frame_len < 1 || frame_len > 2048 || hop < 1) return fail(e, CVAD_E_INVALID, "feeder: frame_len outside [1, 2048] or hop < 1");
    if (capacity_frames < 2) capacity_frames = 8;
    cvad_feeder *f = new cvad_feeder();
    f->eng = e;
    f->max_streams = max_streams;
    f->pcm_format = pcm_format;
    f->frame_len = frame_len;
    f->hop = hop;
    f->src_rate = src_rate;
    f->es = pcm_format == CVAD_PCM_F32 ? 4 : 2;
    f->max_step_frames = capacity_frames;
    // rows start small (the arena is max_streams rows of pinned memory) and grow when a producer runs ahead of step()
    f->cap = (size_t)frame_len + (size_t)(std::min(capacity_frames, 3) + 1) * (size_t)std::max(hop, frame_len);
    f->cap += (-(int64_t)f->cap) & 7;
    const size_t bytes = (size_t)max_streams * f->cap * f->es;
    if (e) {
        cudaSetDevice(e->device);
        void *p = nullptr;
        if (cudaMallocHost(&p, bytes) != cudaSuccess) {
            cudaGetLastError();
            delete f;
            return fail(e, CVAD_E_CUDA, "feeder: cudaMallocHost of the stream arena failed");
        }
        f->arena = static_cast<unsigned char *>(p);
    } else {
        f->arena = static_cast<unsigned char *>(std::malloc(bytes));
        if (!f->arena) { delete f; return CVAD_E_CAPACITY; }
    }
    f->slot.resize((size_t)max_streams);
    f->fill.assign((size_t)max_streams, 0);
    f->opn.assign((size_t)max_streams, 0);
    f->pay.assign((size_t)max_streams, 0);
    f->act.assign((size_t)max_streams, 0);
    f->skp.assign((size_t)max_streams, 0);
    const unsigned hw = std::thread::hardware_concurrency();
    f->threads = hw >= 16 ? 6 : (hw >= 8 ? 4 : (hw >= 4 ? 2 : 1));
    if (f->threads > 1) f->pool.reset(new FeederPool(f->threads - 1));
    f->mark.assign((size_t)max_streams, 0u);
    *out = f;
    return CVAD_OK;
}

int cvad_feeder_destroy(cvad_feeder *f) {
    if (!f) return CVAD_OK;
    for (int w = 0; w < 2; ++w)
        if (f->stage[w]) { if (f->eng) cudaFreeHost(f->stage[w]); else std::free(f->stage[w]); }
    if (f->arena) { if (f->eng) cudaFreeHost(f->arena); else std::free(f->arena); }
    delete f;
    return CVAD_OK;
}

const char *cvad_feeder_last_error(const cvad_feeder *f) { return f ? f->err.c_str() : ""; }

int cvad_feeder_open(cvad_feeder *f, int slot, int src_rate, int payload, double vad_start_probability,
                     int enable_denoising) {
    if (!f) return CVAD_E_INVALID;
    if (slot < 0 || slot >= f->max_streams) return ffail(f, CVAD_E_CAPACITY, "slot id out of range");
    if (payload < CVAD_PAYLOAD_NONE || payload > CVAD_PAYLOAD_FRAMES) return ffail(f, CVAD_E_INVALID, "unknown payload mode");
    if (src_rate == 0) src_rate = f->src_rate ? f->src_rate : 16000;
    if (f->src_rate == 0) {
        if (src_rate != 16000 && rate_index(src_rate) < 0)
            return ffail(f, CVAD_E_INVALID, "sample_rate must be 8000, 16000, 24000 or 48000");
    } else if (src_rate != f->src_rate) {
        return ffail(f, CVAD_E_INVALID, "this feeder takes one source rate for all streams");
    }
    std::lock_guard<std::mutex> lk(f->mu);
    cvad_feeder::Slot &s = f->slot[slot];
    f->opn[slot] = 1;
    f->pay[slot] = (uint8_t)payload;
    f->act[slot] = 0;
    s.rate = src_rate;
    s.n_in = rate_n_in(src_rate);
    s.denoise = enable_denoising != 0;
    s.start_p = vad_start_probability;
    f->skp[slot] = 0;
    s.pre_roll.clear();
    s.segment.clear();
    f->fill[slot] = 0;
    return CVAD_OK;
}

int cvad_feeder_close(cvad_feeder *f, int slot) {
    if (!f) return CVAD_E_INVALID;
    if (slot < 0 || slot >= f->max_streams) return ffail(f, CVAD_E_CAPACITY, "slot id out of range");
    std::lock_guard<std::mutex> lk(f->mu);
    cvad_feeder::Slot &s = f->slot[slot];
    f->opn[slot] = 0;
    f->act[slot] = 0;
    std::vector<float>().swap(s.pre_roll);
    std::vector<float>().swap(s.segment);
    f->fill[slot] = 0;
    return CVAD_OK;
}

int cvad_feeder_clear(cvad_feeder *f, int slot) {
    if (!f) return CVAD_E_INVALID;
    if (slot < 0 || slot >= f->max_streams) return ffail(f, CVAD_E_CAPACITY, "slot id out of range");
    std::lock_guard<std::mutex> lk(f->mu);
    cvad_feeder::Slot &s = f->slot[slot];
    f->act[slot] = 0;
    f->skp[slot] = 0;
    s.pre_roll.clear();
    s.segment.clear();
    f->fill[slot] = 0;
    return CVAD_OK;
}

int cvad_feeder_is_active(cvad_feeder *f, int slot) {
    if (!f || slot < 0 || slot >= f->max_streams) return CVAD_E_INVALID;
    return f->act[slot] ? 1 : 0;
}

int64_t cvad_feeder_pending(cvad_feeder *f, int slot) {
    if (!f || slot < 0 || slot >= f->max_streams) return CVAD_E_INVALID;
    std::lock_guard<std::mutex> lk(f->mu);
    return f->fill[slot];
}

// Rows grow (all of them: the arena stays one rectangular pinned block) when a producer runs ahead of step().
static int feeder_grow_arena(cvad_feeder *f, int64_t need) {
    if (need <= (int64_t)f->cap) return CVAD_OK;
    size_t cap = std::max<size_t>((size_t)need, 2 * f->cap);
    cap += (-(int64_t)cap) & 7;
    const size_t bytes = (size_t)f->max_streams * cap * f->es;
    if (bytes > kFeederArenaLimit)
        return ffail(f, CVAD_E_CAPACITY, "stream buffer full: step() the feeder before pushing more audio");
    unsigned char *p = nullptr;
    if (f->eng) {
        void *q = nullptr;
        if (cudaMallocHost(&q, bytes) != cudaSuccess) { cudaGetLastError(); return ffail(f, CVAD_E_CUDA, "cudaMallocHost failed"); }
        p = static_cast<unsigned char *>(q);
    } else {
        p = static_cast<unsigned char *>(std::malloc(bytes));
        if (!p) return ffail(f, CVAD_E_CAPACITY, "out of host memory");
    }
    for (int s = 0; s < f->max_streams; ++s)
        if (f->fill[s] > 0)
            std::memcpy(p + (size_t)s * cap * f->es, f->arena + (size_t)s * f->cap * f->es, (size_t)f->fill[s] * f->es);
    if (f->eng) cudaFreeHost(f->arena); else std::free(f->arena);
    f->arena = p;
    f->cap = cap;
    return CVAD_OK;
}

static int feeder_push_locked(cvad_feeder *f, int slot, const void *samples, int64_t n) {
    if (!f->opn[slot]) return ffail(f, CVAD_E_INVALID, "stream is not open");
    int64_t &skip = f->skp[slot];
    if (skip > 0) {
        const int64_t d = std::min(skip, n);
        samples = static_cast<const unsigned char *>(samples) + (size_t)d * f->es;
        n -= d;
        skip -= d;
        if (n == 0) return CVAD_OK;
    }
    const int64_t have = f->fill[slot];
    if (have + n > (int64_t)f->cap) {
        const int rc = feeder_grow_arena(f, have + n);
        if (rc) return rc;
    }
    std::memcpy(f->arena + ((size_t)slot * f->cap + (size_t)have) * f->es, samples, (size_t)n * f->es);
    f->fill[slot] = have + n;
    return CVAD_OK;
}

static bool feeder_all_finite(const float *x, int64_t n) {
    // AudioUtils.validate_audio_data (audio.py:227-228): exponent all ones <=> NaN or Inf
    const uint32_t *u = reinterpret_cast<const uint32_t *>(x);
    uint32_t bad = 0;
    for (int64_t i = 0; i < n; ++i) bad |= ((u[i] & 0x7f800000u) == 0x7f800000u);
    return bad == 0;
}

int cvad_feeder_push(cvad_feeder *f, int slot, const void *samples, int64_t n_samples) {
    if (!f) return CVAD_E_INVALID;
    if (slot < 0 || slot >= f->max_streams) return ffail(f, CVAD_E_CAPACITY, "slot id out of range");
    if (!samples || n_samples <= 0) return ffail(f, CVAD_E_INVALID, "Audio data is empty");
    if (f->pcm_format == CVAD_PCM_F32 && !feeder_all_finite(static_cast<const float *>(samples), n_samples))
        return ffail(f, CVAD_E_INVALID, "Audio data contains infinite or NaN values");
    std::lock_guard<std::mutex> lk(f->mu);
    return feeder_push_locked(f, slot, samples, n_samples);
}

int cvad_feeder_push_many(cvad_feeder *f, int n, const int32_t *slots, const void *block, int64_t row_stride,
                          int64_t n_samples) {
    if (!f) return CVAD_E_INVALID;
    if (n < 0 || !slots) return ffail(f, CVAD_E_INVALID, "push_many: bad slot list");
    if (!block || n_samples <= 0) return ffail(f, CVAD_E_INVALID, "Audio data is empty");
    if (row_stride < n_samples) return ffail(f, CVAD_E_INVALID, "push_many: row_stride < n_samples");
    const unsigned char *b = static_cast<const unsigned char *>(block);
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= f->max_streams) return ffail(f, CVAD_E_CAPACITY, "slot id out of range");
        if (f->pcm_format == CVAD_PCM_F32 &&
            !feeder_all_finite(reinterpret_cast<const float *>(b + (size_t)i * (size_t)row_stride * f->es), n_samples))
            return ffail(f, CVAD_E_INVALID, "Audio data contains infinite or NaN values");
    }
    std::lock_guard<std::mutex> lk(f->mu);
    int64_t need = 0;
    for (int i = 0; i < n; ++i) {
        if (!f->opn[slots[i]]) return ffail(f, CVAD_E_INVALID, "push_many: a stream is not open");
        need = std::max(need, f->fill[slots[i]] + n_samples);
    }
    if (const int rc = feeder_grow_arena(f, need)) return rc;
    // rows of distinct slots are independent (the arena has room for all of them now): copy them on the pool
    bool distinct = true;
    if (++f->mark_gen == 0u) { std::fill(f->mark.begin(), f->mark.end(), 0u); f->mark_gen = 1u; }
    for (int i = 0; i < n && distinct; ++i) {
        distinct = f->mark[slots[i]] != f->mark_gen;
        f->mark[slots[i]] = f->mark_gen;
    }
    const size_t bytes = (size_t)n * (size_t)n_samples * f->es;
    const int nt = (distinct && f->pool && bytes > (1u << 20)) ? std::min(f->threads, n) : 1;
    auto rows = [&](int i0, int i1) {
        for (int i = i0; i < i1; ++i)
            feeder_push_locked(f, slots[i], b + (size_t)i * (size_t)row_stride * f->es, n_samples);
    };
    if (nt <= 1) rows(0, n);
    else f->pool->run(nt, [&](int t) { rows((int)((int64_t)n * t / nt), (int)((int64_t)n * (t + 1) / nt)); });
    return CVAD_OK;
}

static void feeder_fill_result(cvad_feeder *f, cvad_feeder_result *r) {
    std::memset(r, 0, sizeof(*r));
    const int n = (int)f->ids.size();
    r->n_streams = n;
    r->max_frames = f->tmax;
    int64_t tot = 0;
    for (int k = 0; k < n; ++k) tot += f->counts[k];
    r->n_frames_total = tot;
    r->slots = f->ids.data();
    r->counts = f->counts.data();
    r->probs = f->probs.data();
    r->flags = f->flags.data();
    r->n_events = (int32_t)f->events.size();
    r->events = f->events.data();
    r->n_deliveries = (int32_t)f->deliveries.size();
    r->deliveries = f->deliveries.data();
    r->raw = f->planes ? nullptr : f->stage[f->cur];     // the row block (hooks, multi-frame steps); NULL after a step in rounds
    r->raw_stride = f->planes ? 0 : f->row;
}

int cvad_feeder_step(cvad_feeder *f, cvad_feeder_result *r) {
    if (!f || !r) return CVAD_E_INVALID;
    if (!f->eng) return ffail(f, CVAD_E_NOGPU, "feeder has no engine: there is no CPU fallback");
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();
    int rc = feeder_gather(f, true);
    if (rc) return rc;
    const auto t1 = clk::now();
    const int n = (int)f->ids.size(), T = f->tmax;
    f->events.clear();
    f->probs.assign((size_t)n * T, 0.f);
    f->flags.assign((size_t)n * T, 0);
    f->status.assign((size_t)n, 0);
    // A few frames per stream, most streams with fewer than the maximum (arrival jitter): frame by frame, each round
    // over the streams that still have one -- every round is a one-frame step (the fused kernel), and only round 0
    // touches every stream.  Many frames for everybody (a producer that batches) stay one multi-frame step.
    const bool rounds = n > 0 && f->planes;
    if (rounds) {
        // Round r runs the streams that hold an r-th frame.  Rounds are SUBMITTED back to back (cvad_step_submit: the engine
        // orders their kernels, the copies of round r + 1 run under the kernel of round r) and collected afterwards, so the
        // packing of round r + 1 and the unpacking of round r - 1 happen while the GPU works on round r.
        const size_t flen_al = (size_t)f->plane_row;
        struct Round {
            std::vector<int32_t> slots, k;
            std::vector<float> probs;
            std::vector<uint8_t> flags, status;
            std::vector<cvad_event> events;
            int nev = 0, ticket = -1;
        };
        std::vector<Round> rd((size_t)T);
        int n_rounds = 0;
        for (int r = 0; r < T; ++r) {
            Round &q = rd[(size_t)r];
            for (int k = 0; k < n; ++k)
                if (f->counts[k] > r) { q.k.push_back(k); q.slots.push_back(f->ids[k]); }
            if (q.k.empty()) break;
            n_rounds = r + 1;
        }
        static const bool trace = std::getenv("CVAD_FEEDER_TRACE") != nullptr;     // development aid: per-round timings on stderr
        auto collect = [&](int r) -> int {
            Round &q = rd[(size_t)r];
            const auto tc0 = clk::now();
            const int rcc = cvad_step_collect(f->eng, q.ticket);
            q.ticket = -1;
            if (trace)
                std::fprintf(stderr, "[feeder] round %d: %d streams, collect %.3f ms\n", r, (int)q.k.size(),
                             std::chrono::duration<double, std::milli>(clk::now() - tc0).count());
            if (rcc) return ffail(f, rcc, cvad_last_error(f->eng));
            const int nr = (int)q.k.size();
            for (int i = 0; i < nr; ++i) {
                if (q.status[i]) return ffail(f, CVAD_E_INVALID, "Audio data contains infinite or NaN values");
                f->probs[(size_t)q.k[i] * T + r] = q.probs[i];
                f->flags[(size_t)q.k[i] * T + r] = q.flags[i];
            }
            for (int i = 0; i < std::min(q.nev, (int)q.events.size()); ++i) {
                cvad_event ev = q.events[i];
                ev.stream = q.k[ev.stream];
                ev.frame = r;
                f->events.push_back(ev);
            }
            return CVAD_OK;
        };
        int failed = CVAD_OK;
        for (int r = 0; r < n_rounds && !failed; ++r) {
            Round &q = rd[(size_t)r];
            const auto tr0 = clk::now();
            const int nr = (int)q.k.size();
            // plane r: the r-th frames of exactly the streams of this round, in their order (feeder_gather)
            const void *audio = f->stage[f->cur] + (size_t)f->plane_off[r] * flen_al * f->es;
            q.probs.assign((size_t)nr, 0.f);
            q.flags.assign((size_t)nr, 0);
            q.status.assign((size_t)nr, 0);
            q.events.resize((size_t)std::max(16, 2 * nr));
            cvad_step_args a{};
            a.n_streams = nr;
            a.slots = q.slots.data();
            a.audio = audio;
            a.pcm_format = f->pcm_format;
            a.stream_stride = (int64_t)flen_al;
            a.max_frames = 1;
            a.frame_len = f->frame_len;
            a.hop = f->hop;
            a.src_rate = f->src_rate;
            a.probs_out = q.probs.data();
            a.flags_out = q.flags.data();
            a.status_out = q.status.data();
            a.events_out = q.events.data();
            a.max_events = (int32_t)q.events.size();
            a.n_events_out = &q.nev;
            const auto tr1 = clk::now();
            rc = cvad_step_submit(f->eng, &a, &q.ticket);
            if (trace)
                std::fprintf(stderr, "[feeder] round %d: %d streams, prepare %.3f ms, submit %.3f ms\n", r, nr,
                             std::chrono::duration<double, std::milli>(tr1 - tr0).count(),
                             std::chrono::duration<double, std::milli>(clk::now() - tr1).count());
            if (rc) { q.ticket = -1; failed = ffail(f, rc, cvad_last_error(f->eng)); break; }
            if (r > 0) failed = collect(r - 1);
        }
        // the last round (and, after a failure, whatever is still in flight: its buffers must outlive the copies)
        for (int r = 0; r < n_rounds; ++r)
            if (rd[(size_t)r].ticket >= 0) {
                const int rcc = collect(r);
                if (!failed) failed = rcc;
            }
        if (failed) { f->events.clear(); return failed; }
        std::sort(f->events.begin(), f->events.end(), [](const cvad_event &x, const cvad_event &y) {
            if (x.stream != y.stream) return x.stream < y.stream;
            if (x.frame != y.frame) return x.frame < y.frame;
            return x.kind < y.kind;
        });
    } else if (n > 0) {
        const int max_events = std::max(16, 2 * n * T);
        f->events.resize((size_t)max_events);
        int nev = 0;
        cvad_step_args a{};
        a.n_streams = n;
        a.slots = f->ids.data();
        a.audio = f->stage[f->cur];
        a.pcm_format = f->pcm_format;
        a.stream_stride = f->row;
        a.n_frames = f->counts.data();
        a.max_frames = T;
        a.frame_len = f->frame_len;
        a.hop = f->hop;
        a.src_rate = f->src_rate ? f->src_rate : 16000;
        a.src_rates = f->src_rate == 0 ? f->rates.data() : nullptr;
        a.probs_out = f->probs.data();
        a.flags_out = f->flags.data();
        a.status_out = f->status.data();
        a.events_out = f->events.data();
        a.max_events = max_events;
        a.n_events_out = &nev;
        rc = cvad_step(f->eng, &a);
        if (rc) { f->events.clear(); return ffail(f, rc, cvad_last_error(f->eng)); }
        f->events.resize((size_t)std::min(nev, max_events));
        for (int k = 0; k < n; ++k)
            if (f->status[k]) {   // cannot happen through cvad_feeder_push (it validates), kept for raw arena writers
                f->events.clear();
                return ffail(f, CVAD_E_INVALID, "Audio data contains infinite or NaN values");
            }
    }
    const auto t2 = clk::now();
    feeder_deliver(f);
    feeder_fill_result(f, r);
    const auto t3 = clk::now();
    r->gather_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    r->gpu_ms = std::chrono::duration<double, std::milli>(t2 - t1).count();
    r->deliver_ms = std::chrono::duration<double, std::milli>(t3 - t2).count();
    return CVAD_OK;
}

/* Test hooks for hosts without a GPU: the two host phases of cvad_feeder_step on their own. */
int cvad_feeder_gather_only(cvad_feeder *f, cvad_feeder_result *r) {
    if (!f || !r) return CVAD_E_INVALID;
    int rc = feeder_gather(f);
    if (rc) return rc;
    const int n = (int)f->ids.size(), T = f->tmax;
    f->events.clear();
    f->deliveries.clear();
    f->probs.assign((size_t)n * T, 0.f);
    f->flags.assign((size_t)n * T, 0);
    feeder_fill_result(f, r);
    return CVAD_OK;
}

int cvad_feeder_deliver_only(cvad_feeder *f, const float *probs, const uint8_t *flags, cvad_feeder_result *r) {
    if (!f || !r || !probs || !flags) return CVAD_E_INVALID;
    const int n = (int)f->ids.size(), T = f->tmax;
    f->probs.assign(probs, probs + (size_t)n * T);
    f->flags.assign(flags, flags + (size_t)n * T);
    feeder_deliver(f);
    feeder_fill_result(f, r);
    return CVAD_OK;
}

}  // extern "C"

// ---- row snapshots (layout in include/cutter_vad_b200.h, above cvad_feeder_export)
namespace {

struct SnapHeader {
    uint32_t magic, version;
    int32_t pcm_format, frame_len, hop, src_rate, n, zero;
};
struct SnapRow {
    int32_t rate, n_in, payload, denoise;
    double start_p;
    int32_t active, zero;
    int64_t skip, n_pending, n_pre_roll, n_segment;
};
static_assert(sizeof(SnapHeader) == 32 && sizeof(SnapRow) == 64, "feeder snapshot layout");

// range and distinctness of a slot list (mark / mark_gen as in push_many; caller holds the lock)
int feeder_check_slots(cvad_feeder *f, int n, const int32_t *slots) {
    if (n < 0 || (n > 0 && !slots)) return ffail(f, CVAD_E_INVALID, "bad slot list");
    if (++f->mark_gen == 0u) { std::fill(f->mark.begin(), f->mark.end(), 0u); f->mark_gen = 1u; }
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= f->max_streams) return ffail(f, CVAD_E_CAPACITY, "slot id out of range");
        if (f->mark[slots[i]] == f->mark_gen) return ffail(f, CVAD_E_INVALID, "slot " + std::to_string(slots[i]) + " is listed twice");
        f->mark[slots[i]] = f->mark_gen;
    }
    return CVAD_OK;
}

}  // namespace

extern "C" {

int cvad_feeder_export(cvad_feeder *f, int n, const int32_t *slots, void *out, size_t out_bytes, size_t *needed) {
    if (!f) return CVAD_E_INVALID;
    std::lock_guard<std::mutex> lk(f->mu);
    if (const int rc = feeder_check_slots(f, n, slots)) return rc;
    size_t total = sizeof(SnapHeader);
    for (int i = 0; i < n; ++i) {
        const int s = slots[i];
        if (!f->opn[s]) return ffail(f, CVAD_E_INVALID, "export: stream " + std::to_string(s) + " is not open");
        total += sizeof(SnapRow) + (size_t)f->fill[s] * f->es +
                 (f->slot[s].pre_roll.size() + f->slot[s].segment.size()) * sizeof(float);
    }
    if (needed) *needed = total;
    if (!out) return CVAD_OK;
    if (out_bytes < total) return ffail(f, CVAD_E_CAPACITY, "export: out_bytes < needed");
    unsigned char *p = static_cast<unsigned char *>(out);
    const SnapHeader hd{CVAD_FEEDER_SNAPSHOT_MAGIC, CVAD_FEEDER_SNAPSHOT_VERSION, f->pcm_format, f->frame_len, f->hop,
                        f->src_rate, n, 0};
    std::memcpy(p, &hd, sizeof(hd));
    p += sizeof(hd);
    for (int i = 0; i < n; ++i) {
        const int s = slots[i];
        const cvad_feeder::Slot &sl = f->slot[s];
        const SnapRow r{sl.rate, sl.n_in, f->pay[s], sl.denoise ? 1 : 0, sl.start_p, f->act[s] ? 1 : 0, 0, f->skp[s],
                        f->fill[s], (int64_t)sl.pre_roll.size(), (int64_t)sl.segment.size()};
        std::memcpy(p, &r, sizeof(r));
        p += sizeof(r);
        const size_t pb = (size_t)f->fill[s] * f->es;
        if (pb) std::memcpy(p, f->arena + (size_t)s * f->cap * f->es, pb);
        p += pb;
        if (!sl.pre_roll.empty()) std::memcpy(p, sl.pre_roll.data(), sl.pre_roll.size() * sizeof(float));
        p += sl.pre_roll.size() * sizeof(float);
        if (!sl.segment.empty()) std::memcpy(p, sl.segment.data(), sl.segment.size() * sizeof(float));
        p += sl.segment.size() * sizeof(float);
    }
    return CVAD_OK;
}

int cvad_feeder_import(cvad_feeder *f, int n, const int32_t *slots, const void *in, size_t in_bytes) {
    if (!f) return CVAD_E_INVALID;
    if (!in) return ffail(f, CVAD_E_INVALID, "import: blob is NULL");
    std::lock_guard<std::mutex> lk(f->mu);
    if (const int rc = feeder_check_slots(f, n, slots)) return rc;
    // the whole blob is checked before any slot changes
    const unsigned char *b = static_cast<const unsigned char *>(in);
    SnapHeader hd{};
    if (in_bytes < sizeof(hd)) return ffail(f, CVAD_E_INVALID, "import: blob shorter than its header");
    std::memcpy(&hd, b, sizeof(hd));
    if (hd.magic != CVAD_FEEDER_SNAPSHOT_MAGIC) return ffail(f, CVAD_E_INVALID, "import: not a feeder snapshot (bad magic)");
    if (hd.version != CVAD_FEEDER_SNAPSHOT_VERSION)
        return ffail(f, CVAD_E_INVALID, "import: feeder snapshot version " + std::to_string(hd.version) + " is not supported");
    if (hd.pcm_format != f->pcm_format) return ffail(f, CVAD_E_INVALID, "import: the blob's PCM format differs from this feeder's");
    if (hd.src_rate != f->src_rate || hd.frame_len != f->frame_len || hd.hop != f->hop)
        return ffail(f, CVAD_E_INVALID, "import: the blob's framing (frame_len, hop, source rate) differs from this feeder's");
    if (hd.n != n) return ffail(f, CVAD_E_INVALID, "import: the blob holds " + std::to_string(hd.n) + " rows, not n");
    std::vector<size_t> at((size_t)n);
    size_t pos = sizeof(hd);
    int64_t longest = 0;
    for (int i = 0; i < n; ++i) {
        SnapRow r{};
        if (in_bytes - pos < sizeof(r)) return ffail(f, CVAD_E_INVALID, "import: blob truncated at row " + std::to_string(i));
        std::memcpy(&r, b + pos, sizeof(r));
        at[(size_t)i] = pos;
        const std::string row = "import: row " + std::to_string(i) + ": ";
        const int want_rate = f->src_rate ? f->src_rate : r.rate;
        if (r.rate != want_rate || (r.rate != 16000 && rate_index(r.rate) < 0))
            return ffail(f, CVAD_E_INVALID, row + "source rate " + std::to_string(r.rate) + " does not fit this feeder");
        if (r.n_in != rate_n_in(r.rate)) return ffail(f, CVAD_E_INVALID, row + "n_in does not match its rate");
        if (r.payload < CVAD_PAYLOAD_NONE || r.payload > CVAD_PAYLOAD_FRAMES) return ffail(f, CVAD_E_INVALID, row + "unknown payload mode");
        if ((r.denoise != 0 && r.denoise != 1) || (r.active != 0 && r.active != 1) || !(r.start_p >= 0.0 && r.start_p <= 1.0))
            return ffail(f, CVAD_E_INVALID, row + "bad denoise / active flag or start probability");
        if (r.skip < 0 || r.n_pending < 0 || r.n_pre_roll < 0 || r.n_segment < 0)
            return ffail(f, CVAD_E_INVALID, row + "negative length");
        pos += sizeof(r);
        const uint64_t tail = (uint64_t)r.n_pending * f->es + ((uint64_t)r.n_pre_roll + (uint64_t)r.n_segment) * sizeof(float);
        if ((uint64_t)(in_bytes - pos) < tail || r.n_pending > (int64_t)(in_bytes / f->es) ||
            r.n_pre_roll > (int64_t)in_bytes || r.n_segment > (int64_t)in_bytes)
            return ffail(f, CVAD_E_INVALID, row + "blob truncated");
        pos += (size_t)tail;
        longest = std::max(longest, r.n_pending);
    }
    if (pos != in_bytes) return ffail(f, CVAD_E_INVALID, "import: " + std::to_string(in_bytes - pos) + " bytes after the last row");
    if (const int rc = feeder_grow_arena(f, longest)) return rc;
    for (int i = 0; i < n; ++i) {
        SnapRow r{};
        std::memcpy(&r, b + at[(size_t)i], sizeof(r));
        const unsigned char *p = b + at[(size_t)i] + sizeof(r);
        const int s = slots[i];
        cvad_feeder::Slot &sl = f->slot[s];
        f->opn[s] = 1;
        f->pay[s] = (uint8_t)r.payload;
        f->act[s] = (uint8_t)r.active;
        f->skp[s] = r.skip;
        sl.rate = r.rate;
        sl.n_in = r.n_in;
        sl.denoise = r.denoise != 0;
        sl.start_p = r.start_p;
        const size_t pb = (size_t)r.n_pending * f->es;
        if (pb) std::memcpy(f->arena + (size_t)s * f->cap * f->es, p, pb);
        f->fill[s] = r.n_pending;
        p += pb;
        // a row that carries no audio keeps none (its payload mode may have been lowered since the export)
        const bool audio = r.payload >= CVAD_PAYLOAD_SEGMENTS;
        sl.pre_roll.resize(audio ? (size_t)r.n_pre_roll : 0);
        if (!sl.pre_roll.empty()) std::memcpy(sl.pre_roll.data(), p, sl.pre_roll.size() * sizeof(float));
        p += (size_t)r.n_pre_roll * sizeof(float);
        sl.segment.resize(audio ? (size_t)r.n_segment : 0);
        if (!sl.segment.empty()) std::memcpy(sl.segment.data(), p, sl.segment.size() * sizeof(float));
    }
    return CVAD_OK;
}

}  // extern "C"
