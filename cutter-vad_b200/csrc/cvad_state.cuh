// cvad_state.cuh -- bulk export / import of per-slot state as cvad_stream_state records (stream snapshots).
//
// A slot's state is spread over the engine's arrays: h / c in the [slot / 8][128][slot % 8] layout of cvad::state_at,
// one word per slot for the state machine, frames_done and the thresholds.  export_states_kernel gathers it into
// records, import_states_kernel scatters records back; both walk the records as 268 consecutive 4-byte words, so the
// record side (the side a copy reads or writes) is coalesced and the state side is 4-byte gathers, which is fine at
// ~1 KB per stream.  validate_states_kernel runs before every import: one warp per record, and the first bad record's
// index is kept with an atomicMin, so that the scatter runs only when every record passed.
// Included by cvad_capi.cu (one translation unit), after quiesce / stage_slots.
#pragma once

static_assert(sizeof(cvad_stream_state) == 1072, "cvad_stream_state must be 1,072 bytes without padding");
static_assert(offsetof(cvad_stream_state, frames_done) == 1024 && offsetof(cvad_stream_state, is_voice_active) == 1048 &&
              offsetof(cvad_stream_state, enable_denoising) == 1068, "cvad_stream_state layout");

namespace {

constexpr int kRecWords = (int)(sizeof(cvad_stream_state) / 4);   // 268
constexpr unsigned kNoBadRecord = 0xFFFFFFFFu;

struct StateArrays {
    float *h, *c;
    int *act, *sc, *ec, *n_start, *n_end;
    long long *fd;
    double *start_p, *end_p;
    unsigned char *denoise;
};

StateArrays state_arrays(cvad_engine *e) {
    return {e->h_state, e->c_state, e->sm_active, e->sm_scount, e->sm_ecount, e->n_start, e->n_end,
            e->frames_done, e->start_p, e->end_p, e->denoise};
}

// record word w of slot `slot` (the 64-bit fields are two little-endian words each)
__device__ __forceinline__ uint32_t state_word(const StateArrays &S, int slot, int w) {
    if (w < 128) return __float_as_uint(S.h[cvad::state_at(w, slot)]);
    if (w < 256) return __float_as_uint(S.c[cvad::state_at(w - 128, slot)]);
    switch (w) {
        case 256: case 257: return reinterpret_cast<const uint32_t *>(S.fd + slot)[w - 256];
        case 258: case 259: return reinterpret_cast<const uint32_t *>(S.start_p + slot)[w - 258];
        case 260: case 261: return reinterpret_cast<const uint32_t *>(S.end_p + slot)[w - 260];
        case 262: return (uint32_t)S.act[slot];
        case 263: return (uint32_t)S.sc[slot];
        case 264: return (uint32_t)S.ec[slot];
        case 265: return (uint32_t)S.n_start[slot];
        case 266: return (uint32_t)S.n_end[slot];
        default: return (uint32_t)S.denoise[slot];
    }
}

__device__ __forceinline__ void set_state_word(const StateArrays &S, int slot, int w, uint32_t v) {
    if (w < 128) { S.h[cvad::state_at(w, slot)] = __uint_as_float(v); return; }
    if (w < 256) { S.c[cvad::state_at(w - 128, slot)] = __uint_as_float(v); return; }
    switch (w) {
        case 256: case 257: reinterpret_cast<uint32_t *>(S.fd + slot)[w - 256] = v; break;
        case 258: case 259: reinterpret_cast<uint32_t *>(S.start_p + slot)[w - 258] = v; break;
        case 260: case 261: reinterpret_cast<uint32_t *>(S.end_p + slot)[w - 260] = v; break;
        case 262: S.act[slot] = (int)v; break;
        case 263: S.sc[slot] = (int)v; break;
        case 264: S.ec[slot] = (int)v; break;
        case 265: S.n_start[slot] = (int)v; break;
        case 266: S.n_end[slot] = (int)v; break;
        default: S.denoise[slot] = (unsigned char)v; break;
    }
}

// records k = 0..n-1 of slots[k] (slots == nullptr: first + k)
__global__ void export_states_kernel(StateArrays S, const int *slots, int first, int n, uint32_t *out) {
    const long long total = (long long)n * kRecWords;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i / kRecWords), w = (int)(i - (long long)k * kRecWords);
        out[i] = state_word(S, slots ? slots[k] : first + k, w);
    }
}

__global__ void import_states_kernel(StateArrays S, const int *slots, int n, const uint32_t *in) {
    const long long total = (long long)n * kRecWords;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i / kRecWords), w = (int)(i - (long long)k * kRecWords);
        set_state_word(S, slots ? slots[k] : k, w, in[i]);
    }
}

// one warp per record; *first_bad = the smallest index of a record that breaks a rule (kNoBadRecord when none does)
__global__ void validate_states_kernel(const cvad_stream_state *in, int n, unsigned *first_bad) {
    const int k = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (k >= n) return;
    const cvad_stream_state &r = in[k];
    bool ok = true;
    for (int j = lane; j < 128; j += 32) ok = ok && isfinite(r.h[j]) && isfinite(r.c[j]);
    if (lane == 0) {
        ok = ok && (r.is_voice_active == 0 || r.is_voice_active == 1) && r.voice_start_frame_count >= 0 &&
             r.voice_end_frame_count >= 0 && r.frames_done >= 0 && r.vad_start_probability >= 0.0 &&
             r.vad_start_probability <= 1.0 && r.vad_end_probability >= 0.0 && r.vad_end_probability <= 1.0 &&
             r.n_start >= 1 && r.n_end >= 1 && (r.enable_denoising == 0 || r.enable_denoising == 1);
    }
    if (!__all_sync(0xFFFFFFFFu, ok) && lane == 0) atomicMin(first_bad, (unsigned)k);
}

int state_grid(cvad_engine *e, int n) {
    const long long blocks = ((long long)n * kRecWords + 255) / 256;
    return (int)std::min<long long>(std::max<long long>(blocks, 1), (long long)e->num_sms * 16);
}

// where a caller's record buffer lives: 0 = pageable host, 1 = pinned host, 2 = device memory of the engine's device
int record_buffer_kind(cvad_engine *e, const void *p, int *kind) {
    if (is_host_pinned_or_device(p, true)) {
        cudaPointerAttributes at{};
        CU_TRY(e, cudaPointerGetAttributes(&at, p));
        if (at.device != e->device)
            return fail(e, CVAD_E_INVALID, "records are in device memory of another device: copy them to the engine's device first");
        // the kernels read and write device records in place, with 8-byte loads of frames_done and the probabilities
        if (reinterpret_cast<uintptr_t>(p) % alignof(cvad_stream_state) != 0)
            return fail(e, CVAD_E_INVALID, "device records must be 8-byte aligned");
        *kind = 2;
    } else {
        *kind = is_host_pinned_or_device(p, false) ? 1 : 0;
    }
    return CVAD_OK;
}

// range and distinctness of a host slot list, then its device copy (nullptr for slots == nullptr)
int stage_state_slots(cvad_engine *e, int n, const int32_t *slots, const int **d_slots) {
    *d_slots = nullptr;
    if (!slots) {
        if (n > e->max_streams) return fail(e, CVAD_E_CAPACITY, "n exceeds max_streams");
        return CVAD_OK;
    }
    std::vector<uint8_t> seen((size_t)e->max_streams, 0);
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= e->max_streams) return fail(e, CVAD_E_CAPACITY, "slot id out of range");
        if (seen[(size_t)slots[i]]) return fail(e, CVAD_E_INVALID, "slot " + std::to_string(slots[i]) + " is listed twice");
        seen[(size_t)slots[i]] = 1;
    }
    return stage_slots(e, n, slots, d_slots);
}

}  // namespace

extern "C" {

int cvad_model_fingerprint(const cvad_engine *e, uint64_t *out) {
    if (!e || !out) return CVAD_E_INVALID;
    *out = e->fingerprint;
    return CVAD_OK;
}

int cvad_export_states(cvad_engine *e, int n, const int32_t *slots, cvad_stream_state *out) {
    if (!e) return CVAD_E_INVALID;
    if (n < 0) return fail(e, CVAD_E_INVALID, "n < 0");
    if (n == 0) return CVAD_OK;
    if (!out) return fail(e, CVAD_E_INVALID, "out is NULL");
    CU_TRY(e, cudaSetDevice(e->device));
    int rc = quiesce(e);
    if (rc) return rc;
    int kind = 0;
    const int *ds = nullptr;
    if ((rc = record_buffer_kind(e, out, &kind)) || (rc = stage_state_slots(e, n, slots, &ds))) return rc;
    const size_t bytes = (size_t)n * sizeof(cvad_stream_state);
    uint32_t *dst = reinterpret_cast<uint32_t *>(out);
    if (kind != 2) {
        if ((rc = grow(e, e->d_state_blk, bytes))) return rc;
        dst = static_cast<uint32_t *>(e->d_state_blk.p);
    }
    export_states_kernel<<<state_grid(e, n), 256, 0, e->stream>>>(state_arrays(e), ds, 0, n, dst);
    CU_TRY(e, cudaGetLastError());
    if (kind == 1) {
        CU_TRY(e, cudaMemcpyAsync(out, dst, bytes, cudaMemcpyDeviceToHost, e->stream));
    } else if (kind == 0) {
        if ((rc = grow_host(e, e->h_state_blk, bytes))) return rc;
        CU_TRY(e, cudaMemcpyAsync(e->h_state_blk.p, dst, bytes, cudaMemcpyDeviceToHost, e->stream));
    }
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    if (kind == 0) std::memcpy(out, e->h_state_blk.p, bytes);
    return CVAD_OK;
}

int cvad_import_states(cvad_engine *e, int n, const int32_t *slots, const cvad_stream_state *in) {
    if (!e) return CVAD_E_INVALID;
    if (n < 0) return fail(e, CVAD_E_INVALID, "n < 0");
    if (n == 0) return CVAD_OK;
    if (!in) return fail(e, CVAD_E_INVALID, "in is NULL");
    CU_TRY(e, cudaSetDevice(e->device));
    int rc = quiesce(e);
    if (rc) return rc;
    int kind = 0;
    const int *ds = nullptr;
    if ((rc = record_buffer_kind(e, in, &kind)) || (rc = stage_state_slots(e, n, slots, &ds))) return rc;
    // 1. the records on the device (device input is read in place), the check word behind them
    const size_t bytes = (size_t)n * sizeof(cvad_stream_state);          // a multiple of 16
    const size_t at = kind == 2 ? 0 : bytes;
    if ((rc = grow(e, e->d_state_blk, at + 16))) return rc;
    unsigned char *blk = static_cast<unsigned char *>(e->d_state_blk.p);
    const cvad_stream_state *rec = kind == 2 ? in : reinterpret_cast<const cvad_stream_state *>(blk);
    unsigned *d_bad = reinterpret_cast<unsigned *>(blk + at);
    if (kind == 1) {
        CU_TRY(e, cudaMemcpyAsync(blk, in, bytes, cudaMemcpyHostToDevice, e->stream));
    } else if (kind == 0) {
        if ((rc = grow_host(e, e->h_state_blk, bytes))) return rc;
        std::memcpy(e->h_state_blk.p, in, bytes);
        CU_TRY(e, cudaMemcpyAsync(blk, e->h_state_blk.p, bytes, cudaMemcpyHostToDevice, e->stream));
    }
    CU_TRY(e, cudaMemsetAsync(d_bad, 0xFF, sizeof(unsigned), e->stream));
    // 2. every record is checked before any slot is written
    validate_states_kernel<<<(unsigned)(((long long)n * 32 + 255) / 256), 256, 0, e->stream>>>(rec, n, d_bad);
    CU_TRY(e, cudaGetLastError());
    unsigned bad = 0;
    CU_TRY(e, cudaMemcpyAsync(&bad, d_bad, sizeof(unsigned), cudaMemcpyDeviceToHost, e->stream));
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    if (bad != kNoBadRecord)
        return fail(e, CVAD_E_INVALID, "import: record " + std::to_string(bad) +
                    " is invalid (h and c must be finite, is_voice_active and enable_denoising 0 or 1, counts and"
                    " frames_done >= 0, probabilities within [0, 1], n_start and n_end >= 1); no slot was changed");
    // 3. all passed: scatter
    import_states_kernel<<<state_grid(e, n), 256, 0, e->stream>>>(state_arrays(e), ds, n,
                                                                   reinterpret_cast<const uint32_t *>(rec));
    CU_TRY(e, cudaGetLastError());
    CU_TRY(e, cudaStreamSynchronize(e->stream));
    return CVAD_OK;
}

}  // extern "C"
