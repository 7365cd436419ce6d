// cvad_pack.cuh -- the bytes the kernels read: the canonical weight blobs and the resampling operators repacked into
// the kernels' streaming layouts.  Each layout fact is stated once here: the v5 blob view (V5Blob), the FP32 STFT
// column order (put_stft_fp32), the tensor-core STFT row map (stft_tiles), the v5 tile order (v5_tiles), the split of a
// weight into BF16 or FP16 parts (emit_tiles, with the SWIZZLE_128B offset of cvad::tc::sw128_offset) and the
// resampling operator (build_resample_operator).
// Included by cvad_capi.cu (one translation unit) after the kernel headers whose sizes it uses; plain C++17 plus the
// host conversions of cuda_fp16.h, no device code.  Device allocation and upload stay in cvad_capi.cu.
#pragma once

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include <cuda_fp16.h>

namespace {

// ---- canonical v5 blob (include/cutter_vad_b200.h, oracle/silero_ref.c), viewed as named arrays
struct V5Blob {
    const float *basis;                              // [258][256]
    const float *e0w, *e0b;                          // [128][129][3]
    const float *e1w, *e1b;                          // [64][128][3]
    const float *e2w, *e2b;                          // [64][64][3]
    const float *e3w, *e3b;                          // [128][64][3]
    const float *wih, *whh, *bih, *bhh;              // [512][128] x 2, [512] x 2 (gates i, f, g, o)
    const float *decw, *decb;                        // [128], [1]

    explicit V5Blob(const float *p) {
        auto take = [&](size_t n) { const float *r = p; p += n; return r; };
        basis = take(258 * 256);
        e0w = take(128 * 129 * 3); e0b = take(128);
        e1w = take(64 * 128 * 3); e1b = take(64);
        e2w = take(64 * 64 * 3); e2b = take(64);
        e3w = take(128 * 64 * 3); e3b = take(128);
        wih = take(512 * 128); whh = take(512 * 128); bih = take(512); bhh = take(512);
        decw = take(128); decb = take(1);
    }
};

// ---- FP32 kernels (cvad_v5.cuh, cvad_v4.cuh)
struct Fp32Packed {
    std::vector<float> w_fe, b_fe, w_rec, b_rec, w_dec;
};

// The STFT basis [258][256] as the FP32 front ends stream it: [k][n], output column n = basis row 0 (n = 0), 128 (n = 1),
// then the real and imaginary parts of bins 1..127 interleaved
void put_stft_fp32(float *o, const float *basis) {
    for (int k = 0; k < 256; ++k)
        for (int n = 0; n < 256; ++n) {
            int row;
            if (n == 0) row = 0;
            else if (n == 1) row = 128;
            else row = (n & 1) ? 129 + (n >> 1) : (n >> 1);
            o[k * 256 + n] = basis[row * 256 + k];
        }
}

Fp32Packed pack_v5(const float *blob) {
    const V5Blob b(blob);
    Fp32Packed P;
    P.w_fe.assign(cvad::kFeStreamFloats, 0.f);
    float *o = P.w_fe.data();
    put_stft_fp32(o, b.basis);
    o += 65536;
    for (int c = 0; c < 129; ++c)
        for (int t = 0; t < 3; ++t)
            for (int oc = 0; oc < 128; ++oc) o[(c * 3 + t) * 128 + oc] = b.e0w[(oc * 129 + c) * 3 + t];
    o += 129 * 384;
    for (int c = 0; c < 128; ++c)
        for (int t = 0; t < 3; ++t)
            for (int oc = 0; oc < 64; ++oc) o[(c * 3 + t) * 64 + oc] = b.e1w[(oc * 128 + c) * 3 + t];
    o += 128 * 192;
    for (int c = 0; c < 64; ++c)
        for (int t = 0; t < 2; ++t)
            for (int oc = 0; oc < 64; ++oc) o[(c * 2 + t) * 64 + oc] = b.e2w[(oc * 64 + c) * 3 + (t + 1)];
    o += 64 * 128;
    for (int c = 0; c < 64; ++c)
        for (int oc = 0; oc < 128; ++oc) o[c * 128 + oc] = b.e3w[(oc * 64 + c) * 3 + 1];

    P.b_fe.resize(cvad::kFeBiasFloats);
    std::memcpy(P.b_fe.data(), b.e0b, 128 * 4);
    std::memcpy(P.b_fe.data() + 128, b.e1b, 64 * 4);
    std::memcpy(P.b_fe.data() + 192, b.e2b, 64 * 4);
    std::memcpy(P.b_fe.data() + 256, b.e3b, 128 * 4);

    P.w_rec.resize(cvad::kRecStreamFloats);
    P.b_rec.resize(512);
    for (int n = 0; n < 512; ++n) {
        const int unit = n >> 2, gate = n & 3;
        const int row = gate * 128 + unit;
        for (int k = 0; k < 128; ++k) {
            P.w_rec[k * 512 + n] = b.wih[row * 128 + k];
            P.w_rec[(128 + k) * 512 + n] = b.whh[row * 128 + k];
        }
        P.b_rec[n] = b.bih[row] + b.bhh[row];
    }
    P.w_dec.resize(129);
    std::memcpy(P.w_dec.data(), b.decw, 128 * 4);
    P.w_dec[128] = b.decb[0];
    return P;
}

// ---- v4 weight repack (canonical blob order: oracle/silero_ref.c "Silero VAD v4")
Fp32Packed pack_v4(const float *blob) {
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

    Fp32Packed P;
    P.w_fe.assign(cvad::kV4FeStreamFloats, 0.f);
    put_stft_fp32(P.w_fe.data(), basis);
    float *o = P.w_fe.data() + cvad::kV4OffFirst;
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

// ---- tensor-core operands: (rows x 64 K) tiles of 16-bit parts in the SWIZZLE_128B K-major layout
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

// How a weight w is split into parts: each part is w's remainder rounded to nearest (BF16, or FP16 after scaling w by
// the power of two `scale`), the next part takes what it left.  BF16 x 3 holds w to 24 bits, FP16 x 2 to 22.
struct Parts {
    int n;
    bool fp16;
    float scale;   // FP16 only
};
constexpr Parts kBf16x3{3, false, 1.f}, kBf16x1{1, false, 1.f};
Parts fp16x2(float scale) { return {2, true, scale}; }

// Append the part tiles of W(r, k), r < rows, k in [k0, k0 + 64): part p of every weight forms one tile, the parts one
// after another
template <typename F>
void emit_tiles(std::vector<unsigned char> &out, const Parts &p, int rows, int k0, F W) {
    const size_t tile = (size_t)rows * 128;
    const size_t at = out.size();
    out.resize(at + p.n * tile, 0);
    for (int r = 0; r < rows; ++r)
        for (int kk = 0; kk < 64; ++kk) {
            float x = p.fp16 ? W(r, k0 + kk) * p.scale : W(r, k0 + kk);
            const size_t off = at + cvad::tc::sw128_offset((uint32_t)r, (uint32_t)kk, (uint32_t)rows);
            for (int part = 0; part < p.n; ++part) {
                uint16_t b;
                if (p.fp16) {
                    const __half h = __float2half_rn(x);
                    b = __half_as_ushort(h);
                    x -= __half2float(h);
                } else {
                    b = bf16_rn_bits(x);
                    x -= bf16_val(b);
                }
                std::memcpy(&out[off + part * tile], &b, 2);
            }
        }
}

// Scale that brings maxabs to [2^14, 2^15), and its inverse
float pow2_scale_for(float maxabs, float *inv) {
    if (!(maxabs > 0.f)) { *inv = 1.f; return 1.f; }
    int ex;
    std::frexp(maxabs, &ex);                 // maxabs = m * 2^ex, m in [0.5, 1)  ->  maxabs in [2^(ex-1), 2^ex)
    const float s = std::ldexp(1.0f, 15 - ex);
    *inv = std::ldexp(1.0f, ex - 15);
    return s;
}

// The tensor-core STFT block (v5's front end and v4tc_stft_kernel): blk 0 = basis rows 0..127 (re bins 0..127), blk 1 =
// row 128 (re bin 128), then rows 130..256 (im bins 1..127); each blk as K blocks 0..3.  tile(layer, rows, k0, W) as in
// v5_tiles; `basis` is any [258][256] array in the basis' row order.
template <typename Tile>
void stft_tiles(const float *basis, Tile &&tile) {
    for (int blk = 0; blk < 2; ++blk)
        for (int kb = 0; kb < 4; ++kb)
            tile(0, 128, kb * 64, [&](int m, int k) {
                const int row = blk == 0 ? m : (m == 0 ? 128 : 129 + m);
                return basis[row * 256 + k];
            });
}

// The v5 tensor-core tiles in the order cvad_v5tc.cuh consumes them: tile(layer, rows, k0, W) for each (rows x 64 K)
// tile of element function W(row, k).  Layers index the per-layer scales: 0 STFT, 1..4 enc0..enc3 (the front-end stream),
// 5 W_ih and 6 W_hh (the recurrent stream: gate x kb, K = [x 128 | h 128]).
template <typename Tile>
void v5_tiles(const V5Blob &b, Tile &&tile) {
    stft_tiles(b.basis, tile);
    static const int taps0[3] = {1, 0, 2}, taps1[3] = {1, 2, 0};
    for (int kb = 0; kb < 2; ++kb)
        for (int ti = 0; ti < 3; ++ti)
            tile(1, 128, kb * 64, [&](int o, int c) { return b.e0w[(o * 129 + c) * 3 + taps0[ti]]; });
    for (int kb = 0; kb < 2; ++kb)
        for (int ti = 0; ti < 3; ++ti)
            tile(2, 64, kb * 64, [&](int o, int c) { return b.e1w[(o * 128 + c) * 3 + taps1[ti]]; });
    for (int tap = 1; tap <= 2; ++tap)
        tile(3, 64, 0, [&](int o, int c) { return b.e2w[(o * 64 + c) * 3 + tap]; });
    tile(4, 128, 0, [&](int o, int c) { return b.e3w[(o * 64 + c) * 3 + 1]; });
    for (int g = 0; g < 4; ++g)
        for (int kb = 0; kb < 4; ++kb)
            tile(kb < 2 ? 5 : 6, 128, kb * 64, [&](int u, int k) {
                const int row = g * 128 + u;
                return k < 128 ? b.wih[row * 128 + k] : b.whh[row * 128 + (k - 128)];
            });
}

// ---- v5 tensor-core repack: every GEMM weight as three BF16 parts, plus the FP32 side tables
struct V5TcPacked {
    std::vector<unsigned char> w_fe, w_rec;
    std::vector<float> nyq_w, b_rec;
};

V5TcPacked pack_v5_tc(const float *blob) {
    const V5Blob b(blob);
    V5TcPacked P;
    P.w_fe.reserve(cvad::tc5::kFeStreamBytes);
    v5_tiles(b, [&](int layer, int rows, int k0, auto W) { emit_tiles(layer < 5 ? P.w_fe : P.w_rec, kBf16x3, rows, k0, W); });
    P.nyq_w.assign(128 * 4, 0.f);
    for (int o = 0; o < 128; ++o)
        for (int t = 0; t < 3; ++t) P.nyq_w[o * 4 + t] = b.e0w[(o * 129 + 128) * 3 + t];
    P.b_rec.resize(512);
    for (int n = 0; n < 512; ++n) P.b_rec[n] = b.bih[n] + b.bhh[n];
    return P;
}

// ---- v5 FP16-split repack (CVAD_MATH_TC16): the same tile order with TWO FP16 parts per weight, every layer scaled
// by the power of two that brings its largest weight to [2^14, 2^15) (inverse returned in inv_w: stft, enc0..3, W_ih, W_hh)
struct V5HPacked {
    std::vector<unsigned char> w_fe, w_rec;
    float inv_w[8] = {0};
};

V5HPacked pack_v5_tc16(const float *blob) {
    const V5Blob b(blob);
    auto maxabs = [](const float *w, size_t n) { float m = 0.f; for (size_t i = 0; i < n; ++i) m = std::max(m, std::fabs(w[i])); return m; };
    V5HPacked P;
    float s[7];
    s[0] = pow2_scale_for(maxabs(b.basis, 258 * 256), &P.inv_w[0]);
    s[1] = pow2_scale_for(maxabs(b.e0w, 128 * 129 * 3), &P.inv_w[1]);
    s[2] = pow2_scale_for(maxabs(b.e1w, 64 * 128 * 3), &P.inv_w[2]);
    s[3] = pow2_scale_for(maxabs(b.e2w, 64 * 64 * 3), &P.inv_w[3]);
    s[4] = pow2_scale_for(maxabs(b.e3w, 128 * 64 * 3), &P.inv_w[4]);
    // one scale for [W_ih | W_hh]: the recurrent kernel accumulates both halves of K in the same TMEM columns
    s[5] = pow2_scale_for(std::max(maxabs(b.wih, 512 * 128), maxabs(b.whh, 512 * 128)), &P.inv_w[5]);
    s[6] = s[5];
    P.inv_w[6] = P.inv_w[5];
    P.w_fe.reserve(cvad::tc5::kFeStreamBytesH);
    v5_tiles(b, [&](int layer, int rows, int k0, auto W) {
        emit_tiles(layer < 5 ? P.w_fe : P.w_rec, fp16x2(s[layer]), rows, k0, W);
    });
    return P;
}

// v4 tensor-core STFT: the basis as 24 BF16x3 tiles
std::vector<unsigned char> pack_v4_stft_tc(const float *blob) {
    std::vector<unsigned char> out;
    out.reserve(cvad::tc5::kV4StftStreamBytes);
    stft_tiles(blob, [&](int, int rows, int k0, auto W) { emit_tiles(out, kBf16x3, rows, k0, W); });
    return out;
}

// v4 FFT path: delta = (the file's float32 STFT basis) - (periodic Hann x DFT-256, evaluated in double) -- what the
// exact-basis FFT lacks.  Scaled by 2^24 it is O(1) and goes to the tensor cores as ONE BF16 part per weight
// (8 tiles, the STFT block of the tile order).  Returns max |delta| (7.7e-8 for the reference's file).
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
    stft_tiles(delta.data(), [&](int, int rows, int k0, auto W) { emit_tiles(out, kBf16x1, rows, k0, W); });
    return worst;
}

// ---- resampling operators
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

// One source rate's operator in every form a resampler kernel reads: R^T [n_in][512] for resample_kernel, and R as
// tiles for resample_tc_kernel (K block kb-major, then output block of 128 samples, then part) -- BF16x3, and FP16x2
// scaled so that its largest entry lies in [2^14, 2^15), `inv` the inverse of that scale.
struct ResampleOperator {
    std::vector<float> rt;
    std::vector<unsigned char> tc, tc16;
    float inv = 1.f;
};

ResampleOperator build_resample_operator(int n_in) {
    ResampleOperator op;
    build_resample_rt(n_in, op.rt);
    float mx = 0.f;
    for (float v : op.rt) mx = std::max(mx, std::fabs(v));
    const Parts h = fp16x2(pow2_scale_for(mx, &op.inv));
    op.tc.reserve((size_t)512 * n_in * 6);
    op.tc16.reserve((size_t)512 * n_in * 4);
    for (int kb = 0; kb < n_in / 64; ++kb)
        for (int blk = 0; blk < 4; ++blk) {
            auto R = [&](int r, int m) { return op.rt[(size_t)m * 512 + blk * 128 + r]; };
            emit_tiles(op.tc, kBf16x3, 128, kb * 64, R);
            emit_tiles(op.tc16, h, 128, kb * 64, R);
        }
    return op;
}

}  // namespace
