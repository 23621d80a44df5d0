// vbx_synth.cu — deterministic synthetic speech-like audio generated on the device (SURVEY.md §8d "Synthetic audio").
//
// Bench / parity-at-scale infrastructure, not part of the reference's path: the corpora BASELINE.json names (1 h … 1000 h of
// synthetic audio) are far too large to synthesise on the host inside a bench run, and tiling a few host-made utterances
// times the data-dependent kernels (Laguerre, Brent) on little variety.  Every utterance here is distinct and a function of
// (seed, utterance index) only, so any rank / any chunking regenerates the same samples; parity runs copy the samples
// device → host and feed exactly those to the CPU oracle (never regenerated on the host).
//
// Per utterance u: a piecewise-linear f0 contour (80–300 Hz, one knot per 0.25 s, 30 % of the segments unvoiced); the
// source is a unit impulse train at the running period when voiced and 0.1·N(0,1) when unvoiced; it is shaped by a cascade
// of 4 (fs <= 16 kHz) or 5 two-pole resonators (centres uniform in [300,900], [900,2200], [2200,3200], [3200,4200],
// [4200,5500] Hz, bandwidths uniform 50–300 Hz, fixed per utterance, fp64 filter state); the result is scaled to peak 0.5
// and white noise at −40 dB re peak is added (mandatory: without a noise floor LPC is ill-posed even in f64, SURVEY §7.3).
// One thread per utterance, counter-based RNG (splitmix64 finaliser over (seed, utterance, stream, index)); two passes:
// the first finds the peak, the second regenerates the same samples and writes them scaled (fp32, or int16 PCM ·32767, or
// that int16 PCM G.711-encoded).
#include <cmath>
#include <type_traits>

#include "vbx_internal.cuh"

namespace {

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__device__ __forceinline__ uint64_t rng_key(uint64_t seed, uint64_t u, uint64_t stream, uint64_t i) {
    return mix64(mix64(seed + u * 0x9E3779B97F4A7C15ULL) + stream * 0xD1B54A32D192ED03ULL + i);
}
__device__ __forceinline__ double rng_uniform(uint64_t seed, uint64_t u, uint64_t stream, uint64_t i) {
    return (double)(rng_key(seed, u, stream, i) >> 11) * (1.0 / 9007199254740992.0);
}
// N(0,1) number i of a stream: Box–Muller over the pair (i >> 1), fp32 transcendental functions
__device__ __forceinline__ float rng_normal(uint64_t seed, uint64_t u, uint64_t stream, uint64_t i) {
    const uint64_t k = rng_key(seed, u, stream, i >> 1);
    const float u1 = ((float)(uint32_t)(k >> 40) + 1.0f) * (1.0f / 16777216.0f);  // (0, 1]
    const float u2 = (float)(uint32_t)((k >> 8) & 0xffffffu) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, c;
    sincospif(2.0f * u2, &s, &c);
    return (i & 1) ? r * s : r * c;
}

enum { STREAM_F0 = 1, STREAM_VOICED = 2, STREAM_SOURCE = 3, STREAM_FORMANT = 4, STREAM_FLOOR = 5 };

struct Resonators {
    double a1[5], a2[5];  // y[n] = x[n] + a1·y[n−1] + a2·y[n−2]
    int n;
};

template <bool WRITE, typename TOut>
__device__ __forceinline__ double synth_pass(uint64_t seed, uint64_t u, int64_t n_samples, double fs, const Resonators& R, double scale,
                                             TOut* out) {
    const int64_t seg = (int64_t)llrint(0.25 * fs);
    double y1[5] = {0, 0, 0, 0, 0}, y2[5] = {0, 0, 0, 0, 0};
    double phase = 0.0, peak = 0.0;
    int64_t k = -1;
    double f_lo = 0.0, f_hi = 0.0;
    bool voiced = false;
    const double inv_fs = 1.0 / fs, inv_seg = 1.0 / (double)seg;
    int64_t in_seg = seg;  // forces the knot load at i = 0
    for (int64_t i = 0; i < n_samples; ++i) {
        if (in_seg == seg) {
            in_seg = 0;
            ++k;
            f_lo = 80.0 + 220.0 * rng_uniform(seed, u, STREAM_F0, (uint64_t)k);
            f_hi = 80.0 + 220.0 * rng_uniform(seed, u, STREAM_F0, (uint64_t)k + 1);
            voiced = rng_uniform(seed, u, STREAM_VOICED, (uint64_t)k) >= 0.30;
        }
        const double f0 = f_lo + (f_hi - f_lo) * ((double)in_seg * inv_seg);
        ++in_seg;
        const double before = floor(phase);
        phase += f0 * inv_fs;
        const bool pulse = floor(phase) > before;
        double x = voiced ? (pulse ? 1.0 : 0.0) : 0.1 * (double)rng_normal(seed, u, STREAM_SOURCE, (uint64_t)i);
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            if (r < R.n) {
                const double y = fma(R.a1[r], y1[r], fma(R.a2[r], y2[r], x));
                y2[r] = y1[r];
                y1[r] = y;
                x = y;
            }
        }
        if (WRITE) {
            const double v = x * scale + 0.005 * (double)rng_normal(seed, u, STREAM_FLOOR, (uint64_t)i);  // −40 dB re the 0.5 peak
            if constexpr (std::is_same<TOut, float>::value) {
                out[i] = v;
            } else {
                double q = rint(v * 32767.0);
                q = q < -32768.0 ? -32768.0 : (q > 32767.0 ? 32767.0 : q);
                if constexpr (std::is_same<TOut, vbx_mulaw8>::value) out[i].code = (uint8_t)vbx_mulaw_encode((int)q);
                else if constexpr (std::is_same<TOut, vbx_alaw8>::value) out[i].code = (uint8_t)vbx_alaw_encode((int)q);
                else out[i] = (TOut)q;
            }
        } else {
            const double a = fabs(x);
            if (a > peak) peak = a;
        }
    }
    return peak;
}

template <typename TOut>
__global__ void __launch_bounds__(64) synth_speech_kernel(TOut* out, int64_t n_utts, int64_t n_samples, double fs, uint64_t seed,
                                                          int64_t first_utt) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_utts) return;
    const uint64_t u = (uint64_t)(first_utt + t);
    const double lo[5] = {300., 900., 2200., 3200., 4200.}, hi[5] = {900., 2200., 3200., 4200., 5500.};
    Resonators R;
    R.n = fs <= 16000.0 ? 4 : 5;
    const double PI = 3.14159265358979323846;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
        const double fc = lo[r] + (hi[r] - lo[r]) * rng_uniform(seed, u, STREAM_FORMANT, 2 * r);
        const double bw = 50.0 + 250.0 * rng_uniform(seed, u, STREAM_FORMANT, 2 * r + 1);
        const double rad = exp(-PI * bw / fs);
        R.a1[r] = 2.0 * rad * cos(2.0 * PI * fc / fs);
        R.a2[r] = -rad * rad;
    }
    const double peak = synth_pass<false, TOut>(seed, u, n_samples, fs, R, 0.0, nullptr);
    const double scale = 0.5 / (peak > 1e-30 ? peak : 1e-30);
    synth_pass<true, TOut>(seed, u, n_samples, fs, R, scale, out + t * n_samples);
}

}  // namespace

extern "C" int vbx_synth_speech(vbx_ctx* ctx, void* out, int32_t dtype, int64_t n_utts, int64_t n_samples, double sample_rate,
                                uint64_t seed, int64_t first_utt) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || vbx_dtype_is_pcm(dtype), "dtype must be VBX_F32, VBX_I16, VBX_MULAW8 or VBX_ALAW8");
    VBX_REQUIRE(ctx, n_utts >= 0 && n_samples >= 0 && first_utt >= 0, "negative sizes");
    VBX_REQUIRE(ctx, sample_rate >= 8000.0 && sample_rate <= 192000.0, "sample_rate must be in 8000..192000");
    if (n_utts == 0 || n_samples == 0) return VBX_OK;
    VBX_REQUIRE(ctx, out != nullptr, "out is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_utts + 63) / 64;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many utterances for one launch");
    if (dtype == VBX_I16)
        synth_speech_kernel<int16_t><<<(unsigned)grid, 64, 0, ctx->stream>>>((int16_t*)out, n_utts, n_samples, sample_rate, seed, first_utt);
    else if (dtype == VBX_MULAW8)
        synth_speech_kernel<vbx_mulaw8><<<(unsigned)grid, 64, 0, ctx->stream>>>((vbx_mulaw8*)out, n_utts, n_samples, sample_rate, seed,
                                                                               first_utt);
    else if (dtype == VBX_ALAW8)
        synth_speech_kernel<vbx_alaw8><<<(unsigned)grid, 64, 0, ctx->stream>>>((vbx_alaw8*)out, n_utts, n_samples, sample_rate, seed,
                                                                              first_utt);
    else
        synth_speech_kernel<float><<<(unsigned)grid, 64, 0, ctx->stream>>>((float*)out, n_utts, n_samples, sample_rate, seed, first_utt);
    VBX_CHECK_LAUNCH(ctx, "synth_speech_kernel");
    return VBX_OK;
}
