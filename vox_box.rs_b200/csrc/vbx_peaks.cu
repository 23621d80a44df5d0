// vbx_peaks.cu — per-frame and per-segment peak amplitudes of a vbx_frames view (vbx_frame_peaks).
//
// The local peak of frame f is max |x| over its frame_len samples as loaded (I16 and decoded G.711 scaled by 1/32767), before
// any window.
// The global peak of segment u is the same max over every sample its frames span,
// [u·segment_stride, u·segment_stride + (J−1)·frame_stride + frame_len): with hop > frame_len that includes the gaps
// between frames.  NaN samples are skipped (a fold from 0 with `>`, so a NaN never wins; an all-NaN frame has peak 0).
// Max is exact, so the results do not depend on the reduction order.
//
// One warp per frame: the lanes stride over the frame (coalesced), then over the gap to the next frame of the segment if
// there is one (global peak only).  The warps of a CTA hold consecutive frames, so the CTA folds the frames of each
// segment it touches before one atomicMax per (CTA, segment): peaks are non-negative and never NaN, and non-negative
// doubles order like their bit patterns, so the atomic works on the 64-bit pattern.
#include <type_traits>

#include "vbx_internal.cuh"

namespace {

constexpr int kPeakWarps = 8;

template <typename TIn>
__global__ void __launch_bounds__(32 * kPeakWarps) frame_peaks_kernel(const TIn* __restrict__ base, int64_t n_frames, int64_t stride,
                                                                     int64_t seg_frames, int64_t seg_stride, int n,
                                                                     double* __restrict__ local_out,
                                                                     unsigned long long* __restrict__ global_out) {
    __shared__ double s_val[kPeakWarps];
    __shared__ int64_t s_seg[kPeakWarps];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t f = (int64_t)blockIdx.x * kPeakWarps + warp;
    const bool live = f < n_frames;
    int64_t seg = -1;
    double loc = 0.0, glo = 0.0;
    if (live) {
        seg = f / seg_frames;
        const int64_t j = f - seg * seg_frames;
        const TIn* x = base + seg * seg_stride + j * stride;
        for (int i = lane; i < n; i += 32) {
            const double a = fabs(vbx_load_sample_d<TIn>(x + i));
            if (a > loc) loc = a;
        }
        glo = loc;
        if (global_out && stride > n && j + 1 < seg_frames) {  // samples between this frame's end and the next frame's start
            for (int64_t i = n + lane; i < stride; i += 32) {
                const double a = fabs(vbx_load_sample_d<TIn>(x + i));
                if (a > glo) glo = a;
            }
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) {
            const double o = __shfl_xor_sync(FULL, loc, m), g = __shfl_xor_sync(FULL, glo, m);
            if (o > loc) loc = o;
            if (g > glo) glo = g;
        }
        if constexpr (vbx_pcm<TIn>::value) {  // monotone, so max(|v| / 32767) = max|v| / 32767 exactly
            loc = loc / 32767.0;
            glo = glo / 32767.0;
        }
        if (local_out && lane == 0) local_out[f] = loc;
    }
    if (!global_out) return;
    if (lane == 0) {
        s_val[warp] = glo;
        s_seg[warp] = seg;
    }
    __syncthreads();
    // thread w heads the run of warps that share warp w's segment
    const int w = threadIdx.x;
    if (w < kPeakWarps && s_seg[w] >= 0 && (w == 0 || s_seg[w - 1] != s_seg[w])) {
        double m = s_val[w];
        for (int k = w + 1; k < kPeakWarps && s_seg[k] == s_seg[w]; ++k)
            if (s_val[k] > m) m = s_val[k];
        atomicMax(global_out + s_seg[w], (unsigned long long)__double_as_longlong(m));
    }
}

}  // namespace

int vbx_launch_frame_peaks(vbx_ctx* ctx, const vbx_frames* fr, double* local_out, double* global_out) {
    if (fr->n_frames == 0 || (!local_out && !global_out)) return VBX_OK;
    const int64_t J = vbx_frames_per_segment(fr);
    const int64_t seg_stride = fr->frames_per_segment > 0 ? fr->segment_stride : 0;
    if (global_out) VBX_CUDA(ctx, cudaMemsetAsync(global_out, 0, (size_t)(fr->n_frames / J) * sizeof(double), ctx->stream));
    const int64_t grid = (fr->n_frames + kPeakWarps - 1) / kPeakWarps;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
    auto* g = reinterpret_cast<unsigned long long*>(global_out);
    if (fr->dtype == VBX_I16)
        frame_peaks_kernel<int16_t><<<(unsigned)grid, 32 * kPeakWarps, 0, ctx->stream>>>(
            (const int16_t*)fr->base, fr->n_frames, fr->frame_stride, J, seg_stride, fr->frame_len, local_out, g);
    else if (fr->dtype == VBX_MULAW8)
        frame_peaks_kernel<vbx_mulaw8><<<(unsigned)grid, 32 * kPeakWarps, 0, ctx->stream>>>(
            (const vbx_mulaw8*)fr->base, fr->n_frames, fr->frame_stride, J, seg_stride, fr->frame_len, local_out, g);
    else if (fr->dtype == VBX_ALAW8)
        frame_peaks_kernel<vbx_alaw8><<<(unsigned)grid, 32 * kPeakWarps, 0, ctx->stream>>>(
            (const vbx_alaw8*)fr->base, fr->n_frames, fr->frame_stride, J, seg_stride, fr->frame_len, local_out, g);
    else if (fr->dtype == VBX_F64)
        frame_peaks_kernel<double><<<(unsigned)grid, 32 * kPeakWarps, 0, ctx->stream>>>(
            (const double*)fr->base, fr->n_frames, fr->frame_stride, J, seg_stride, fr->frame_len, local_out, g);
    else
        frame_peaks_kernel<float><<<(unsigned)grid, 32 * kPeakWarps, 0, ctx->stream>>>(
            (const float*)fr->base, fr->n_frames, fr->frame_stride, J, seg_stride, fr->frame_len, local_out, g);
    VBX_CHECK_LAUNCH(ctx, "frame_peaks_kernel");
    return VBX_OK;
}

// segment u's samples as the planar equivalent holds them (all of a contiguous single-segment view's extent):
// base[u*segment_stride + k*s], k < vbx_planar_len
double vbx_host_peak(const vbx_frames* fr, int64_t u) {
    const int64_t n = vbx_planar_len(fr), s = vbx_sample_step(fr);
    const int64_t first = fr->frames_per_segment > 0 ? u * fr->segment_stride : 0;
    double m = 0.0;
    if (vbx_dtype_is_pcm(fr->dtype)) {
        int a = 0;
        for (int64_t k = 0; k < n; ++k) {
            const int64_t i = first + k * s;
            int v;
            if (fr->dtype == VBX_I16) v = ((const int16_t*)fr->base)[i];
            else if (fr->dtype == VBX_MULAW8) v = vbx_mulaw_decode(((const uint8_t*)fr->base)[i]);
            else v = vbx_alaw_decode(((const uint8_t*)fr->base)[i]);
            if (v < 0) v = -v;
            if (v > a) a = v;
        }
        m = (double)a / 32767.0;
    } else if (fr->dtype == VBX_F64) {
        const double* x = (const double*)fr->base;
        for (int64_t k = 0; k < n; ++k) {
            const double a = fabs(x[first + k * s]);
            if (a > m) m = a;
        }
    } else {
        const float* x = (const float*)fr->base;
        float mf = 0.f;
        for (int64_t k = 0; k < n; ++k) {
            const float a = fabsf(x[first + k * s]);
            if (a > mf) mf = a;
        }
        m = (double)mf;
    }
    return m;
}

extern "C" {

int vbx_frame_peaks(vbx_ctx* ctx, const vbx_frames* frames, double* local_out, double* global_out) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_check_frames(ctx, frames, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    if (frames->n_frames == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    vbx_frames pv;  // the planar equivalent of an interleaved view
    st = vbx_planarize(ctx, frames, &pv);
    if (st != VBX_OK) return st;
    return vbx_launch_frame_peaks(ctx, &pv, local_out, global_out);
}

}  // extern "C"
