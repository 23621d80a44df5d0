// vbx_interleave.cu — interleaved views (vbx_frames.sample_step > 1): the planar copy every frame-view path runs on.
//
// The header defines an interleaved view by its planar equivalent P[u][k] = base[u*segment_stride + k*s], k < S, in rows of
// S' = S rounded up to 64 samples.  vbx_planarize builds exactly that array on the device, in the view's own dtype (bytes are
// moved, never converted: G.711 stays one byte per sample and is decoded by the loaders as usual), and hands the caller the
// planar view, so the tuned kernels and their planners never see a sample step.  The padding [S, S') of every row is zeroed.
//
// interleave_gather_kernel: the channels-as-segments layout, where all segments' samples of time k lie inside the s samples
// [k*s, k*s + s) ((U-1)*segment_stride < s; a single segment always qualifies).  A CTA owns the times [k0, k0 + K) of every
// segment: it reads the contiguous interleaved span of those times with 16-byte loads (only the unaligned head and tail of
// the span go byte by byte, so no load leaves the view's extent), splits it in shared memory, and writes each segment's row
// with 16-byte stores.  interleave_gather_strided_kernel: any other geometry, one thread per output sample.
// A `lead` of zeros before every row lets the host pipeline give a chunk's frames the alignment they have in the planar
// equivalent of the whole view (vbx_pipeline.cuh).
// Both are copies bound by HBM bandwidth: each interleaved byte is read once and each planar byte written once.
#include "vbx_internal.cuh"

namespace {

constexpr int kGatherThreads = 256;
constexpr int64_t kGatherTileBytes = 16384;  // interleaved bytes a CTA stages
constexpr int64_t kGatherMaxFrameBytes = 512;  // s * sample size the tiled kernel takes (64 times = 32 KB of shared memory)

template <typename T>
__global__ void __launch_bounds__(kGatherThreads) interleave_gather_kernel(const T* __restrict__ base, int64_t extent,
                                                                           int64_t seg_stride, int64_t step, int U, int64_t S,
                                                                           int64_t lead, int64_t row, int K, T* __restrict__ out) {
    extern __shared__ uint4 smem_v[];
    unsigned char* sm = reinterpret_cast<unsigned char*>(smem_v);
    constexpr int E = (int)sizeof(T);
    constexpr int W = 16 / E;  // samples per 16-byte store
    const int64_t k0 = (int64_t)blockIdx.x * K;  // output positions [k0, k0 + K) hold the times [k0 - lead, k0 - lead + K)
    const int64_t t0 = k0 - lead > 0 ? k0 - lead : 0;
    // the interleaved span of those times that the view can read: samples [t0*s, min((k0-lead+K)*s, extent))
    const int64_t s_lo = t0 * step;
    int64_t s_hi = (k0 - lead + K) * step;
    if (s_hi > extent) s_hi = extent;
    const uintptr_t lo = reinterpret_cast<uintptr_t>(base + s_lo);
    const uintptr_t hi = reinterpret_cast<uintptr_t>(base + (s_hi > s_lo ? s_hi : s_lo));
    const uintptr_t a0 = lo & ~(uintptr_t)15;
    const int nq = (int)((hi - a0 + 15) >> 4);
    for (int q = threadIdx.x; q < nq; q += kGatherThreads) {
        const uintptr_t a = a0 + ((uintptr_t)q << 4);
        if (a >= lo && a + 16 <= hi) {
            smem_v[q] = __ldg(reinterpret_cast<const uint4*>(a));
        } else {
            for (int b = 0; b < 16; ++b)
                if (a + b >= lo && a + b < hi) sm[16 * q + b] = __ldg(reinterpret_cast<const unsigned char*>(a + b));
        }
    }
    __syncthreads();
    const T* tile = reinterpret_cast<const T*>(sm + (lo - a0));  // tile[t*s + u*seg_stride] = time t0 + t of segment u
    const int nv = K / W;
    for (int i = threadIdx.x; i < U * nv; i += kGatherThreads) {
        const int u = i / nv, v = i - u * nv;
        const int64_t k = k0 + (int64_t)v * W;
        if (k >= row) continue;
        union { uint4 q; T x[W]; } pk;
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int64_t t = k + w - lead;
            pk.x[w] = (t >= 0 && t < S) ? tile[(t - t0) * step + (int64_t)u * seg_stride] : (T)0;
        }
        *reinterpret_cast<uint4*>(out + (int64_t)u * row + k) = pk.q;  // row and k are multiples of 64 samples: aligned
    }
}

template <typename T>
__global__ void __launch_bounds__(kGatherThreads) interleave_gather_strided_kernel(const T* __restrict__ base, int64_t seg_stride,
                                                                                   int64_t step, int64_t U, int64_t S, int64_t lead,
                                                                                   int64_t row, T* __restrict__ out) {
    const int64_t total = U * row;
    for (int64_t i = (int64_t)blockIdx.x * kGatherThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kGatherThreads) {
        const int64_t u = i / row, t = i - u * row - lead;
        out[i] = (t >= 0 && t < S) ? __ldg(base + u * seg_stride + t * step) : (T)0;
    }
}

template <typename T>
int launch_gather(vbx_ctx* ctx, const vbx_frames* fr, int64_t U, int64_t S, int64_t lead, int64_t row, void* out) {
    const int64_t s = vbx_sample_step(fr);
    const int64_t seg = fr->frames_per_segment > 0 ? fr->segment_stride : 0;
    const T* base = reinterpret_cast<const T*>(fr->base);
    constexpr int64_t E = sizeof(T);
    if (U <= s && (U == 1 || (U - 1) * seg < s) && s * E <= kGatherMaxFrameBytes) {
        int64_t K = (kGatherTileBytes / (s * E)) & ~(int64_t)63;
        if (K < 64) K = 64;
        const int64_t grid = (row + K - 1) / K;
        VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "interleaved view too long for one gather launch");
        const size_t smem = (size_t)(K * s * E) + 32;  // the span, plus the aligned-down head and the rounded-up tail
        VBX_CUDA(ctx, cudaFuncSetAttribute(interleave_gather_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        interleave_gather_kernel<T><<<(unsigned)grid, kGatherThreads, smem, ctx->stream>>>(base, vbx_frames_extent(fr), seg, s, (int)U,
                                                                                           S, lead, row, (int)K, (T*)out);
        VBX_CHECK_LAUNCH(ctx, "interleave_gather_kernel");
        return VBX_OK;
    }
    int64_t grid = (U * row + kGatherThreads - 1) / kGatherThreads;
    if (grid > (int64_t)ctx->sm_count * 64) grid = (int64_t)ctx->sm_count * 64;
    interleave_gather_strided_kernel<T><<<(unsigned)grid, kGatherThreads, 0, ctx->stream>>>(base, seg, s, U, S, lead, row, (T*)out);
    VBX_CHECK_LAUNCH(ctx, "interleave_gather_strided_kernel");
    return VBX_OK;
}

}  // namespace

int vbx_planarize(vbx_ctx* ctx, const vbx_frames* fr, vbx_frames* out, int64_t lead) {
    *out = *fr;
    if (fr->sample_step <= 1 || fr->n_frames == 0) return VBX_OK;
    const int64_t J = vbx_frames_per_segment(fr), U = fr->n_frames / J, S = vbx_planar_len(fr);
    const int64_t row = (lead + S + 63) & ~(int64_t)63;
    const size_t es = vbx_dtype_size(fr->dtype);
    const size_t bytes = (size_t)U * (size_t)row * es;
    if (bytes > ctx->planar_bytes) {
        // grow-only; kernels of an earlier call on the context's stream may still read the old copy
        VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->planar) cudaFree(ctx->planar);
        ctx->planar = nullptr;
        ctx->planar_bytes = 0;
        const cudaError_t e = cudaMalloc(&ctx->planar, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return vbx_fail(ctx, VBX_ERR_NOMEM, "planar copy of an interleaved view: cudaMalloc(%zu) failed: %s", bytes,
                            cudaGetErrorString(e));
        }
        ctx->planar_bytes = bytes;
    }
    int st;
    if (es == 1) st = launch_gather<uint8_t>(ctx, fr, U, S, lead, row, ctx->planar);
    else if (es == 2) st = launch_gather<uint16_t>(ctx, fr, U, S, lead, row, ctx->planar);
    else if (es == 4) st = launch_gather<uint32_t>(ctx, fr, U, S, lead, row, ctx->planar);
    else st = launch_gather<unsigned long long>(ctx, fr, U, S, lead, row, ctx->planar);
    if (st != VBX_OK) return st;
    out->base = (const char*)ctx->planar + (size_t)lead * es;
    out->frame_stride = fr->frame_stride / vbx_sample_step(fr);
    out->segment_stride = row;
    out->sample_step = 0;
    return VBX_OK;
}
