// vbx_pipeline.cuh — chunked H2D / compute / D2H overlap for the `_host` entry points.
//
// A host-pointer call is split into chunks of whole segments (utterances) — or of frame ranges when the
// view is a single segment — and run as a three-stage pipeline on three streams: the copy-in stream
// uploads chunk k+1 while the context's stream computes chunk k and the copy-out stream downloads the
// results of chunk k−1 (PCIe is full duplex).  Device buffers are double buffered and come from a
// dedicated block of the context (the kernels keep using the scratch arena, serialised on the compute
// stream).  Pinned host memory is what makes the copies asynchronous; with pageable memory the result is
// the same, only the overlap is lost.
//
// An interleaved view whose segments share memory (the channels of one recording: segment_stride below a segment's extent)
// is cut by TIME instead: chunk k is frames [j0, j1) of every segment.  It uploads the interleaved span those frames cover,
// once for all channels, the device call gathers the channels (vbx_planarize) and runs on the sub-view of J' = j1 − j0
// frames per segment, and each output comes back with one cudaMemcpy2DAsync to rows u*J + j0 .. of every segment u.
// Consecutive chunks share only the frame overlap of their boundary, (frame_len − hop) samples of every channel, exactly as
// the frame chunks of a single-segment view do; every other interleaved byte crosses PCIe once.  The pipeline gathers each
// interleaved chunk itself, placing the chunk's first frame at the offset (mod 64 samples) it has in the planar equivalent of
// the whole view, so that every frame is read at the alignment the device call reads it at and the results are the device
// call's bit for bit.
#pragma once
#include "vbx_internal.cuh"

// the host pipeline cuts this view into time ranges of every segment (see above)
static inline bool vbx_chunk_by_time(const vbx_frames* fr) {
    if (fr->frames_per_segment <= 0 || vbx_sample_step(fr) <= 1) return false;
    const int64_t seg_extent = (fr->frames_per_segment - 1) * fr->frame_stride + ((int64_t)fr->frame_len - 1) * vbx_sample_step(fr) + 1;
    return fr->segment_stride < seg_extent;
}

struct vbx_host_out {
    void* host;              // destination (host), may be null = output not requested
    size_t bytes_per_frame;  // bytes produced per frame
    void* dev;               // filled per chunk: device address of this chunk's block
};

// launch(chunk_frames_view_on_device, first_frame, first_segment, outs_with_dev_set) -> status.  When the view is cut by
// time (vbx_chunk_by_time), first_frame is the chunk's first frame j0 inside every segment and first_segment is 0.
template <class Launch>
static int vbx_run_chunked(vbx_ctx* ctx, const vbx_frames* fr, vbx_host_out* outs, int n_outs, Launch launch,
                           int max_chunks = 0 /* 0 = no limit; paths with a latency-bound per-chunk kernel ask for few, large chunks */,
                           size_t target_bytes = (size_t)24 << 20 /* input bytes per chunk; compute-bound paths ask for more */) {
    const int64_t F = fr->n_frames;
    const size_t es = vbx_dtype_size(fr->dtype);
    const bool by_time = vbx_chunk_by_time(fr);
    const bool segmented = fr->frames_per_segment > 0 && !by_time;
    const int64_t J = vbx_frames_per_segment(fr), U = F / J;
    const int64_t frame_extent = ((int64_t)fr->frame_len - 1) * vbx_sample_step(fr) + 1;  // samples one frame spans
    // chunkable units: segments, frames, or (by time) the frame index j of every segment at once
    const int64_t n_units = segmented ? U : (by_time ? J : F);
    const int64_t unit_frames = segmented ? J : (by_time ? U : 1);
    const int64_t unit_stride = segmented ? fr->segment_stride : fr->frame_stride;  // samples between unit starts
    const int64_t unit_extent = segmented ? (J - 1) * fr->frame_stride + frame_extent
                                          : (by_time ? (U - 1) * fr->segment_stride + frame_extent : frame_extent);
    size_t out_per_frame = 0;
    for (int i = 0; i < n_outs; ++i) out_per_frame += outs[i].host ? outs[i].bytes_per_frame : 0;
    // chunk size: `target_bytes` of input per chunk (24 MB unless the caller says otherwise; VBX_HOST_CHUNK_MB overrides)
    size_t target = target_bytes;
    if (const char* e = getenv("VBX_HOST_CHUNK_MB")) target = (size_t)atoll(e) << 20;
    int64_t units_per_chunk = (int64_t)(target / ((size_t)unit_stride * es + 1)) + 1;
    if (max_chunks > 0 && !getenv("VBX_HOST_CHUNK_MB")) {
        const int64_t floor_units = (n_units + max_chunks - 1) / max_chunks;
        if (units_per_chunk < floor_units) units_per_chunk = floor_units;
    }
    if (units_per_chunk > n_units) units_per_chunk = n_units;
    if (units_per_chunk < 1) units_per_chunk = 1;
    const int64_t n_chunks = (n_units + units_per_chunk - 1) / units_per_chunk;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t in_chunk = al((size_t)((units_per_chunk - 1) * unit_stride + unit_extent) * es);
    size_t out_chunk = 0;
    for (int i = 0; i < n_outs; ++i)
        if (outs[i].host) out_chunk += al((size_t)units_per_chunk * unit_frames * outs[i].bytes_per_frame);
    const int nbuf = n_chunks > 1 ? 2 : 1;
    int st = vbx_pipe_reserve(ctx, nbuf * (in_chunk + out_chunk));
    if (st != VBX_OK) return st;
    char* blk = (char*)ctx->pipe;
    cudaEvent_t ev_in[2], ev_comp[2], ev_out[2];
    for (int b = 0; b < 2; ++b) {
        ev_in[b] = ctx->ev_pipe[b];
        ev_comp[b] = ctx->ev_pipe[2 + b];
        ev_out[b] = ctx->ev_pipe[4 + b];
    }
    int rc = VBX_OK;
    // a CUDA error inside the loop must not return before the drain below: copies may still touch caller memory
#define PIPE_CUDA(call)                                                                                              \
    {                                                                                                                \
        cudaError_t e__ = (call);                                                                                    \
        if (e__ != cudaSuccess) {                                                                                    \
            rc = vbx_fail(ctx, VBX_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            break;                                                                                                   \
        }                                                                                                            \
    }
    for (int64_t c = 0; c < n_chunks && rc == VBX_OK; ++c) {
        const int b = (int)(c & 1);
        const int64_t u0 = c * units_per_chunk;
        const int64_t nu = (n_units - u0 < units_per_chunk) ? n_units - u0 : units_per_chunk;
        const int64_t nf = nu * unit_frames;
        char* d_in = blk + (size_t)b * (in_chunk + out_chunk);
        char* d_out = d_in + in_chunk;
        const size_t bytes_in = (size_t)((nu - 1) * unit_stride + unit_extent) * es;
        // the input buffer b is free once the compute of chunk c−2 is done
        if (c >= 2) PIPE_CUDA(cudaStreamWaitEvent(ctx->s_h2d, ev_comp[b], 0));
        PIPE_CUDA(cudaMemcpyAsync(d_in, (const char*)fr->base + (size_t)u0 * unit_stride * es, bytes_in,
                                      cudaMemcpyHostToDevice, ctx->s_h2d));
        PIPE_CUDA(cudaEventRecord(ev_in[b], ctx->s_h2d));
        // compute: needs its input, and its output buffer b free (D2H of chunk c−2 done)
        PIPE_CUDA(cudaStreamWaitEvent(ctx->stream, ev_in[b], 0));
        if (c >= 2) PIPE_CUDA(cudaStreamWaitEvent(ctx->stream, ev_out[b], 0));
        vbx_frames ifr = *fr;
        ifr.base = d_in;
        ifr.n_frames = nf;
        if (by_time) ifr.frames_per_segment = nu;
        // an interleaved chunk is gathered here, with its first frame at the offset (mod 64 samples) it has in the planar
        // equivalent of the whole view: the kernels then see every frame at the alignment the device call gives it
        vbx_frames dfr;
        const int64_t first_frame = segmented ? 0 : u0;  // index of the chunk's first frame inside its segment(s)
        rc = vbx_planarize(ctx, &ifr, &dfr, (first_frame * (fr->frame_stride / vbx_sample_step(fr))) % 64);
        if (rc != VBX_OK) break;
        size_t off = 0;
        for (int i = 0; i < n_outs; ++i) {
            outs[i].dev = nullptr;
            if (outs[i].host) {
                outs[i].dev = d_out + off;
                off += al((size_t)units_per_chunk * unit_frames * outs[i].bytes_per_frame);
            }
        }
        rc = launch(&dfr, by_time ? u0 : u0 * unit_frames, segmented ? u0 : 0, outs);
        if (rc != VBX_OK) break;
        PIPE_CUDA(cudaEventRecord(ev_comp[b], ctx->stream));
        PIPE_CUDA(cudaStreamWaitEvent(ctx->s_d2h, ev_comp[b], 0));
        for (int i = 0; i < n_outs && rc == VBX_OK; ++i) {
            if (!outs[i].host) continue;
            const size_t bpf = outs[i].bytes_per_frame;
            // by time: the chunk's [U][nu] rows go to rows u*J + u0 of the caller's [U][J]
            const cudaError_t ec =
                by_time ? cudaMemcpy2DAsync((char*)outs[i].host + (size_t)u0 * bpf, (size_t)J * bpf, outs[i].dev, (size_t)nu * bpf,
                                            (size_t)nu * bpf, (size_t)U, cudaMemcpyDeviceToHost, ctx->s_d2h)
                        : cudaMemcpyAsync((char*)outs[i].host + (size_t)u0 * unit_frames * bpf, outs[i].dev, (size_t)nf * bpf,
                                          cudaMemcpyDeviceToHost, ctx->s_d2h);
            if (ec != cudaSuccess) rc = vbx_fail(ctx, VBX_ERR_CUDA, "host pipeline: D2H copy failed: %s", cudaGetErrorString(ec));
        }
        if (rc != VBX_OK) break;
        PIPE_CUDA(cudaEventRecord(ev_out[b], ctx->s_d2h));
    }
    // drain all three streams (also on error, so that no copy is still touching caller memory)
#undef PIPE_CUDA
    const cudaError_t e1 = cudaStreamSynchronize(ctx->s_h2d);
    const cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    const cudaError_t e3 = cudaStreamSynchronize(ctx->s_d2h);
    if (rc == VBX_OK) {
        cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) return vbx_fail(ctx, VBX_ERR_CUDA, "host pipeline failed: %s", cudaGetErrorString(e));
    }
    return rc;
}
