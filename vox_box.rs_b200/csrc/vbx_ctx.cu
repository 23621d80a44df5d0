// vbx_ctx.cu — context, memory helpers, window tables, timing, pipe-peak calibration.
#include <cmath>

#include "vbx_internal.cuh"

extern "C" {
// lib.rs:27-28
VBX_API const double VBX_MALE_FORMANT_ESTIMATES[4] = {320., 1440., 2760., 3200.};
VBX_API const double VBX_FEMALE_FORMANT_ESTIMATES[4] = {480., 1760., 3200., 3520.};
}

int vbx_fail(vbx_ctx* ctx, int status, const char* fmt, ...) {
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
        va_end(ap);
    }
    return status;
}

void vbx_prof_mark(vbx_ctx* ctx, const char* name) {
    if (ctx->prof_used >= ctx->prof_events.size()) {
        if (ctx->prof_events.size() >= 65536) return;  // pool exhausted: stop recording, totals stay a lower bound
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); return; }
        ctx->prof_events.push_back(e);
    }
    cudaEventRecord(ctx->prof_events[ctx->prof_used], ctx->stream);
    if (ctx->prof_used > 0) ctx->prof_names.push_back(name);
    ctx->prof_used++;
}

int vbx_launch_begin(vbx_ctx* ctx, const char* name, cudaStream_t stream) {
    if (stream == ctx->stream || !ctx->prof_on || ctx->prof_ranges.size() >= 65536) return -1;
    vbx_ctx::ProfRange r;
    r.name = name;
    if (cudaEventCreate(&r.e0) != cudaSuccess) { cudaGetLastError(); return -1; }
    if (cudaEventCreate(&r.e1) != cudaSuccess) { cudaGetLastError(); cudaEventDestroy(r.e0); return -1; }
    cudaEventRecord(r.e0, stream);
    ctx->prof_ranges.push_back(r);
    return (int)ctx->prof_ranges.size() - 1;
}
int vbx_launch_end(vbx_ctx* ctx, int slot, const char* name, cudaStream_t stream) {
    if (slot >= 0 && slot < (int)ctx->prof_ranges.size()) cudaEventRecord(ctx->prof_ranges[slot].e1, stream);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return vbx_fail(ctx, VBX_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e));
    ctx->launches++;
    if (stream == ctx->stream && ctx->prof_on) vbx_prof_mark(ctx, name);
    return VBX_OK;
}

int vbx_arena_reserve(vbx_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->arena_bytes) return VBX_OK;
    // a tracker of an earlier vbx_find_formants call may still read the block from the side stream
    if (ctx->s_side) cudaStreamSynchronize(ctx->s_side);
    // grow-only; the stream is drained first so no in-flight kernel still uses the old block
    VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->arena) cudaFree(ctx->arena);
    ctx->arena = nullptr;
    ctx->arena_bytes = 0;
    size_t want = bytes + (bytes >> 2) + (1 << 20);
    cudaError_t e = cudaMalloc(&ctx->arena, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        want = bytes;
        e = cudaMalloc(&ctx->arena, want);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "scratch arena: cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    ctx->arena_bytes = want;
    return VBX_OK;
}

int vbx_hard_list_reserve(vbx_ctx* ctx, int64_t n) {
    if (n <= ctx->hard_cap) return VBX_OK;
    // grow-only; a fix-up launch of an earlier call may still read the list from the side stream
    if (ctx->s_side) VBX_CUDA(ctx, cudaStreamSynchronize(ctx->s_side));
    VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->hard_list) cudaFree(ctx->hard_list);
    ctx->hard_list = nullptr;
    ctx->hard_cap = 0;
    const cudaError_t e = cudaMalloc(&ctx->hard_list, (size_t)n * sizeof(int));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "roots fix-up list: cudaMalloc(%zu) failed: %s", (size_t)n * sizeof(int), cudaGetErrorString(e));
    }
    ctx->hard_cap = n;
    return VBX_OK;
}

int vbx_scratch_get(vbx_ctx* ctx, size_t bytes, void** out) {
    if (ctx->sub_scratch) {
        if (bytes > ctx->sub_scratch_bytes)
            return vbx_fail(ctx, VBX_ERR_NOMEM, "internal: callee scratch (%zu bytes) exceeds the caller's reservation (%zu)", bytes,
                            ctx->sub_scratch_bytes);
        *out = ctx->sub_scratch;
        return VBX_OK;
    }
    int st = vbx_arena_reserve(ctx, bytes);
    if (st != VBX_OK) return st;
    *out = ctx->arena;
    return VBX_OK;
}

int vbx_pipe_reserve(vbx_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->pipe_bytes) return VBX_OK;
    VBX_CUDA(ctx, cudaDeviceSynchronize());
    if (ctx->pipe) cudaFree(ctx->pipe);
    ctx->pipe = nullptr;
    ctx->pipe_bytes = 0;
    cudaError_t e = cudaMalloc(&ctx->pipe, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "host pipeline block: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    ctx->pipe_bytes = bytes;
    return VBX_OK;
}

int vbx_pinned_reserve(vbx_ctx* ctx, size_t bytes) {
    if (bytes <= ctx->pinned_bytes) return VBX_OK;
    VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pinned_bytes = 0;
    size_t want = bytes + (bytes >> 2) + (1 << 20);
    cudaError_t e = cudaMallocHost(&ctx->pinned, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "pinned staging: cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    ctx->pinned_bytes = want;
    return VBX_OK;
}

// Window tables are computed on the host in f64 exactly as the reference's callers do:
//  - HANN_SYMMETRIC: sample::window::Window::<_, Hanning>::new(n): phase starts at 0 and is
//    ACCUMULATED, phase = (phase + 1/(n-1)) % 1.0, value 0.5·(1 − cos(2π·phase));
//  - HANN_PERIODIC:  lib.rs:66-70, phase = i · (1/n);
//  - HANN_LAG: the autocorrelation of the Hann window, HanningLag (periodic.rs:236-247), same phases
//    as HANN_SYMMETRIC — a table for the pitch path, not a frame window;
//  - NONE: ones (the multiply by 1.0 is exact).
void vbx_window_fill_host(int kind, int n, double* out) {
    const double PI = 3.14159265358979323846264338327950288;
    if (kind == VBX_WINDOW_HANN_SYMMETRIC) {
        double step = 1.0 / ((double)n - 1.0), phase = 0.0;
        for (int i = 0; i < n; ++i) {
            out[i] = 0.5 * (1.0 - cos(2.0 * PI * phase));
            phase = fmod(phase + step, 1.0);
        }
    } else if (kind == VBX_WINDOW_HANN_PERIODIC) {
        double len_inv = 1.0 / (double)n;
        for (int i = 0; i < n; ++i) out[i] = 0.5 * (1.0 - cos(2.0 * PI * ((double)i * len_inv)));
    } else if (kind == VBX_WINDOW_HANN_LAG) {
        // periodic.rs:236-247 HanningLag::at_phase over Window::new(n)'s accumulated phases (periodic.rs:400)
        double step = 1.0 / ((double)n - 1.0), phase = 0.0;
        const double pi_2 = PI * 2.0;
        for (int i = 0; i < n; ++i) {
            const double v = phase * pi_2;
            out[i] = (1.0 - phase) * (2.0 / 3.0 + (1.0 / 3.0) * cos(v)) + (1.0 / pi_2) * sin(v);
            phase = fmod(phase + step, 1.0);
        }
    } else {
        for (int i = 0; i < n; ++i) out[i] = 1.0;
    }
}

int vbx_get_window(vbx_ctx* ctx, int kind, int n, const double** dev_out, int sample_dtype) {
    const bool pcm = vbx_dtype_is_pcm(sample_dtype);
    uint64_t key = ((uint64_t)(uint32_t)(kind | (pcm ? 0x100 : 0)) << 32) | (uint32_t)n;
    auto it = ctx->windows.find(key);
    if (it != ctx->windows.end()) {
        *dev_out = it->second;
        return VBX_OK;
    }
    std::vector<double> host(n);
    vbx_window_fill_host(kind, n, host.data());
    if (pcm)
        for (auto& v : host) v = v / 32767.0;  // sample / 32767 · w  ==  sample · (w / 32767) to an ulp of f64
    double* dev = nullptr;
    cudaError_t e = cudaMalloc(&dev, (size_t)n * sizeof(double));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "window table: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    // synchronous copy from pageable memory: `host` dies at scope exit
    VBX_CUDA(ctx, cudaMemcpy(dev, host.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
    ctx->windows[key] = dev;
    *dev_out = dev;
    return VBX_OK;
}

int vbx_check_frames(vbx_ctx* ctx, const vbx_frames* fr, bool allow_f64) {
    VBX_REQUIRE(ctx, fr != nullptr, "frames descriptor is NULL");
    VBX_REQUIRE(ctx, fr->n_frames >= 0, "n_frames < 0");
    VBX_REQUIRE(ctx, fr->frame_len >= 1, "frame_len must be >= 1 (the reference indexes self[0])");
    VBX_REQUIRE(ctx, fr->frame_stride >= 1, "frame_stride must be >= 1");
    VBX_REQUIRE(ctx, fr->dtype == VBX_F32 || vbx_dtype_is_pcm(fr->dtype) || (allow_f64 && fr->dtype == VBX_F64),
                allow_f64 ? "frames dtype must be VBX_F32, VBX_I16, VBX_MULAW8, VBX_ALAW8 or VBX_F64"
                          : "frames dtype must be VBX_F32, VBX_I16, VBX_MULAW8 or VBX_ALAW8");
    VBX_REQUIRE(ctx, fr->window >= VBX_WINDOW_NONE && fr->window <= VBX_WINDOW_HANN_PERIODIC, "unknown window kind");
    VBX_REQUIRE(ctx, fr->sample_step >= 0, "frames.sample_step < 0");
    VBX_REQUIRE(ctx, fr->frames_per_segment >= 0, "frames_per_segment < 0");
    if (fr->frames_per_segment > 0) {
        VBX_REQUIRE(ctx, fr->n_frames % fr->frames_per_segment == 0, "n_frames must be a multiple of frames_per_segment");
        VBX_REQUIRE(ctx, fr->segment_stride >= 0, "segment_stride < 0");
    }
    const int64_t s = vbx_sample_step(fr);
    VBX_REQUIRE(ctx, fr->frame_stride % s == 0, "frame_stride (%lld) must be a multiple of sample_step (%lld)",
                (long long)fr->frame_stride, (long long)s);
    // extent = (U-1)*segment_stride + (J-1)*frame_stride + (N-1)*s + 1 samples, and its bytes, must fit int64
    if (fr->n_frames > 0) {
        const int64_t J = vbx_frames_per_segment(fr), U = fr->n_frames / J;
        int64_t a = 0, b = 0, c = 0, e = 0;
        const bool ovf = __builtin_mul_overflow(U - 1, fr->frames_per_segment > 0 ? fr->segment_stride : 0, &a) ||
                         __builtin_mul_overflow(J - 1, fr->frame_stride, &b) ||
                         __builtin_mul_overflow((int64_t)fr->frame_len - 1, s, &c) || __builtin_add_overflow(a, b, &e) ||
                         __builtin_add_overflow(e, c + 1, &e) || __builtin_mul_overflow(e, (int64_t)vbx_dtype_size(fr->dtype), &e);
        VBX_REQUIRE(ctx, !ovf, "the view's extent overflows int64");
    }
    VBX_REQUIRE(ctx, fr->n_frames == 0 || fr->base != nullptr, "frames.base is NULL");
    return VBX_OK;
}

// ------------------------------------------------------------------------------------------
// pipe-peak calibration kernels: 8 independent FMA chains per thread, 1024 threads/SM resident
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) vbx_fma_peak_kernel(T* out, int iters, T a, T b) {
    T v0 = (T)threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            v0 = fma(v0, a, b); v1 = fma(v1, a, b); v2 = fma(v2, a, b); v3 = fma(v3, a, b);
            v4 = fma(v4, a, b); v5 = fma(v5, a, b); v6 = fma(v6, a, b); v7 = fma(v7, a, b);
        }
    }
    T s = v0 + v1 + v2 + v3 + v4 + v5 + v6 + v7;
    if (s == (T)123456789) out[blockIdx.x * blockDim.x + threadIdx.x] = s;  // never true; keeps the chains alive
}

template <typename T>
static int measure_one(vbx_ctx* ctx, double* tflops) {
    const int blocks = ctx->sm_count * 8, threads = 256, iters = 2048;
    T* sink = (T*)ctx->arena;
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        VBX_CUDA(ctx, cudaEventRecord(ctx->ev_start, ctx->stream));
        vbx_fma_peak_kernel<T><<<blocks, threads, 0, ctx->stream>>>(sink, iters, (T)0.999, (T)0.001);
        VBX_CHECK_LAUNCH(ctx, "vbx_fma_peak_kernel");
        VBX_CUDA(ctx, cudaEventRecord(ctx->ev_stop, ctx->stream));
        VBX_CUDA(ctx, cudaEventSynchronize(ctx->ev_stop));
        float ms = 0;
        VBX_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        if (rep > 0 && ms < best) best = ms;
    }
    double fmas = (double)blocks * threads * (double)iters * 64.0;
    *tflops = 2.0 * fmas / (best * 1e-3) / 1e12;
    return VBX_OK;
}

extern "C" {

int vbx_version(void) { return 100; }

const char* vbx_status_str(int status) {
    switch (status) {
    case VBX_OK: return "ok";
    case VBX_ERR_LPC: return "Denum was <= 0.0";
    case VBX_ERR_PITCH: return "pitch candidate strength is NaN";
    case VBX_ERR_POLYNOMIAL: return "Failed to find roots";
    case VBX_ERR_WORKSPACE: return "Not enough workspace allocated";
    case VBX_ERR_CUDA: return "CUDA error";
    case VBX_ERR_BADARG: return "bad argument";
    case VBX_ERR_NOMEM: return "out of memory";
    default: return "unknown status";
    }
}

int vbx_ctx_create(int device, vbx_ctx** out) {
    if (!out) return VBX_ERR_BADARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        cudaGetLastError();
        return VBX_ERR_CUDA;  // no CPU fallback: the product path needs a CUDA device
    }
    if (device < 0 || device >= count) return VBX_ERR_BADARG;
    if (cudaSetDevice(device) != cudaSuccess) return VBX_ERR_CUDA;
    vbx_ctx* ctx = new vbx_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return VBX_ERR_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->s_h2d, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->s_d2h, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_start) != cudaSuccess || cudaEventCreate(&ctx->ev_stop) != cudaSuccess) {
        delete ctx;
        return VBX_ERR_CUDA;
    }
    for (int i = 0; i < 6; ++i)
        if (cudaEventCreateWithFlags(&ctx->ev_pipe[i], cudaEventDisableTiming) != cudaSuccess) {
            delete ctx;
            return VBX_ERR_CUDA;
        }
    if (cudaMalloc(&ctx->tile_counter, 256) != cudaSuccess) { delete ctx; return VBX_ERR_CUDA; }
    {
        // the tracker's CTAs should be dispatched ahead of the queued LPC / roots grids: highest priority
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&ctx->s_side, cudaStreamNonBlocking, hi) != cudaSuccess) { delete ctx; return VBX_ERR_CUDA; }
        for (int i = 0; i < 4; ++i)
            if (cudaEventCreateWithFlags(&ctx->ev_side[i], cudaEventDisableTiming) != cudaSuccess) { delete ctx; return VBX_ERR_CUDA; }
    }
    *out = ctx;
    return VBX_OK;
}

int vbx_ctx_destroy(vbx_ctx* ctx) {
    if (!ctx) return VBX_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto& kv : ctx->windows) cudaFree(kv.second);
    vbx_mfcc_cache_free(ctx);
    for (auto e : ctx->prof_events) cudaEventDestroy(e);
    if (ctx->work_counters) cudaFree(ctx->work_counters);
    if (ctx->tile_counter) cudaFree(ctx->tile_counter);
    if (ctx->hard_list) cudaFree(ctx->hard_list);
    if (ctx->arena) cudaFree(ctx->arena);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->pipe) cudaFree(ctx->pipe);
    if (ctx->planar) cudaFree(ctx->planar);
    for (int i = 0; i < 6; ++i) cudaEventDestroy(ctx->ev_pipe[i]);
    for (int i = 0; i < 4; ++i) cudaEventDestroy(ctx->ev_side[i]);
    for (auto& r : ctx->prof_ranges) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    if (ctx->s_side) cudaStreamDestroy(ctx->s_side);
    cudaStreamDestroy(ctx->s_h2d);
    cudaStreamDestroy(ctx->s_d2h);
    cudaEventDestroy(ctx->ev_start);
    cudaEventDestroy(ctx->ev_stop);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return VBX_OK;
}

int vbx_sync(vbx_ctx* ctx) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->s_side) VBX_CUDA(ctx, cudaStreamSynchronize(ctx->s_side));
    return VBX_OK;
}

void* vbx_ctx_stream(vbx_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
const char* vbx_last_error(vbx_ctx* ctx) { return ctx ? ctx->err : "no context"; }
int vbx_device_sm_count(vbx_ctx* ctx) { return ctx ? ctx->sm_count : 0; }
int64_t vbx_kernel_launches(vbx_ctx* ctx) { return ctx ? ctx->launches : 0; }

int vbx_malloc(vbx_ctx* ctx, size_t bytes, void** dev_out) {
    if (!ctx || !dev_out) return VBX_ERR_BADARG;
    *dev_out = nullptr;
    if (bytes == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaMalloc(dev_out, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    return VBX_OK;
}
int vbx_free(vbx_ctx* ctx, void* dev) {
    if (!ctx) return VBX_ERR_BADARG;
    if (dev) VBX_CUDA(ctx, cudaFree(dev));
    return VBX_OK;
}
int vbx_malloc_host(vbx_ctx* ctx, size_t bytes, void** host_out) {
    if (!ctx || !host_out) return VBX_ERR_BADARG;
    *host_out = nullptr;
    if (bytes == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaHostAlloc(host_out, bytes, cudaHostAllocPortable);  // pinned for every device's copy engines (vbx_multi)
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    return VBX_OK;
}
int vbx_free_host(vbx_ctx* ctx, void* host) {
    if (!ctx) return VBX_ERR_BADARG;
    if (host) VBX_CUDA(ctx, cudaFreeHost(host));
    return VBX_OK;
}
int vbx_memcpy_h2d(vbx_ctx* ctx, void* dev, const void* host, size_t bytes) {
    if (!ctx) return VBX_ERR_BADARG;
    if (bytes) VBX_CUDA(ctx, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return VBX_OK;
}
int vbx_memcpy_d2h(vbx_ctx* ctx, void* host, const void* dev, size_t bytes) {
    if (!ctx) return VBX_ERR_BADARG;
    if (bytes) VBX_CUDA(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return VBX_OK;
}
int vbx_memcpy_d2d(vbx_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx) return VBX_ERR_BADARG;
    if (bytes) VBX_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return VBX_OK;
}
int vbx_memset(vbx_ctx* ctx, void* dev, int value, size_t bytes) {
    if (!ctx) return VBX_ERR_BADARG;
    if (bytes) VBX_CUDA(ctx, cudaMemsetAsync(dev, value, bytes, ctx->stream));
    return VBX_OK;
}

int vbx_timer_start(vbx_ctx* ctx) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_CUDA(ctx, cudaEventRecord(ctx->ev_start, ctx->stream));
    return VBX_OK;
}
int vbx_timer_stop_ms(vbx_ctx* ctx, float* ms_out) {
    if (!ctx || !ms_out) return VBX_ERR_BADARG;
    VBX_CUDA(ctx, cudaEventRecord(ctx->ev_stop, ctx->stream));
    VBX_CUDA(ctx, cudaEventSynchronize(ctx->ev_stop));
    VBX_CUDA(ctx, cudaEventElapsedTime(ms_out, ctx->ev_start, ctx->ev_stop));
    return VBX_OK;
}

int vbx_profile_begin(vbx_ctx* ctx) {
    if (!ctx) return VBX_ERR_BADARG;
    ctx->prof_used = 0;
    ctx->prof_names.clear();
    ctx->prof_totals.clear();
    for (auto& r : ctx->prof_ranges) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    ctx->prof_ranges.clear();
    cudaSetDevice(ctx->device);
    if (!ctx->work_counters) {
        if (cudaMalloc(&ctx->work_counters, VBX_N_WORK_COUNTERS * sizeof(unsigned long long)) != cudaSuccess) {
            cudaGetLastError();
            ctx->work_counters = nullptr;
        }
    }
    if (ctx->work_counters) cudaMemsetAsync(ctx->work_counters, 0, VBX_N_WORK_COUNTERS * sizeof(unsigned long long), ctx->stream);
    ctx->prof_on = true;
    vbx_prof_mark(ctx, "begin");
    return VBX_OK;
}

int vbx_profile_end(vbx_ctx* ctx) {
    if (!ctx) return VBX_ERR_BADARG;
    ctx->prof_on = false;
    VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->s_side) VBX_CUDA(ctx, cudaStreamSynchronize(ctx->s_side));
    for (auto& r : ctx->prof_ranges) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.e0, r.e1) != cudaSuccess) { cudaGetLastError(); continue; }
        auto& t = ctx->prof_totals[r.name];
        t.first += ms;
        t.second += 1;
    }
    for (size_t i = 1; i < ctx->prof_used; ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->prof_events[i - 1], ctx->prof_events[i]) != cudaSuccess) { cudaGetLastError(); continue; }
        auto& t = ctx->prof_totals[ctx->prof_names[i - 1]];
        t.first += ms;
        t.second += 1;
    }
    return VBX_OK;
}

int vbx_profile_counters(vbx_ctx* ctx, uint64_t* out, int32_t n) {
    if (!ctx || !out || n < 0) return VBX_ERR_BADARG;
    unsigned long long host[VBX_N_WORK_COUNTERS] = {0};
    if (ctx->work_counters) {
        VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        VBX_CUDA(ctx, cudaMemcpy(host, ctx->work_counters, sizeof(host), cudaMemcpyDeviceToHost));
    }
    for (int i = 0; i < n; ++i) out[i] = i < VBX_N_WORK_COUNTERS ? (uint64_t)host[i] : 0;
    return VBX_OK;
}

int vbx_profile_count(vbx_ctx* ctx) { return ctx ? (int)ctx->prof_totals.size() : 0; }

int vbx_profile_entry(vbx_ctx* ctx, int index, char* name_out, int name_len, double* ms_total, int64_t* launches) {
    if (!ctx || index < 0 || index >= (int)ctx->prof_totals.size()) return VBX_ERR_BADARG;
    auto it = ctx->prof_totals.begin();
    std::advance(it, index);
    if (name_out && name_len > 0) snprintf(name_out, name_len, "%s", it->first.c_str());
    if (ms_total) *ms_total = it->second.first;
    if (launches) *launches = it->second.second;
    return VBX_OK;
}

int vbx_measure_peaks(vbx_ctx* ctx, double* fp32_tflops, double* fp64_tflops) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_arena_reserve(ctx, 1 << 20);
    if (st != VBX_OK) return st;
    double a = 0, b = 0;
    st = measure_one<float>(ctx, &a);
    if (st != VBX_OK) return st;
    st = measure_one<double>(ctx, &b);
    if (st != VBX_OK) return st;
    if (fp32_tflops) *fp32_tflops = a;
    if (fp64_tflops) *fp64_tflops = b;
    return VBX_OK;
}

int vbx_window_table_host(int window, int32_t n, double* out) {
    if (n < 1 || !out || window < VBX_WINDOW_NONE || window > VBX_WINDOW_HANN_LAG) return VBX_ERR_BADARG;
    vbx_window_fill_host(window, n, out);
    return VBX_OK;
}

}  // extern "C"
