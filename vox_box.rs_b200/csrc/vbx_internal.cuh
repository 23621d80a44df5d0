// vbx_internal.cuh — shared internals of libvoxbox_b200 (context, error plumbing, device helpers).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/voxbox_b200.h"

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
struct vbx_mfcc_cache;  // vbx_mfcc.cu: device tables per (N, num_coeffs, bounds, fs)
void vbx_mfcc_cache_free(struct vbx_ctx* ctx);

struct vbx_ctx {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;  // max dynamic shared memory per block (opt-in)
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    int64_t launches = 0;
    char err[512] = {0};
    // scratch arena (device) and pinned staging (host) — grow-only, reused across calls
    void* arena = nullptr;
    size_t arena_bytes = 0;
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
    // A caller inside the library that already holds arena pointers (vbx_find_formants) hands its callees their scratch
    // as a sub-range of its own single reservation: while set, vbx_scratch_get serves from here and never touches the arena.
    void* sub_scratch = nullptr;
    size_t sub_scratch_bytes = 0;
    // host-call pipeline (vbx_pipeline.cuh): copy-in / copy-out streams, events, double-buffered device block
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_pipe[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    void* pipe = nullptr;
    size_t pipe_bytes = 0;
    // side stream of vbx_find_formants (the latency-bound tracker of frame chunk c runs there while the main stream computes
    // the LPC / roots of chunk c + 1); ev_side: [0..1] chunk c's resonances ready, [2..3] the roots fix-up of the chunk that
    // used buffer set 0 / 1 done (the set may be reused); [2] also the join after the last chunk's tracker
    cudaStream_t s_side = nullptr;
    cudaEvent_t ev_side[4] = {nullptr, nullptr, nullptr, nullptr};
    // window tables (device, f64), keyed by (kind << 32 | n)
    std::map<uint64_t, double*> windows;
    // per-kernel timing (vbx_profile_*): an event after every launch; a kernel's time = the gap to the previous event
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_events;   // pool, created lazily
    std::vector<const char*> prof_names;    // name of the launch that precedes event i+1 (event 0 = begin marker)
    size_t prof_used = 0;
    std::map<std::string, std::pair<double, int64_t>> prof_totals;  // name -> (ms, launches)
    // launches on the side stream are timed as explicit (start, stop) event pairs on that stream
    struct ProfRange { const char* name; cudaEvent_t e0, e1; };
    std::vector<ProfRange> prof_ranges;
    // executed-work counters of the data-dependent kernels (device, VBX_N_WORK_COUNTERS × u64; zeroed by vbx_profile_begin,
    // incremented only while profiling is on): see vbx_profile_counters in the header
    unsigned long long* work_counters = nullptr;
    int reserve_sms = 0;               // SMs the persistent kernels leave free for a co-running side-stream kernel
    unsigned* tile_counter = nullptr;  // device: [0] the persistent kernels' dynamic tile cursor, [1..2] lengths of fix-up lists
    int* hard_list = nullptr;          // device: frames the pair-deflation roots kernel hands to the f64 fix-up launch
    int64_t hard_cap = 0;              // entries of hard_list (vbx_hard_list_reserve: as many as a roots launch has frames)
    vbx_mfcc_cache* mfcc_cache = nullptr;
    bool mfcc_fft_f32 = false;  // MFCC transform precision (default fp64)
    // planar copy of an interleaved view (vbx_planarize): grow-only, written and read on the context's stream only
    void* planar = nullptr;
    size_t planar_bytes = 0;
};

enum { VBX_WORK_ROOTS_HORNER = 0, VBX_WORK_ROOTS_ROUNDS = 1, VBX_WORK_REFINE_TERMS = 2, VBX_WORK_REFINE_EVALS = 3, VBX_N_WORK_COUNTERS = 8 };
// device pointer of the counter block while profiling is on, else null (kernels skip the accounting)
static inline unsigned long long* vbx_work_ptr(vbx_ctx* ctx) { return ctx->prof_on ? ctx->work_counters : nullptr; }

int vbx_fail(vbx_ctx* ctx, int status, const char* fmt, ...);
void vbx_prof_mark(vbx_ctx* ctx, const char* name);        // records "launch `name` was just enqueued" (profiling on)
// A launch on `stream` placed between these two.  On the context's stream, end does what VBX_CHECK_LAUNCH does; on a side
// stream, where the begin / end markers of vbx_prof_mark do not apply, the launch is timed as its own (start, stop) event pair
// on that stream (begin returns its slot, or -1).  end checks and counts the launch either way.
int vbx_launch_begin(vbx_ctx* ctx, const char* name, cudaStream_t stream);
int vbx_launch_end(vbx_ctx* ctx, int slot, const char* name, cudaStream_t stream);
int vbx_arena_reserve(vbx_ctx* ctx, size_t bytes);         // ensures ctx->arena has >= bytes
int vbx_pinned_reserve(vbx_ctx* ctx, size_t bytes);        // ensures ctx->pinned has >= bytes
int vbx_hard_list_reserve(vbx_ctx* ctx, int64_t n);        // ensures ctx->hard_list has >= n entries
// scratch for a kernel launcher: the caller-provided sub-range if one is set (see vbx_ctx::sub_scratch), else the arena
int vbx_scratch_get(vbx_ctx* ctx, size_t bytes, void** out);
// scratch the LPC stage of vbx_find_formants may ask for through vbx_scratch_get (0 when the fused kernels apply)
size_t vbx_lpc_scratch_bytes(vbx_ctx* ctx, const vbx_frames* fr, int n_lags);
size_t vbx_burg_scratch_bytes(vbx_ctx* ctx, const vbx_frames* fr);
int vbx_pipe_reserve(vbx_ctx* ctx, size_t bytes);          // ensures ctx->pipe has >= bytes
// vbx_peaks.cu: per-frame (local_out [F]) and per-segment (global_out [n_segments]) max |x| of a device view, either may be
// null; and the same max over the whole extent of a host view (the global peak of a single-segment view)
int vbx_launch_frame_peaks(vbx_ctx* ctx, const vbx_frames* fr, double* local_out, double* global_out);
// sample dtypes whose samples load as integer PCM values (int16, or G.711 decoded to int16): their 1/32767 scale lives in the
// window table
static inline bool vbx_dtype_is_pcm(int dt) { return dt == VBX_I16 || dt == VBX_MULAW8 || dt == VBX_ALAW8; }
// cached device table (ones for NONE).  An integer-PCM sample_dtype folds the PCM scale into the table: w[i] / 32767
// (tests/lib.rs:17-19 scale every sample by 1/(i32::MAX >> 16) before any arithmetic).  int16 and G.711 views share it.
int vbx_get_window(vbx_ctx* ctx, int kind, int n, const double** dev_out, int sample_dtype = VBX_F32);
void vbx_window_fill_host(int kind, int n, double* out);

#define VBX_CUDA(ctx, call)                                                                          \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return vbx_fail((ctx), VBX_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                            __FILE__, __LINE__);                                                     \
    } while (0)

#define VBX_CHECK_LAUNCH(ctx, name)                                                                  \
    do {                                                                                             \
        cudaError_t e__ = cudaGetLastError();                                                        \
        if (e__ != cudaSuccess)                                                                      \
            return vbx_fail((ctx), VBX_ERR_CUDA, "launch of %s failed: %s", (name), cudaGetErrorString(e__)); \
        (ctx)->launches++;                                                                           \
        if ((ctx)->prof_on) vbx_prof_mark((ctx), (name));                                            \
    } while (0)

#define VBX_REQUIRE(ctx, cond, ...)                                                                  \
    do {                                                                                             \
        if (!(cond)) return vbx_fail((ctx), VBX_ERR_BADARG, __VA_ARGS__);                            \
    } while (0)

static inline size_t vbx_dtype_size(int dt) {
    return dt == VBX_F64 ? 8 : (dt == VBX_I16 ? 2 : ((dt == VBX_MULAW8 || dt == VBX_ALAW8) ? 1 : 4));
}

// validates a vbx_frames descriptor (device or host pointers alike)
int vbx_check_frames(vbx_ctx* ctx, const vbx_frames* fr, bool allow_f64 = false);
// number of samples spanned by the strided view (0 if n_frames == 0)
static inline int64_t vbx_frames_per_segment(const vbx_frames* fr) {
    return fr->frames_per_segment > 0 ? fr->frames_per_segment : fr->n_frames;
}
// samples between consecutive samples of a frame (vbx_frames.sample_step: 0 and 1 are contiguous)
static inline int64_t vbx_sample_step(const vbx_frames* fr) { return fr->sample_step > 1 ? fr->sample_step : 1; }
static inline int64_t vbx_frames_extent(const vbx_frames* fr) {
    if (fr->n_frames <= 0) return 0;
    const int64_t J = vbx_frames_per_segment(fr), segs = fr->n_frames / J;
    return (segs - 1) * (fr->frames_per_segment > 0 ? fr->segment_stride : 0) + (J - 1) * fr->frame_stride +
           ((int64_t)fr->frame_len - 1) * vbx_sample_step(fr) + 1;
}
// Interleaved views (sample_step > 1, vbx_interleave.cu).  The planar equivalent of the header: segment u's channel samples
// P[u][k] = base[u*segment_stride + k*s], k < vbx_planar_len, in rows of vbx_planar_row samples.
static inline int64_t vbx_planar_len(const vbx_frames* fr) {
    return ((vbx_frames_per_segment(fr) - 1) * fr->frame_stride) / vbx_sample_step(fr) + fr->frame_len;
}
static inline int64_t vbx_planar_row(const vbx_frames* fr) { return (vbx_planar_len(fr) + 63) & ~(int64_t)63; }
// *out = the planar equivalent of *fr: for an interleaved view, gathered on the context's stream into ctx->planar (a grow-only
// buffer of its own, never the scratch arena or a caller's sub-range of it); any other view is copied unchanged.  Every
// frame-view entry point that launches kernels calls this once after its argument checks.  lead > 0 (the host pipeline) puts
// `lead` zero samples before every row, so that the view starts at planar offset lead (rows: lead + S rounded up to 64).
int vbx_planarize(vbx_ctx* ctx, const vbx_frames* fr, vbx_frames* out, int64_t lead = 0);
// max |x| over segment u's channel samples (a host view; the global peak vbx_frame_peaks defines), dtype scaling included
double vbx_host_peak(const vbx_frames* fr, int64_t u);

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
#ifdef __CUDACC__
template <typename T> __device__ __forceinline__ T vbx_ldg(const T* p) { return __ldg(p); }

// G.711 (VBX_MULAW8 / VBX_ALAW8): one byte per sample.  The tag types give the kernels one instantiation per law.
struct vbx_mulaw8 { uint8_t code; };
struct vbx_alaw8 { uint8_t code; };

// code -> the 16-bit linear value of ITU-T G.711 (g711.c's ulaw2linear / alaw2linear).  Arithmetic rather than a table: the
// 32 lanes of a warp load 32 different codes, which a constant-memory table would serialise.
__host__ __device__ __forceinline__ int vbx_mulaw_decode(unsigned b) {
    const unsigned u = ~b & 0xffu;
    const int t = (int)(((u & 0x0fu) << 3) + 0x84u) << ((u & 0x70u) >> 4);
    return (u & 0x80u) ? 0x84 - t : t - 0x84;
}
__host__ __device__ __forceinline__ int vbx_alaw_decode(unsigned b) {
    const unsigned a = (b ^ 0x55u) & 0xffu;
    const unsigned seg = (a & 0x70u) >> 4;
    int t = (int)((a & 0x0fu) << 4) + (seg ? 0x108 : 8);
    if (seg > 1) t <<= seg - 1;
    return (a & 0x80u) ? t : -t;
}
// int16 -> code, as audioop.lin2ulaw / lin2alaw(x, 2): g711.c's 14-bit mu-law encoder on x >> 2, 13-bit A-law encoder on x >> 3
__host__ __device__ __forceinline__ unsigned vbx_mulaw_encode(int x) {
    int v = x >> 2;
    unsigned mask = 0xffu;
    if (v < 0) { v = -v; mask = 0x7fu; }
    if (v > 8159) v = 8159;
    v += 0x84 >> 2;
    int seg = 0;
    while (seg < 8 && v > (0x40 << seg) - 1) ++seg;  // seg_uend = {0x3F, 0x7F, ..., 0x1FFF}
    if (seg >= 8) return 0x7fu ^ mask;
    return (((unsigned)seg << 4) | (((unsigned)v >> (seg + 1)) & 0x0fu)) ^ mask;
}
__host__ __device__ __forceinline__ unsigned vbx_alaw_encode(int x) {
    int v = x >> 3;
    unsigned mask = 0xd5u;
    if (v < 0) { v = -v - 1; mask = 0x55u; }
    int seg = 0;
    while (seg < 8 && v > (0x20 << seg) - 1) ++seg;  // seg_aend = {0x1F, 0x3F, ..., 0xFFF}
    if (seg >= 8) return 0x7fu ^ mask;
    const unsigned q = seg < 2 ? ((unsigned)v >> 1) & 0x0fu : ((unsigned)v >> seg) & 0x0fu;
    return (((unsigned)seg << 4) | q) ^ mask;
}

template <typename TIn> struct vbx_g711 { static constexpr bool value = false; };
template <> struct vbx_g711<vbx_mulaw8> { static constexpr bool value = true; };
template <> struct vbx_g711<vbx_alaw8> { static constexpr bool value = true; };
// sample types that load as integer PCM values (the 1/32767 scale lives in the window table)
template <typename TIn> struct vbx_pcm { static constexpr bool value = vbx_g711<TIn>::value; };
template <> struct vbx_pcm<int16_t> { static constexpr bool value = true; };

// the value of one G.711 code (the low byte of `code`)
template <typename TIn> __device__ __forceinline__ float vbx_decode8(unsigned code);
template <> __device__ __forceinline__ float vbx_decode8<vbx_mulaw8>(unsigned code) { return (float)vbx_mulaw_decode(code & 0xffu); }
template <> __device__ __forceinline__ float vbx_decode8<vbx_alaw8>(unsigned code) { return (float)vbx_alaw_decode(code & 0xffu); }
// the 16 samples of one 16-byte load of G.711 codes, in memory order
template <typename TIn> __device__ __forceinline__ void vbx_decode16(const uint4& v, float (&x)[16]) {
    const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int h = 0; h < 4; ++h)
#pragma unroll
        for (int b = 0; b < 4; ++b) x[4 * h + b] = vbx_decode8<TIn>(w[h] >> (8 * b));
}

// sample load with dtype dispatch (F32, raw I16 PCM, or G.711 decoded to the int16 value: the 1/32767 scale lives in the
// window table, vbx_get_window)
template <typename TIn> __device__ __forceinline__ float vbx_load_sample(const TIn* p);
template <> __device__ __forceinline__ float vbx_load_sample<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float vbx_load_sample<int16_t>(const int16_t* p) { return (float)__ldg(p); }
template <> __device__ __forceinline__ float vbx_load_sample<vbx_mulaw8>(const vbx_mulaw8* p) {
    return vbx_decode8<vbx_mulaw8>(__ldg(reinterpret_cast<const unsigned char*>(p)));
}
template <> __device__ __forceinline__ float vbx_load_sample<vbx_alaw8>(const vbx_alaw8* p) {
    return vbx_decode8<vbx_alaw8>(__ldg(reinterpret_cast<const unsigned char*>(p)));
}
// double-valued loader for the paths that also accept f64 samples (Burg / find_formants)
template <typename TIn> __device__ __forceinline__ double vbx_load_sample_d(const TIn* p) { return (double)vbx_load_sample<TIn>(p); }
template <> __device__ __forceinline__ double vbx_load_sample_d<double>(const double* p) { return __ldg(p); }

template <typename TOut> __device__ __forceinline__ void vbx_store(TOut* p, double v) { *p = (TOut)v; }

__device__ __forceinline__ double vbx_shfl_xor(double v, int mask) { return __shfl_xor_sync(0xffffffffu, v, mask); }
#endif
