// vbx_multi.cu — the whole box behind one handle: utterance sharding over the GPUs of a node with a host-side gather.
//
// SURVEY §8(e): the path shards by utterance (frames are independent; the McCandless tracker carries state only inside
// an utterance), so there is NO data-path collective: device i runs the complete kernel chain on a contiguous range of
// the caller's utterances and its results land directly in the caller's single host buffer at that range's rows — that
// is the "gather".  One worker thread per device owns that device's vbx_ctx (contexts are single-threaded by contract)
// and runs the ordinary `_host` pipeline (vbx_pipeline.cuh: chunked H2D / kernels / D2H on three streams) on its range,
// so all devices stage and compute concurrently.  A worker binds itself to the CPUs the kernel reports as local to its
// GPU's PCIe root (sysfs local_cpulist) before it creates its context, so the context's staging allocations and the
// copy-engine doorbells stay on the GPU's NUMA node.  A Rust (or any) host drives 1…8 GPUs through this C ABI with no
// torch / NCCL / MPI in the process.
#include <sched.h>

#include <condition_variable>
#include <cstdlib>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "vbx_internal.cuh"

struct vbx_multi {
    int n = 0;
    std::vector<int> devices;
    std::vector<vbx_ctx*> ctxs;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    std::function<int(int, vbx_ctx*)> job;
    uint64_t generation = 0;
    int pending = 0;
    bool stop = false;
    std::vector<int> status;
    std::vector<int> create_status;
    char err[640] = {0};
};

namespace {

// CPUs local to the device's PCIe root: /sys/bus/pci/devices/<domain:bus:dev.fn>/local_cpulist ("0-31,64-95")
void bind_to_device_cpus(int device) {
    if (const char* e = getenv("VBX_MULTI_NO_BIND"))
        if (e[0] == '1') return;
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) { cudaGetLastError(); return; }
    for (char* p = bdf; *p; ++p) *p = (char)tolower(*p);
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", bdf);
    FILE* f = fopen(path, "r");
    if (!f) return;
    char line[1024] = {0};
    const bool got = fgets(line, sizeof(line), f) != nullptr;
    fclose(f);
    if (!got) return;
    cpu_set_t allowed, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return;
    int count = 0;
    for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k == 1) b = a;
        if (k < 1) continue;
        for (int c = a; c <= b && c < CPU_SETSIZE; ++c)
            if (CPU_ISSET(c, &allowed)) { CPU_SET(c, &want); ++count; }
    }
    if (count > 0) sched_setaffinity(0, sizeof(want), &want);
}

void worker_main(vbx_multi* m, int idx) {
    bind_to_device_cpus(m->devices[idx]);
    vbx_ctx* ctx = nullptr;
    const int st = vbx_ctx_create(m->devices[idx], &ctx);
    uint64_t seen = 0;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->ctxs[idx] = ctx;
        m->create_status[idx] = st;
        --m->pending;
    }
    m->cv_done.notify_all();
    while (true) {
        std::function<int(int, vbx_ctx*)> job;
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_job.wait(lk, [&] { return m->stop || m->generation != seen; });
            if (m->stop) break;
            seen = m->generation;
            job = m->job;
        }
        const int rc = ctx ? job(idx, ctx) : VBX_ERR_CUDA;
        {
            std::lock_guard<std::mutex> lk(m->mu);
            m->status[idx] = rc;
            --m->pending;
        }
        m->cv_done.notify_all();
    }
    if (ctx) vbx_ctx_destroy(ctx);
}

// runs fn(idx, ctx) on every worker concurrently; returns the first non-OK status (message copied into m->err)
int run_all(vbx_multi* m, std::function<int(int, vbx_ctx*)> fn) {
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->job = std::move(fn);
        m->pending = m->n;
        ++m->generation;
    }
    m->cv_job.notify_all();
    {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv_done.wait(lk, [&] { return m->pending == 0; });
    }
    for (int i = 0; i < m->n; ++i)
        if (m->status[i] != VBX_OK) {
            snprintf(m->err, sizeof(m->err), "device %d: %s", m->devices[i], m->ctxs[i] ? m->ctxs[i]->err : "no context");
            return m->status[i];
        }
    return VBX_OK;
}

struct Shard {
    vbx_frames fr;    // this device's sub-view (host pointers)
    int64_t frame0;   // first frame of the sub-view inside the caller's batch (row offset of every per-frame output)
    int64_t seg0;     // first segment (row offset of per-segment state)
};

// Contiguous ranges of segments (utterances), or of frames when the view is one segment and `by_frames_ok`.
Shard shard_of(const vbx_frames* fr, int n_parts, int part, bool by_frames_ok) {
    Shard s;
    s.fr = *fr;
    s.frame0 = 0;
    s.seg0 = 0;
    const size_t es = vbx_dtype_size(fr->dtype);
    if (fr->frames_per_segment > 0) {
        const int64_t J = fr->frames_per_segment, U = fr->n_frames / J;
        int64_t lo, hi;
        vbx_multi_partition(U, n_parts, part, &lo, &hi);
        s.fr.base = (const char*)fr->base + (size_t)lo * fr->segment_stride * es;
        s.fr.n_frames = (hi - lo) * J;
        s.frame0 = lo * J;
        s.seg0 = lo;
    } else if (by_frames_ok) {
        int64_t lo, hi;
        vbx_multi_partition(fr->n_frames, n_parts, part, &lo, &hi);
        s.fr.base = (const char*)fr->base + (size_t)lo * fr->frame_stride * es;
        s.fr.n_frames = hi - lo;
        s.frame0 = lo;
    } else if (part != 0) {
        s.fr.n_frames = 0;  // one sequential segment: device 0 takes it all
    }
    return s;
}

inline void* row(void* p, int64_t r, size_t bytes_per_row) { return p ? (char*)p + (size_t)r * bytes_per_row : nullptr; }

}  // namespace

extern "C" {

void vbx_multi_partition(int64_t n_units, int32_t n_parts, int32_t part, int64_t* lo, int64_t* hi) {
    if (n_parts < 1) n_parts = 1;
    if (part < 0) part = 0;
    if (part >= n_parts) part = n_parts - 1;
    if (n_units < 0) n_units = 0;
    // floor(n·p / parts) without overflow for n < 2^62 / parts
    const int64_t q = n_units / n_parts, r = n_units % n_parts;
    const int64_t a = q * part + (r * part) / n_parts, b = q * (part + 1) + (r * (part + 1)) / n_parts;
    if (lo) *lo = a;
    if (hi) *hi = b;
}

int vbx_multi_create(int32_t n_devices, const int32_t* devices, vbx_multi** out) {
    if (!out) return VBX_ERR_BADARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        cudaGetLastError();
        return VBX_ERR_CUDA;  // no CPU fallback
    }
    if (n_devices <= 0) n_devices = count;  // 0 = every visible device
    if (n_devices > count && !devices) return VBX_ERR_BADARG;
    vbx_multi* m = new vbx_multi();
    m->n = n_devices;
    for (int i = 0; i < n_devices; ++i) {
        const int d = devices ? devices[i] : i;
        if (d < 0 || d >= count) { delete m; return VBX_ERR_BADARG; }
        m->devices.push_back(d);
    }
    m->ctxs.assign(n_devices, nullptr);
    m->status.assign(n_devices, VBX_OK);
    m->create_status.assign(n_devices, VBX_OK);
    m->pending = n_devices;
    for (int i = 0; i < n_devices; ++i) m->workers.emplace_back(worker_main, m, i);
    {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv_done.wait(lk, [&] { return m->pending == 0; });
    }
    for (int i = 0; i < n_devices; ++i)
        if (m->create_status[i] != VBX_OK) {
            const int st = m->create_status[i];
            vbx_multi_destroy(m);
            return st;
        }
    *out = m;
    return VBX_OK;
}

int vbx_multi_destroy(vbx_multi* m) {
    if (!m) return VBX_OK;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->stop = true;
    }
    m->cv_job.notify_all();
    for (auto& t : m->workers)
        if (t.joinable()) t.join();
    delete m;
    return VBX_OK;
}

int32_t vbx_multi_device_count(vbx_multi* m) { return m ? m->n : 0; }
vbx_ctx* vbx_multi_ctx(vbx_multi* m, int32_t i) { return (m && i >= 0 && i < m->n) ? m->ctxs[i] : nullptr; }
const char* vbx_multi_last_error(vbx_multi* m) { return m ? m->err : "no handle"; }
int64_t vbx_multi_kernel_launches(vbx_multi* m) {
    int64_t n = 0;
    if (m)
        for (auto* c : m->ctxs) n += c ? c->launches : 0;
    return n;
}

int vbx_multi_lpc_host(vbx_multi* m, const vbx_frames* frames, int32_t p, void* r_out, void* ac_out, void* kc_out, int32_t out_dtype) {
    if (!m || !frames) return VBX_ERR_BADARG;
    const size_t os = vbx_dtype_size(out_dtype);
    return run_all(m, [=](int i, vbx_ctx* ctx) -> int {
        const Shard s = shard_of(frames, m->n, i, true);
        if (s.fr.n_frames == 0) return VBX_OK;
        return vbx_lpc_host(ctx, &s.fr, p, row(r_out, s.frame0, (size_t)(p + 1) * os), row(ac_out, s.frame0, (size_t)(p + 1) * os),
                            row(kc_out, s.frame0, (size_t)p * os), out_dtype);
    });
}

int vbx_multi_find_formants_host(vbx_multi* m, const vbx_frames* frames, double sample_rate, int32_t n_coeffs, int32_t lpc_method,
                                 void* est_inout, int32_t n_formants, void* tracks_out, void* resonances_out, int32_t* nres_out,
                                 uint8_t* status_out, int32_t dtype) {
    if (!m || !frames) return VBX_ERR_BADARG;
    const size_t pair = (dtype == VBX_F64) ? 16 : 8;
    return run_all(m, [=](int i, vbx_ctx* ctx) -> int {
        // the tracker is sequential inside a segment: a single-segment view is not split (device 0 takes it)
        const Shard s = shard_of(frames, m->n, i, false);
        if (s.fr.n_frames == 0) return VBX_OK;
        return vbx_find_formants_host(ctx, &s.fr, sample_rate, n_coeffs, lpc_method, row(est_inout, s.seg0, (size_t)n_formants * pair),
                                      n_formants, row(tracks_out, s.frame0, (size_t)n_formants * pair),
                                      row(resonances_out, s.frame0, (size_t)VBX_MAX_RESONANCES * pair),
                                      (int32_t*)row(nres_out, s.frame0, 4), (uint8_t*)row(status_out, s.frame0, 1), dtype);
    });
}

int vbx_multi_pitch_host(vbx_multi* m, const vbx_frames* frames, double sample_rate, double threshold, double min_hz, double max_hz,
                         int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int32_t out_dtype) {
    return vbx_multi_pitch_with_peaks_host(m, frames, sample_rate, threshold, 0.0, nullptr, nullptr, min_hz, max_hz, max_candidates,
                                           cand_out, n_cand_out, status_out, out_dtype);
}

// A single-segment view is split into frame ranges, so its missing global peak is taken over the whole view first, as
// vbx_pitch_with_peaks_host does for its chunks; every device then reads the same value.
int vbx_multi_pitch_with_peaks_host(vbx_multi* m, const vbx_frames* frames, double sample_rate, double threshold,
                                    double silence_threshold, const double* local_peaks, const double* global_peaks, double min_hz,
                                    double max_hz, int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out,
                                    int32_t out_dtype) {
    if (!m || !frames) return VBX_ERR_BADARG;
    const size_t pair = (out_dtype == VBX_F64) ? 16 : 8;
    const bool segmented = frames->frames_per_segment > 0;
    double whole = 0.0;
    const double* global = global_peaks;
    if (silence_threshold > 0.0 && !global && !segmented && frames->n_frames > 0 && frames->base && frames->frame_len >= 1 &&
        frames->frame_stride >= 1 && (frames->dtype == VBX_F32 || vbx_dtype_is_pcm(frames->dtype) || frames->dtype == VBX_F64)) {
        whole = vbx_host_peak(frames, 0);
        global = &whole;
    }
    return run_all(m, [=](int i, vbx_ctx* ctx) -> int {
        const Shard s = shard_of(frames, m->n, i, true);
        if (s.fr.n_frames == 0) return VBX_OK;
        return vbx_pitch_with_peaks_host(ctx, &s.fr, sample_rate, threshold, silence_threshold,
                                         local_peaks ? local_peaks + s.frame0 : nullptr,
                                         global ? global + (segmented ? s.seg0 : 0) : nullptr, min_hz, max_hz, max_candidates,
                                         row(cand_out, s.frame0, (size_t)max_candidates * pair), (int32_t*)row(n_cand_out, s.frame0, 4),
                                         (uint8_t*)row(status_out, s.frame0, 1), out_dtype);
    });
}

int vbx_multi_mfcc_host(vbx_multi* m, const vbx_frames* frames, int32_t num_coeffs, int32_t n_keep, double freq_lo, double freq_hi,
                        double sample_rate, void* out, int32_t out_dtype) {
    if (!m || !frames) return VBX_ERR_BADARG;
    const size_t os = vbx_dtype_size(out_dtype);
    return run_all(m, [=](int i, vbx_ctx* ctx) -> int {
        const Shard s = shard_of(frames, m->n, i, true);
        if (s.fr.n_frames == 0) return VBX_OK;
        return vbx_mfcc_host(ctx, &s.fr, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, row(out, s.frame0, (size_t)n_keep * os),
                             out_dtype);
    });
}

// Host→device copy bandwidth of the first n_active devices, all copying at once from pinned buffers their own (NUMA-bound)
// worker allocated: the probe behind tools/h2d_probe.py (which link saturates as more GPUs stage concurrently).
int vbx_multi_h2d_bandwidth(vbx_multi* m, size_t bytes_per_device, int32_t reps, int32_t n_active, double* gbs_out) {
    if (!m || !gbs_out || bytes_per_device == 0 || reps < 1) return VBX_ERR_BADARG;
    if (n_active <= 0 || n_active > m->n) n_active = m->n;
    for (int i = 0; i < m->n; ++i) gbs_out[i] = 0.0;
    return run_all(m, [=](int i, vbx_ctx* ctx) -> int {
        if (i >= n_active) return VBX_OK;
        cudaSetDevice(ctx->device);
        void *h = nullptr, *d = nullptr;
        if (cudaMallocHost(&h, bytes_per_device) != cudaSuccess) { cudaGetLastError(); return vbx_fail(ctx, VBX_ERR_NOMEM, "probe: cudaMallocHost failed"); }
        if (cudaMalloc(&d, bytes_per_device) != cudaSuccess) { cudaGetLastError(); cudaFreeHost(h); return vbx_fail(ctx, VBX_ERR_NOMEM, "probe: cudaMalloc failed"); }
        memset(h, 1, bytes_per_device);
        cudaMemcpyAsync(d, h, bytes_per_device, cudaMemcpyHostToDevice, ctx->stream);  // warm-up
        cudaStreamSynchronize(ctx->stream);
        cudaEventRecord(ctx->ev_start, ctx->stream);
        for (int r = 0; r < reps; ++r) cudaMemcpyAsync(d, h, bytes_per_device, cudaMemcpyHostToDevice, ctx->stream);
        cudaEventRecord(ctx->ev_stop, ctx->stream);
        cudaEventSynchronize(ctx->ev_stop);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop);
        gbs_out[i] = ms > 0.f ? (double)bytes_per_device * reps / (ms * 1e-3) / 1e9 : 0.0;
        cudaFree(d);
        cudaFreeHost(h);
        const cudaError_t e = cudaGetLastError();
        return e == cudaSuccess ? VBX_OK : vbx_fail(ctx, VBX_ERR_CUDA, "probe: %s", cudaGetErrorString(e));
    });
}

}  // extern "C"
