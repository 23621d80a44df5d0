// vbx_lpc.cu — windowed autocorrelation (fp64 accumulate) + Levinson–Durbin, fused.
//
// Replaces, batched over frames:
//   periodic.rs:265-289  Autocorrelate::autocorrelate_mut   r[lag] = x[0] + Σ_{i>=1} x[i]·x[i+lag]
//   spectrum.rs:63-84    LPC::lpc_mut (Levinson–Durbin)
// with the window multiply of the reference's callers (Windower::hanning / lib.rs:66-70) fused
// into the load.
//
// Kernel shape (DESIGN.md §K1/K2): a CTA stages the contiguous audio span of G overlapping frames
// in shared memory once (padded so that frame starts fall in distinct banks), then every group of K
// lanes owns one frame.  A lane walks its part of the frame sequentially with the last L windowed
// samples in a register ring and L fp64 accumulators (L = p+1 lags, all static indices): per sample
// 1 LDS (sample) + 1 LDS.64 (window) + 1 DMUL + L DFMA, no cross-lane traffic in the loop.  K>1
// partial sums are combined with shuffles; Levinson then runs one thread per frame out of shared
// memory and the results leave through a coalesced store.
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "vbx_internal.cuh"
#include "vbx_pipeline.cuh"

namespace {

constexpr int kMaxThreads = 128;

struct LpcParams {
    const void* base;      // samples
    const double* win;     // [n] device window table (ones for WINDOW_NONE)
    void* r_out;           // [F][L]   or null
    void* ac_out;          // [F][L]   or null
    void* kc_out;          // [F][L-1] or null
    int64_t n_frames;
    int64_t stride;        // frame stride in samples
    int64_t seg_frames;    // frames per segment (utterance); a CTA's frames lie in one segment unless `straddle`
    int64_t seg_stride;    // samples between segment starts
    int ctas_per_seg;
    int threads;           // CTA size (multiple of 32, <= kMaxThreads)
    unsigned sv_magic;     // floor(2^32 / sv) + 1: s / sv == __umulhi(s, sv_magic) for s·sv < 2^32
    int n;                 // frame length
    int k;                 // lanes per frame (power of two <= 32)
    int frames_per_cta;    // G = kThreads / k
    int sv;                // virtual stride inside shared memory: min(stride, n)
    int pad;               // 0/1: one pad word after every sv samples so that (sv+pad) is odd
    int part;              // samples per lane part: ceil(n / k)
    int span_words;        // shared-memory words reserved for the padded span
    int out_f64;           // outputs are double (else float)
    int do_levinson;
    int straddle;          // lpc_fused16_kernel: CTAs take G consecutive frames of the batch, across segment boundaries
};

// Levinson–Durbin exactly as spectrum.rs:63-84 (no zero guard: err == 0 propagates inf/NaN).
template <int P>
__device__ __forceinline__ void levinson(const double* __restrict__ r, double* __restrict__ ac, double* __restrict__ kc) {
    double a[P + 1];
    double err = r[0];
    a[0] = 1.0;
#pragma unroll
    for (int i = 1; i <= P; ++i) a[i] = 0.0;
#pragma unroll
    for (int i = 1; i <= P; ++i) {
        double acc = r[i];
#pragma unroll
        for (int j = 1; j < i; ++j) acc = acc + a[j] * r[i - j];
        const double k = (-acc) / err;
        kc[i - 1] = k;
        a[i] = k;
        // ac[j] += k·tmp[i-j] for j in 1..i-1 with tmp = the pre-update copy (spectrum.rs:76-81):
        // updated pairwise so both ends read old values and no copy is needed
#pragma unroll
        for (int j = 1; 2 * j < i; ++j) {
            const double lo = a[j], hi = a[i - j];
            a[j] = lo + k * hi;
            a[i - j] = hi + k * lo;
        }
        if ((i & 1) == 0) a[i / 2] = a[i / 2] + k * a[i / 2];
        err = err * (1.0 - k * k);
    }
#pragma unroll
    for (int i = 0; i <= P; ++i) ac[i] = a[i];
}

// Common epilogue of the fused kernels: the frame leaders park r in shared memory (the span is dead by
// then), Levinson runs one thread per frame, and r / ac / kc leave through coalesced stores.
template <int L>
__device__ __forceinline__ void lpc_finish(const LpcParams& P, const double (&acc)[L], bool leader, int g, int Gc, int64_t g0,
                                           double* s_out) {
    const int tid = threadIdx.x, nthreads = P.threads, G = P.frames_per_cta;
    __syncthreads();  // everyone is done reading the span; reuse it as output staging

    double* s_r = s_out;                  // [G][L]
    double* s_ac = s_r + G * L;           // [G][L]
    double* s_kc = s_ac + G * L;          // [G][L-1]
    if (leader) {
#pragma unroll
        for (int lag = 0; lag < L; ++lag) s_r[g * L + lag] = acc[lag];
    }
    __syncthreads();
    if (P.do_levinson && tid < Gc) {
        double r[L], ac[L], kc[L - 1];
#pragma unroll
        for (int lag = 0; lag < L; ++lag) r[lag] = s_r[tid * L + lag];
        levinson<L - 1>(r, ac, kc);
#pragma unroll
        for (int lag = 0; lag < L; ++lag) s_ac[tid * L + lag] = ac[lag];
#pragma unroll
        for (int j = 0; j < L - 1; ++j) s_kc[tid * (L - 1) + j] = kc[j];
    }
    __syncthreads();

    // ---- coalesced write-out --------------------------------------------------------------
    auto store = [&](void* out, const double* src, int per_frame) {
        if (!out) return;
        const int total = Gc * per_frame;
        const int64_t off = g0 * per_frame;
        if (P.out_f64) {
            double* o = reinterpret_cast<double*>(out) + off;
            for (int idx = tid; idx < total; idx += nthreads) o[idx] = src[idx];
        } else {
            float* o = reinterpret_cast<float*>(out) + off;
            for (int idx = tid; idx < total; idx += nthreads) o[idx] = (float)src[idx];
        }
    };
    store(P.r_out, s_r, L);
    if (P.do_levinson) {
        store(P.ac_out, s_ac, L);
        store(P.kc_out, s_kc, L - 1);
    }
}

template <int L, typename TIn>
__global__ void __launch_bounds__(kMaxThreads, (L <= 13 ? 5 : 1)) lpc_fused_kernel(const LpcParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_win = reinterpret_cast<double*>(smem_raw);                 // [n]
    float* s_span = reinterpret_cast<float*>(s_win + P.n);               // padded span
    double* s_out = reinterpret_cast<double*>(s_win + P.n);              // staging, reuses the span after a barrier

    const int tid = threadIdx.x;
    const int G = P.frames_per_cta;
    const int64_t seg = blockIdx.x / P.ctas_per_seg;
    const int64_t j0 = (int64_t)(blockIdx.x - seg * P.ctas_per_seg) * G;  // first frame of this CTA inside its segment
    const int64_t g0 = seg * P.seg_frames + j0;                           // ... and in the batch (output row)
    const int Gc = (int)min((int64_t)G, P.seg_frames - j0);
    const int n = P.n, sv = P.sv, pad = P.pad;
    const TIn* __restrict__ base = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride;

    // ---- stage window + span -------------------------------------------------------------
    const int nthreads = P.threads;
    for (int i = tid; i < n; i += nthreads) s_win[i] = __ldg(P.win + i);
    if (P.stride <= (int64_t)n) {
        // overlapped / packed frames: one contiguous run of (Gc-1)·stride + n samples, copied with many
        // independent loads in flight per thread; word s lands at s + pad·(s / sv)
        const TIn* src = base + j0 * P.stride;
        const int total = (Gc - 1) * sv + n;
        const unsigned magic = P.sv_magic;
        auto phys = [&](int s_) -> int { return pad ? s_ + (int)__umulhi((unsigned)s_, magic) : s_; };
        int done = 0;
        if (sizeof(TIn) == 4 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            // 16-byte loads, 8 in flight per thread.  With pad == 0 the copy is the identity; with
            // sv % 4 == 0 the four words of a load stay inside one sv-block (one division per load)
            const float4* src4 = reinterpret_cast<const float4*>(src);
            const int n4 = total >> 2;
            for (int v0 = tid; v0 < n4; v0 += 8 * nthreads) {
                float4 a[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int v = v0 + u * nthreads;
                    if (v < n4) a[u] = __ldg(src4 + v);
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int v = v0 + u * nthreads;
                    if (v < n4) {
                        if (pad == 0 || (sv & 3) == 0) {
                            float* dst = s_span + phys(4 * v);
                            dst[0] = a[u].x;
                            dst[1] = a[u].y;
                            dst[2] = a[u].z;
                            dst[3] = a[u].w;
                        } else {
                            s_span[phys(4 * v)] = a[u].x;
                            s_span[phys(4 * v + 1)] = a[u].y;
                            s_span[phys(4 * v + 2)] = a[u].z;
                            s_span[phys(4 * v + 3)] = a[u].w;
                        }
                    }
                }
            }
            done = n4 << 2;
        }
        if (sizeof(TIn) == 2 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            // int16 PCM: 16-byte loads of 8 samples, 4 in flight per thread
            const uint4* src8 = reinterpret_cast<const uint4*>(src);
            const int n8 = total >> 3;
            for (int v0 = tid; v0 < n8; v0 += 4 * nthreads) {
                uint4 a[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int v = v0 + u * nthreads;
                    if (v < n8) a[u] = __ldg(src8 + v);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int v = v0 + u * nthreads;
                    if (v < n8) {
                        const unsigned w[4] = {a[u].x, a[u].y, a[u].z, a[u].w};
#pragma unroll
                        for (int h = 0; h < 4; ++h) {
                            s_span[phys(8 * v + 2 * h)] = (float)(short)(w[h] & 0xffffu);
                            s_span[phys(8 * v + 2 * h + 1)] = (float)(short)(w[h] >> 16);
                        }
                    }
                }
            }
            done = n8 << 3;
        }
        if constexpr (vbx_g711<TIn>::value) {
            if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
                // G.711: 16-byte loads of 16 codes, 4 in flight per thread, decoded as they land
                const uint4* src16 = reinterpret_cast<const uint4*>(src);
                const int n16 = total >> 4;
                for (int v0 = tid; v0 < n16; v0 += 4 * nthreads) {
                    uint4 a[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int v = v0 + u * nthreads;
                        if (v < n16) a[u] = __ldg(src16 + v);
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int v = v0 + u * nthreads;
                        if (v < n16) {
                            float x[16];
                            vbx_decode16<TIn>(a[u], x);
#pragma unroll
                            for (int e = 0; e < 16; ++e) s_span[phys(16 * v + e)] = x[e];
                        }
                    }
                }
                done = n16 << 4;
            }
        }
        for (int s0 = done + tid; s0 < total; s0 += 8 * nthreads) {
            float a[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int s_ = s0 + u * nthreads;
                if (s_ < total) a[u] = vbx_load_sample<TIn>(src + s_);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int s_ = s0 + u * nthreads;
                if (s_ < total) s_span[phys(s_)] = a[u];
            }
        }
    } else {
        // gapped frames: each frame's n samples land in consecutive blocks of sv == n words
        const int warp = tid >> 5, lane = tid & 31;
        for (int g = warp; g < Gc; g += nthreads / 32) {
            const TIn* src = base + (j0 + g) * P.stride;
            for (int j = lane; j < n; j += 32) s_span[g * (sv + pad) + j] = vbx_load_sample<TIn>(src + j);
        }
    }
    __syncthreads();

    // ---- per-lane partial autocorrelation -------------------------------------------------
    const int k = P.k;
    const int g = tid / k, q = tid - g * k;
    double acc[L], h[L];
#pragma unroll
    for (int j = 0; j < L; ++j) { acc[j] = 0.0; h[j] = 0.0; }
    double x0 = 0.0;  // frame sample 0 (windowed) for the reference's "+ x[0]" seed
    if (g < Gc) {
        const int i_begin = q * P.part;
        const int i_end = min(n, i_begin + P.part);
        // running position in the padded span: pos(i) = g·(sv+pad) + i + pad·(i / sv)
        int i = (q == 0) ? 0 : max(0, i_begin - (L - 1));
        int blk = i / sv;
        int pos = g * (sv + pad) + i + pad * blk;
        int left = sv - (i - blk * sv);  // samples until the next pad word
        auto fetch = [&](int idx) -> double {
            double v = (double)s_span[pos] * s_win[idx];
            ++pos;
            if (--left == 0) { pos += pad; left = sv; }
            return v;
        };
        if (q != 0) {
            // history: h[j] = xw[i_begin - L + j], j = 1..L-1 (i_begin >= L-1 is guaranteed by the host)
#pragma unroll
            for (int j = 1; j < L; ++j) { h[j] = fetch(i); ++i; }
        }
        // full chunks of L samples: ring slot u holds xw[i+u]; lag products use static slots.  A chunk
        // that contains no pad word reads its samples at immediate offsets (no per-sample bookkeeping).
        if (pad == 0) left = 0x3fffffff;
        for (; i + L <= i_end; i += L) {
            float xf[L];
            if (left > L) {
#pragma unroll
                for (int u = 0; u < L; ++u) xf[u] = s_span[pos + u];
                pos += L;
                left -= L;
            } else {
#pragma unroll
                for (int u = 0; u < L; ++u) {
                    xf[u] = s_span[pos];
                    ++pos;
                    if (--left == 0) { pos += pad; left = sv; }
                }
            }
#pragma unroll
            for (int u = 0; u < L; ++u) {
                const double xn = (double)xf[u] * s_win[i + u];
                h[u] = xn;
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(xn, h[(u - lag + L) % L], acc[lag]);
            }
            if (q == 0 && i == 0) {
                // reference quirk (periodic.rs:284): the fold is seeded with x[0] and skips the i = 0
                // product, so r[lag] = true_r[lag] − x0·x[lag] + x0.  After the first chunk h[j] = xw[j].
                x0 = h[0];
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(x0, 1.0 - h[lag], acc[lag]);
            }
        }
        // tail chunk (< L samples): zero-fed slots contribute nothing
        if (i < i_end) {
            const bool first = (q == 0 && i == 0);
#pragma unroll
            for (int u = 0; u < L; ++u) {
                const double xn = (i + u < i_end) ? fetch(i + u) : 0.0;
                h[u] = xn;
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(xn, h[(u - lag + L) % L], acc[lag]);
            }
            if (first) {  // n < L: lags >= n see x[lag] = 0, r[lag] = x0 as in the reference
                x0 = h[0];
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(x0, 1.0 - h[lag], acc[lag]);
            }
        }
    }
    // combine the K parts of a frame (K consecutive lanes, K | 32)
    for (int m = 1; m < k; m <<= 1) {
#pragma unroll
        for (int lag = 0; lag < L; ++lag) acc[lag] += vbx_shfl_xor(acc[lag], m);
    }
    lpc_finish<L>(P, acc, g < Gc && q == 0, g, Gc, g0, s_out);
}

#include "vbx_lpc16.cuh"
#include "vbx_lpca.cuh"

// Generic fallback (any n_lags / frame length): one CTA per frame, windowed frame as fp64 in
// shared memory when it fits, lags strided over warps with a shuffle reduction.
template <typename TIn>
__global__ void __launch_bounds__(256) autocorr_generic_kernel(const TIn* __restrict__ base, const double* __restrict__ win,
                                                               int64_t stride, int64_t seg_frames, int64_t seg_stride, int n,
                                                               int n_lags, void* r_out, int out_f64, int use_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_x = reinterpret_cast<double*>(smem_raw);
    const int64_t f = blockIdx.x;
    const int64_t seg = f / seg_frames;
    const TIn* x = base + seg * seg_stride + (f - seg * seg_frames) * stride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    if (use_smem) {
        for (int i = tid; i < n; i += blockDim.x) s_x[i] = vbx_load_sample_d<TIn>(x + i) * __ldg(win + i);
        __syncthreads();
    }
    auto xw = [&](int i) -> double {
        return use_smem ? s_x[i] : vbx_load_sample_d<TIn>(x + i) * __ldg(win + i);
    };
    const double x0 = xw(0);
    for (int lag = warp; lag < n_lags; lag += nwarps) {
        double acc = 0.0;
        for (int i = 1 + lane; i + lag < n; i += 32) acc = fma(xw(i), xw(i + lag), acc);
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) acc += vbx_shfl_xor(acc, m);
        if (lane == 0) {
            const double r = x0 + acc;
            if (out_f64) reinterpret_cast<double*>(r_out)[f * n_lags + lag] = r;
            else reinterpret_cast<float*>(r_out)[f * n_lags + lag] = (float)r;
        }
    }
}

// periodic.rs:291-304  `impl Autocorrelate for VecDeque<T>`: the same fold on a ring buffer.  One CTA per ring; the
// logical sequence x[i] = ring[(head + i) mod capacity] is unrolled into shared memory as f64 when it fits.
template <typename T>
__global__ void __launch_bounds__(256) autocorr_ring_kernel(const T* __restrict__ rings, int64_t capacity, const int64_t* __restrict__ heads,
                                                            int n, int n_lags, void* r_out, int out_f64, int use_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_x = reinterpret_cast<double*>(smem_raw);
    const int64_t b = blockIdx.x;
    const T* ring = rings + b * capacity;
    const int64_t head = heads ? heads[b] % capacity : 0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    auto at = [&](int i) -> double {
        int64_t j = head + i;
        if (j >= capacity) j -= capacity;
        return (double)ring[j];
    };
    if (use_smem) {
        for (int i = tid; i < n; i += blockDim.x) s_x[i] = at(i);
        __syncthreads();
    }
    auto x = [&](int i) -> double { return use_smem ? s_x[i] : at(i); };
    const double x0 = x(0);
    for (int lag = warp; lag < n_lags; lag += nwarps) {
        double acc = 0.0;
        for (int i = 1 + lane; i + lag < n; i += 32) acc = fma(x(i), x(i + lag), acc);
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) acc += vbx_shfl_xor(acc, m);
        if (lane == 0) {
            const double r = x0 + acc;
            if (out_f64) reinterpret_cast<double*>(r_out)[b * n_lags + lag] = r;
            else reinterpret_cast<float*>(r_out)[b * n_lags + lag] = (float)r;
        }
    }
}

// Stand-alone Levinson: one thread per frame, r read from global (f32 or f64).
template <int PORD>
__global__ void __launch_bounds__(128) levinson_kernel(const void* __restrict__ r_in, int r_f64, int64_t n_frames,
                                                       int r_stride, void* ac_out, void* kc_out, int out_f64) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    double r[PORD + 1], ac[PORD + 1], kc[PORD];
#pragma unroll
    for (int i = 0; i <= PORD; ++i)
        r[i] = r_f64 ? reinterpret_cast<const double*>(r_in)[f * r_stride + i]
                     : (double)reinterpret_cast<const float*>(r_in)[f * r_stride + i];
    levinson<PORD>(r, ac, kc);
    if (ac_out) {
#pragma unroll
        for (int i = 0; i <= PORD; ++i) {
            if (out_f64) reinterpret_cast<double*>(ac_out)[f * (PORD + 1) + i] = ac[i];
            else reinterpret_cast<float*>(ac_out)[f * (PORD + 1) + i] = (float)ac[i];
        }
    }
    if (kc_out) {
#pragma unroll
        for (int i = 0; i < PORD; ++i) {
            if (out_f64) reinterpret_cast<double*>(kc_out)[f * PORD + i] = kc[i];
            else reinterpret_cast<float*>(kc_out)[f * PORD + i] = (float)kc[i];
        }
    }
}

constexpr int kMaxFastLags = 25;  // fused kernel instantiated for 2..25 lags (LPC orders 1..24)
constexpr int kMaxLevinsonOrder = 32;

typedef void (*lpc_kernel_t)(const LpcParams);
typedef void (*lpca_kernel_t)(const LpcParams, const LpcaExtra);
typedef void (*lpcp_kernel_t)(const LpcParams, const LpcaExtra, const int, unsigned*);
typedef void (*lev_kernel_t)(const void*, int, int64_t, int, void*, void*, int);

// Kernel tables indexed by a template argument: t[I] = make(std::integral_constant<int, I>()) for I = Lo..Hi.
template <int Lo, int Hi, typename T, typename Make>
void fill_table(T* t, Make make) {
    t[Lo] = make(std::integral_constant<int, Lo>());
    if constexpr (Lo < Hi) fill_table<Lo + 1, Hi>(t, make);
}

// The two shifted window rows of lpc_fuseda_kernel, E = [0, 0, w…, 0…] and O = [0, 0, 0, w…, 0…] ([2][wt] f64), cached per
// (window kind, n, sample dtype) next to the plain tables.
int get_window_rows_aligned(vbx_ctx* ctx, int kind, int n, int wt, const double** dev_out, int sample_dtype) {
    const bool pcm = vbx_dtype_is_pcm(sample_dtype);
    const uint64_t key = ((uint64_t)(uint32_t)(kind | (pcm ? 0x100 : 0) | 0x200) << 32) | (uint32_t)n;
    auto it = ctx->windows.find(key);
    if (it != ctx->windows.end()) {
        *dev_out = it->second;
        return VBX_OK;
    }
    std::vector<double> w(n), rows((size_t)2 * wt, 0.0);
    vbx_window_fill_host(kind, n, w.data());
    for (int i = 0; i < n; ++i) {
        const double v = pcm ? w[i] / 32767.0 : w[i];
        rows[(size_t)2 + i] = v;        // E
        rows[(size_t)wt + 3 + i] = v;   // O
    }
    double* dev = nullptr;
    cudaError_t e = cudaMalloc(&dev, rows.size() * sizeof(double));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "window rows: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    VBX_CUDA(ctx, cudaMemcpy(dev, rows.data(), rows.size() * sizeof(double), cudaMemcpyHostToDevice));
    ctx->windows[key] = dev;
    *dev_out = dev;
    return VBX_OK;
}

// Choose lanes-per-frame K for a CTA of kMaxThreads: the smallest power of two whose CTA span fits the
// shared-memory budget, keeping each lane's part >= 2L samples.  Returns false if no fused
// configuration fits.
bool plan_fused(const vbx_ctx* ctx, int n, int64_t stride, int L, LpcParams* P, size_t* smem_bytes) {
    const int sv = (int)(stride < (int64_t)n ? stride : n);
    const int pad = ((sv & 1) == 0) ? 1 : 0;
    const size_t budget_soft = 72 * 1024;  // 3 CTAs / SM
    const size_t budget_hard = ctx->smem_optin;
    int best_k = 0;
    size_t best_bytes = 0;
    for (int k = 1; k <= 32; k <<= 1) {
        const int G = kMaxThreads / k;
        const int part = (n + k - 1) / k;
        if (k > 1 && part < 2 * L) break;
        const int64_t span = (int64_t)(G - 1) * sv + n;
        if (span * (int64_t)sv >= (1LL << 32)) continue;  // sv_magic validity
        const int64_t span_words = span + pad * (span / sv + 1) + 4;
        const size_t stage_bytes = (size_t)G * (3 * L - 1) * sizeof(double);
        size_t span_bytes = (size_t)span_words * sizeof(float);
        span_bytes = (span_bytes + 15) & ~(size_t)15;
        const size_t bytes = (size_t)n * sizeof(double) + (span_bytes > stage_bytes ? span_bytes : stage_bytes);
        if (bytes > budget_hard) continue;
        best_k = k;
        best_bytes = bytes;
        P->k = k;
        P->frames_per_cta = G;
        P->part = part;
        P->span_words = (int)span_words;
        if (bytes <= budget_soft) break;
    }
    if (!best_k) return false;
    P->sv = sv;
    P->pad = pad;
    P->threads = kMaxThreads;
    P->sv_magic = sv > 1 ? (unsigned)((1ULL << 32) / (unsigned)sv) + 1u : 0u;
    *smem_bytes = best_bytes;
    return true;
}

// Plan for lpc_fused16_kernel (vbx_lpc16.cuh): 16-aligned framings with at most 16 lags.  Two lanes per frame (a pair of
// warps per 32 frames); the CTA size is chosen as described in the loop below (C2: 128 threads = 64 frames, 4 CTAs / SM).
// VBX_LPC16=0 disables the kernel.
bool plan_fused16(const vbx_ctx* ctx, int n, int64_t stride, int L, LpcParams* P, size_t* smem_bytes) {
    if (L < 2 || L > kChunk || (n % kChunk) != 0) return false;
    const int sv = (int)(stride < (int64_t)n ? stride : n);
    if ((sv % kChunk) != 0) return false;
    if (const char* e = getenv("VBX_LPC16")) {
        if (atoi(e) == 0) return false;
    }
    const int pad = 4;  // sv / 4 is even, so (sv + 4) / 4 is odd: frame starts walk through all 8 bank groups
    const size_t sm_bytes = 228 * 1024, cta_overhead = 1024;
    int best_threads = 0, best_score = 0;
    size_t best_bytes = 0;
    int best_words = 0;
    for (int threads = 64; threads <= 256; threads += 64) {
        const int G = threads / 2;
        const int64_t span = (int64_t)(G - 1) * sv + n;
        if (span * (int64_t)sv >= (1LL << 32)) continue;
        // room for a span staged as two pieces (a CTA that crosses into the next utterance, P.straddle)
        const int64_t span_words = (int64_t)G * (sv + pad) + 2 * ((int64_t)n + pad * (n / sv + 1)) + 8;
        const size_t stage_bytes = (size_t)G * (3 * L - 1) * sizeof(double);
        size_t span_bytes = ((size_t)span_words * sizeof(float) + 15) & ~(size_t)15;
        const size_t bytes = (size_t)n * sizeof(double) + (span_bytes > stage_bytes ? span_bytes : stage_bytes);
        if (bytes > ctx->smem_optin) continue;
        int ctas = (int)(sm_bytes / (bytes + cta_overhead));
        const int by_regs = 65536 / (96 * threads);
        if (ctas > by_regs) ctas = by_regs;
        if (ctas > 32) ctas = 32;
        // Measured on C2 (profiles/r1_lpc16_cta_sweep.txt): 128 threads with 4 CTAs / SM beats both more, smaller CTAs
        // (window reload and span overlap per CTA) and fewer, larger ones (coarser waves, more padding frames in an
        // utterance's last CTA); more than 16 resident warps buys nothing (the kernel is dispatch-bound).  So: reach 16
        // resident warps with at least 3 CTAs, then prefer the CTA size closest to 128.
        const int warps = ctas * threads / 32;
        const int d = threads > 128 ? threads - 128 : 128 - threads;
        const int score = (warps < 16 ? warps : 16) * 1000 + (ctas >= 3 ? 500 : 0) + (256 - d);
        if (score > best_score) {
            best_threads = threads;
            best_score = score;
            best_bytes = bytes;
            best_words = (int)span_words;
        }
    }
    if (!best_threads) return false;
    P->k = 2;
    P->threads = best_threads;
    P->frames_per_cta = best_threads / 2;
    P->part = 0;
    P->span_words = best_words;
    P->sv = sv;
    P->pad = pad;
    P->sv_magic = (unsigned)((1ULL << 32) / (unsigned)sv) + 1u;
    *smem_bytes = best_bytes;
    return true;
}

enum class LpcKind { fused16, persistent, aligned, general, generic };

struct LpcPlan {
    LpcKind kind;
    LpcParams P;   // everything but the window, the outputs and the Levinson flag, which launch_lpc adds
    LpcaExtra X;   // persistent / aligned: geometry of the window rows (launch_lpc adds the rows themselves)
    size_t smem;   // dynamic shared memory per CTA
    int64_t ctas;  // CTAs of the one-shot kernels, tiles of the persistent one
};

// The one place that picks the LPC kernel for a view.  vbx_lpc_scratch_bytes asks it too, so the scratch that
// vbx_find_formants reserves for the LPC stage always matches the path launch_lpc takes.  In order of preference:
// lpc_fused16_kernel (16-aligned framings, <= 16 lags), lpc_fusedp_kernel (fp32, overlapped or packed frames, <= 13 lags,
// enough tiles for every SM), lpc_fuseda_kernel (the same framings), lpc_fused_kernel (<= 25 lags), and the generic
// autocorrelation + stand-alone Levinson.  f64 samples (the single-frame trait calls of the Rust shim on [f64]) take the
// generic kernels: the fused ones stage fp32 / int16 samples.  VBX_LPC_FORCE_GENERIC=1 (tests) sends every view there.
LpcPlan plan_lpc(const vbx_ctx* ctx, const vbx_frames* fr, int L) {
    LpcPlan pl{};
    pl.kind = LpcKind::generic;
    const char* force = getenv("VBX_LPC_FORCE_GENERIC");
    if (fr->dtype == VBX_F64 || (force && force[0] == '1')) return pl;
    const int n = fr->frame_len;
    const int64_t stride = fr->frame_stride;
    LpcParams& P = pl.P;
    if (plan_fused16(ctx, n, stride, L, &P, &pl.smem)) pl.kind = LpcKind::fused16;
    else if (plan_fusedp(ctx, fr, L, &P, &pl.X, &pl.smem)) pl.kind = LpcKind::persistent;
    else if (plan_fuseda(ctx, n, stride, L, vbx_dtype_size(fr->dtype), &P, &pl.X, &pl.smem)) pl.kind = LpcKind::aligned;
    else if (L >= 2 && L <= kMaxFastLags && plan_fused(ctx, n, stride, L, &P, &pl.smem)) pl.kind = LpcKind::general;
    else return pl;
    P.base = fr->base;
    P.n_frames = fr->n_frames;
    P.stride = stride;
    P.seg_frames = vbx_frames_per_segment(fr);
    P.seg_stride = fr->frames_per_segment > 0 ? fr->segment_stride : 0;
    P.ctas_per_seg = (int)((P.seg_frames + P.frames_per_cta - 1) / P.frames_per_cta);
    P.n = n;
    // 16-aligned kernel, several utterances of at least one CTA's worth of overlapped frames: CTAs take G consecutive
    // frames of the batch (an utterance of 998 frames otherwise leaves 26 of its last CTA's 64 frame slots empty)
    P.straddle = (pl.kind == LpcKind::fused16 && P.n_frames > P.seg_frames && P.seg_frames >= P.frames_per_cta &&
                  stride <= (int64_t)n) ? 1 : 0;
    pl.ctas = P.straddle ? (P.n_frames + P.frames_per_cta - 1) / P.frames_per_cta
                         : (P.n_frames / P.seg_frames) * P.ctas_per_seg;
    return pl;
}

// Launches the fused kernel a plan names.  Instantiated for fp32, int16 and G.711 samples: plan_lpc sends f64 samples to the
// generic kernels.
template <typename TIn>
int launch_fused(vbx_ctx* ctx, const vbx_frames* fr, int L, LpcPlan& pl) {
    // kernel tables: filled once, thread-safely (C++11 static initialisation)
    struct Tables {
        lpc_kernel_t chunk16[kChunk + 1] = {nullptr};
        lpcp_kernel_t persistent[kLpcaMaxLags + 1] = {nullptr};
        lpca_kernel_t aligned[kLpcaMaxLags + 1] = {nullptr};
        lpc_kernel_t general[kMaxFastLags + 1] = {nullptr};
        Tables() {
            fill_table<2, kChunk>(chunk16, [](auto l) -> lpc_kernel_t { return lpc_fused16_kernel<decltype(l)::value, TIn>; });
            fill_table<2, kLpcaMaxLags>(persistent, [](auto l) -> lpcp_kernel_t { return lpc_fusedp_kernel<decltype(l)::value>; });
            fill_table<2, kLpcaMaxLags>(aligned, [](auto l) -> lpca_kernel_t { return lpc_fuseda_kernel<decltype(l)::value, TIn>; });
            fill_table<2, kMaxFastLags>(general, [](auto l) -> lpc_kernel_t { return lpc_fused_kernel<decltype(l)::value, TIn>; });
        }
    };
    static const Tables tables;
    auto launch = [&](auto kern, int64_t grid, const char* name, auto... args) -> int {
        VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
        VBX_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
        kern<<<(unsigned)grid, pl.P.threads, pl.smem, ctx->stream>>>(args...);
        VBX_CHECK_LAUNCH(ctx, name);
        return VBX_OK;
    };
    if (pl.kind == LpcKind::fused16) return launch(tables.chunk16[L], pl.ctas, "lpc_fused16_kernel", pl.P);
    if (pl.kind == LpcKind::general) return launch(tables.general[L], pl.ctas, "lpc_fused_kernel", pl.P);
    // the aligned-down 16-sample-chunk walk (vbx_lpca.cuh)
    int st = get_window_rows_aligned(ctx, fr->window, fr->frame_len, pl.X.wt, &pl.X.tabs, fr->dtype);
    if (st != VBX_OK) return st;
    if (pl.kind == LpcKind::aligned) return launch(tables.aligned[L], pl.ctas, "lpc_fuseda_kernel", pl.P, pl.X);
    // enough tiles for every SM: the persistent, TMA-fed, warp-specialised CTA (one per SM)
    int grid = ctx->sm_count - (ctx->reserve_sms > 0 && ctx->reserve_sms < ctx->sm_count / 2 ? ctx->reserve_sms : 0);
    if (pl.ctas < grid) grid = (int)pl.ctas;
    VBX_CUDA(ctx, cudaMemsetAsync(ctx->tile_counter, 0, sizeof(unsigned), ctx->stream));
    return launch(tables.persistent[L], grid, "lpc_fusedp_kernel", pl.P, pl.X, (int)pl.ctas, ctx->tile_counter);
}

template <typename TIn>
int launch_lpc(vbx_ctx* ctx, const vbx_frames* fr, int L, void* r_out, void* ac_out, void* kc_out, int out_dtype,
               bool do_levinson) {
    const double* win = nullptr;
    int st = vbx_get_window(ctx, fr->window, fr->frame_len, &win, fr->dtype);
    if (st != VBX_OK) return st;
    if constexpr (!std::is_same<TIn, double>::value) {
        LpcPlan pl = plan_lpc(ctx, fr, L);
        if (pl.kind != LpcKind::generic) {
            pl.P.win = win;
            pl.P.r_out = r_out;
            pl.P.ac_out = ac_out;
            pl.P.kc_out = kc_out;
            pl.P.out_f64 = (out_dtype == VBX_F64);
            pl.P.do_levinson = do_levinson ? 1 : 0;
            return launch_fused<TIn>(ctx, fr, L, pl);
        }
    }

    // fallback: generic autocorrelation (+ stand-alone Levinson through a scratch r buffer)
    void* r_tmp = r_out;
    int r_dtype = out_dtype;
    if (do_levinson && (!r_out || out_dtype != VBX_F64)) {
        st = vbx_scratch_get(ctx, (size_t)fr->n_frames * L * sizeof(double), &r_tmp);
        if (st != VBX_OK) return st;
        r_dtype = VBX_F64;
        VBX_REQUIRE(ctx, r_tmp != ac_out && r_tmp != kc_out, "internal: the r scratch aliases an output");
    }
    const size_t xs = (size_t)fr->frame_len * sizeof(double);
    const int use_smem = xs <= ctx->smem_optin ? 1 : 0;
    if (use_smem)
        VBX_CUDA(ctx, cudaFuncSetAttribute(autocorr_generic_kernel<TIn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xs));
    VBX_REQUIRE(ctx, fr->n_frames <= 0x7fffffffLL, "too many frames for one launch");
    autocorr_generic_kernel<TIn><<<(unsigned)fr->n_frames, 256, use_smem ? xs : 0, ctx->stream>>>(
        reinterpret_cast<const TIn*>(fr->base), win, fr->frame_stride, vbx_frames_per_segment(fr), fr->segment_stride,
        fr->frame_len, L, r_tmp, r_dtype == VBX_F64, use_smem);
    VBX_CHECK_LAUNCH(ctx, "autocorr_generic_kernel");
    if (do_levinson) {
        st = vbx_lpc_levinson(ctx, r_tmp, r_dtype, fr->n_frames, L, L - 1, ac_out, kc_out, out_dtype);
        if (st != VBX_OK) return st;
        if (r_out && r_tmp != r_out) {
            // r was requested in f32 as well: convert with a second generic pass (rare path)
            autocorr_generic_kernel<TIn><<<(unsigned)fr->n_frames, 256, use_smem ? xs : 0, ctx->stream>>>(
                reinterpret_cast<const TIn*>(fr->base), win, fr->frame_stride, vbx_frames_per_segment(fr), fr->segment_stride,
                fr->frame_len, L, r_out, 0, use_smem);
            VBX_CHECK_LAUNCH(ctx, "autocorr_generic_kernel");
        }
    }
    return VBX_OK;
}

// Argument checks of the autocorrelation and LPC entry points.  The host twins run them before they size their buffers
// from n_lags, the device calls before they launch.
int lpc_check(vbx_ctx* ctx, const vbx_frames* fr, int n_lags, const void* r_out, int out_dtype, bool do_levinson) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_check_frames(ctx, fr, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, do_levinson || r_out || fr->n_frames == 0, "r_out is NULL");
    VBX_REQUIRE(ctx, !do_levinson || n_lags >= 2, "LPC order must be >= 1");
    VBX_REQUIRE(ctx, n_lags >= 1, "n_lags must be >= 1");
    VBX_REQUIRE(ctx, n_lags <= fr->frame_len, "n_lags (%d) > frame_len (%d): the reference's `self.len() - lag` underflows",
                n_lags, fr->frame_len);
    VBX_REQUIRE(ctx, !do_levinson || n_lags - 1 <= kMaxLevinsonOrder, "LPC order > %d not supported", kMaxLevinsonOrder);
    return VBX_OK;
}

int lpc_dispatch(vbx_ctx* ctx, const vbx_frames* fr, int n_lags, void* r_out, void* ac_out, void* kc_out, int out_dtype,
                 bool do_levinson) {
    int st = lpc_check(ctx, fr, n_lags, r_out, out_dtype, do_levinson);
    if (st != VBX_OK || fr->n_frames == 0) return st;
    cudaSetDevice(ctx->device);
    vbx_frames pv;  // the planar equivalent of an interleaved view
    st = vbx_planarize(ctx, fr, &pv);
    if (st != VBX_OK) return st;
    fr = &pv;
    if (fr->dtype == VBX_I16)
        return launch_lpc<int16_t>(ctx, fr, n_lags, r_out, ac_out, kc_out, out_dtype, do_levinson);
    if (fr->dtype == VBX_MULAW8)
        return launch_lpc<vbx_mulaw8>(ctx, fr, n_lags, r_out, ac_out, kc_out, out_dtype, do_levinson);
    if (fr->dtype == VBX_ALAW8)
        return launch_lpc<vbx_alaw8>(ctx, fr, n_lags, r_out, ac_out, kc_out, out_dtype, do_levinson);
    if (fr->dtype == VBX_F64)
        return launch_lpc<double>(ctx, fr, n_lags, r_out, ac_out, kc_out, out_dtype, do_levinson);
    return launch_lpc<float>(ctx, fr, n_lags, r_out, ac_out, kc_out, out_dtype, do_levinson);
}

// host twin: chunked H2D / kernels / D2H pipeline (vbx_pipeline.cuh)
int lpc_host(vbx_ctx* ctx, const vbx_frames* fr, int n_lags, void* r_out, void* ac_out, void* kc_out, int out_dtype,
             bool do_levinson) {
    int st = lpc_check(ctx, fr, n_lags, r_out, out_dtype, do_levinson);
    if (st != VBX_OK || fr->n_frames == 0) return st;
    cudaSetDevice(ctx->device);
    const size_t os = vbx_dtype_size(out_dtype);
    vbx_host_out outs[3] = {{r_out, (size_t)n_lags * os, nullptr},
                            {do_levinson ? ac_out : nullptr, (size_t)n_lags * os, nullptr},
                            {do_levinson ? kc_out : nullptr, (size_t)(n_lags - 1) * os, nullptr}};
    return vbx_run_chunked(ctx, fr, outs, 3, [&](const vbx_frames* dfr, int64_t, int64_t, vbx_host_out* o) -> int {
        return lpc_dispatch(ctx, dfr, n_lags, o[0].dev, o[1].dev, o[2].dev, out_dtype, do_levinson);
    });
}

}  // namespace

// scratch launch_lpc asks vbx_scratch_get for when called as vbx_lpc(.., r_out = NULL, ..) (vbx_find_formants' LPC stage)
size_t vbx_lpc_scratch_bytes(vbx_ctx* ctx, const vbx_frames* fr, int n_lags) {
    return plan_lpc(ctx, fr, n_lags).kind == LpcKind::generic ? (size_t)fr->n_frames * n_lags * sizeof(double) : 0;
}

extern "C" {

int vbx_autocorrelate(vbx_ctx* ctx, const vbx_frames* frames, int32_t n_lags, void* r_out, int32_t out_dtype) {
    return lpc_dispatch(ctx, frames, n_lags, r_out, nullptr, nullptr, out_dtype, false);
}
int vbx_autocorrelate_host(vbx_ctx* ctx, const vbx_frames* frames, int32_t n_lags, void* r_out, int32_t out_dtype) {
    return lpc_host(ctx, frames, n_lags, r_out, nullptr, nullptr, out_dtype, false);
}

int vbx_autocorrelate_ring(vbx_ctx* ctx, const void* rings, int32_t dtype, int64_t n_rings, int64_t capacity, const int64_t* heads,
                           int32_t n, int32_t n_lags, void* r_out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_rings >= 0 && capacity >= 1, "bad sizes");
    VBX_REQUIRE(ctx, n >= 1 && n <= capacity, "n must be in 1..capacity (the deque holds n samples)");
    VBX_REQUIRE(ctx, n_lags >= 1 && n_lags <= n, "n_lags must be in 1..n (`self.len() - lag` underflows in the reference)");
    if (n_rings == 0) return VBX_OK;
    VBX_REQUIRE(ctx, rings && r_out, "rings / r_out is NULL");
    VBX_REQUIRE(ctx, n_rings <= 0x7fffffffLL, "too many rings for one launch");
    cudaSetDevice(ctx->device);
    const size_t xs = (size_t)n * sizeof(double);
    const int use_smem = xs <= ctx->smem_optin ? 1 : 0;
    if (dtype == VBX_F64) {
        if (use_smem) VBX_CUDA(ctx, cudaFuncSetAttribute(autocorr_ring_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xs));
        autocorr_ring_kernel<double><<<(unsigned)n_rings, 256, use_smem ? xs : 0, ctx->stream>>>((const double*)rings, capacity, heads, n, n_lags,
                                                                                          r_out, out_dtype == VBX_F64, use_smem);
    } else {
        if (use_smem) VBX_CUDA(ctx, cudaFuncSetAttribute(autocorr_ring_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xs));
        autocorr_ring_kernel<float><<<(unsigned)n_rings, 256, use_smem ? xs : 0, ctx->stream>>>((const float*)rings, capacity, heads, n, n_lags,
                                                                                         r_out, out_dtype == VBX_F64, use_smem);
    }
    VBX_CHECK_LAUNCH(ctx, "autocorr_ring_kernel");
    return VBX_OK;
}

int vbx_lpc(vbx_ctx* ctx, const vbx_frames* frames, int32_t p, void* r_out, void* ac_out, void* kc_out, int32_t out_dtype) {
    return lpc_dispatch(ctx, frames, p + 1, r_out, ac_out, kc_out, out_dtype, true);
}
int vbx_lpc_host(vbx_ctx* ctx, const vbx_frames* frames, int32_t p, void* r_out, void* ac_out, void* kc_out,
                 int32_t out_dtype) {
    return lpc_host(ctx, frames, p + 1, r_out, ac_out, kc_out, out_dtype, true);
}

int vbx_lpc_levinson(vbx_ctx* ctx, const void* r, int32_t r_dtype, int64_t n_frames, int32_t r_stride, int32_t p,
                     void* ac_out, void* kc_out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    struct Tables {
        lev_kernel_t t[kMaxLevinsonOrder + 1] = {nullptr};
        Tables() { fill_table<1, kMaxLevinsonOrder>(t, [](auto p) -> lev_kernel_t { return levinson_kernel<decltype(p)::value>; }); }
    };
    static const Tables tables;  // filled once, thread-safely
    const lev_kernel_t* table = tables.t;
    VBX_REQUIRE(ctx, p >= 1 && p <= kMaxLevinsonOrder, "LPC order must be in 1..%d", kMaxLevinsonOrder);
    VBX_REQUIRE(ctx, r_stride >= p + 1, "r_stride must be >= p + 1 (lpc_mut reads self[0..=p])");
    VBX_REQUIRE(ctx, r_dtype == VBX_F32 || r_dtype == VBX_F64, "r_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_frames >= 0, "n_frames < 0");
    if (n_frames == 0) return VBX_OK;
    VBX_REQUIRE(ctx, r != nullptr, "r is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_frames + 127) / 128;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
    table[p]<<<(unsigned)grid, 128, 0, ctx->stream>>>(r, r_dtype == VBX_F64, n_frames, r_stride, ac_out, kc_out,
                                                      out_dtype == VBX_F64);
    VBX_CHECK_LAUNCH(ctx, "levinson_kernel");
    return VBX_OK;
}

}  // extern "C"
