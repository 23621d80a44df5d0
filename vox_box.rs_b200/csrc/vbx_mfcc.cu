// vbx_mfcc.cu — MFCC (FFT → quirky triangular band energies → log10 clamp → DCT-II), batched.
//
// Replaces, batched over frames:
//   spectrum.rs:371-373,401-441  MFCC::mfcc           (incl. its quirks: |X| — not |X|² — with a RISING weight
//                                                      on the falling slope, log10(..).max(1e-10), one step above f_hi)
//   spectrum.rs:375-381          hz_to_mel, mel_to_hz
//   spectrum.rs:384-398          dct, dct_mut          (direct DCT-II ×2, f64)
// rustfft 1.0 `FFT::new(len, false).process` (crate source not in the reference tree) is the
// unnormalised forward DFT X_k = Σ x_n e^{−2πikn/N}; it is computed here by a shared-memory Stockham
// FFT (radices 4/2/3/5, twiddles from an f64 table), as a real-input transform of N/2 complex points
// when N is even; fp64 by default, fp32 on request (vbx_mfcc_set_fft_precision).  Lengths with other
// prime factors use a direct DFT.
//
// Kernel shape (DESIGN.md §K8): a CTA owns `fpc` frames; every pass spreads the (frame, butterfly)
// pairs over all threads; the band sums run one thread per (frame, band) in fp64 with host-built
// f64 slope tables; the DCT one thread per (frame, coefficient) against a host-built f64 cosine table.
#include <algorithm>
#include <cmath>
#include <vector>

#include <type_traits>

#include "vbx_internal.cuh"
#include "vbx_pipeline.cuh"

namespace {

constexpr int kMaxPasses = 24;

struct MfccParams {
    const void* base;
    const double* win;    // [N]
    const double2* tw;    // [N] exp(−2πik/N), f64 (rounded to the transform's precision when staged)
    const double* wu;     // [N] rising-slope weight of the band whose up-slope holds bin k (0 elsewhere)
    const double* wd;     // [N] weight of the band whose "down"-slope holds bin k
    const int* bins;      // [num_coeffs + 2]
    const double* dct;    // [n_keep][num_coeffs] cos(πk(2n+1)/(2M))
    void* out;            // [F][n_keep]
    void* energies_out;   // [F][num_coeffs] or null (the log-energies before the DCT)
    int64_t n_frames, stride, seg_frames, seg_stride;
    int n, mc;            // frame length; complex FFT size (N/2 packed, N complex, or N direct)
    int ms;               // per-frame buffer stride in float2 (mc, or mc + 1 so that the Nyquist bin fits)
    int klo, khi;         // stored spectrum indices [klo, khi): bins k, folded to min(k, N−k) in the real-packed mode
    int mode;             // 0 real-packed FFT, 1 complex FFT (odd N), 2 direct DFT
    int n_pass;
    int radix[kMaxPasses];
    int num_coeffs, n_keep;
    int kmin, kmax;       // filter-bank bins used: [kmin, kmax)
    int fpc;              // frames per CTA
    int out_f64;
};

template <typename R> struct cxt { R x, y; };
template <typename R> __device__ __forceinline__ cxt<R> mk(R x, R y) { cxt<R> r; r.x = x; r.y = y; return r; }
template <typename R> __device__ __forceinline__ cxt<R> cmulf(cxt<R> a, cxt<R> b) { return mk<R>(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
template <typename R> __device__ __forceinline__ cxt<R> caddf(cxt<R> a, cxt<R> b) { return mk<R>(a.x + b.x, a.y + b.y); }
template <typename R> __device__ __forceinline__ cxt<R> csubf(cxt<R> a, cxt<R> b) { return mk<R>(a.x - b.x, a.y - b.y); }
template <typename R> __device__ __forceinline__ cxt<R> mulnegi(cxt<R> a) { return mk<R>(a.y, -a.x); }  // (−i)·a

// one radix-R Stockham butterfly: inputs src[j + t·T], twiddled by W_{Ls·R}^{k·t}, outputs dst[(j−k)·R + k + u·Ls]
#include "vbx_mfcc_fast.cuh"  // inside the anonymous namespace: uses cxt<> and the complex helpers above
#include "vbx_mfcc_lane5.cuh" // five lanes per frame for 400-sample frames (uses mfcc_fast::bfly)

template <int R, typename TR>
__device__ __forceinline__ void butterfly(const cxt<TR>* __restrict__ src, cxt<TR>* __restrict__ dst, const cxt<TR>* __restrict__ tw,
                                          int j, int T, int Ls, int tw_stride /* N / (Ls·R) */) {
    typedef cxt<TR> C;
    const int k = j % Ls;
    C v[R];
#pragma unroll
    for (int t = 0; t < R; ++t) {
        v[t] = src[j + t * T];
        if (t > 0 && Ls > 1) v[t] = cmulf(v[t], tw[k * t * tw_stride]);
    }
    C y[R];
    if (R == 2) {
        y[0] = caddf(v[0], v[1]);
        y[1] = csubf(v[0], v[1]);
    } else if (R == 3) {
        const TR s3 = (TR)0.86602540378443864676372317075294;
        const C t1 = caddf(v[1], v[2]);
        const C t2 = mk<TR>(v[0].x - (TR)0.5 * t1.x, v[0].y - (TR)0.5 * t1.y);
        const C d = csubf(v[1], v[2]);
        const C t3 = mulnegi(mk<TR>(s3 * d.x, s3 * d.y));
        y[0] = caddf(v[0], t1);
        y[1] = caddf(t2, t3);
        y[2] = csubf(t2, t3);
    } else if (R == 4) {
        const C a0 = caddf(v[0], v[2]), a1 = csubf(v[0], v[2]);
        const C a2 = caddf(v[1], v[3]), a3 = mulnegi(csubf(v[1], v[3]));
        y[0] = caddf(a0, a2);
        y[1] = caddf(a1, a3);
        y[2] = csubf(a0, a2);
        y[3] = csubf(a1, a3);
    } else {  // R == 5
        const TR c1 = (TR)0.30901699437494742410229341718282, c2 = (TR)-0.80901699437494742410229341718282;
        const TR s1 = (TR)0.95105651629515357211643933337938, s2 = (TR)0.58778525229247312916870595463907;
        const C t1 = caddf(v[1], v[4]), t2 = caddf(v[2], v[3]);
        const C t3 = csubf(v[1], v[4]), t4 = csubf(v[2], v[3]);
        y[0] = mk<TR>(v[0].x + t1.x + t2.x, v[0].y + t1.y + t2.y);
        const C a1 = mk<TR>(v[0].x + c1 * t1.x + c2 * t2.x, v[0].y + c1 * t1.y + c2 * t2.y);
        const C a2 = mk<TR>(v[0].x + c2 * t1.x + c1 * t2.x, v[0].y + c2 * t1.y + c1 * t2.y);
        const C b1 = mulnegi(mk<TR>(s1 * t3.x + s2 * t4.x, s1 * t3.y + s2 * t4.y));
        const C b2 = mulnegi(mk<TR>(s2 * t3.x - s1 * t4.x, s2 * t3.y - s1 * t4.y));
        y[1] = caddf(a1, b1);
        y[4] = csubf(a1, b1);
        y[2] = caddf(a2, b2);
        y[3] = csubf(a2, b2);
    }
    const int o = (j - k) * R + k;
#pragma unroll
    for (int u = 0; u < R; ++u) dst[o + u * Ls] = y[u];
}

template <typename TIn, typename TR>
__global__ void __launch_bounds__(256) mfcc_kernel(const MfccParams P) {
    typedef cxt<TR> C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = P.n, mc = P.mc, G = P.fpc;
    C* s_tw = reinterpret_cast<C*>(smem_raw);                             // [n]
    const int ms = P.ms;
    C* bufA = s_tw + n;                                                   // [G][ms]
    C* bufB = bufA + (size_t)G * ms;                                      // [G][ms]
    double* s_e = reinterpret_cast<double*>(bufB + (size_t)G * ms);       // [G][num_coeffs]
    const int tid = threadIdx.x, nth = blockDim.x;
    const int64_t f_first = (int64_t)blockIdx.x * G;
    const int nf = (int)min((int64_t)G, P.n_frames - f_first);

    for (int i = tid; i < n; i += nth) { const double2 w = __ldg(P.tw + i); s_tw[i] = mk<TR>((TR)w.x, (TR)w.y); }
    // ---- load + window -----------------------------------------------------------------------------------
    for (int q = 0; q < nf; ++q) {
        const int64_t f = f_first + q;
        const int64_t seg = f / P.seg_frames;
        const TIn* __restrict__ x = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride + (f - seg * P.seg_frames) * P.stride;
        if (P.mode == 0) {
            for (int i = tid; i < mc; i += nth) {
                const TR re = (TR)(vbx_load_sample_d<TIn>(x + 2 * i) * __ldg(P.win + 2 * i));
                const TR im = (TR)(vbx_load_sample_d<TIn>(x + 2 * i + 1) * __ldg(P.win + 2 * i + 1));
                bufA[(size_t)q * ms + i] = mk<TR>(re, im);
            }
        } else {
            for (int i = tid; i < n; i += nth)
                bufA[(size_t)q * ms + i] = mk<TR>((TR)(vbx_load_sample_d<TIn>(x + i) * __ldg(P.win + i)), (TR)0);
        }
    }
    __syncthreads();

    // ---- transform -------------------------------------------------------------------------------------------
    C* src = bufA;
    C* dst = bufB;
    if (P.mode != 2) {
        int Ls = 1;
        for (int pass = 0; pass < P.n_pass; ++pass) {
            const int R = P.radix[pass];
            const int T = mc / R;
            const int tw_stride = n / (Ls * R);
            // twiddle W_{Ls·R}^{kt} = exp(−2πi·kt/(Ls·R)) = tw_N[kt · N/(Ls·R)]  (Ls·R divides mc, mc divides N)
            const int items = nf * T;
            for (int it = tid; it < items; it += nth) {
                const int q = it / T, j = it - q * T;
                const C* s = src + (size_t)q * ms;
                C* d = dst + (size_t)q * ms;
                if (R == 4) butterfly<4, TR>(s, d, s_tw, j, T, Ls, tw_stride);
                else if (R == 2) butterfly<2, TR>(s, d, s_tw, j, T, Ls, tw_stride);
                else if (R == 3) butterfly<3, TR>(s, d, s_tw, j, T, Ls, tw_stride);
                else butterfly<5, TR>(s, d, s_tw, j, T, Ls, tw_stride);
            }
            __syncthreads();
            C* t = src; src = dst; dst = t;
            Ls *= R;
        }
    }
    // ---- power / magnitude of the needed bins → dst[idx] = (|X|², |X|) -------------------------------------------
    const int nb = P.khi - P.klo;
    {
        const int items = nf * nb;
        for (int it = tid; it < items; it += nth) {
            const int q = it / nb, k = P.klo + (it - q * nb);
            const C* z = src + (size_t)q * ms;
            C X;
            if (P.mode == 0) {  // k in [0, N/2]
                const C zk = z[k == mc ? 0 : k];
                const C zc = z[k == 0 ? 0 : mc - k];
                const C zm = mk<TR>(zc.x, -zc.y);
                const C E = mk<TR>((TR)0.5 * (zk.x + zm.x), (TR)0.5 * (zk.y + zm.y));
                const C O = mk<TR>((TR)0.5 * (zk.x - zm.x), (TR)0.5 * (zk.y - zm.y));
                X = caddf(E, mulnegi(cmulf(s_tw[k], O)));
            } else if (P.mode == 1) {
                X = z[k];
            } else {
                TR re = 0, im = 0;
                int idx = 0;
                for (int i = 0; i < n; ++i) {
                    const TR xv = z[i].x;
                    const C w = s_tw[idx];
                    re = fma(xv, w.x, re);
                    im = fma(xv, w.y, im);
                    idx += k;
                    if (idx >= n) idx -= n;
                }
                X = mk<TR>(re, im);
            }
            const TR pw = X.x * X.x + X.y * X.y;
            dst[(size_t)q * ms + k] = mk<TR>(pw, sqrt(pw));
        }
    }
    __syncthreads();
    // ---- band energies (spectrum.rs:421-435), f64 sums ---------------------------------------------------------------
    const int M = P.num_coeffs;
    {
        const int items = nf * M;
        for (int it = tid; it < items; it += nth) {
            const int q = it / M, w = it - q * M;
            const C* pk = dst + (size_t)q * ms;
            const int b0 = __ldg(P.bins + w), b1 = __ldg(P.bins + w + 1), b2 = __ldg(P.bins + w + 2);
            const bool fold = (P.mode == 0);  // |X_{N−k}| = |X_k| for a real signal
            double up = 0., down = 0.;
            for (int k = b0; k < b1; ++k) up = up + (double)pk[(fold && 2 * k > n) ? n - k : k].x * __ldg(P.wu + k);
            for (int k = b1; k < b2; ++k) down = down + (double)pk[(fold && 2 * k > n) ? n - k : k].y * __ldg(P.wd + k);
            double e = log10(up + down);
            e = (e > 1.0e-10) ? e : 1.0e-10;  // f64::max(1e-10): NaN → 1e-10
            s_e[q * M + w] = e;
            if (P.energies_out) {
                const size_t o = (size_t)(f_first + q) * M + w;
                if (P.out_f64) reinterpret_cast<double*>(P.energies_out)[o] = e;
                else reinterpret_cast<float*>(P.energies_out)[o] = (float)e;
            }
        }
    }
    __syncthreads();
    // ---- DCT-II ×2, first n_keep rows (spectrum.rs:391-398) -------------------------------------------------------------
    {
        const int K = P.n_keep, items = nf * K;
        for (int it = tid; it < items; it += nth) {
            const int q = it / K, k = it - q * K;
            const double* e = s_e + q * M;
            const double* c = P.dct + (size_t)k * M;
            double acc = 0.;
            for (int m = 0; m < M; ++m) acc = acc + e[m] * __ldg(c + m);
            const double v = 2. * acc;
            const size_t o = (size_t)(f_first + q) * K + k;
            if (P.out_f64) reinterpret_cast<double*>(P.out)[o] = v;
            else reinterpret_cast<float*>(P.out)[o] = (float)v;
        }
    }
}

// stand-alone dct / dct_mut (spectrum.rs:384-398): thread per (signal, k)
template <typename T>
__global__ void __launch_bounds__(128) dct_kernel(const T* __restrict__ signal, int64_t n_signals, int n, T* coeffs) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_signals * n) return;
    const int64_t s = e / n;
    const int k = (int)(e - s * n);
    double acc = 0.;
    for (int m = 0; m < n; ++m) {
        // cos(π·k·(2m+1)/(2n)) with the argument reduced exactly: k(2m+1) mod 4n
        const long long num = ((long long)k * (2 * m + 1)) % (4LL * n);
        acc = acc + (double)signal[s * n + m] * cospi((double)num / (2. * (double)n));
    }
    coeffs[e] = (T)(2. * acc);
}

// ---- host-side tables (cached per parameter set in the context) ------------------------------------------------
struct MfccTables {
    int n, num_coeffs, n_keep;
    double f_lo, f_hi, fs;
    double2* tw = nullptr;
    double *wu = nullptr, *wd = nullptr, *dct = nullptr;
    int* bins = nullptr;
    int4* items = nullptr;  // [num_coeffs + 1] intervals between bin edges {j, first bin, end bin, 0}, longest first
    mfcc_lane5::Tables* l5 = nullptr;  // mfcc_lane5_kernel's tables (400-sample frames only)
    int l5_prog_len = 0, l5_pw_len = 0;
    int kmin = 0, kmax = 0;
    int bad = 0;  // a bin the reference would panic on
};

double hz_to_mel_host(double hz) { return 1125. * log1p(hz / 700.); }
double mel_to_hz_host(double mel) { return 700. * (exp(mel / 1125.) - 1.); }

}  // namespace

// cache lives in the context (vbx_internal.cuh keeps it opaque: a vector of void*)
struct vbx_mfcc_cache {
    std::vector<MfccTables> tables;
};

namespace {

int get_tables(vbx_ctx* ctx, int n, int num_coeffs, int n_keep, double f_lo, double f_hi, double fs, const MfccTables** out) {
    if (!ctx->mfcc_cache) ctx->mfcc_cache = new vbx_mfcc_cache();
    auto& cache = ctx->mfcc_cache->tables;
    for (auto& t : cache)
        if (t.n == n && t.num_coeffs == num_coeffs && t.n_keep == n_keep && t.f_lo == f_lo && t.f_hi == f_hi && t.fs == fs) {
            *out = &t;
            return VBX_OK;
        }
    MfccTables t;
    t.n = n; t.num_coeffs = num_coeffs; t.n_keep = n_keep; t.f_lo = f_lo; t.f_hi = f_hi; t.fs = fs;
    // spectrum.rs:411-414
    const double mel_range = hz_to_mel_host(f_hi) - hz_to_mel_host(f_lo);
    std::vector<int> bins(num_coeffs + 2);
    for (int i = 0; i < num_coeffs + 2; ++i) {
        const double point = ((double)i / (double)num_coeffs) * mel_range + hz_to_mel_host(f_lo);
        const double b = floor((double)(n + 1) * mel_to_hz_host(point) / fs);
        // `as usize` saturates: negative / NaN → 0
        long long bi = (b > 0.0) ? (b > 2e9 ? 2000000000LL : (long long)b) : 0;
        bins[i] = (int)bi;
    }
    std::vector<double> wu(n, 0.0), wd(n, 0.0);
    for (int w = 0; w < num_coeffs && !t.bad; ++w) {
        const int b0 = bins[w], b1 = bins[w + 1], b2 = bins[w + 2];
        if (b1 < b0 || b2 < b1) { t.bad = 1; break; }  // usize subtraction underflow panics
        if ((b1 > b0 && b1 - 1 >= n) || (b2 > b1 && b2 - 1 >= n)) { t.bad = 1; break; }  // index panic
        for (int k = b0, i = 0; k < b1; ++k, ++i) wu[k] = (double)i / (double)(b1 - b0);
        for (int k = b1, i = 0; k < b2; ++k, ++i) wd[k] = (double)i / (double)(b2 - b1);
    }
    if (!t.bad) {
        t.kmin = bins[0];
        t.kmax = bins[num_coeffs + 1];
        if (t.kmax < t.kmin) t.kmax = t.kmin;
    }
    const double PI = 3.14159265358979323846264338327950288;
    std::vector<double2> tw(n);
    for (int k = 0; k < n; ++k) {
        const double ang = -2.0 * PI * (double)k / (double)n;
        tw[k] = make_double2(cos(ang), sin(ang));
    }
    std::vector<double> dct((size_t)n_keep * num_coeffs);
    for (int k = 0; k < n_keep; ++k)
        for (int m = 0; m < num_coeffs; ++m)
            dct[(size_t)k * num_coeffs + m] = cos(PI * (double)k * (2. * (double)m + 1.) / (2. * (double)num_coeffs));  // spectrum.rs:395
    auto up = [&](const void* host, size_t bytes, void** dev) -> int {
        cudaError_t e = cudaMalloc(dev, bytes ? bytes : 1);
        if (e != cudaSuccess) { cudaGetLastError(); return vbx_fail(ctx, VBX_ERR_NOMEM, "mfcc tables: cudaMalloc failed"); }
        if (bytes) VBX_CUDA(ctx, cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice));
        return VBX_OK;
    };
    int st;
    if ((st = up(tw.data(), tw.size() * sizeof(double2), (void**)&t.tw)) != VBX_OK) return st;
    if ((st = up(wu.data(), wu.size() * 8, (void**)&t.wu)) != VBX_OK) return st;
    if ((st = up(wd.data(), wd.size() * 8, (void**)&t.wd)) != VBX_OK) return st;
    if ((st = up(dct.data(), dct.size() * 8, (void**)&t.dct)) != VBX_OK) return st;
    if ((st = up(bins.data(), bins.size() * 4, (void**)&t.bins)) != VBX_OK) return st;
    // the intervals between consecutive bin edges, longest first: work items of mfcc_warp_kernel's band stage
    std::vector<int4> items;
    if (!t.bad) {
        for (int j = 0; j <= num_coeffs; ++j) items.push_back(make_int4(j, bins[j], bins[j + 1], 0));
        std::stable_sort(items.begin(), items.end(), [](const int4& a, const int4& b) { return a.z - a.y > b.z - b.y; });
    }
    if ((st = up(items.data(), items.size() * sizeof(int4), (void**)&t.items)) != VBX_OK) return st;
    if (!t.bad && n == mfcc_lane5::N && num_coeffs + 1 <= mfcc_lane5::kMaxItems && t.kmax <= n) {
        std::vector<mfcc_lane5::Tables> l5(1);
        if (mfcc_lane5::build_tables(l5[0], bins.data(), num_coeffs, wu.data(), wd.data())) {
            t.l5_prog_len = l5[0].prog_len;
            t.l5_pw_len = l5[0].pw_len;
            if ((st = up(l5.data(), sizeof(mfcc_lane5::Tables), (void**)&t.l5)) != VBX_OK) return st;
        }
    }
    cache.push_back(t);
    *out = &cache.back();
    return VBX_OK;
}

// factor mc into radices 4, 2, 3, 5 (in that order of preference); false if another prime remains
bool plan_radices(int mc, int* radix, int* n_pass) {
    int np = 0, m = mc;
    while (m % 4 == 0 && np < kMaxPasses) { radix[np++] = 4; m /= 4; }
    while (m % 2 == 0 && np < kMaxPasses) { radix[np++] = 2; m /= 2; }
    while (m % 3 == 0 && np < kMaxPasses) { radix[np++] = 3; m /= 3; }
    while (m % 5 == 0 && np < kMaxPasses) { radix[np++] = 5; m /= 5; }
    *n_pass = np;
    return m == 1;
}

// ---- specialised warp-per-frame kernels for the common even frame lengths (vbx_mfcc_fast.cuh) ------------------------
template <typename TIn, typename TR, int MC, int R0, int R1, int R2, int R3, int FW>
int launch_fast_one(vbx_ctx* ctx, const mfcc_fast::FastParams& Q) {
    constexpr int N = 2 * MC, MS = MC + 1;
    const size_t cs = sizeof(TR) * 2;
    int warps = 4;
    constexpr int WB = FW * MS + ((FW * MS) >> 3) + 1;
    constexpr int TWN = MS + (R1 - 1) * R0 + (R2 - 1) * R0 * R1 + (R3 - 1) * R0 * R1 * R2;  // mfcc_warp_kernel's twiddle tables
    auto bytes = [&](int w) {
        return (size_t)TWN * cs + (size_t)w * WB * cs +
               ((size_t)Q.n_keep * (Q.num_coeffs + 1) + 2 + 2 * (size_t)N + (size_t)w * FW * (2 * Q.num_coeffs + 1)) * sizeof(double);
    };
    while (warps > 1 && bytes(warps) > 56 * 1024) --warps;  // 4 CTAs / SM
    const size_t smem = bytes(warps);
    VBX_REQUIRE(ctx, smem <= ctx->smem_optin, "MFCC: shared memory");
    auto kern = mfcc_fast::mfcc_warp_kernel<TIn, TR, MC, R0, R1, R2, R3, FW>;
    VBX_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VBX_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    const int64_t n_groups = (Q.n_frames + FW - 1) / FW;
    int64_t grid = (n_groups + warps - 1) / warps;
    const int64_t cap = (int64_t)ctx->sm_count * 16;  // persistent: warps loop over frame groups
    if (grid > cap) grid = cap;
    kern<<<(unsigned)grid, warps * 32, smem, ctx->stream>>>(Q);
    VBX_CHECK_LAUNCH(ctx, "mfcc_warp_kernel");
    return VBX_OK;
}

// returns 1 if a specialisation handled the call, 0 if none exists for this frame length, < 0 on error (−status)
template <typename TIn, typename TR>
int launch_fast(vbx_ctx* ctx, int n, const mfcc_fast::FastParams& Q) {
    int st;
    switch (n) {
#define VBX_MFCC_CASE(NN, R0, R1, R2, R3, FW) \
    case NN: st = launch_fast_one<TIn, TR, NN / 2, R0, R1, R2, R3, FW>(ctx, Q); return st == VBX_OK ? 1 : -st;
        VBX_MFCC_CASE(160, 8, 5, 2, 1, 4)
        VBX_MFCC_CASE(200, 5, 5, 4, 1, 4)
        VBX_MFCC_CASE(256, 8, 4, 4, 1, 4)
        VBX_MFCC_CASE(320, 8, 5, 4, 1, 2)
        VBX_MFCC_CASE(400, 8, 5, 5, 1, 2)
        VBX_MFCC_CASE(480, 8, 5, 3, 2, 2)
        VBX_MFCC_CASE(512, 8, 8, 4, 1, 2)
        VBX_MFCC_CASE(640, 8, 8, 5, 1, 2)
        VBX_MFCC_CASE(800, 8, 5, 5, 2, 1)
        VBX_MFCC_CASE(1024, 8, 8, 8, 1, 1)
#undef VBX_MFCC_CASE
    default: return 0;
    }
}

template <typename TIn>
int launch_mfcc(vbx_ctx* ctx, const vbx_frames* fr, int num_coeffs, int n_keep, double f_lo, double f_hi, double fs, void* out,
                void* energies_out, int out_dtype) {
    const int n = fr->frame_len;
    const double* win = nullptr;
    int st = vbx_get_window(ctx, fr->window, n, &win, fr->dtype);
    if (st != VBX_OK) return st;
    const MfccTables* t = nullptr;
    st = get_tables(ctx, n, num_coeffs, n_keep, f_lo, f_hi, fs, &t);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, !t->bad, "mfcc: a filter-bank bin falls outside the spectrum (the reference panics): lower freq_bounds.1");
    MfccParams P;
    memset(&P, 0, sizeof(P));
    P.base = fr->base; P.win = win; P.tw = t->tw; P.wu = t->wu; P.wd = t->wd; P.bins = t->bins; P.dct = t->dct;
    P.out = out; P.energies_out = energies_out;
    P.n_frames = fr->n_frames; P.stride = fr->frame_stride;
    P.seg_frames = vbx_frames_per_segment(fr);
    P.seg_stride = fr->frames_per_segment > 0 ? fr->segment_stride : 0;
    P.n = n; P.num_coeffs = num_coeffs; P.n_keep = n_keep; P.kmin = t->kmin; P.kmax = t->kmax;
    P.out_f64 = (out_dtype == VBX_F64);
    if ((n % 2) == 0 && n >= 4 && plan_radices(n / 2, P.radix, &P.n_pass)) { P.mode = 0; P.mc = n / 2; }
    else if (plan_radices(n, P.radix, &P.n_pass) && n >= 2) { P.mode = 1; P.mc = n; }
    else { P.mode = 2; P.mc = n; P.n_pass = 0; }
    if (getenv("VBX_MFCC_FORCE_DIRECT")) { P.mode = 2; P.mc = n; P.n_pass = 0; }
    if (P.mode == 0) {
        P.ms = P.mc + 1;
        const int last = P.kmax - 1;  // bins above N/2 fold back
        P.klo = P.kmin;
        P.khi = P.kmax;
        if (P.kmax > P.kmin && 2 * last > n) {
            P.khi = P.mc + 1;
            if (n - last < P.klo) P.klo = n - last;
            if (2 * P.kmin > n) P.klo = n - last;
        }
    } else {
        P.ms = P.mc;
        P.klo = P.kmin;
        P.khi = P.kmax;
    }
    // transform precision: fp64 by default (parity first: a band whose sum is ~1 sits on the log10 clamp and an
    // fp32 FFT's ~1e-6 relative error then exceeds the 1e-5 norm-wise bound on quiet frames); fp32 is opt-in
    const bool f32 = ctx->mfcc_fft_f32;
    // (f64 samples — single windowed frames from the Rust shim's trait calls — take the generic kernel)
    // 400-sample frames, fp64 transform, sample pairs loadable as one word: five lanes per frame (vbx_mfcc_lane5.cuh)
    if constexpr (!std::is_same<TIn, double>::value) {
        const char* e5 = getenv("VBX_MFCC_LANE5");
        const size_t pair_bytes = 2 * sizeof(TIn);
        const bool aligned = (reinterpret_cast<uintptr_t>(P.base) % pair_bytes) == 0 && (P.stride % 2) == 0 && (P.seg_stride % 2) == 0;
        const mfcc_lane5::Smem L(num_coeffs, n_keep, t->l5_prog_len, t->l5_pw_len);
        if (t->l5 && !f32 && aligned && !(e5 && e5[0] == '0') && !getenv("VBX_MFCC_GENERIC") && L.total <= ctx->smem_optin) {
            mfcc_lane5::Params Q;
            Q.base = P.base; Q.win = P.win; Q.dct = P.dct; Q.t = t->l5; Q.prog_len = t->l5_prog_len; Q.pw_len = t->l5_pw_len;
            Q.out = P.out; Q.energies_out = P.energies_out;
            Q.n_frames = P.n_frames; Q.stride = P.stride; Q.seg_frames = P.seg_frames; Q.seg_stride = P.seg_stride;
            Q.num_coeffs = num_coeffs; Q.n_keep = n_keep; Q.out_f64 = P.out_f64;
            auto kern = mfcc_lane5::mfcc_lane5_kernel<TIn>;
            VBX_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
            const int64_t n_groups = (P.n_frames + mfcc_lane5::FW - 1) / mfcc_lane5::FW;
            int64_t grid = (n_groups + mfcc_lane5::PAIRS - 1) / mfcc_lane5::PAIRS;
            if (grid > ctx->sm_count) grid = ctx->sm_count;  // persistent: one CTA per SM, warps loop over groups of six frames
            kern<<<(unsigned)grid, mfcc_lane5::WARPS * 32, L.total, ctx->stream>>>(Q);
            VBX_CHECK_LAUNCH(ctx, "mfcc_lane5_kernel");
            return VBX_OK;
        }
    }
    if constexpr (!std::is_same<TIn, double>::value)
    if (P.mode == 0 && !getenv("VBX_MFCC_GENERIC") && P.kmax <= n && num_coeffs <= 128 && n_keep * num_coeffs <= 2048) {
        mfcc_fast::FastParams Q;
        Q.base = P.base; Q.win = P.win; Q.tw = P.tw; Q.wu = P.wu; Q.wd = P.wd; Q.bins = P.bins; Q.items = t->items;
        Q.dct = P.dct;
        Q.out = P.out; Q.energies_out = P.energies_out;
        Q.n_frames = P.n_frames; Q.stride = P.stride; Q.seg_frames = P.seg_frames; Q.seg_stride = P.seg_stride;
        Q.num_coeffs = num_coeffs; Q.n_keep = n_keep; Q.klo = P.klo; Q.khi = P.khi; Q.out_f64 = P.out_f64; Q.warps_per_cta = 0;
        const int r = f32 ? launch_fast<TIn, float>(ctx, n, Q) : launch_fast<TIn, double>(ctx, n, Q);
        if (r < 0) return -r;
        if (r == 1) return VBX_OK;
    }
    const size_t cs = f32 ? sizeof(float) * 2 : sizeof(double) * 2;
    // frames per CTA: as many as fit ~56 KB of shared memory (4 CTAs / SM), at most 16
    const size_t fixed = (size_t)n * cs;
    const size_t per_frame = (size_t)2 * P.ms * cs + (size_t)num_coeffs * sizeof(double);
    int fpc = 16;
    while (fpc > 1 && fixed + fpc * per_frame > 56 * 1024) --fpc;
    const size_t smem = fixed + fpc * per_frame;
    VBX_REQUIRE(ctx, smem <= ctx->smem_optin, "frame_len %d does not fit the MFCC kernel's shared memory", n);
    P.fpc = fpc;
    void (*kern)(const MfccParams) = f32 ? mfcc_kernel<TIn, float> : mfcc_kernel<TIn, double>;
    VBX_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t grid = (fr->n_frames + fpc - 1) / fpc;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
    kern<<<(unsigned)grid, 256, smem, ctx->stream>>>(P);
    VBX_CHECK_LAUNCH(ctx, "mfcc_kernel");
    return VBX_OK;
}

int mfcc_check(vbx_ctx* ctx, const vbx_frames* fr, int num_coeffs, int n_keep, double fs, const void* out, int out_dtype) {
    int st = vbx_check_frames(ctx, fr, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, num_coeffs >= 1 && num_coeffs <= 4096, "num_coeffs must be in 1..4096");
    VBX_REQUIRE(ctx, n_keep >= 1 && n_keep <= num_coeffs, "n_keep must be in 1..num_coeffs");
    VBX_REQUIRE(ctx, fs > 0, "sample_rate must be > 0");
    VBX_REQUIRE(ctx, fr->n_frames == 0 || out != nullptr, "out is NULL");
    return VBX_OK;
}

}  // namespace

void vbx_mfcc_cache_free(vbx_ctx* ctx) {
    if (!ctx->mfcc_cache) return;
    for (auto& t : ctx->mfcc_cache->tables) {
        cudaFree(t.tw); cudaFree(t.wu); cudaFree(t.wd); cudaFree(t.dct); cudaFree(t.bins); cudaFree(t.items); cudaFree(t.l5);
    }
    delete ctx->mfcc_cache;
    ctx->mfcc_cache = nullptr;
}

extern "C" {

int vbx_mfcc_set_fft_precision(vbx_ctx* ctx, int32_t dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    ctx->mfcc_fft_f32 = (dtype == VBX_F32);
    return VBX_OK;
}

double vbx_hz_to_mel(double hz) { return hz_to_mel_host(hz); }
double vbx_mel_to_hz(double mel) { return mel_to_hz_host(mel); }

int vbx_mfcc(vbx_ctx* ctx, const vbx_frames* frames, int32_t num_coeffs, int32_t n_keep, double freq_lo, double freq_hi,
             double sample_rate, void* out, void* energies_out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = mfcc_check(ctx, frames, num_coeffs, n_keep, sample_rate, out, out_dtype);
    if (st != VBX_OK) return st;
    if (frames->n_frames == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    vbx_frames pv;  // the planar equivalent of an interleaved view
    st = vbx_planarize(ctx, frames, &pv);
    if (st != VBX_OK) return st;
    frames = &pv;
    if (frames->dtype == VBX_I16)
        return launch_mfcc<int16_t>(ctx, frames, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, out, energies_out, out_dtype);
    if (frames->dtype == VBX_MULAW8)
        return launch_mfcc<vbx_mulaw8>(ctx, frames, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, out, energies_out, out_dtype);
    if (frames->dtype == VBX_ALAW8)
        return launch_mfcc<vbx_alaw8>(ctx, frames, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, out, energies_out, out_dtype);
    if (frames->dtype == VBX_F64)
        return launch_mfcc<double>(ctx, frames, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, out, energies_out, out_dtype);
    return launch_mfcc<float>(ctx, frames, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, out, energies_out, out_dtype);
}

int vbx_mfcc_host(vbx_ctx* ctx, const vbx_frames* frames, int32_t num_coeffs, int32_t n_keep, double freq_lo, double freq_hi,
                  double sample_rate, void* out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = mfcc_check(ctx, frames, num_coeffs, n_keep, sample_rate, out, out_dtype);
    if (st != VBX_OK) return st;
    if (frames->n_frames == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    vbx_host_out outs[1] = {{out, (size_t)n_keep * vbx_dtype_size(out_dtype), nullptr}};
    // chunked H2D / kernels / D2H pipeline (vbx_pipeline.cuh)
    return vbx_run_chunked(ctx, frames, outs, 1, [&](const vbx_frames* dfr, int64_t, int64_t, vbx_host_out* o) -> int {
        return vbx_mfcc(ctx, dfr, num_coeffs, n_keep, freq_lo, freq_hi, sample_rate, o[0].dev, nullptr, out_dtype);
    });
}

int vbx_dct(vbx_ctx* ctx, const void* signal, int32_t dtype, int64_t n_signals, int32_t n, void* coeffs) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_signals >= 0 && n >= 0, "negative sizes");
    if (n_signals == 0 || n == 0) return VBX_OK;
    VBX_REQUIRE(ctx, signal && coeffs, "signal / coeffs is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_signals * n + 127) / 128;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many signals for one launch");
    if (dtype == VBX_F64) dct_kernel<double><<<(unsigned)grid, 128, 0, ctx->stream>>>((const double*)signal, n_signals, n, (double*)coeffs);
    else dct_kernel<float><<<(unsigned)grid, 128, 0, ctx->stream>>>((const float*)signal, n_signals, n, (float*)coeffs);
    VBX_CHECK_LAUNCH(ctx, "dct_kernel");
    return VBX_OK;
}

}  // extern "C"
