// vbx_formants.cu — the formant path: Burg LPC, polynomial roots, resonances, McCandless tracker.
//
// Replaces, batched over frames / utterances:
//   spectrum.rs:94-146    LPC::{lpc_praat_mut, lpc_praat}        (Burg, Praat NUMburg form)
//   polynomial.rs:10-205  Polynomial::{laguerre, find_roots(_mut), div_polynomial(_mut), degree, off_low}
//   spectrum.rs:149-210   Resonance::from_root, ToResonance::to_resonance
//   spectrum.rs:216-369   EstimateFormants::estimate_formants, FormantExtractor
//   lib.rs:26-116         find_formants (+ work-size helpers)
//
// Kernel shapes (DESIGN.md §K2b–K5):
//   burg_warp_kernel<C>   one warp per frame; the forward/backward error vectors live in registers
//                         (C consecutive elements per lane), fp64; one neighbour shuffle per order.
//   lpc_roots_kernel<P>   one thread per frame; the polynomial lives in registers; Laguerre + forward
//                         deflation in fp32 (or fp64), fp64 Newton polish on the original polynomial,
//                         resonances computed and rank-sorted in fp64.
//   tracker_kernel        one thread per utterance, sequential over its frames (McCandless step).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "vbx_complex.cuh"
#include "vbx_internal.cuh"
#include "vbx_pipeline.cuh"
#include "vbx_roots_kernel.cuh"

namespace {

// =============================================================================================
// Burg
// =============================================================================================
struct BurgParams {
    const void* base;
    const double* win;
    void* coeffs_out;      // [F][p]
    uint8_t* status_out;   // [F] or null
    int64_t n_frames, stride, seg_frames, seg_stride;
    int n, p, out_f64;
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += vbx_shfl_xor(v, m);
    return v;
}

// spectrum.rs:116-140.  b1[j] = x[j], b2[j] = x[j+1] for j in [0, n−1); lane ℓ owns j in [ℓC, ℓC+C).
template <int C, typename TIn>
__global__ void __launch_bounds__(128) burg_warp_kernel(const BurgParams P) {
    const int lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (f >= P.n_frames) return;
    const int64_t seg = f / P.seg_frames;
    const TIn* __restrict__ x = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride + (f - seg * P.seg_frames) * P.stride;
    const int n = P.n, p = P.p;
    const int j0 = lane * C;
    double b1[C], b2[C];
    {
        // xw[j0 .. j0+C] (C+1 values): b1[c] = xw[j0+c], b2[c] = xw[j0+c+1]; entries j >= n−1 are zero
        double prev = (j0 < n) ? vbx_load_sample_d<TIn>(x + j0) * __ldg(P.win + j0) : 0.0;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int j = j0 + c + 1;
            const double nxt = (j < n) ? vbx_load_sample_d<TIn>(x + j) * __ldg(P.win + j) : 0.0;
            const bool valid = (j0 + c) < n - 1;
            b1[c] = valid ? prev : 0.0;
            b2[c] = valid ? nxt : 0.0;
            prev = nxt;
        }
    }
    double co[32], aa[32];  // p <= 32; indexed with lane-uniform runtime indices (local memory, tiny)
    int status = VBX_OK;
    for (int i = 1; i <= p; ++i) {
        // num = Σ b1·b2, denum = Σ b1² + b2² over j < n − i
        const int m = (n - i) - j0;  // this lane's elements c < m take part
        double num0 = 0.0, num1 = 0.0, den0 = 0.0, den1 = 0.0, den2 = 0.0, den3 = 0.0;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            if (c < m) {
                if (c & 1) {
                    num1 = fma(b1[c], b2[c], num1);
                    den1 = fma(b1[c], b1[c], den1);
                    den3 = fma(b2[c], b2[c], den3);
                } else {
                    num0 = fma(b1[c], b2[c], num0);
                    den0 = fma(b1[c], b1[c], den0);
                    den2 = fma(b2[c], b2[c], den2);
                }
            }
        }
        const double num = warp_sum(num0 + num1);
        const double denum = warp_sum((den0 + den1) + (den2 + den3));
        if (!(denum > 0.0)) {  // `denum <= 0` ⇒ Err(LPC("Denum was <= 0.0")); NaN falls through in the reference
            if (denum <= 0.0) { status = VBX_ERR_LPC; break; }
        }
        const double k = 2.0 * num / denum;
        co[i - 1] = k;
        for (int j = 1; j < i; ++j) co[j - 1] = aa[j - 1] - k * aa[i - j - 1];
        if (i < p) {
            for (int j = 1; j <= i; ++j) aa[j - 1] = co[j - 1];
            const double a = aa[i - 1];
            // b1[j] −= a·b2[j]; b2[j] = b2[j+1] − a·b1[j+1] (old values), j < n − i − 1
            const double nb1 = __shfl_down_sync(0xffffffffu, b1[0], 1);
            const double nb2 = __shfl_down_sync(0xffffffffu, b2[0], 1);
            const double e1 = (lane == 31) ? 0.0 : nb1, e2 = (lane == 31) ? 0.0 : nb2;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const double o1 = b1[c], o2 = b2[c];
                const double n1 = (c + 1 < C) ? b1[c + 1] : e1;
                const double n2 = (c + 1 < C) ? b2[c + 1] : e2;
                b1[c] = fma(-a, o2, o1);
                b2[c] = fma(-a, n1, n2);
            }
        }
    }
    if (lane == 0) {
        if (P.status_out) P.status_out[f] = (uint8_t)status;
        for (int j = 0; j < p; ++j) {
            const double v = (status == VBX_OK) ? -co[j] : nan("");
            if (P.out_f64) reinterpret_cast<double*>(P.coeffs_out)[f * p + j] = v;
            else reinterpret_cast<float*>(P.coeffs_out)[f * p + j] = (float)v;
        }
    }
}

// Any frame length: one CTA per frame, b1/b2 in shared memory (or a global scratch when too long).
template <typename TIn>
__global__ void __launch_bounds__(256) burg_block_kernel(const BurgParams P, double* scratch, int use_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double s_red[2][8];
    __shared__ double s_co[32], s_aa[32];
    __shared__ int s_status;
    const int64_t f = blockIdx.x;
    const int64_t seg = f / P.seg_frames;
    const TIn* __restrict__ x = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride + (f - seg * P.seg_frames) * P.stride;
    const int n = P.n, p = P.p, tid = threadIdx.x, T = blockDim.x;
    double* b1 = use_smem ? reinterpret_cast<double*>(smem_raw) : scratch + (size_t)f * 2 * n;
    double* b2 = b1 + n;
    for (int j = tid; j < n - 1; j += T) {
        b1[j] = vbx_load_sample_d<TIn>(x + j) * __ldg(P.win + j);
        b2[j] = vbx_load_sample_d<TIn>(x + j + 1) * __ldg(P.win + j + 1);
    }
    if (tid == 0) s_status = VBX_OK;
    __syncthreads();
    for (int i = 1; i <= p; ++i) {
        double num = 0.0, den = 0.0;
        for (int j = tid; j < n - i; j += T) {
            num = fma(b1[j], b2[j], num);
            den = fma(b1[j], b1[j], den);
            den = fma(b2[j], b2[j], den);
        }
        num = warp_sum(num);
        den = warp_sum(den);
        if ((tid & 31) == 0) { s_red[0][tid >> 5] = num; s_red[1][tid >> 5] = den; }
        __syncthreads();
        if (tid == 0) {
            double sn = 0.0, sd = 0.0;
            for (int w = 0; w < (T >> 5); ++w) { sn += s_red[0][w]; sd += s_red[1][w]; }
            if (sd <= 0.0) s_status = VBX_ERR_LPC;
            else {
                const double k = 2.0 * sn / sd;
                s_co[i - 1] = k;
                for (int j = 1; j < i; ++j) s_co[j - 1] = s_aa[j - 1] - k * s_aa[i - j - 1];
                if (i < p) for (int j = 1; j <= i; ++j) s_aa[j - 1] = s_co[j - 1];
            }
        }
        __syncthreads();
        if (s_status != VBX_OK) break;
        if (i < p) {
            const double a = s_aa[i - 1];
            for (int t0 = 0; t0 < n - i - 1; t0 += T) {
                const int j = t0 + tid;
                double v1 = 0.0, v2 = 0.0;
                const bool act = j < n - i - 1;
                if (act) { v1 = fma(-a, b2[j], b1[j]); v2 = fma(-a, b1[j + 1], b2[j + 1]); }
                __syncthreads();
                if (act) { b1[j] = v1; b2[j] = v2; }
            }
            __syncthreads();
        }
    }
    if (tid == 0) {
        const int status = s_status;
        if (P.status_out) P.status_out[f] = (uint8_t)status;
        for (int j = 0; j < p; ++j) {
            const double v = (status == VBX_OK) ? -s_co[j] : nan("");
            if (P.out_f64) reinterpret_cast<double*>(P.coeffs_out)[f * p + j] = v;
            else reinterpret_cast<float*>(P.coeffs_out)[f * p + j] = (float)v;
        }
    }
}

typedef void (*burg_kernel_t)(const BurgParams);
template <typename TIn> burg_kernel_t pick_burg(int c_needed, int* c_out) {
#define VBX_BURG_CASE(CC) if (c_needed <= CC) { *c_out = CC; return burg_warp_kernel<CC, TIn>; }
    VBX_BURG_CASE(4) VBX_BURG_CASE(8) VBX_BURG_CASE(13) VBX_BURG_CASE(16) VBX_BURG_CASE(20) VBX_BURG_CASE(26)
    VBX_BURG_CASE(32) VBX_BURG_CASE(36)
#undef VBX_BURG_CASE
    *c_out = 0;
    return nullptr;
}

// the block kernel keeps b1/b2 in shared memory when 2·n doubles fit (VBX_BURG_FORCE_GLOBAL=1: never, for tests)
bool burg_block_uses_smem(const vbx_ctx* ctx, int frame_len) {
    if (const char* e = getenv("VBX_BURG_FORCE_GLOBAL"))
        if (e[0] == '1') return false;
    return (size_t)2 * frame_len * sizeof(double) <= ctx->smem_optin - 1024;
}
bool burg_uses_warp_kernel(int frame_len) {
    return (frame_len - 1 + 31) / 32 <= 36 && !getenv("VBX_BURG_FORCE_BLOCK") && !getenv("VBX_BURG_FORCE_GLOBAL");
}

template <typename TIn>
int launch_burg(vbx_ctx* ctx, const vbx_frames* fr, int p, void* coeffs_out, uint8_t* status_out, int out_dtype) {
    const double* win = nullptr;
    int st = vbx_get_window(ctx, fr->window, fr->frame_len, &win, fr->dtype);
    if (st != VBX_OK) return st;
    BurgParams P;
    P.base = fr->base; P.win = win; P.coeffs_out = coeffs_out; P.status_out = status_out;
    P.n_frames = fr->n_frames; P.stride = fr->frame_stride;
    P.seg_frames = vbx_frames_per_segment(fr);
    P.seg_stride = fr->frames_per_segment > 0 ? fr->segment_stride : 0;
    P.n = fr->frame_len; P.p = p; P.out_f64 = (out_dtype == VBX_F64);
    int C = 0;
    burg_kernel_t kern = pick_burg<TIn>((fr->frame_len - 1 + 31) / 32, &C);
    if (kern && burg_uses_warp_kernel(fr->frame_len)) {
        const int warps = 4;
        const int64_t grid = (fr->n_frames + warps - 1) / warps;
        VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
        kern<<<(unsigned)grid, warps * 32, 0, ctx->stream>>>(P);
        VBX_CHECK_LAUNCH(ctx, "burg_warp_kernel");
        return VBX_OK;
    }
    const size_t need = (size_t)2 * fr->frame_len * sizeof(double);
    const int use_smem = burg_block_uses_smem(ctx, fr->frame_len) ? 1 : 0;
    double* scratch = nullptr;
    if (!use_smem) {
        // global b1/b2 rows: from the caller's reservation inside vbx_find_formants (which holds arena pointers), else the arena
        void* sp = nullptr;
        st = vbx_scratch_get(ctx, need * (size_t)fr->n_frames, &sp);
        if (st != VBX_OK) return st;
        scratch = reinterpret_cast<double*>(sp);
    } else {
        VBX_CUDA(ctx, cudaFuncSetAttribute(burg_block_kernel<TIn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
    }
    VBX_REQUIRE(ctx, fr->n_frames <= 0x7fffffffLL, "too many frames for one launch");
    burg_block_kernel<TIn><<<(unsigned)fr->n_frames, 256, use_smem ? need : 0, ctx->stream>>>(P, scratch, use_smem);
    VBX_CHECK_LAUNCH(ctx, "burg_block_kernel");
    return VBX_OK;
}

// =============================================================================================
// roots → resonances
// =============================================================================================
using namespace vbx_roots;

// The fp32 path without a request for the roots themselves runs lpc_roots_pair_kernel (conjugate-pair deflation,
// vbx_roots_kernel.cuh).  Its caller then launches launch_roots_fixup for the frames the kernel listed.
bool roots_use_pair_kernel(int precision, const void* roots_out) { return precision != 1 && !roots_out; }

// The f64 fix-up launch behind lpc_roots_pair_kernel (see there): redoes the frames of the pair kernel's list (Q.hard_list /
// Q.hard_count) with the reference's own algorithm, on `stream` once the pair kernel's results are visible there.  One CTA per
// SM at most walks the list (an empty list costs a few µs, a flagged frame ~0.25 ms of single-thread latency — which is why
// vbx_find_formants puts this launch on its side stream).
int launch_roots_fixup(vbx_ctx* ctx, const RootsParams& Q, int p, cudaStream_t stream) {
    RootsParams Q2 = Q;
    Q2.frame_list = Q.hard_list;
    Q2.frame_count = Q.hard_count;
    Q2.hard_list = nullptr;
    Q2.hard_count = nullptr;
    Q2.work = nullptr;
    const size_t smem_fix = roots_rt_smem_bytes(p, false);
    VBX_CUDA(ctx, cudaFuncSetAttribute(lpc_roots_rt_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_fix));
    const char* name = "lpc_roots_rt_kernel<double> (fix-up launch)";
    const int slot = vbx_launch_begin(ctx, name, stream);
    // one CTA per SM at most: enough for the few frames speech flags; a batch that flags most of its frames (tonal input) walks
    // the list at low occupancy, a latency not measured (DESIGN.md K3+K4)
    const int64_t grid = std::min<int64_t>((Q.n_frames + kRootsThreads - 1) / kRootsThreads, ctx->sm_count);
    lpc_roots_rt_kernel<double><<<(unsigned)grid, kRootsThreads, smem_fix, stream>>>(Q2, p);
    return vbx_launch_end(ctx, slot, name, stream);
}

// Launches the roots kernel only: after lpc_roots_pair_kernel (roots_use_pair_kernel), the caller launches the fix-up.
int launch_lpc_roots(vbx_ctx* ctx, const RootsParams& Q, int p, int precision /*-1 or 0 fast f32+polish, 1 f64*/) {
    const int64_t grid = (Q.n_frames + kRootsThreads - 1) / kRootsThreads;
    const bool f32 = (precision != 1);
    if (roots_use_pair_kernel(precision, Q.roots_out)) {
        const size_t smem_pair = roots_pair_smem_bytes(p);
        VBX_CUDA(ctx, cudaFuncSetAttribute(lpc_roots_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pair));
        RootsParams Q1 = Q;
        if (const char* e = getenv("VBX_ROOTS_FORCE_HARD")) Q1.hard_mod = atoi(e);
        VBX_CUDA(ctx, cudaMemsetAsync(Q1.hard_count, 0, sizeof(unsigned), ctx->stream));
        lpc_roots_pair_kernel<<<(unsigned)grid, kRootsThreads, smem_pair, ctx->stream>>>(Q1, p);
        VBX_CHECK_LAUNCH(ctx, "lpc_roots_pair_kernel");
        return VBX_OK;
    }
    const size_t smem = roots_rt_smem_bytes(p, f32);
    if (f32) {
        VBX_CUDA(ctx, cudaFuncSetAttribute(lpc_roots_rt_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lpc_roots_rt_kernel<float><<<(unsigned)grid, kRootsThreads, smem, ctx->stream>>>(Q, p);
    } else {
        VBX_CUDA(ctx, cudaFuncSetAttribute(lpc_roots_rt_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lpc_roots_rt_kernel<double><<<(unsigned)grid, kRootsThreads, smem, ctx->stream>>>(Q, p);
    }
    VBX_CHECK_LAUNCH(ctx, "lpc_roots_rt_kernel");
    return VBX_OK;
}

// ---------------------------------------------------------------------------------------------
// generic Polynomial::find_roots_mut / laguerre / div_polynomial_mut on complex coefficient arrays
// (any content, len <= 64): one thread per polynomial, arrays in local memory, the reference's own
// control flow incl. degree()/off_low() handling (polynomial.rs:92-152).
// ---------------------------------------------------------------------------------------------
constexpr int kMaxPolyLen = 64;

template <typename T> __device__ inline bool cx_is_zero(vcx<T> a) { return a.re == (T)0 && a.im == (T)0; }
template <typename T> __device__ inline int poly_degree_dev(const vcx<T>* c, int len) {
    for (int i = len - 1; i >= 0; --i)
        if (!cx_is_zero(c[i])) return i;
    return 0;
}
template <typename T> __device__ inline int poly_off_low_dev(const vcx<T>* c, int len) {
    for (int i = 0; i < len; ++i)
        if (!cx_is_zero(c[i])) return i;
    return 0;
}
// polynomial.rs:155-195
template <typename T> __device__ inline int div_polynomial_dev(vcx<T>* self, int len, vcx<T> other, vcx<T>* rem) {
    for (int i = 0; i < len; ++i) rem[i] = self[i];
    if (cx_is_zero(other)) return VBX_ERR_POLYNOMIAL;  // "Tried to divide by zero"
    const int ns = poly_degree_dev(self, len);
    if (ns < 1) return VBX_ERR_BADARG;  // (0..(ns − 1 + 1)).rev() with ns == 0: `ns - ds` underflows in the reference
    for (int i = ns - 1; i >= 0; --i) {
        self[i] = rem[i + 1];
        rem[i] = csub(rem[i], cmul(self[i], other));
    }
    for (int k = 1; k < ns + 1; ++k) rem[poly_degree_dev(rem, len)] = cmk<T>((T)0, (T)0);
    const int l = poly_degree_dev(self, len);
    const int cnt = (l + 1) - ns - 1 + 1;
    if (cnt < 0) return VBX_ERR_BADARG;
    for (int k = 0; k < cnt; ++k) self[poly_degree_dev(self, len)] = cmk<T>((T)0, (T)0);
    return VBX_OK;
}

template <typename T>
__global__ void __launch_bounds__(64) find_roots_generic_kernel(const T* __restrict__ coeffs, int64_t n_polys, int len,
                                                                T* roots_out, uint8_t* status_out) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_polys) return;
    vcx<T> self[kMaxPolyLen], c[kMaxPolyLen], rem[kMaxPolyLen], zr[kMaxPolyLen + 1];
    for (int i = 0; i < len; ++i) self[i] = cmk<T>(coeffs[((size_t)f * len + i) * 2], coeffs[((size_t)f * len + i) * 2 + 1]);
    for (int i = 0; i <= len; ++i) zr[i] = cmk<T>((T)0, (T)0);
    int status = VBX_OK;
    const int hi = poly_degree_dev(self, len);
    int zi = 0;
    if (hi < 1) status = VBX_ERR_POLYNOMIAL;  // "Zero degree polynomial: no roots to be found."
    else {
        const int lo = poly_off_low_dev(self, len);
        int m = hi - lo;
        const int clen = hi - lo + 1;
        for (int i = 0; i < lo; ++i) { zr[i] = cmk<T>((T)0, (T)0); ++zi; }
        if (lo > 0) status = VBX_ERR_BADARG;  // polynomial.rs:110-112 indexes un-shifted ⇒ the reference panics
        else {
            for (int i = 0; i < clen; ++i) c[i] = self[i];
            for (int k = m; k >= 3 && status == VBX_OK; --k) {
                const vcx<T> z = laguerre_solve_rt<T>(c, clen, cmk<T>((T)-2, (T)-2));
                zr[zi++] = z;
                if (div_polynomial_dev<T>(c, clen, cneg(z), rem) != VBX_OK) status = VBX_ERR_POLYNOMIAL;  // "Failed to find roots"
                m = m - 1;
            }
            if (status == VBX_OK && m == 2) {
                const vcx<T> a2 = cadd(c[2], c[2]);
                const vcx<T> d = csqrt_principal(csub(cmul(c[1], c[1]), cmul(cmul(cmk<T>((T)4, (T)0), c[2]), c[0])));
                const vcx<T> x = cneg(c[1]);
                zr[zi] = cdiv(cadd(x, d), a2);
                zr[zi + 1] = cdiv(csub(x, d), a2);
                zi += 2;
            }
            if (status == VBX_OK && m == 1) { zr[zi] = cdiv(cneg(c[0]), c[1]); zi += 1; }
        }
    }
    if (status_out) status_out[f] = (uint8_t)status;
    // write-back: roots, one extra (zero) element, rest zero (polynomial.rs:145-150); on error the input is kept
    for (int i = 0; i < len; ++i) {
        vcx<T> v = (status == VBX_OK) ? ((i <= zi) ? zr[i] : cmk<T>((T)0, (T)0)) : self[i];
        roots_out[((size_t)f * len + i) * 2] = v.re;
        roots_out[((size_t)f * len + i) * 2 + 1] = v.im;
    }
}

template <typename T>
__global__ void __launch_bounds__(64) laguerre_generic_kernel(const T* __restrict__ coeffs, int64_t n_polys, int len, T sre,
                                                              T sim, T* z_out) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_polys) return;
    vcx<T> c[kMaxPolyLen];
    for (int i = 0; i < len; ++i) c[i] = cmk<T>(coeffs[((size_t)f * len + i) * 2], coeffs[((size_t)f * len + i) * 2 + 1]);
    const vcx<T> z = laguerre_solve_rt<T>(c, len, cmk<T>(sre, sim));
    z_out[f * 2] = z.re;
    z_out[f * 2 + 1] = z.im;
}

template <typename T>
__global__ void __launch_bounds__(64) div_polynomial_generic_kernel(T* coeffs, int64_t n_polys, int len, const T* __restrict__ other,
                                                                    int other_per_poly, T* rem_out, uint8_t* status_out) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_polys) return;
    vcx<T> self[kMaxPolyLen], rem[kMaxPolyLen];
    for (int i = 0; i < len; ++i) self[i] = cmk<T>(coeffs[((size_t)f * len + i) * 2], coeffs[((size_t)f * len + i) * 2 + 1]);
    const size_t oi = other_per_poly ? (size_t)f * 2 : 0;
    const int st = div_polynomial_dev<T>(self, len, cmk<T>(other[oi], other[oi + 1]), rem);
    if (status_out) status_out[f] = (uint8_t)st;
    for (int i = 0; i < len; ++i) {
        coeffs[((size_t)f * len + i) * 2] = self[i].re;
        coeffs[((size_t)f * len + i) * 2 + 1] = self[i].im;
        if (rem_out) {
            rem_out[((size_t)f * len + i) * 2] = rem[i].re;
            rem_out[((size_t)f * len + i) * 2 + 1] = rem[i].im;
        }
    }
}

// roots (complex, any count) → resonances, to_resonance / find_formants semantics
template <typename T>
__global__ void __launch_bounds__(128) roots_to_resonances_kernel(const T* __restrict__ roots, int64_t n_frames, int n_roots,
                                                                  double fs, int strict_im, void* res_out, int out_f64, int R,
                                                                  int32_t* nres_out) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    double rf[kMaxPolyLen], rb[kMaxPolyLen];
    int cnt = 0;
    for (int k = 0; k < n_roots; ++k) {
        double fr_, bw_;
        if (from_root_f64((double)roots[((size_t)f * n_roots + k) * 2], (double)roots[((size_t)f * n_roots + k) * 2 + 1], fs,
                          strict_im != 0, &fr_, &bw_)) {
            rf[cnt] = fr_; rb[cnt] = bw_; ++cnt;
        }
    }
    // stable insertion sort ascending by frequency
    for (int i = 1; i < cnt; ++i) {
        const double kf = rf[i], kb = rb[i];
        int j = i - 1;
        while (j >= 0 && rf[j] > kf) { rf[j + 1] = rf[j]; rb[j + 1] = rb[j]; --j; }
        rf[j + 1] = kf; rb[j + 1] = kb;
    }
    for (int s = 0; s < R; ++s) {
        const double a = s < cnt ? rf[s] : 0.0, b = s < cnt ? rb[s] : 0.0;
        if (out_f64) { reinterpret_cast<double*>(res_out)[((size_t)f * R + s) * 2] = a; reinterpret_cast<double*>(res_out)[((size_t)f * R + s) * 2 + 1] = b; }
        else { reinterpret_cast<float*>(res_out)[((size_t)f * R + s) * 2] = (float)a; reinterpret_cast<float*>(res_out)[((size_t)f * R + s) * 2 + 1] = (float)b; }
    }
    if (nres_out) nres_out[f] = cnt;
}

// =============================================================================================
// McCandless tracker
// =============================================================================================
struct TrackParams {
    const void* res;        // [F][R] resonance pairs
    const int32_t* nres;    // [F] count of real resonances, zero padding behind them (read by tracker_idx_kernel only)
    const uint8_t* status;  // per-frame status (frames with an error leave the estimates untouched) or null
    void* est_inout;        // [n_segments][n_est]
    void* tracks_out;       // [F][n_est] or null
    int64_t n_segments, seg_frames;
    int R, n_res_eff;       // stored slots per frame; number of resonances the step sees (zero padded up to it)
    int n_est, res_f64, out_f64;
    int64_t j_begin, j_count;  // the frames [j_begin, j_begin + j_count) of every segment are stepped through (state in est_inout)
};

// One warp per utterance (segment).  Lane j holds resonance j of the current frame (32 lanes = the 32
// zero-padded slots find_formants passes, lib.rs:114); the nearest-peak search of step 2 is a warp
// arg-min; the <= 6 formant slots and estimates live in registers, identically in every lane, so the
// sequential steps 3-5 run without divergence; the next frame's resonances are prefetched while the
// current step runs.  Step 4 only ever touches slots for resonance indices j < 6 (all three of its
// conditions need j or j±1 to be a slot index), so it is unrolled over j = 0..5.
__device__ __forceinline__ double ld_pair(const void* p, int f64, size_t idx) {
    return f64 ? reinterpret_cast<const double*>(p)[idx] : (double)reinterpret_cast<const float*>(p)[idx];
}
__device__ __forceinline__ void st_pair(void* p, int f64, size_t idx, double v) {
    if (f64) reinterpret_cast<double*>(p)[idx] = v;
    else reinterpret_cast<float*>(p)[idx] = (float)v;
}

__global__ void __launch_bounds__(128) tracker_kernel(const TrackParams T) {
    constexpr int NS = VBX_MAX_FORMANT_SLOTS;
    const int lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= T.n_segments) return;
    const int n_est = T.n_est, n6 = n_est < NS ? n_est : NS;
    const unsigned FULL = 0xffffffffu;
    double ef[NS], eb[NS];  // estimates 0..5 (uniform across lanes)
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        ef[k] = (k < n_est) ? ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + k) * 2) : 0.0;
        eb[k] = (k < n_est) ? ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + k) * 2 + 1) : 0.0;
    }
    // estimates beyond the 6 slots never change (the zip at spectrum.rs:235 stops at 6 slots)
    double xf = 0.0, xb = 0.0;
    if (lane >= NS && lane < n_est) {
        xf = ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + lane) * 2);
        xb = ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + lane) * 2 + 1);
    }
    const int64_t f0 = u * T.seg_frames + T.j_begin;
    auto load_res = [&](int64_t f, double& rf, double& rb, int& st) {
        rf = 0.0; rb = 0.0;
        if (lane < T.R && lane < T.n_res_eff) {
            rf = ld_pair(T.res, T.res_f64, ((size_t)f * T.R + lane) * 2);
            rb = ld_pair(T.res, T.res_f64, ((size_t)f * T.R + lane) * 2 + 1);
        }
        st = T.status ? (int)T.status[f] : 0;
    };
    double nrf, nrb;
    int nst;
    load_res(f0, nrf, nrb, nst);
    for (int64_t j = 0; j < T.j_count; ++j) {
        const int64_t f = f0 + j;
        const double rf = nrf, rb = nrb;
        const int st = nst;
        if (j + 1 < T.j_count) load_res(f + 1, nrf, nrb, nst);  // prefetch
        if (st == VBX_OK) {
            double sf[NS], sb[NS];
            bool some[NS];
            // step 2: nearest resonance per estimate, first wins ties
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                some[k] = false; sf[k] = 0.0; sb[k] = 0.0;
                if (k < n6) {
                    double d = (lane < T.n_res_eff) ? fabs(rf - ef[k]) : INFINITY;
                    // the reference's fold starts from res[0] and replaces only on `<`: a NaN distance never wins
                    if (d != d) d = INFINITY;
                    double dmin = d;
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) dmin = fmin(dmin, __shfl_xor_sync(FULL, dmin, off));
                    // first (lowest index) resonance at the minimum distance
                    const int idx = __ffs(__ballot_sync(FULL, d == dmin)) - 1;
                    sf[k] = __shfl_sync(FULL, rf, idx);
                    sb[k] = __shfl_sync(FULL, rb, idx);
                    some[k] = true;
                }
            }
            // step 3: remove duplicates (w = last kept slot)
            int w = 0;
            bool has_unassigned = false;
#pragma unroll
            for (int r = 1; r < NS; ++r) {
                if (some[r]) {
                    double wf = 0.0, wb = 0.0, we = 0.0;
                    bool wsome = false;
#pragma unroll
                    for (int q = 0; q < NS; ++q)
                        if (q == w) { wf = sf[q]; wb = sb[q]; we = ef[q]; wsome = some[q]; }
                    if (wsome && sf[r] == wf && sb[r] == wb) {
                        has_unassigned = true;
                        if (fabs(sf[r] - ef[r]) < fabs(sf[r] - we)) {
#pragma unroll
                            for (int q = 0; q < NS; ++q)
                                if (q == w) some[q] = false;
                            w = r;
                        } else {
                            some[r] = false;
                        }
                    } else {
                        w = r;
                    }
                }
            }
            // step 4: unassigned peaks; the resonance index j doubles as the slot index (j < 6 only)
            if (has_unassigned) {
#pragma unroll
                for (int jj = 0; jj < NS; ++jj) {
                    if (jj < T.n_res_eff) {
                        const double pf = __shfl_sync(FULL, rf, jj), pb = __shfl_sync(FULL, rb, jj);
                        bool contained = false;
#pragma unroll
                        for (int q = 0; q < NS; ++q) contained = contained || (some[q] && sf[q] == pf && sb[q] == pb);
                        if (!contained) {
                            if (!some[jj]) {
                                some[jj] = true; sf[jj] = pf; sb[jj] = pb;
                            } else if (jj > 0 && !some[jj > 0 ? jj - 1 : 0]) {
                                // swap(j, j−1); slots[j] = peak
                                some[jj - 1 >= 0 ? jj - 1 : 0] = true; sf[jj - 1 >= 0 ? jj - 1 : 0] = sf[jj]; sb[jj - 1 >= 0 ? jj - 1 : 0] = sb[jj];
                                sf[jj] = pf; sb[jj] = pb;
                            } else if (jj + 1 < NS && !some[jj + 1 < NS ? jj + 1 : NS - 1]) {
                                some[jj + 1 < NS ? jj + 1 : NS - 1] = true; sf[jj + 1 < NS ? jj + 1 : NS - 1] = sf[jj]; sb[jj + 1 < NS ? jj + 1 : NS - 1] = sb[jj];
                                sf[jj] = pf; sb[jj] = pb;
                            }
                        }
                    }
                }
            }
            // step 5: stable sort, None first then ascending frequency (adjacent swaps on strict <)
#pragma unroll
            for (int pass = 0; pass < NS - 1; ++pass) {
#pragma unroll
                for (int q = 0; q < NS - 1 - pass; ++q) {
                    // is slot[q+1] < slot[q] ?
                    bool less;
                    if (!some[q + 1]) less = some[q];
                    else if (!some[q]) less = false;
                    else less = sf[q + 1] < sf[q];
                    if (less) {
                        const double tf = sf[q], tb = sb[q]; const bool ts = some[q];
                        sf[q] = sf[q + 1]; sb[q] = sb[q + 1]; some[q] = some[q + 1];
                        sf[q + 1] = tf; sb[q + 1] = tb; some[q + 1] = ts;
                    }
                }
            }
            // winners (Some, f > 0) overwrite the leading estimates
            int k = 0;
#pragma unroll
            for (int q = 0; q < NS; ++q) {
                if (some[q] && sf[q] > 0.0 && k < n_est) {
#pragma unroll
                    for (int t = 0; t < NS; ++t)
                        if (t == k) { ef[t] = sf[q]; eb[t] = sb[q]; }
                    ++k;
                }
            }
        }
        if (T.tracks_out && lane < n_est) {
            double of = xf, ob = xb;
#pragma unroll
            for (int t = 0; t < NS; ++t)
                if (t == lane) { of = ef[t]; ob = eb[t]; }
            st_pair(T.tracks_out, T.out_f64, ((size_t)f * n_est + lane) * 2, of);
            st_pair(T.tracks_out, T.out_f64, ((size_t)f * n_est + lane) * 2 + 1, ob);
        }
    }
    if (lane < n6) {
        double of = 0.0, ob = 0.0;
#pragma unroll
        for (int t = 0; t < NS; ++t)
            if (t == lane) { of = ef[t]; ob = eb[t]; }
        st_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + lane) * 2, of);
        st_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + lane) * 2 + 1, ob);
    }
}

// ---------------------------------------------------------------------------------------------
// McCandless tracker for the fused find_formants path, one THREAD per utterance, slots held as INDICES.
//
// The warp-per-utterance kernel above spends ~1100 warp instructions per frame step (warp-wide arg-min
// butterflies, every lane repeating the serial slot logic on (frequency, bandwidth) pairs), so a launch
// costs ~3 ms however few utterances it gets and ~30 % of the C3 step at scale.  In the fused path the
// frame's resonances are known to be: `nres` distinct entries sorted by ascending frequency (all > 50 Hz),
// followed by zero padding up to 32 (lib.rs:94-114).  That lets a slot be a small integer:
//   −1 = None, i in [0, nres) = resonance i, nres = "the (0, 0) pad" (all pads are the same value; only the
//   first can win the strict `<` of step 2),
// and turns the step into integer logic: equality of slots = equality of indices; the two distances step 3
// compares are the step-2 minima bd[r], bd[w] (both slots hold the same resonance); the sort by frequency
// is a sort of the keys (None < pad < index order) through a 12-comparator network; only the ≤ 6 winners'
// values are fetched.  Rows are streamed through shared memory with cp.async one frame ahead (16-byte
// chunks, [chunk][thread] layout), nres/status are prefetched one frame ahead, and a warp advances 32
// utterances per instruction.
// ---------------------------------------------------------------------------------------------
constexpr int kTrkThreads = 64;        // stand-alone launches: many small CTAs, one or two warps per SM
constexpr int kTrkThreadsPacked = 512; // vbx_find_formants' side stream: few big CTAs (see estimate_formants_impl)

template <bool RES_F64>
__global__ void __launch_bounds__(kTrkThreadsPacked) tracker_idx_kernel(const TrackParams T, const int chunks_per_row) {
    extern __shared__ __align__(16) unsigned char trk_smem[];
    constexpr int NS = VBX_MAX_FORMANT_SLOTS;
    const int TT = blockDim.x;
    constexpr int NONE = -1;
    const int tid = threadIdx.x;
    const int64_t u = (int64_t)blockIdx.x * TT + tid;
    if (u >= T.n_segments) return;
    const int n_est = T.n_est, n6 = n_est < NS ? n_est : NS;
    const int R = T.R;
    const int n_stored = R < T.n_res_eff ? R : T.n_res_eff;
    const size_t row_bytes = (size_t)R * (RES_F64 ? 16 : 8);
    uint4* buf = reinterpret_cast<uint4*>(trk_smem);  // [2][chunks_per_row][TT] 16-byte chunks
    const char* res_base = reinterpret_cast<const char*>(T.res) + ((size_t)u * T.seg_frames + T.j_begin) * row_bytes;
    auto issue = [&](int64_t j, int b) {
        const char* src = res_base + (size_t)j * row_bytes;
        for (int c = 0; c < chunks_per_row; ++c) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(buf + ((size_t)b * chunks_per_row + c) * TT + tid);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + (size_t)c * 16) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto entry = [&](int b, int i, double& f, double& bw) {  // stored entry i of the staged row b
        if (RES_F64) {
            const double2 v = *reinterpret_cast<const double2*>(buf + ((size_t)b * chunks_per_row + i) * TT + tid);
            f = v.x; bw = v.y;
        } else {
            const float2 v = *(reinterpret_cast<const float2*>(buf + ((size_t)b * chunks_per_row + (i >> 1)) * TT + tid) + (i & 1));
            f = (double)v.x; bw = (double)v.y;
        }
    };
    double ef[NS], eb[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        ef[k] = (k < n_est) ? ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + k) * 2) : 0.0;
        eb[k] = (k < n_est) ? ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + k) * 2 + 1) : 0.0;
    }
    const int64_t f0 = u * T.seg_frames + T.j_begin;
    int st_next = 0, nres_next = 0;
    if (T.j_count > 0) {
        issue(0, 0);
        st_next = T.status ? (int)T.status[f0] : 0;
        nres_next = T.nres[f0];
    }
    for (int64_t j = 0; j < T.j_count; ++j) {
        const int64_t f = f0 + j;
        const int b = (int)(j & 1);
        const int st = st_next, nres_f = nres_next;
        if (j + 1 < T.j_count) {
            issue(j + 1, b ^ 1);
            st_next = T.status ? (int)T.status[f + 1] : 0;
            nres_next = T.nres[f + 1];
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        if (st == VBX_OK) {
            const int n_real = nres_f < n_stored ? nres_f : n_stored;
            const bool has_pad = n_real < T.n_res_eff;
            const int pad = n_real;  // canonical index of the (0, 0) padding
            // step 2: nearest resonance per estimate (fold from entry 0, replace on strict `<`, NaN never wins)
            double bd[NS];
            int slot[NS];
            {
                double f_, b_;
                if (n_real > 0) entry(b, 0, f_, b_); else f_ = 0.0;
#pragma unroll
                for (int k = 0; k < NS; ++k) { bd[k] = fabs(f_ - ef[k]); slot[k] = 0; }
            }
            for (int i = 1; i < n_real; ++i) {
                double f_, b_;
                entry(b, i, f_, b_);
#pragma unroll
                for (int k = 0; k < NS; ++k) {
                    const double d = fabs(f_ - ef[k]);
                    if (d < bd[k]) { bd[k] = d; slot[k] = i; }
                }
            }
            if (has_pad && n_real > 0) {
#pragma unroll
                for (int k = 0; k < NS; ++k) {
                    const double d = fabs(0.0 - ef[k]);
                    if (d < bd[k]) { bd[k] = d; slot[k] = pad; }
                }
            }
#pragma unroll
            for (int k = 0; k < NS; ++k)
                if (k >= n6) slot[k] = NONE;
            // step 3: remove duplicates; w = last kept slot (a Some slot whenever it is consulted)
            int w = 0, wv = slot[0];
            double wbd = bd[0];
            bool has_unassigned = false;
#pragma unroll
            for (int r = 1; r < NS; ++r) {
                if (slot[r] != NONE) {
                    if (wv != NONE && slot[r] == wv) {
                        has_unassigned = true;
                        if (bd[r] < wbd) {
#pragma unroll
                            for (int q = 0; q < NS; ++q)
                                if (q == w) slot[q] = NONE;
                            w = r; wbd = bd[r];  // wv unchanged (same resonance)
                        } else {
                            slot[r] = NONE;
                        }
                    } else {
                        w = r; wv = slot[r]; wbd = bd[r];
                    }
                }
            }
            // step 4: unassigned peaks; the resonance index doubles as the slot index, so only indices < 6 can act
            if (has_unassigned) {
#pragma unroll
                for (int jj = 0; jj < NS; ++jj) {
                    if (jj < T.n_res_eff) {
                        const int c = jj < n_real ? jj : pad;
                        bool contained = false;
#pragma unroll
                        for (int q = 0; q < NS; ++q) contained = contained || (slot[q] == c);
                        if (!contained) {
                            if (slot[jj] == NONE) {
                                slot[jj] = c;
                            } else if (jj > 0 && slot[jj > 0 ? jj - 1 : 0] == NONE) {
                                slot[jj > 0 ? jj - 1 : 0] = slot[jj];
                                slot[jj] = c;
                            } else if (jj + 1 < NS && slot[jj + 1 < NS ? jj + 1 : NS - 1] == NONE) {
                                slot[jj + 1 < NS ? jj + 1 : NS - 1] = slot[jj];
                                slot[jj] = c;
                            }
                        }
                    }
                }
            }
            // step 5: sort — None first, then ascending frequency: pad (0 Hz) < resonance 0 < resonance 1 < …
            int key[NS];
#pragma unroll
            for (int q = 0; q < NS; ++q) key[q] = (slot[q] == NONE) ? -1 : (slot[q] == pad ? 0 : slot[q] + 1);
#define VBX_CE(a, b) { const int lo = min(key[a], key[b]), hi = max(key[a], key[b]); key[a] = lo; key[b] = hi; }
            VBX_CE(0, 5) VBX_CE(1, 3) VBX_CE(2, 4) VBX_CE(1, 2) VBX_CE(3, 4) VBX_CE(0, 3) VBX_CE(2, 5) VBX_CE(0, 1) VBX_CE(2, 3)
            VBX_CE(4, 5) VBX_CE(1, 2) VBX_CE(3, 4)
#undef VBX_CE
            // winners (Some, f > 0 ⇔ key > 0) overwrite the leading estimates, in order
            int z = 0;
#pragma unroll
            for (int q = 0; q < NS; ++q) z += (key[q] <= 0) ? 1 : 0;
#pragma unroll
            for (int t = 0; t < NS; ++t) {
                int kk = 0;
#pragma unroll
                for (int q = 0; q < NS; ++q)
                    if (q == z + t) kk = key[q];
                if (z + t < NS && t < n_est) entry(b, kk - 1, ef[t], eb[t]);
            }
        }
        if (T.tracks_out) {
#pragma unroll
            for (int t = 0; t < NS; ++t)
                if (t < n_est) {
                    st_pair(T.tracks_out, T.out_f64, ((size_t)f * n_est + t) * 2, ef[t]);
                    st_pair(T.tracks_out, T.out_f64, ((size_t)f * n_est + t) * 2 + 1, eb[t]);
                }
            for (int t = NS; t < n_est; ++t) {  // estimates beyond the 6 slots never change (spectrum.rs:235 zip)
                st_pair(T.tracks_out, T.out_f64, ((size_t)f * n_est + t) * 2, ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + t) * 2));
                st_pair(T.tracks_out, T.out_f64, ((size_t)f * n_est + t) * 2 + 1, ld_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + t) * 2 + 1));
            }
        }
    }
#pragma unroll
    for (int t = 0; t < NS; ++t)
        if (t < n6) {
            st_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + t) * 2, ef[t]);
            st_pair(T.est_inout, T.out_f64, ((size_t)u * n_est + t) * 2 + 1, eb[t]);
        }
}

// ---------------------------------------------------------------------------------------------
// lib.rs:57-61 — the linear resampler inside find_formants (sample::interpolate::Linear +
// Converter::scale_sample_hz): output k interpolates between source samples idx[k] and idx[k]+1 with
// weight w[k]; (idx, w) follow from the converter's ACCUMULATED interpolation value (interp += 1/ratio,
// whole frames peeled off while interp >= 1), which depends only on (ratio, k) — so the table is built
// once on the host, sequentially, exactly as the converter steps, and every frame reuses it.  A source
// index beyond the frame reads equilibrium (0).  Output: packed [F][rlen] f64 (the reference resamples in
// S = f64; rounding the resampled frame to fp32 would leak into Burg).
// ---------------------------------------------------------------------------------------------
template <typename TIn>
__global__ void __launch_bounds__(256) resample_kernel(const TIn* __restrict__ base, int64_t n_frames, int64_t stride,
                                                       int64_t seg_frames, int64_t seg_stride, int n, double scale,
                                                       const int* __restrict__ idx, const double* __restrict__ w, int rlen,
                                                       const double* __restrict__ win /* [rlen] or null */, int row_len, int copy_only,
                                                       double* __restrict__ out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_frames * row_len) return;
    const int64_t f = e / row_len;
    const int k = (int)(e - f * row_len);
    if (k >= rlen) {  // the untouched tail of the reference's resampled_buf: zeros (0·window = 0)
        out[e] = 0.0;
        return;
    }
    const int64_t seg = f / seg_frames;
    const TIn* x = base + seg * seg_stride + (f - seg * seg_frames) * stride;
    double v;
    if (copy_only) {  // resample_ratio == 1: lib.rs:62-64 copies
        v = vbx_load_sample_d<TIn>(x + k) * scale;
    } else {
        const int i = __ldg(idx + k);
        const double left = (i < n) ? vbx_load_sample_d<TIn>(x + i) * scale : 0.0;
        const double right = (i + 1 < n) ? vbx_load_sample_d<TIn>(x + i + 1) * scale : 0.0;
        v = left + (right - left) * __ldg(w + k);
    }
    out[e] = win ? v * __ldg(win + k) : v;
}

}  // namespace

size_t vbx_burg_scratch_bytes(vbx_ctx* ctx, const vbx_frames* fr) {
    if (burg_uses_warp_kernel(fr->frame_len) || burg_block_uses_smem(ctx, fr->frame_len)) return 0;
    return (size_t)2 * fr->frame_len * sizeof(double) * (size_t)fr->n_frames;
}

extern "C" {

int64_t vbx_find_formants_real_work_size(int64_t buf_len, int64_t n_coeffs) { return buf_len * 2 + n_coeffs * 23 + 2; }  // lib.rs:30-32
int64_t vbx_find_formants_complex_work_size(int64_t n_coeffs) { return n_coeffs * 7 + 4; }                                   // lib.rs:34-36
int64_t vbx_find_roots_work_size(int64_t len) { return len * 6 + 4; }                                                          // polynomial.rs:75-77

int vbx_lpc_burg(vbx_ctx* ctx, const vbx_frames* frames, int32_t p, void* coeffs_out, uint8_t* status_out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_check_frames(ctx, frames, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, p >= 1 && p <= 32, "Burg order must be in 1..32");
    VBX_REQUIRE(ctx, frames->frame_len >= 2, "frame_len must be >= 2 (b2[len-2] is indexed)");
    VBX_REQUIRE(ctx, p < frames->frame_len, "Burg order must be < frame_len (`self.len() - i` underflows)");
    if (frames->n_frames == 0) return VBX_OK;
    VBX_REQUIRE(ctx, coeffs_out != nullptr, "coeffs_out is NULL");
    cudaSetDevice(ctx->device);
    vbx_frames pv;  // the planar equivalent of an interleaved view
    st = vbx_planarize(ctx, frames, &pv);
    if (st != VBX_OK) return st;
    frames = &pv;
    if (frames->dtype == VBX_I16) return launch_burg<int16_t>(ctx, frames, p, coeffs_out, status_out, out_dtype);
    if (frames->dtype == VBX_MULAW8) return launch_burg<vbx_mulaw8>(ctx, frames, p, coeffs_out, status_out, out_dtype);
    if (frames->dtype == VBX_ALAW8) return launch_burg<vbx_alaw8>(ctx, frames, p, coeffs_out, status_out, out_dtype);
    if (frames->dtype == VBX_F64) return launch_burg<double>(ctx, frames, p, coeffs_out, status_out, out_dtype);
    return launch_burg<float>(ctx, frames, p, coeffs_out, status_out, out_dtype);
}

// Checks the arguments of a roots -> resonances call and fills *Q (nothing to launch when n_frames == 0).  The fix-up list of
// the pair kernel (hard_list, hard_count, hard_cap) is left for the caller to set.
static int lpc_roots_params(vbx_ctx* ctx, const void* lpc, int32_t lpc_dtype, int64_t n_frames, int32_t lpc_stride, int32_t p,
                            int32_t lpc_has_leading_one, double sample_rate, int32_t strict_im, const uint8_t* status_in,
                            void* res_out, int32_t res_slots, int32_t* nres_out, void* roots_out, uint8_t* status_out,
                            int32_t out_dtype, int32_t precision, int64_t in_J, int64_t out_J, int64_t out_j0, RootsParams* Q) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, lpc_dtype == VBX_F32 || lpc_dtype == VBX_F64, "lpc_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_frames >= 0, "n_frames < 0");
    VBX_REQUIRE(ctx, lpc_stride >= p + (lpc_has_leading_one ? 1 : 0), "lpc_stride too small for the order");
    VBX_REQUIRE(ctx, !res_out || res_slots >= 1, "res_slots must be >= 1");
    VBX_REQUIRE(ctx, precision >= -1 && precision <= 1, "precision must be -1 (default), 0 (f32 + f64 polish) or 1 (f64)");
    if (n_frames == 0) return VBX_OK;
    VBX_REQUIRE(ctx, lpc != nullptr, "lpc is NULL");
    cudaSetDevice(ctx->device);
    VBX_REQUIRE(ctx, p >= 2 && p <= kMaxRootsOrder, "LPC order for root finding must be in 2..%d", kMaxRootsOrder);
    VBX_REQUIRE(ctx, n_frames <= 0x7fffffffLL, "too many frames for one launch");  // frame indices of the fix-up list are int
    Q->lpc = lpc; Q->status_in = status_in; Q->res_out = res_out; Q->nres_out = nres_out; Q->roots_out = roots_out;
    Q->status_out = status_out; Q->n_frames = n_frames; Q->fs = sample_rate; Q->lpc_stride = lpc_stride;
    Q->lpc_has_one = lpc_has_leading_one ? 1 : 0; Q->lpc_f64 = (lpc_dtype == VBX_F64); Q->out_f64 = (out_dtype == VBX_F64);
    Q->R = res_slots; Q->strict_im = strict_im ? 1 : 0; Q->polish_steps = 2;
    Q->work = vbx_work_ptr(ctx);
    Q->in_J = in_J; Q->out_J = out_J; Q->out_j0 = out_j0;
    Q->hard_list = nullptr; Q->hard_count = nullptr; Q->hard_cap = 0; Q->hard_mod = 0; Q->frame_list = nullptr; Q->frame_count = nullptr;
    return VBX_OK;
}

int vbx_lpc_to_resonances(vbx_ctx* ctx, const void* lpc, int32_t lpc_dtype, int64_t n_frames, int32_t lpc_stride, int32_t p,
                          int32_t lpc_has_leading_one, double sample_rate, int32_t strict_im, const uint8_t* status_in,
                          void* res_out, int32_t res_slots, int32_t* nres_out, void* roots_out, uint8_t* status_out,
                          int32_t out_dtype, int32_t precision) {
    RootsParams Q;
    int st = lpc_roots_params(ctx, lpc, lpc_dtype, n_frames, lpc_stride, p, lpc_has_leading_one, sample_rate, strict_im, status_in,
                              res_out, res_slots, nres_out, roots_out, status_out, out_dtype, precision, 0, 0, 0, &Q);
    if (st != VBX_OK || n_frames == 0) return st;
    if (!roots_use_pair_kernel(precision, roots_out)) return launch_lpc_roots(ctx, Q, p, precision);
    // the pair kernel's fix-up list: set 0 of the context's lists, its length in tile_counter[1]
    st = vbx_hard_list_reserve(ctx, n_frames);
    if (st != VBX_OK) return st;
    Q.hard_list = ctx->hard_list;
    Q.hard_count = ctx->tile_counter + 1;
    Q.hard_cap = (int)ctx->hard_cap;
    st = launch_lpc_roots(ctx, Q, p, precision);
    if (st != VBX_OK) return st;
    return launch_roots_fixup(ctx, Q, p, ctx->stream);
}

int vbx_find_roots(vbx_ctx* ctx, const void* coeffs, int32_t dtype, int64_t n_polys, int32_t len, void* roots_out,
                   uint8_t* status_out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, len >= 1 && len <= kMaxPolyLen, "polynomial length must be in 1..%d", kMaxPolyLen);
    VBX_REQUIRE(ctx, n_polys >= 0, "n_polys < 0");
    if (n_polys == 0) return VBX_OK;
    VBX_REQUIRE(ctx, coeffs && roots_out, "coeffs / roots_out is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_polys + 63) / 64;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many polynomials for one launch");
    if (dtype == VBX_F64)
        find_roots_generic_kernel<double><<<(unsigned)grid, 64, 0, ctx->stream>>>((const double*)coeffs, n_polys, len, (double*)roots_out, status_out);
    else
        find_roots_generic_kernel<float><<<(unsigned)grid, 64, 0, ctx->stream>>>((const float*)coeffs, n_polys, len, (float*)roots_out, status_out);
    VBX_CHECK_LAUNCH(ctx, "find_roots_generic_kernel");
    return VBX_OK;
}

int vbx_laguerre(vbx_ctx* ctx, const void* coeffs, int32_t dtype, int64_t n_polys, int32_t len, double start_re,
                 double start_im, void* z_out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, len >= 1 && len <= kMaxPolyLen, "polynomial length must be in 1..%d", kMaxPolyLen);
    VBX_REQUIRE(ctx, n_polys >= 0, "n_polys < 0");
    if (n_polys == 0) return VBX_OK;
    VBX_REQUIRE(ctx, coeffs && z_out, "coeffs / z_out is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_polys + 63) / 64;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many polynomials for one launch");
    if (dtype == VBX_F64)
        laguerre_generic_kernel<double><<<(unsigned)grid, 64, 0, ctx->stream>>>((const double*)coeffs, n_polys, len, start_re, start_im, (double*)z_out);
    else
        laguerre_generic_kernel<float><<<(unsigned)grid, 64, 0, ctx->stream>>>((const float*)coeffs, n_polys, len, (float)start_re, (float)start_im, (float*)z_out);
    VBX_CHECK_LAUNCH(ctx, "laguerre_generic_kernel");
    return VBX_OK;
}

int vbx_div_polynomial(vbx_ctx* ctx, void* coeffs_inout, int32_t dtype, int64_t n_polys, int32_t len, const void* other,
                       int32_t other_per_poly, void* rem_out, uint8_t* status_out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, len >= 1 && len <= kMaxPolyLen, "polynomial length must be in 1..%d", kMaxPolyLen);
    VBX_REQUIRE(ctx, n_polys >= 0, "n_polys < 0");
    if (n_polys == 0) return VBX_OK;
    VBX_REQUIRE(ctx, coeffs_inout && other, "coeffs / other is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_polys + 63) / 64;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many polynomials for one launch");
    if (dtype == VBX_F64)
        div_polynomial_generic_kernel<double><<<(unsigned)grid, 64, 0, ctx->stream>>>((double*)coeffs_inout, n_polys, len, (const double*)other, other_per_poly, (double*)rem_out, status_out);
    else
        div_polynomial_generic_kernel<float><<<(unsigned)grid, 64, 0, ctx->stream>>>((float*)coeffs_inout, n_polys, len, (const float*)other, other_per_poly, (float*)rem_out, status_out);
    VBX_CHECK_LAUNCH(ctx, "div_polynomial_generic_kernel");
    return VBX_OK;
}

int vbx_roots_to_resonances(vbx_ctx* ctx, const void* roots, int32_t dtype, int64_t n_frames, int32_t n_roots,
                            double sample_rate, int32_t strict_im, void* res_out, int32_t res_slots, int32_t* nres_out,
                            int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_roots >= 0 && n_roots <= kMaxPolyLen, "n_roots must be in 0..%d", kMaxPolyLen);
    VBX_REQUIRE(ctx, res_slots >= 1 && n_frames >= 0, "res_slots must be >= 1");
    if (n_frames == 0) return VBX_OK;
    VBX_REQUIRE(ctx, (roots || n_roots == 0) && res_out, "roots / res_out is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_frames + 127) / 128;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
    if (dtype == VBX_F64)
        roots_to_resonances_kernel<double><<<(unsigned)grid, 128, 0, ctx->stream>>>((const double*)roots, n_frames, n_roots, sample_rate, strict_im, res_out, out_dtype == VBX_F64, res_slots, nres_out);
    else
        roots_to_resonances_kernel<float><<<(unsigned)grid, 128, 0, ctx->stream>>>((const float*)roots, n_frames, n_roots, sample_rate, strict_im, res_out, out_dtype == VBX_F64, res_slots, nres_out);
    VBX_CHECK_LAUNCH(ctx, "roots_to_resonances_kernel");
    return VBX_OK;
}

// nres (optional, internal): per-frame count of real resonances when every stored entry behind it is known to be (0, 0)
static int estimate_formants_impl(vbx_ctx* ctx, const void* resonances, int32_t res_dtype, int32_t res_slots, int32_t n_resonances,
                                  int64_t n_segments, int64_t frames_per_segment, const uint8_t* status_in, void* est_inout,
                                  int32_t n_estimates, void* tracks_out, int32_t dtype, const int32_t* nres,
                                  int64_t j_begin = 0, int64_t j_count = -1, cudaStream_t stream = nullptr, bool packed = false) {
    if (!ctx) return VBX_ERR_BADARG;
    if (!stream) stream = ctx->stream;
    if (j_count < 0) j_count = frames_per_segment - j_begin;
    VBX_REQUIRE(ctx, res_dtype == VBX_F32 || res_dtype == VBX_F64, "res_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, res_slots >= 1, "res_slots must be >= 1");
    VBX_REQUIRE(ctx, n_resonances >= 1 && n_resonances <= VBX_MAX_RESONANCES, "n_resonances must be in 1..%d (resonances[0] is indexed)", VBX_MAX_RESONANCES);
    VBX_REQUIRE(ctx, n_estimates >= 0 && n_estimates <= VBX_MAX_RESONANCES, "n_estimates must be in 0..%d", VBX_MAX_RESONANCES);
    VBX_REQUIRE(ctx, n_segments >= 0 && frames_per_segment >= 0, "negative counts");
    if (n_segments == 0 || frames_per_segment == 0 || n_estimates == 0) return VBX_OK;
    VBX_REQUIRE(ctx, resonances && est_inout, "resonances / est_inout is NULL");
    cudaSetDevice(ctx->device);
    TrackParams T;
    T.res = resonances; T.nres = nres; T.status = status_in; T.est_inout = est_inout; T.tracks_out = tracks_out;
    T.n_segments = n_segments; T.seg_frames = frames_per_segment; T.R = res_slots; T.n_res_eff = n_resonances;
    T.n_est = n_estimates; T.res_f64 = (res_dtype == VBX_F64); T.out_f64 = (dtype == VBX_F64);
    T.j_begin = j_begin; T.j_count = j_count;
    // fused path (per-frame counts known, rows sorted and zero padded): the index-based thread-per-utterance kernel,
    // when the rows can be staged with 16-byte cp.async chunks.  Arbitrary caller resonances (vbx_estimate_formants) or
    // odd fp32 row lengths: the value-based warp-per-utterance kernel.
    const size_t pair_bytes = (res_dtype == VBX_F64) ? 16 : 8;
    const size_t row_bytes = (size_t)res_slots * pair_bytes;
    const bool aligned = (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(resonances) & 15) == 0);
    const int chunks = (int)(row_bytes / 16);
    // On vbx_find_formants' side stream the tracker runs next to the LPC / roots grids of the following frame chunk.  Spread as
    // 64-thread CTAs over every SM, each of its warps competes with 8-16 busy warps for issue slots and the (purely latency-
    // bound) step chain runs 4-5x slower — slower than the main stream's chunk, so the tracker became the critical path
    // (measured: 1.2 ms per chunk against 0.27 alone).  `packed` launches it as 512-thread CTAs instead: ~n_segments / 512 of
    // them, each filling most of an SM's shared memory, so they cannot share an SM with the persistent LPC kernel's CTA — which
    // leaves exactly that many SMs free (ctx->reserve_sms).  Whichever kernel the block scheduler places first, the tracker ends
    // up alone on its SMs (0.69 ms per chunk, hidden); with small CTAs the outcome depended on the launch race.
    int trk_threads = packed ? kTrkThreadsPacked : kTrkThreads;
    while (trk_threads > 32 && (size_t)2 * chunks * trk_threads * 16 > ctx->smem_optin) trk_threads >>= 1;
    const size_t smem = (size_t)2 * chunks * trk_threads * 16;
    if (nres && aligned && smem <= ctx->smem_optin) {
        const int64_t grid = (n_segments + trk_threads - 1) / trk_threads;
        VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many segments for one launch");
        void (*kern)(const TrackParams, const int) = (res_dtype == VBX_F64) ? tracker_idx_kernel<true> : tracker_idx_kernel<false>;
        VBX_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int slot = vbx_launch_begin(ctx, "tracker_idx_kernel", stream);
        kern<<<(unsigned)grid, trk_threads, smem, stream>>>(T, chunks);
        return vbx_launch_end(ctx, slot, "tracker_idx_kernel", stream);
    }
    const int64_t grid = (n_segments + 3) / 4;  // one warp per segment
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many segments for one launch");
    const int slot = vbx_launch_begin(ctx, "tracker_kernel", stream);
    tracker_kernel<<<(unsigned)grid, 128, 0, stream>>>(T);
    return vbx_launch_end(ctx, slot, "tracker_kernel", stream);
}

int vbx_estimate_formants(vbx_ctx* ctx, const void* resonances, int32_t res_dtype, int32_t res_slots, int32_t n_resonances,
                          int64_t n_segments, int64_t frames_per_segment, const uint8_t* status_in, void* est_inout,
                          int32_t n_estimates, void* tracks_out, int32_t dtype) {
    return estimate_formants_impl(ctx, resonances, res_dtype, res_slots, n_resonances, n_segments, frames_per_segment, status_in,
                                  est_inout, n_estimates, tracks_out, dtype, nullptr);
}

// lib.rs:40-116 find_formants, batched: LPC (Burg on the frame as windowed by frames->window — HANN_PERIODIC
// for the reference's own in-line window — or autocorrelation + Levinson) → roots → resonances (im > 0,
// sorted, zero padded to 32) → McCandless step per frame, sequential inside each segment (utterance).
int vbx_find_formants(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, int32_t n_coeffs, int32_t lpc_method,
                      void* est_inout, int32_t n_formants, void* tracks_out, void* resonances_out, int32_t* nres_out,
                      uint8_t* status_out, int32_t dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_check_frames(ctx, frames, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, lpc_method == VBX_LPC_BURG || lpc_method == VBX_LPC_AUTOCORR, "unknown lpc_method");
    VBX_REQUIRE(ctx, n_coeffs >= 2 && n_coeffs <= kMaxRootsOrder, "n_coeffs must be in 2..%d", kMaxRootsOrder);
    VBX_REQUIRE(ctx, n_coeffs < frames->frame_len, "n_coeffs must be < frame_len");
    VBX_REQUIRE(ctx, n_formants >= 0 && n_formants <= VBX_MAX_RESONANCES, "n_formants must be in 0..%d", VBX_MAX_RESONANCES);
    const int64_t F = frames->n_frames;
    if (F == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    // an interleaved view is gathered into the context's planar buffer, not into the arena block reserved below
    vbx_frames pv;
    st = vbx_planarize(ctx, frames, &pv);
    if (st != VBX_OK) return st;
    frames = &pv;
    const int p = n_coeffs;
    const int64_t J = vbx_frames_per_segment(frames), segs = F / J;
    const bool track = (n_formants > 0 && est_inout);
    // Frame chunks.  The tracker is sequential over the frames of an utterance (998 steps of ~2 µs however many utterances
    // there are), so run after everything else it would add its whole latency to the call.  Instead the frames of EVERY
    // utterance are processed in K chunks [j_c, j_c+1): the main stream computes LPC + roots of chunk c + 1 while the side
    // stream steps the tracker through chunk c (its state lives in est_inout), and only the last chunk's tracker — 1/K of
    // the latency — is exposed.  Per-frame results (resonances, counts, status) are laid out [utterance][frame] as the
    // caller sees them, so chunks touch disjoint rows; only the LPC coefficients are chunk-local (written and consumed on
    // the main stream).  VBX_FORMANT_CHUNKS=<K> overrides the choice (1 = the single pass).
    int K = 1;
    if (track) {
        K = 6;   // with tapered chunks C3 measures 9.66 / 9.40 / 9.32 / 9.37 / 9.36 / 9.46 / 9.52 / 9.66 ms for K = 3 / 4 / 5 / 6 / 7 / 8 / 10 / 12
        if (J / 32 < K) K = (int)(J / 32);
        if (F / 65536 < K) K = (int)(F / 65536);
        if (const char* e = getenv("VBX_FORMANT_CHUNKS")) K = atoi(e);
        if (K > J) K = (int)J;
        if (K < 1) K = 1;
    }
    // chunk boundaries on multiples of 32 frames (the LPC kernels' tile): only an utterance's last tile is partial
    // The last chunk's tracker is the only one nobody overlaps, so the last two chunks are shorter than the others (3/4 and
    // 1/2 of a share): the exposed tail shrinks with the chunk, the chunks before it grow by 10 %.
    const bool taper = K >= 4;
    auto chunk_begin = [&](int c) -> int64_t {
        if (c <= 0) return 0;
        if (c >= K) return J;
        int64_t j;
        if (taper) {
            const double total = (double)K - 0.75;   // K − 2 full shares + 0.75 + 0.5
            const double cum = (c <= K - 2) ? (double)c : (double)(K - 2) + 0.75;
            j = (int64_t)((double)J * cum / total);
        } else {
            j = (J * c) / K;
        }
        if (J >= 64 * (int64_t)K) j = ((j + 16) / 32) * 32;
        return j < J ? j : J;
    };
    int64_t Jc_max = 1;
    for (int c = 0; c < K; ++c) Jc_max = std::max<int64_t>(Jc_max, chunk_begin(c + 1) - chunk_begin(c));
    // With overlap, chunk c's roots fix-up runs on the side stream and reads the chunk-local LPC rows, LPC status and fix-up
    // list; chunk c + 1 works on a second set of them, and chunk c + 2 waits for that fix-up before it reuses the first.
    const bool overlap = track && K > 1;
    const int nbuf = overlap ? 2 : 1;
    // scratch: nbuf × (lpc [segs·Jc_max][p+1] f64) | nbuf × (lpc status [segs·Jc_max]) | status [F] | resonances [F][p] pairs |
    // nres [F] (the last three only when the caller does not ask for them)
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const int64_t Fc_max = segs * Jc_max;
    const size_t lpc_bytes = al((size_t)Fc_max * (p + 1) * sizeof(double));
    const size_t stl_bytes = al((size_t)Fc_max);
    const size_t st_bytes = status_out ? 0 : al((size_t)F);
    const size_t res_es = (dtype == VBX_F64) ? 16 : 8;
    const bool own_res = (resonances_out == nullptr);
    const int R = own_res ? p : VBX_MAX_RESONANCES;
    const size_t res_bytes = own_res ? al((size_t)F * R * res_es) : 0;
    const size_t nres_bytes = nres_out ? 0 : al((size_t)F * sizeof(int32_t));
    // the LPC stage's own scratch (Burg rows that do not fit shared memory, the r rows of the non-fused autocorrelation
    // path) is part of THIS reservation: a callee that grew the arena would free the block the pointers below point into
    vbx_frames cfr = *frames;  // the largest chunk's view, for the scratch queries
    cfr.n_frames = Fc_max;
    cfr.frames_per_segment = Jc_max;
    const size_t sub_bytes = al(lpc_method == VBX_LPC_BURG ? vbx_burg_scratch_bytes(ctx, &cfr) : vbx_lpc_scratch_bytes(ctx, &cfr, p + 1));
    const size_t lst_bytes = nbuf * (lpc_bytes + stl_bytes);
    const size_t own_bytes = lst_bytes + st_bytes + res_bytes + nres_bytes;
    st = vbx_arena_reserve(ctx, own_bytes + sub_bytes);
    if (st != VBX_OK) return st;
    st = vbx_hard_list_reserve(ctx, nbuf * Fc_max);  // fix-up list(s): Fc_max entries each, counts in tile_counter[1 + b]
    if (st != VBX_OK) return st;
    char* base = (char*)ctx->arena;
    struct SubScratch {  // scoped: the callees of this call see the sub-range, nobody else does
        vbx_ctx* c;
        SubScratch(vbx_ctx* c_, void* p_, size_t b_) : c(c_) { c->sub_scratch = b_ ? p_ : nullptr; c->sub_scratch_bytes = b_; }
        ~SubScratch() { c->sub_scratch = nullptr; c->sub_scratch_bytes = 0; }
    };
    uint8_t* d_st = status_out ? status_out : (uint8_t*)(base + lst_bytes);
    void* d_res = own_res ? (void*)(base + lst_bytes + st_bytes) : resonances_out;
    int32_t* d_nres = nres_out ? nres_out : (int32_t*)(base + lst_bytes + st_bytes + res_bytes);
    bool fixup_queued[2] = {false, false};  // a fix-up launch reads buffer set b (its completion: ev_side[2 + b])
    const size_t es = vbx_dtype_size(frames->dtype);
    const int64_t seg_stride = frames->frames_per_segment > 0 ? frames->segment_stride : 0;
    for (int c = 0; c < K; ++c) {
        const int64_t j0 = chunk_begin(c), j1 = chunk_begin(c + 1), Jc = j1 - j0;
        if (Jc <= 0) continue;
        const int b = c % nbuf;  // buffer set of this chunk
        double* d_lpc = (double*)(base + b * lpc_bytes);
        uint8_t* d_st_lpc = (uint8_t*)(base + nbuf * lpc_bytes + b * stl_bytes);
        if (fixup_queued[b]) {  // chunk c − 2's fix-up still reads this set
            fixup_queued[b] = false;
            if (cudaStreamWaitEvent(ctx->stream, ctx->ev_side[2 + b], 0) != cudaSuccess) {
                st = vbx_fail(ctx, VBX_ERR_CUDA, "find_formants: wait for the roots fix-up failed: %s", cudaGetErrorString(cudaGetLastError()));
                break;
            }
        }
        vbx_frames sub = *frames;
        sub.base = (const char*)frames->base + (size_t)j0 * frames->frame_stride * es;
        sub.n_frames = segs * Jc;
        sub.frames_per_segment = (K > 1 || frames->frames_per_segment > 0) ? Jc : 0;
        sub.segment_stride = seg_stride;
        const uint8_t* lpc_status = nullptr;
        int lpc_stride, has_one;
        {
            SubScratch scoped(ctx, base + own_bytes, sub_bytes);
            if (lpc_method == VBX_LPC_BURG) {
                st = vbx_lpc_burg(ctx, &sub, p, d_lpc, d_st_lpc, VBX_F64);
                lpc_status = d_st_lpc;
                lpc_stride = p;
                has_one = 0;
            } else {
                // the persistent LPC kernel leaves SMs for the co-running tracker: 16 of its warps (512 utterances) per SM
                ctx->reserve_sms = overlap ? (int)((segs + kTrkThreadsPacked - 1) / kTrkThreadsPacked) : 0;
                st = vbx_lpc(ctx, &sub, p, nullptr, d_lpc, nullptr, VBX_F64);
                ctx->reserve_sms = 0;
                lpc_stride = p + 1;
                has_one = 1;
            }
        }
        if (st != VBX_OK) break;
        // roots: always lpc_roots_pair_kernel here (fp32, no roots_out), with buffer set b's fix-up list
        RootsParams Qc;
        st = lpc_roots_params(ctx, d_lpc, VBX_F64, sub.n_frames, lpc_stride, p, has_one, sample_rate, /*strict_im=*/1, lpc_status, d_res,
                              R, d_nres, nullptr, d_st, dtype, -1, K > 1 ? Jc : 0, K > 1 ? J : 0, K > 1 ? j0 : 0, &Qc);
        if (st != VBX_OK) break;
        Qc.hard_list = ctx->hard_list + b * Fc_max;
        Qc.hard_count = ctx->tile_counter + 1 + b;
        Qc.hard_cap = (int)Fc_max;
        st = launch_lpc_roots(ctx, Qc, p, -1);
        if (st != VBX_OK) break;
        if (!overlap) {  // with overlap, the fix-up goes to the side stream below
            st = launch_roots_fixup(ctx, Qc, p, ctx->stream);
            if (st != VBX_OK) break;
        }
        if (!track) continue;
        if (K == 1) {
            st = estimate_formants_impl(ctx, d_res, dtype, R, VBX_MAX_RESONANCES, segs, J, d_st, est_inout, n_formants, tracks_out, dtype,
                                        d_nres);
            if (st != VBX_OK) break;
            continue;
        }
        // chunk c's resonances are ready -> its tracker steps on the side stream (after chunk c − 1's: same stream)
        cudaEvent_t ready = ctx->ev_side[c & 1];
        if (cudaEventRecord(ready, ctx->stream) != cudaSuccess || cudaStreamWaitEvent(ctx->s_side, ready, 0) != cudaSuccess) {
            st = vbx_fail(ctx, VBX_ERR_CUDA, "find_formants: chunk hand-over failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        // (the last chunk's tracker has the device to itself: small CTAs over all SMs, 0.27 ms instead of 0.69)
        // the roots fix-up (rarely any work, but ~0.25 ms of latency when there is) rides the side stream too
        st = launch_roots_fixup(ctx, Qc, p, ctx->s_side);
        if (st != VBX_OK) break;
        if (cudaEventRecord(ctx->ev_side[2 + b], ctx->s_side) != cudaSuccess) {
            st = vbx_fail(ctx, VBX_ERR_CUDA, "find_formants: fix-up event failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        fixup_queued[b] = true;
        st = estimate_formants_impl(ctx, d_res, dtype, R, VBX_MAX_RESONANCES, segs, J, d_st, est_inout, n_formants, tracks_out, dtype,
                                    d_nres, j0, Jc, ctx->s_side, /*packed=*/c + 1 < K);
        if (st != VBX_OK) break;
    }
    if (overlap) {
        // join: whatever follows on the context's stream (and vbx_sync) sees the tracks and the final state.  Done on the
        // error path too, so the side stream never runs behind the caller's back.
        cudaEvent_t done = ctx->ev_side[2];
        if (cudaEventRecord(done, ctx->s_side) != cudaSuccess || cudaStreamWaitEvent(ctx->stream, done, 0) != cudaSuccess) {
            if (st == VBX_OK) st = vbx_fail(ctx, VBX_ERR_CUDA, "find_formants: join failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        if (ctx->prof_on) vbx_prof_mark(ctx, "(wait: last chunk's tracker)");
    }
    return st;
}

}  // extern "C"

// lib.rs:40-116 with resample_ratio != 1 and / or a resampled_buf longer than the resampled frame: resample every frame
// linearly to ceil(ratio·N) samples (f64) — or copy it (ratio 1) — into a zero-tailed row of resampled_buf_len samples, then
// the reference's own chain: periodic Hann at phase idx / resampled_len over the whole row, Burg over the whole row, roots,
// resonances, McCandless step.  frames->window must be VBX_WINDOW_NONE (find_formants windows AFTER resampling, lib.rs:66-70).
extern "C" int vbx_find_formants_buffered(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double resample_ratio,
                                          int64_t resampled_buf_len, int32_t n_coeffs, void* est_inout, int32_t n_formants,
                                          void* tracks_out, void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_check_frames(ctx, frames, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, resample_ratio > 0.0 && resample_ratio <= 64.0, "resample_ratio must be in (0, 64]");
    VBX_REQUIRE(ctx, frames->window == VBX_WINDOW_NONE, "find_formants windows after resampling: pass VBX_WINDOW_NONE");
    const int n = frames->frame_len;
    const int64_t F = frames->n_frames;
    const double rl = ceil(resample_ratio * (double)n);
    VBX_REQUIRE(ctx, rl >= 2.0 && rl <= 1.0e6, "resampled frame length out of range");
    const int rlen = (int)rl;
    VBX_REQUIRE(ctx, resampled_buf_len == 0 || resampled_buf_len >= rlen,
                "resampled_buf_len (%lld) < resampled_len (%d): the reference's assert!(resampled_len <= resampled_buf.len())",
                (long long)resampled_buf_len, rlen);
    VBX_REQUIRE(ctx, resampled_buf_len <= 1000000, "resampled_buf_len out of range");
    const int row_len = resampled_buf_len > 0 ? (int)resampled_buf_len : rlen;
    if (F == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    vbx_frames pv;  // the planar equivalent of an interleaved view
    st = vbx_planarize(ctx, frames, &pv);
    if (st != VBX_OK) return st;
    frames = &pv;
    vbx_frames rfr = *frames;
    if (resample_ratio == 1.0 && row_len == rlen) {  // lib.rs:62-64: plain copy, window over exactly the frame
        rfr.window = VBX_WINDOW_HANN_PERIODIC;
        return vbx_find_formants(ctx, &rfr, sample_rate, n_coeffs, VBX_LPC_BURG, est_inout, n_formants, tracks_out, resonances_out,
                                 nres_out, status_out, dtype);
    }
    const bool copy_only = (resample_ratio == 1.0);
    // the converter's stepping, sequential in f64 (sample 0.10 interpolate::Converter::next)
    std::vector<int> idx(rlen);
    std::vector<double> w(rlen), win(rlen);
    {
        double interp = 0.0;
        const double step = 1.0 / resample_ratio;
        int left = 0;
        for (int k = 0; k < rlen; ++k) {
            while (interp >= 1.0) { ++left; interp -= 1.0; }
            idx[k] = left;
            w[k] = interp;
            interp += step;
        }
    }
    // lib.rs:66-70: window[idx] = Hanning::at_phase(idx · (1 / resampled_len)), host f64 (applied here, so the inner call sees
    // frames that are already windowed; only needed when the row is longer than the resampled frame — otherwise the periodic
    // Hann table of the Burg stage is the same thing)
    const bool window_here = row_len != rlen;
    if (window_here) vbx_window_fill_host(VBX_WINDOW_HANN_PERIODIC, rlen, win.data());
    // a private block: [F][row_len] f64 + the tables (the inner find_formants uses the context arena)
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t out_bytes = al((size_t)F * row_len * sizeof(double)), idx_bytes = al((size_t)rlen * 4), w_bytes = al((size_t)rlen * 8);
    void* blk = nullptr;
    cudaError_t e = cudaMalloc(&blk, out_bytes + idx_bytes + 2 * w_bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return vbx_fail(ctx, VBX_ERR_NOMEM, "find_formants_resampled: cudaMalloc failed: %s", cudaGetErrorString(e));
    }
    double* d_out = (double*)blk;
    int* d_idx = (int*)((char*)blk + out_bytes);
    double* d_w = (double*)((char*)blk + out_bytes + idx_bytes);
    double* d_win = (double*)((char*)blk + out_bytes + idx_bytes + w_bytes);
    auto run = [&]() -> int {
        VBX_CUDA(ctx, cudaMemcpyAsync(d_idx, idx.data(), (size_t)rlen * 4, cudaMemcpyHostToDevice, ctx->stream));
        VBX_CUDA(ctx, cudaMemcpyAsync(d_w, w.data(), (size_t)rlen * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (window_here) VBX_CUDA(ctx, cudaMemcpyAsync(d_win, win.data(), (size_t)rlen * 8, cudaMemcpyHostToDevice, ctx->stream));
        const int64_t total = F * row_len;
        const int64_t grid = (total + 255) / 256;
        VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
        const int64_t J = vbx_frames_per_segment(frames);
        const int64_t seg_stride = frames->frames_per_segment > 0 ? frames->segment_stride : 0;
        const double* wn = window_here ? d_win : nullptr;
        if (frames->dtype == VBX_I16)
            resample_kernel<int16_t><<<(unsigned)grid, 256, 0, ctx->stream>>>((const int16_t*)frames->base, F, frames->frame_stride, J,
                                                                           seg_stride, n, 1.0 / 32767.0, d_idx, d_w, rlen, wn, row_len,
                                                                           copy_only, d_out);
        else if (frames->dtype == VBX_MULAW8)
            resample_kernel<vbx_mulaw8><<<(unsigned)grid, 256, 0, ctx->stream>>>((const vbx_mulaw8*)frames->base, F, frames->frame_stride,
                                                                              J, seg_stride, n, 1.0 / 32767.0, d_idx, d_w, rlen, wn,
                                                                              row_len, copy_only, d_out);
        else if (frames->dtype == VBX_ALAW8)
            resample_kernel<vbx_alaw8><<<(unsigned)grid, 256, 0, ctx->stream>>>((const vbx_alaw8*)frames->base, F, frames->frame_stride,
                                                                             J, seg_stride, n, 1.0 / 32767.0, d_idx, d_w, rlen, wn,
                                                                             row_len, copy_only, d_out);
        else if (frames->dtype == VBX_F64)
            resample_kernel<double><<<(unsigned)grid, 256, 0, ctx->stream>>>((const double*)frames->base, F, frames->frame_stride, J,
                                                                          seg_stride, n, 1.0, d_idx, d_w, rlen, wn, row_len, copy_only, d_out);
        else
            resample_kernel<float><<<(unsigned)grid, 256, 0, ctx->stream>>>((const float*)frames->base, F, frames->frame_stride, J,
                                                                         seg_stride, n, 1.0, d_idx, d_w, rlen, wn, row_len, copy_only, d_out);
        VBX_CHECK_LAUNCH(ctx, "resample_kernel");
        vbx_frames pf;
        pf.base = d_out; pf.n_frames = F; pf.frame_stride = row_len; pf.frames_per_segment = frames->frames_per_segment;
        pf.segment_stride = (frames->frames_per_segment > 0) ? frames->frames_per_segment * (int64_t)row_len : 0;
        pf.frame_len = row_len; pf.dtype = VBX_F64; pf.window = window_here ? VBX_WINDOW_NONE : VBX_WINDOW_HANN_PERIODIC; pf.sample_step = 0;
        int s2 = vbx_find_formants(ctx, &pf, sample_rate, n_coeffs, VBX_LPC_BURG, est_inout, n_formants, tracks_out, resonances_out,
                                   nres_out, status_out, dtype);
        if (s2 != VBX_OK) return s2;
        VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the private block is freed on return
        return VBX_OK;
    };
    st = run();
    cudaStreamSynchronize(ctx->stream);
    cudaFree(blk);
    return st;
}

extern "C" int vbx_find_formants_resampled(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double resample_ratio,
                                           int32_t n_coeffs, void* est_inout, int32_t n_formants, void* tracks_out,
                                           void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype) {
    return vbx_find_formants_buffered(ctx, frames, sample_rate, resample_ratio, 0, n_coeffs, est_inout, n_formants, tracks_out,
                                      resonances_out, nres_out, status_out, dtype);
}

// host twin of vbx_find_formants: chunked H2D / kernels / D2H pipeline over whole utterances (vbx_pipeline.cuh);
// the tracker state travels once (in before the first chunk, out after the last)
extern "C" int vbx_find_formants_host(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, int32_t n_coeffs,
                                      int32_t lpc_method, void* est_inout, int32_t n_formants, void* tracks_out,
                                      void* resonances_out, int32_t* nres_out, uint8_t* status_out, int32_t dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = vbx_check_frames(ctx, frames, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    const int64_t F = frames->n_frames;
    if (F == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    const size_t pair = (dtype == VBX_F64) ? 16 : 8;
    const int64_t J = vbx_frames_per_segment(frames), segs = F / J;
    const size_t est_bytes = (est_inout && n_formants > 0) ? (size_t)segs * n_formants * pair : 0;
    void* d_est = nullptr;
    if (est_bytes) {
        cudaError_t e = cudaMalloc(&d_est, est_bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return vbx_fail(ctx, VBX_ERR_NOMEM, "find_formants_host: cudaMalloc(%zu) failed: %s", est_bytes, cudaGetErrorString(e));
        }
    }
    auto run = [&]() -> int {
        if (est_bytes) VBX_CUDA(ctx, cudaMemcpyAsync(d_est, est_inout, est_bytes, cudaMemcpyHostToDevice, ctx->stream));
        vbx_host_out outs[4] = {{n_formants > 0 ? tracks_out : nullptr, (size_t)n_formants * pair, nullptr},
                                {resonances_out, (size_t)VBX_MAX_RESONANCES * pair, nullptr},
                                {nres_out, 4, nullptr},
                                {status_out, 1, nullptr}};
        int s = vbx_run_chunked(ctx, frames, outs, 4, [&](const vbx_frames* dfr, int64_t, int64_t seg0, vbx_host_out* o) -> int {
            void* est = d_est ? (char*)d_est + (size_t)seg0 * n_formants * pair : nullptr;
            return vbx_find_formants(ctx, dfr, sample_rate, n_coeffs, lpc_method, est, n_formants, o[0].dev, o[1].dev,
                                     (int32_t*)o[2].dev, (uint8_t*)o[3].dev, dtype);
        }, /*max_chunks=*/4);  // the tracker is sequential inside an utterance: a launch costs ~3 ms however few utterances it gets
        if (s != VBX_OK) return s;
        if (est_bytes) {
            VBX_CUDA(ctx, cudaMemcpyAsync(est_inout, d_est, est_bytes, cudaMemcpyDeviceToHost, ctx->stream));
            VBX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        return VBX_OK;
    };
    st = run();
    cudaStreamSynchronize(ctx->stream);
    if (d_est) cudaFree(d_est);
    return st;
}
