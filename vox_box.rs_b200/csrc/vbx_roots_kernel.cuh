// vbx_roots_kernel.cuh — LPC coefficients → roots → resonances, one thread per frame (K3 + K4).
// Included by vbx_formants.cu (the launcher) only: lpc_roots_pair_kernel is a plain kernel defined here.
#pragma once
#include "vbx_complex.cuh"
#include "vbx_internal.cuh"

namespace vbx_roots {

constexpr double kPi = 3.14159265358979323846264338327950288;

// spectrum.rs:166-192 from_root (fp64).  Returns true and fills (f, bw) if the root yields a resonance.
static __device__ __noinline__ bool from_root_f64(double re, double im, double fs, bool strict_im, double* f_out, double* bw_out) {
    const double freq_mul = fs / (kPi * 2.0);
    if (strict_im ? !(im > 0.0) : !(im >= 0.0)) return false;
    // (r, θ) = polar(z); a root outside the unit circle is reflected to 1/conj(z) = z/|z|²: same θ, radius 1/r.
    // bw = −2·freq_mul·ln r' with r' = min(r, 1/r)  ⇒  bw = freq_mul·|ln |z|²|.  (The reference converts the
    // reflected root to polar form again; θ and ln r agree with it to an ulp.)
    const double theta = atan2(im, re);
    const double ns = re * re + im * im;
    const double f = freq_mul * theta;
    const double bw = freq_mul * fabs(log(ns));
    if (f > 50.0 && f < fs * 0.5 - 50.0) {
        *f_out = f;
        *bw_out = bw;
        return true;
    }
    return false;
}

struct RootsParams {
    const void* lpc;       // [F][lpc_stride] LPC coefficients (f64 or f32)
    const uint8_t* status_in;  // per-frame status of the LPC stage (or null)
    void* res_out;         // [F][R] resonance pairs, sorted ascending, zero padded
    int32_t* nres_out;     // [F] or null
    void* roots_out;       // [F][P] complex roots in find_roots order (or null)
    uint8_t* status_out;   // [F] or null
    int64_t n_frames;
    double fs;
    int lpc_stride;        // entries per frame in `lpc`
    int lpc_has_one;       // 1: lpc[f] = [1, a1..ap] (Levinson `ac`), 0: [a1..ap] (Burg)
    int lpc_f64, out_f64;
    int R;                 // resonance slots per frame in res_out
    int strict_im;         // 1: keep roots with im > 0 (lib.rs:95), 0: im >= 0 (to_resonance)
    int polish_steps;
    unsigned long long* work;  // executed-work counters (vbx_profile_counters) or null
    // vbx_find_formants runs the frames of every utterance in chunks: input row f (chunk-local, in_J frames per utterance) is
    // output row (f / in_J)·out_J + out_j0 + f % in_J of the caller's [utterance][frame] layout.  out_J == 0: identity.
    int64_t in_J, out_J, out_j0;
    // Frames on which a solve of the pair kernel ran into its 20-iteration cap WITHOUT converging are appended here (capacity
    // hard_cap, at least the launch's frame count: no frame is dropped); the fix-up launch of the f64 reference-order kernel then
    // redoes exactly those frames (frame_list / frame_count set: list entry i is frame frame_list[i]).  hard_mod > 0 (tests):
    // every hard_mod-th frame is treated as hard.
    int* hard_list;
    unsigned* hard_count;
    int hard_cap, hard_mod;
    const int* frame_list;
    const unsigned* frame_count;
};

// ---------------------------------------------------------------------------------------------
// lpc_roots_rt_kernel: runtime loops over the degree, coefficients in shared memory (column layout
// [k][thread], conflict free), one copy of the Laguerre body.  The first version of this kernel was
// statically unrolled over the degree with the polynomial in registers: 250 KB of SASS, instruction-
// cache bound once the grid was many waves deep (profiles/r1_roots_v0_icache.txt: stall_no_inst 82 %,
// 76 Mframes/s at the C3 scale against 540 now).  Arithmetic and its order are the reference's (Horner
// from the deflated degree M, n = P in the formulas).
// ---------------------------------------------------------------------------------------------
constexpr int kRootsThreads = 128;

// approximate reciprocal / principal complex square root for the fp32 fast path (the f64 instantiations fall back to the
// exact operations; they are never used by FAST code).  One MUFU each, flush-to-zero: the callers keep the arguments in
// the normal range.
__device__ __forceinline__ float fast_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ double fast_rcp(double x) { return 1.0 / x; }
__device__ __forceinline__ float fast_rsqrt(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ vcx<float> csqrt_fast(vcx<float> a) {
    const float n2 = a.re * a.re + a.im * a.im;
    // |a|² outside the comfortable fp32 range (an iterate that sits on a root to the last bit makes a1 / a0 huge), zero or
    // NaN: the overflow-safe hypot form
    if (!(n2 >= 1.0e-30f && n2 <= 1.0e30f)) return csqrt_principal(a);
    const float r = n2 * fast_rsqrt(n2);                  // |a|
    // the larger of sqrt((r ± re)/2) is computed directly (no cancellation), the other follows from re·im = a.im / 2
    const float big = 0.5f * (r + fabsf(a.re));
    const float rs = fast_rsqrt(big);
    const float t = big * rs;                             // sqrt(big)
    const float small = 0.5f * fabsf(a.im) * rs;          // |a.im| / (2·sqrt(big))
    const bool neg_im = (a.im < 0.f) || (a.im == 0.f && signbit(a.im));
    if (a.re >= 0.f) return cmk<float>(t, neg_im ? -small : small);
    return cmk<float>(small, neg_im ? -t : t);
}
__device__ __forceinline__ vcx<double> csqrt_fast(vcx<double> a) { return csqrt_principal(a); }

// Laguerre update (polynomial.rs:48-69) from the Horner triple (a0, a1, a2) = (P, P', P''/2) at z: returns the step n/cc.
// FAST (fp32 path, polished in fp64 afterwards): one reciprocal per complex division instead of two IEEE divisions and
// squared magnitudes for the |cc1| > |cc2| choice; the fp64 path keeps the reference's operations one for one.
template <typename TR, bool FAST>
__device__ __forceinline__ vcx<TR> laguerre_step(vcx<TR> a0, vcx<TR> a1, vcx<TR> a2, TR nn, TR nref) {
    if (FAST) {
        // The fp32 iterate is self-correcting and polished in fp64 afterwards, so this path uses the hardware's approximate
        // reciprocal / reciprocal square root (1-2 ulp, one MUFU each) instead of IEEE divisions, hypotf and sqrtf: the step
        // changes in its last bits, the root it converges to does not (~60 instructions fewer per round).
        const TR inv0 = fast_rcp(cnorm_sqr(a0));
        const vcx<TR> ca = cmk<TR>(-(a1.re * a0.re + a1.im * a0.im) * inv0, -(a1.im * a0.re - a1.re * a0.im) * inv0);
        const vcx<TR> ca2 = cmul(ca, ca);
        const vcx<TR> t2 = cmk<TR>((TR)2 * (a2.re * a0.re + a2.im * a0.im) * inv0, (TR)2 * (a2.im * a0.re - a2.re * a0.im) * inv0);
        const vcx<TR> cb = csub(ca2, t2);
        const vcx<TR> c1 = csqrt_fast(cmk<TR>(nn * cb.re - ca2.re, nn * cb.im - ca2.im));
        const vcx<TR> cc1 = cadd(ca, c1), cc2 = csub(ca, c1);
        const TR n1 = cnorm_sqr(cc1), n2 = cnorm_sqr(cc2);
        const vcx<TR> den = (n1 > n2) ? cc1 : cc2;
        const TR invd = nref * fast_rcp((n1 > n2) ? n1 : n2);
        return cmk<TR>(den.re * invd, -den.im * invd);  // n / den = n·conj(den)/|den|²
    } else {
        const vcx<TR> ca = cdiv(cneg(a1), a0);
        const vcx<TR> ca2 = cmul(ca, ca);
        const vcx<TR> t2 = cdiv(cmk<TR>((TR)2 * a2.re, (TR)2 * a2.im), a0);
        const vcx<TR> cb = csub(ca2, t2);
        const vcx<TR> c1 = csqrt_principal(cmk<TR>(nn * cb.re - ca2.re, nn * cb.im - ca2.im));
        const vcx<TR> cc1 = cadd(ca, c1), cc2 = csub(ca, c1);
        const vcx<TR> den = (cnorm(cc1) > cnorm(cc2)) ? cc1 : cc2;
        return cdiv(cmk<TR>(nref, (TR)0), den);
    }
}

// One frame of lpc_roots_rt_kernel: list entry `item` of n_items (the frame itself, or the fix-up list's item-th frame).
template <typename TR>
__device__ __forceinline__ void lpc_roots_rt_frame(const RootsParams& Q, const int P, const int64_t item, const int64_t n_items) {
    extern __shared__ __align__(16) unsigned char roots_smem[];
    constexpr int T = kRootsThreads;
    const unsigned FULL = 0xffffffffu;
    double* a_s = reinterpret_cast<double*>(roots_smem);                    // [P+1][T] original real coefficients
    vcx<TR>* c_s = reinterpret_cast<vcx<TR>*>(a_s + (size_t)(P + 1) * T);   // [P+1][T] working polynomial
    vcx<TR>* r_s = c_s + (size_t)(P + 1) * T;                               // [P][T]   roots in find_roots order
    const int tid = threadIdx.x;
    const bool in_range = item < n_items;
    const int64_t f_raw = Q.frame_list ? (int64_t)Q.frame_list[in_range ? item : 0] : item;
    const int64_t f = in_range ? f_raw : Q.n_frames - 1;
    const int64_t fo = Q.out_J ? (f / Q.in_J) * Q.out_J + Q.out_j0 + (f % Q.in_J) : f;  // output row  // out-of-range lanes shadow the last frame (no stores): warp-wide ops stay full
    const int R = Q.R;
    auto write_res = [&](int slot, double fr_, double bw_) {
        if (Q.out_f64) {
            double* o = reinterpret_cast<double*>(Q.res_out) + ((size_t)fo * R + slot) * 2;
            o[0] = fr_; o[1] = bw_;
        } else {
            float* o = reinterpret_cast<float*>(Q.res_out) + ((size_t)fo * R + slot) * 2;
            o[0] = (float)fr_; o[1] = (float)bw_;
        }
    };
    auto write_root = [&](int k, vcx<double> z) {
        if (Q.out_f64) {
            double* o = reinterpret_cast<double*>(Q.roots_out) + ((size_t)fo * P + k) * 2;
            o[0] = z.re; o[1] = z.im;
        } else {
            float* o = reinterpret_cast<float*>(Q.roots_out) + ((size_t)fo * P + k) * 2;
            o[0] = (float)z.re; o[1] = (float)z.im;
        }
    };
    const bool lpc_failed = Q.status_in && Q.status_in[f] != VBX_OK;  // find_formants returns Err before root finding
    // polynomial in ascending powers: a[k] = coefficient of z^k = lpc_{P-k}, a[P] = 1   (lib.rs:78-91)
    auto lpc_at = [&](int idx) -> double {
        return Q.lpc_f64 ? reinterpret_cast<const double*>(Q.lpc)[(size_t)f * Q.lpc_stride + idx]
                         : (double)reinterpret_cast<const float*>(Q.lpc)[(size_t)f * Q.lpc_stride + idx];
    };
    for (int k = 0; k <= P; ++k) {
        const double v = (k < P) ? lpc_at((P - k) - (Q.lpc_has_one ? 0 : 1)) : (Q.lpc_has_one ? lpc_at(0) : 1.0);
        a_s[k * T + tid] = v;
        c_s[k * T + tid] = cmk<TR>((TR)v, (TR)0);
    }
    constexpr bool FAST = (sizeof(TR) == 4);
    const TR nn = (TR)((P - 1) * P), nref = (TR)P;
    // polynomial.rs:116-128: for m = P down to 3: z = laguerre(coeffs, −2−2i); deflate.  The (degree, iteration)
    // loops are flattened: every lane carries its own degree M and iteration count, so a lane that converges early
    // deflates and starts its next solve at once instead of idling until the slowest lane of the warp is done.  One
    // trip = one Laguerre iteration for every lane; Horner starts at the warp's largest M — the coefficients above a
    // lane's own degree are exact zeros, so the extra steps change nothing (0·z + c = c).
    int M = P, it = 0;
    vcx<TR> z = cmk<TR>((TR)-2, (TR)-2);
    bool active = (P >= 3) && !lpc_failed;
    unsigned work_steps = 0, work_rounds = 0;  // executed Horner steps / rounds of this lane (idle lanes run them too)
#pragma unroll 1
    while (true) {
        const int Mmax = __reduce_max_sync(FULL, active ? M : 0);
        if (Mmax < 3) break;
        work_steps += (unsigned)Mmax;
        ++work_rounds;
        vcx<TR> a0 = c_s[Mmax * T + tid], a1 = cmk<TR>((TR)0, (TR)0), a2 = cmk<TR>((TR)0, (TR)0);
#pragma unroll 4
        for (int j = Mmax - 1; j >= 0; --j) {
            const vcx<TR> cj = c_s[j * T + tid];
            a2 = cfma(a2, z, a1);
            a1 = cfma(a1, z, a0);
            a0 = cfma(a0, z, cj);
        }
        if (active) {
            bool done = false;
            if (cnorm_sqr(a0) <= (TR)1.0e-32) {  // |P(z)| <= 1e-16 (polynomial.rs:47)
                done = true;
            } else {
                const vcx<TR> step = laguerre_step<TR, FAST>(a0, a1, a2, nn, nref);
                z = cadd(z, step);
                if (FAST) {  // converged for the purpose of the fp64 polish that follows
                    const TR eps = (TR)3.0e-7;
                    if (cnorm_sqr(step) <= eps * eps * cnorm_sqr(z)) done = true;
                }
                if (++it == 20) done = true;
            }
            if (done) {
                r_s[(P - M) * T + tid] = z;
                // deflation by the root (polynomial.rs:155-195 with other = −z)
                vcx<TR> carry = c_s[M * T + tid];
                c_s[M * T + tid] = cmk<TR>((TR)0, (TR)0);
#pragma unroll 4
                for (int i = M - 1; i >= 0; --i) {
                    const vcx<TR> old = c_s[i * T + tid];
                    c_s[i * T + tid] = carry;
                    carry = cmk<TR>(old.re + (carry.re * z.re - carry.im * z.im), old.im + (carry.re * z.im + carry.im * z.re));
                }
                --M;
                it = 0;
                z = cmk<TR>((TR)-2, (TR)-2);
                active = (M >= 3);
            }
        }
    }
    if (Q.work) {  // warp-uniform counts: one atomic pair per warp
        if ((tid & 31) == 0) {
            atomicAdd(Q.work + 0, 32ULL * work_steps);
            atomicAdd(Q.work + 1, 32ULL * work_rounds);
        }
    }
    if (lpc_failed) {
        if (in_range) {
            if (Q.status_out) Q.status_out[fo] = Q.status_in[f];
            if (Q.nres_out) Q.nres_out[fo] = 0;
            if (Q.res_out) for (int s = 0; s < R; ++s) write_res(s, 0.0, 0.0);
        }
        return;
    }
    if (!in_range) return;
    if (P >= 2) {
        // polynomial.rs:131-139 quadratic tail: (−c1 ± sqrt(c1² − 4 c2 c0)) / 2c2, "+" first
        const vcx<TR> q0 = c_s[tid], q1 = c_s[T + tid], q2 = c_s[2 * T + tid];
        const vcx<TR> a2 = cadd(q2, q2);
        const vcx<TR> four_ac = cmul(cmul(cmk<TR>((TR)4, (TR)0), q2), q0);
        const vcx<TR> d = csqrt_principal(csub(cmul(q1, q1), four_ac));
        const vcx<TR> x = cneg(q1);
        r_s[(P - 2) * T + tid] = cdiv(cadd(x, d), a2);
        r_s[(P - 1) * T + tid] = cdiv(csub(x, d), a2);
    } else {
        r_s[tid] = cdiv(cneg(c_s[tid]), c_s[T + tid]);  // polynomial.rs:141-144 linear tail
    }
    // resonances: fp64 polish of the roots that can become resonances (two Newton steps on the ORIGINAL
    // polynomial), then from_root; the sorted resonances are staged in the (now free) working-polynomial columns
    // sorted-resonance staging in the thread's OWN column of the (now free) working polynomial: for fp64 a
    // (frequency, bandwidth) pair is one 16-byte element of c_s; for fp32 an element is 8 bytes = one double,
    // so frequencies go to rows 0..P−1 and bandwidths to rows P..2P−1 (row P+cnt is r_s row cnt−1 < k, already
    // consumed).  Any other mapping lands in another thread's column while that thread may still be solving.
    double* rf = reinterpret_cast<double*>(c_s);
    auto stage_put = [&](int i, double fr_, double bw_) {
        if (sizeof(TR) == 8) { rf[(i * T + tid) * 2] = fr_; rf[(i * T + tid) * 2 + 1] = bw_; }
        else { rf[i * T + tid] = fr_; rf[(P + i) * T + tid] = bw_; }
    };
    auto stage_f = [&](int i) -> double { return sizeof(TR) == 8 ? rf[(i * T + tid) * 2] : rf[i * T + tid]; };
    auto stage_b = [&](int i) -> double { return sizeof(TR) == 8 ? rf[(i * T + tid) * 2 + 1] : rf[(P + i) * T + tid]; };
    int cnt = 0;
#pragma unroll 1
    for (int k = 0; k < P; ++k) {
        const vcx<TR> zr = r_s[k * T + tid];
        vcx<double> z = cmk<double>((double)zr.re, (double)zr.im);
        const bool cand = Q.strict_im ? (z.im > 0.0) : (z.im >= 0.0);
        if (cand && FAST && Q.polish_steps > 0) {
            for (int s = 0; s < Q.polish_steps; ++s) {
                vcx<double> p0 = cmk<double>(a_s[P * T + tid], 0.0), p1 = cmk<double>(0.0, 0.0);
#pragma unroll 4
                for (int j = P - 1; j >= 0; --j) {
                    p1 = cfma(p1, z, p0);
                    p0 = cmk<double>(fma(p0.re, z.re, fma(-p0.im, z.im, a_s[j * T + tid])), fma(p0.re, z.im, p0.im * z.re));
                }
                if (cnorm_sqr(p1) == 0.0) break;
                z = csub(z, cdiv(p0, p1));
            }
        }
        if (Q.roots_out) write_root(k, z);
        double fr_, bw_;
        if (cand && from_root_f64(z.re, z.im, Q.fs, Q.strict_im != 0, &fr_, &bw_)) {
            stage_put(cnt, fr_, bw_);
            ++cnt;
        }
    }
    if (Q.status_out) Q.status_out[fo] = VBX_OK;  // NaN/inf roots yield no resonance, silently, as in the reference
    if (Q.nres_out) Q.nres_out[fo] = cnt;
    if (Q.res_out) {
        // stable rank sort by frequency (lib.rs:105-110 / spectrum.rs:207), zero padding behind
#pragma unroll 1
        for (int k = 0; k < cnt; ++k) {
            const double fk = stage_f(k);
            int rank = 0;
#pragma unroll 1
            for (int j = 0; j < cnt; ++j) {
                const double fj = stage_f(j);
                rank += (fj < fk || (fj == fk && j < k)) ? 1 : 0;
            }
            if (rank < R) write_res(rank, fk, stage_b(k));
        }
        for (int s = cnt; s < R; ++s) write_res(s, 0.0, 0.0);
    }
}

// A plain launch covers its frames with its grid (one trip of the loop).  The fix-up launch (frame_list set) walks the list of
// frames the pair kernel flagged with a grid-stride loop, so a grid of any size covers a list of any length.
template <typename TR>
__global__ void __launch_bounds__(kRootsThreads) lpc_roots_rt_kernel(const RootsParams Q, const int P) {
    const int64_t n_items = Q.frame_list ? (int64_t)min(*Q.frame_count, (unsigned)Q.hard_cap) : Q.n_frames;
#pragma unroll 1
    for (int64_t i0 = (int64_t)blockIdx.x * kRootsThreads; i0 < n_items; i0 += (int64_t)gridDim.x * kRootsThreads)  // CTA-uniform
        lpc_roots_rt_frame<TR>(Q, P, i0 + threadIdx.x, n_items);
}

// ---------------------------------------------------------------------------------------------
// lpc_roots_pair_kernel: the fp32 fast path for the fused LPC → resonances call when the caller does not ask for the
// roots themselves.  The LPC polynomial is REAL, so every complex root comes with its conjugate: after a Laguerre solve
// (same update formula and n as polynomial.rs:34-72, started near the unit circle) the pair is divided out as the real
// quadratic x² − 2·Re(z)·x + |z|² (a real root as x − z), the working polynomial stays real and its degree drops by
// two per solve: 5 solves over degrees 12, 10, 8, 6, 4 instead of the reference's 10 over 12 … 3 — 40 instead of 75
// Horner coefficient steps per iteration round and half the Laguerre updates.  The set of roots is the same (they are
// the roots of the same polynomial; each candidate is then polished in fp64 on the ORIGINAL coefficients exactly as in
// lpc_roots_rt_kernel), only the order in which they are found differs — which is why a call that wants `roots_out`
// (find_roots order) takes lpc_roots_rt_kernel instead.  Resonance counts and values are checked against the oracle in
// tests/test_gpu_formants.py, tests/test_gpu_full_size.py and tools/parity_scale.py.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRootsThreads) lpc_roots_pair_kernel(const RootsParams Q, const int P) {
    extern __shared__ __align__(16) unsigned char roots_smem[];
    constexpr int T = kRootsThreads;
    typedef float TR;
    const unsigned FULL = 0xffffffffu;
    double* a_s = reinterpret_cast<double*>(roots_smem);                    // [P+1][T] original real coefficients
    vcx<TR>* r_s = reinterpret_cast<vcx<TR>*>(a_s + (size_t)(P + 1) * T);   // [P][T]   roots (im >= 0 first of a pair)
    // The sorted-resonance staging reuses the root rows as they are consumed: an 8-byte row holds one double, resonance i
    // goes to rows 2i (frequency) and 2i+1 (bandwidth).  Candidate k (im > 0) sits right before its conjugate and at most
    // floor(k / 2) resonances precede it, so rows 2i and 2i+1 <= k + 1 are the candidate's own (already in registers) and
    // its conjugate's (skipped by the loop) or older.
    double* st_s = reinterpret_cast<double*>(r_s);
    float* c_s = reinterpret_cast<float*>(r_s + (size_t)P * T);             // [P+1][T] working polynomial (real)
    const int tid = threadIdx.x;
    const int64_t f_raw = (int64_t)blockIdx.x * T + tid;
    const bool in_range = f_raw < Q.n_frames;
    const int64_t f = in_range ? f_raw : Q.n_frames - 1;
    const int64_t fo = Q.out_J ? (f / Q.in_J) * Q.out_J + Q.out_j0 + (f % Q.in_J) : f;  // output row
    const int R = Q.R;
    auto write_res = [&](int slot, double fr_, double bw_) {
        if (Q.out_f64) {
            double* o = reinterpret_cast<double*>(Q.res_out) + ((size_t)fo * R + slot) * 2;
            o[0] = fr_; o[1] = bw_;
        } else {
            float* o = reinterpret_cast<float*>(Q.res_out) + ((size_t)fo * R + slot) * 2;
            o[0] = (float)fr_; o[1] = (float)bw_;
        }
    };
    const bool lpc_failed = Q.status_in && Q.status_in[f] != VBX_OK;
    auto lpc_at = [&](int idx) -> double {
        return Q.lpc_f64 ? reinterpret_cast<const double*>(Q.lpc)[(size_t)f * Q.lpc_stride + idx]
                         : (double)reinterpret_cast<const float*>(Q.lpc)[(size_t)f * Q.lpc_stride + idx];
    };
    for (int k = 0; k <= P; ++k) {
        const double v = (k < P) ? lpc_at((P - k) - (Q.lpc_has_one ? 0 : 1)) : (Q.lpc_has_one ? lpc_at(0) : 1.0);
        a_s[k * T + tid] = v;
        c_s[k * T + tid] = (float)v;
    }
    const TR nn = (TR)((P - 1) * P), nref = (TR)P;
    int M = P, it = 0, nroots = 0;
    // Start of every solve: a generic point just inside the unit circle, where the roots of an LPC polynomial live.  The
    // reference starts at −2−2i (polynomial.rs:118); since this kernel does not reproduce the reference's root ORDER anyway,
    // it may start closer: 30-45 % fewer Laguerre iterations and fewer solves that run into the 20-iteration cap
    // (measured on the synthetic corpus at 16 and 44.1 kHz), same roots.
    const vcx<TR> z_start = cmk<TR>((TR)0.3, (TR)0.9);
    vcx<TR> z = z_start;
    bool active = (P >= 3) && !lpc_failed;
    bool hard = false, retried = false;
    unsigned work_steps = 0, work_rounds = 0;  // executed Horner steps / rounds of this lane (idle lanes run them too)
#pragma unroll 1
    while (true) {
        const int Mmax = __reduce_max_sync(FULL, active ? M : 0);
        if (Mmax < 3) break;
        work_steps += (unsigned)Mmax;
        ++work_rounds;
        // Horner triple (P, P', P''/2) at z from the warp's largest degree: coefficients above a lane's own degree are 0
        vcx<TR> a0 = cmk<TR>(c_s[Mmax * T + tid], (TR)0), a1 = cmk<TR>((TR)0, (TR)0), a2 = cmk<TR>((TR)0, (TR)0);
#pragma unroll 4
        for (int j = Mmax - 1; j >= 0; --j) {
            const TR cj = c_s[j * T + tid];
            a2 = cfma(a2, z, a1);
            a1 = cfma(a1, z, a0);
            a0 = cfma(a0, z, cmk<TR>(cj, (TR)0));
        }
        if (active) {
            bool done = false;
            if (cnorm_sqr(a0) <= (TR)1.0e-32) {
                done = true;
            } else {
                const vcx<TR> step = laguerre_step<TR, true>(a0, a1, a2, nn, nref);
                z = cadd(z, step);
                // Laguerre converges cubically: a step of 1e-5·|z| means the iterate is already exact to fp32, and the fp64
                // polish that follows squares whatever error is left twice.  (3e-7, the fp32 rounding level, made solves
                // jitter around the threshold for extra iterations: 20 % more Horner work for the same roots; 1e-3 is where
                // resonance counts start to differ — numpy emulation of this kernel, 16 and 44.1 kHz.)
                const TR eps = (TR)1.0e-5;
                ++it;
                if (cnorm_sqr(step) <= eps * eps * cnorm_sqr(z)) {
                    done = true;
                } else if (it == 20) {
                    // The cap without convergence (about one frame in 10^5 on speech-like input).  Dividing a non-root out
                    // would corrupt every later root, so first the same solve is retried from a second start point; if that
                    // hits the cap too, the frame goes to the f64 fix-up launch (the reference's own algorithm).
                    if (!retried) {
                        retried = true;
                        it = 0;
                        z = cmk<TR>((TR)-0.4, (TR)0.85);
                    } else {
                        done = true;
                        hard = true;
                    }
                }
            }
            if (done) {
                // a root this close to the real axis (|arg| < 1e-5: below 0.1 Hz at any audio rate) is divided out as real
                const bool real_root = fabsf(z.im) <= (TR)1.0e-5 * fabsf(z.re);
                if (real_root) {
                    r_s[nroots * T + tid] = cmk<TR>(z.re, (TR)0);
                    ++nroots;
                    // synthetic division by (x − r): b[i−1] = c[i] + r·b[i]
                    TR carry = c_s[M * T + tid];
                    c_s[M * T + tid] = (TR)0;
#pragma unroll 4
                    for (int i = M - 1; i >= 0; --i) {
                        const TR old = c_s[i * T + tid];
                        c_s[i * T + tid] = carry;
                        carry = fmaf(carry, z.re, old);
                    }
                    M -= 1;
                } else {
                    r_s[nroots * T + tid] = cmk<TR>(z.re, fabsf(z.im));
                    r_s[(nroots + 1) * T + tid] = cmk<TR>(z.re, -fabsf(z.im));
                    nroots += 2;
                    // synthetic division by x² + p·x + q, p = −2·Re z, q = |z|²: b[i−2] = c[i] − p·b[i−1] − q·b[i]
                    const TR pq = (TR)-2 * z.re, qq = cnorm_sqr(z);
                    TR b1 = (TR)0, b2 = (TR)0;  // b[i−1+1], b[i+1] of the previous step
#pragma unroll 4
                    for (int i = M; i >= 2; --i) {
                        const TR b0 = fmaf(-pq, b1, fmaf(-qq, b2, c_s[i * T + tid]));
                        c_s[i * T + tid] = b2;   // quotient coefficient of x^i (slots M, M−1 become 0, the rest shift down by 2)
                        b2 = b1;
                        b1 = b0;
                    }
                    // after the loop: b1 = b[0], b2 = b[1]; quotient x^1 and x^0 coefficients
                    c_s[1 * T + tid] = b2;
                    c_s[0 * T + tid] = b1;
                    M -= 2;
                }
                it = 0;
                retried = false;
                z = z_start;
                active = (M >= 3);
            }
        }
    }
    if (Q.work) {  // warp-uniform counts: one atomic pair per warp
        if ((tid & 31) == 0) {
            atomicAdd(Q.work + 0, 32ULL * work_steps);
            atomicAdd(Q.work + 1, 32ULL * work_rounds);
        }
    }
    if (lpc_failed) {
        if (in_range) {
            if (Q.status_out) Q.status_out[fo] = Q.status_in[f];
            if (Q.nres_out) Q.nres_out[fo] = 0;
            if (Q.res_out) for (int s = 0; s < R; ++s) write_res(s, 0.0, 0.0);
        }
        return;
    }
    if (!in_range) return;
    if (Q.hard_mod > 0 && (f_raw % Q.hard_mod) == 0) hard = true;
    if (hard && Q.hard_list) {
        const unsigned idx = atomicAdd(Q.hard_count, 1u);
        if (idx < (unsigned)Q.hard_cap) Q.hard_list[idx] = (int)f_raw;
        if (Q.work) atomicAdd(Q.work + 4, 1ULL);
    }
    // tail: what is left has degree 2, 1 or 0 (real coefficients)
    if (M == 2) {
        const TR q0 = c_s[tid], q1 = c_s[T + tid], q2 = c_s[2 * T + tid];
        const TR disc = q1 * q1 - (TR)4 * q2 * q0;
        const TR inv = (TR)1 / ((TR)2 * q2);
        if (disc < (TR)0) {
            const TR sq = sqrtf(-disc);
            r_s[nroots * T + tid] = cmk<TR>(-q1 * inv, fabsf(sq * inv));
            r_s[(nroots + 1) * T + tid] = cmk<TR>(-q1 * inv, -fabsf(sq * inv));
        } else {
            const TR sq = sqrtf(disc);
            r_s[nroots * T + tid] = cmk<TR>((-q1 + sq) * inv, (TR)0);
            r_s[(nroots + 1) * T + tid] = cmk<TR>((-q1 - sq) * inv, (TR)0);
        }
        nroots += 2;
    } else if (M == 1) {
        r_s[nroots * T + tid] = cmk<TR>(-c_s[tid] / c_s[T + tid], (TR)0);
        nroots += 1;
    }
    // resonances: fp64 polish (Newton on the ORIGINAL polynomial) of the roots that can become resonances, from_root
    int cnt = 0;
#pragma unroll 1
    for (int k = 0; k < nroots; ++k) {
        const vcx<TR> zr = r_s[k * T + tid];
        vcx<double> zz = cmk<double>((double)zr.re, (double)zr.im);
        const bool cand = Q.strict_im ? (zz.im > 0.0) : (zz.im >= 0.0);
        if (cand && Q.polish_steps > 0) {
            for (int s = 0; s < Q.polish_steps; ++s) {
                vcx<double> p0 = cmk<double>(a_s[P * T + tid], 0.0), p1 = cmk<double>(0.0, 0.0);
#pragma unroll 4
                for (int j = P - 1; j >= 0; --j) {
                    p1 = cfma(p1, zz, p0);
                    p0 = cmk<double>(fma(p0.re, zz.re, fma(-p0.im, zz.im, a_s[j * T + tid])), fma(p0.re, zz.im, p0.im * zz.re));
                }
                if (cnorm_sqr(p1) == 0.0) break;
                zz = csub(zz, cdiv(p0, p1));
            }
        }
        double fr_, bw_;
        const bool keep = cand && from_root_f64(zz.re, zz.im, Q.fs, Q.strict_im != 0, &fr_, &bw_);
        if (zr.im > (TR)0) ++k;  // the next row is this root's conjugate (never a candidate): skip it — it may be overwritten below
        if (keep) {
            st_s[(2 * cnt) * T + tid] = fr_;
            st_s[(2 * cnt + 1) * T + tid] = bw_;
            ++cnt;
        }
    }
    if (Q.status_out) Q.status_out[fo] = VBX_OK;
    if (Q.nres_out) Q.nres_out[fo] = cnt;
    if (Q.res_out) {
#pragma unroll 1
        for (int k = 0; k < cnt; ++k) {
            const double fk = st_s[(2 * k) * T + tid];
            int rank = 0;
#pragma unroll 1
            for (int j = 0; j < cnt; ++j) {
                const double fj = st_s[(2 * j) * T + tid];
                rank += (fj < fk || (fj == fk && j < k)) ? 1 : 0;
            }
            if (rank < R) write_res(rank, fk, st_s[(2 * k + 1) * T + tid]);
        }
        for (int s = cnt; s < R; ++s) write_res(s, 0.0, 0.0);
    }
}

static inline size_t roots_pair_smem_bytes(int P) {
    // a_s [P+1] f64, r_s [P] complex f32 (reused as the resonance staging), c_s [P+1] f32
    return (size_t)kRootsThreads * ((size_t)(P + 1) * 8 + (size_t)P * 8 + (size_t)(P + 1) * 4);
}

static inline size_t roots_rt_smem_bytes(int P, bool f32) {
    const size_t cs = f32 ? 8 : 16;
    return (size_t)kRootsThreads * ((size_t)(P + 1) * 8 + (size_t)(P + 1) * cs + (size_t)P * cs);
}

constexpr int kMaxRootsOrder = 24;

}  // namespace vbx_roots
