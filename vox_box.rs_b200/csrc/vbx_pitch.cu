// vbx_pitch.cu — Boersma autocorrelation pitch candidates, batched over frames.
//
// Replaces, batched over frames:
//   periodic.rs:356-358,377-456  Pitched::pitch::<Hanning>          (the whole candidate chain)
//   periodic.rs:362-375          LocalMaxima::local_maxima           (strict 3-point peaks)
//   periodic.rs:29-87            interpolate_sinc                    (with the swapped-neighbour quirk)
//   periodic.rs:103-188          brent_maximize                      (a Brent MINIMISER as written)
//   periodic.rs:89-93,192-230    Interpolation, improve_extremum
//   periodic.rs:232-252          LagType / HanningLag                (lag-window table, host f64)
//   periodic.rs:306-354          Pitch, PitchExtractor               (arg-max: candidates[f][0])
//
// Kernel shapes (DESIGN.md §K6/K7):
//   pitch_lag64_kernel    a CTA stages the windowed frames of `fpc` frames in shared memory as exact
//                         f64 products x·w and computes ALL N lags on the FP64 pipe: a lane owns a
//                         16-lag group and walks the frame in 8-sample steps, the triangle is balanced
//                         by pairing group g with group G-1-g on the same lane (vbx_pitch_lag64.cuh).
//                         A warp per frame then normalises (÷ max|r|), divides by the lag window, finds
//                         the strict local maxima below N/2, interpolates them parabolically, applies
//                         the (min, max) filter and appends the survivors to a global work list.
//   pitch_refine8q_kernel slots of two lanes run the reference's Brent minimiser over the windowed-sinc
//                         interpolant, all in fp64; a CTA takes tiles of the work list, sorts each by
//                         interpolation depth and its slots draw candidates from that order.
//   pitch_finalize_kernel a warp per frame appends the unvoiced candidate, checks for NaN
//                         strengths and rank-sorts by strength (stable, descending).  With peaks
//                         (vbx_pitch_with_peaks) the unvoiced candidate's strength is Boersma's voiceless
//                         strength of the frame instead of the fixed threshold.
#include <cmath>

#include "vbx_internal.cuh"
#include "vbx_pipeline.cuh"

namespace {

constexpr double kPi = 3.14159265358979323846264338327950288;

struct PitchCand {
    int frame;   // frame index inside the slab
    int k;       // rank of the candidate inside its frame (ascending lag)
    double n;    // Brent start abscissa: fs/freq − offset
};

struct PitchParams {
    const void* base;
    const double* win;      // [N] frame window (device, f64)
    const double* lagwin;   // [N] HanningLag table (device, f64)
    double* y;              // [S][N] scratch: r, then the normalised / window-divided lag function
    PitchCand* list;        // [S·cap] work list
    double2* refined;       // [S·cap] (frequency, strength) per work-list entry
    int2* range;            // [S] (first list entry, count) per frame
    unsigned long long* counter;  // [0] number of list entries, [1] tile cursor of the refine kernel
    unsigned long long* work;     // executed-work counters (vbx_profile_counters) or null
    int64_t frame0;         // first frame of this slab inside the batch
    int64_t n_frames;       // frames in this slab
    int64_t stride, seg_frames, seg_stride;
    int n, n16;             // frame length, rounded up to 16
    int G, lpf, fpc, T;     // lag groups of 16, lanes per frame, frames per CTA, steps per lane
    int xs_words;           // shared-memory words per frame
    int ixmax;              // floor(N/2)
    double fs, fmin, fmax, threshold;
    // vbx_pitch_with_peaks: local peak per frame of the batch, global peak per segment (both null for vbx_pitch)
    const double* local_peak;
    const double* global_peak;
    double silence;         // silence threshold b > 0 of voiceless_strength
};

// Boersma (1993) / Praat's voiceless strength of a frame: a + max(0, 2 − ratio·(1 + a)/b), ratio = min(local/global, 1),
// ratio = 0 where global <= 0 or is NaN; a NaN ratio (a NaN local peak) leaves a.  a = voicing threshold, b = silence
// threshold > 0.  The test reference (tests/test_gpu_pitch_peaks.py) evaluates the same expression in the same order.
__device__ __forceinline__ double voiceless_strength(double local, double global, double a, double b) {
    double ratio = 0.0;
    if (global > 0.0) {
        ratio = local / global;
        if (ratio > 1.0) ratio = 1.0;
    }
    const double v = 2.0 - ratio * (1.0 + a) / b;
    return a + (v > 0.0 ? v : 0.0);
}

__device__ __forceinline__ int lag_steps(int n, int g) {  // 8-sample steps lag group g needs
    const int len = n - 16 * g;
    return len > 0 ? (len + 7) >> 3 : 0;
}

// Per frame (one warp), after the lag sweep: normalise, ÷ lag window, local maxima, parabolic, filter.
// `smem` = the CTA's frame buffers (dead after the sweep), `frame_bytes` apart.
__device__ __forceinline__ void pitch_lag_post(const PitchParams& P, unsigned char* smem, size_t frame_bytes, int64_t f_first, int nf) {
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int n = P.n;
    const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
    const unsigned FULL = 0xffffffffu;
    for (int qf = warp; qf < nf; qf += nwarps) {
        double* yrow = P.y + (size_t)(f_first + qf) * n;
        // waves.rs:39-59 max_amplitude: fold from |r[0]| with `>`: a NaN at index 0 sticks, later NaNs never win
        double pm = -1.0;
        for (int i = 1 + lane; i < n; i += 32) {
            const double a = fabs(yrow[i]);
            if (a > pm) pm = a;
        }
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) {
            const double o = __shfl_xor_sync(FULL, pm, m);
            if (o > pm) pm = o;
        }
        const double r0a = fabs(yrow[0]);
        const double mx = (r0a != r0a) ? r0a : (pm > r0a ? pm : r0a);
        const double scale = 1.0 / mx;  // waves.rs:70: no zero guard
        for (int i = lane; i < n; i += 32) yrow[i] = (yrow[i] * scale) / __ldg(P.lagwin + i);
        __syncwarp();
        // periodic.rs:417-439: maxima of y[0..ixmax), parabolic frequency, (min, max) filter
        const int ixmax = P.ixmax;
        const double offset = -(double)ixmax - 1.0;
        // one pass: the start abscissae are parked in the frame's (now dead) sample buffer, the frame's slice of the
        // work list is reserved once the count is known, then the entries are written out
        double* stage = reinterpret_cast<double*>(smem + (size_t)qf * frame_bytes);  // frame_bytes >= (ixmax/2 + 1)·8
        int k = 0;
        for (int base = 1; base + 1 < ixmax; base += 32) {
            const int cidx = base + lane;
            bool keep = false;
            double nn = 0.0;
            if (cidx + 1 < ixmax) {
                const double peak = yrow[cidx], rev = yrow[cidx - 1], fwd = yrow[cidx + 1];
                if (rev < peak && fwd < peak) {
                    const double dr = 0.5 * (fwd - rev);
                    const double d2r = 2. * peak - (rev - fwd);  // sign quirk, periodic.rs:424
                    const double freq = P.fs / ((double)cidx + dr / d2r);
                    keep = (freq == 0.) || (freq > P.fmin && freq < P.fmax);
                    nn = P.fs / freq - offset;
                }
            }
            const unsigned bal = __ballot_sync(FULL, keep);
            if (keep) stage[k + __popc(bal & ((1u << lane) - 1u))] = nn;
            k += __popc(bal);
        }
        const int count = k;
        unsigned long long pos = 0;
        if (lane == 0) {
            pos = atomicAdd(P.counter, (unsigned long long)count);
            P.range[f_first + qf] = make_int2((int)pos, count);
        }
        const int start = (int)__shfl_sync(FULL, pos, 0);
        __syncwarp();  // the staging writes above are read by other lanes below
        for (int i = lane; i < count; i += 32) {
            PitchCand e;
            e.frame = (int)(f_first + qf);
            e.k = i;
            e.n = stage[i];
            P.list[(size_t)start + i] = e;
        }
    }
}

// K6: windowed frame → all-lag autocorrelation → y = (r / max|r|) / lag window → candidates
#include "vbx_pitch_lag64.cuh"

// -------------------------------------------------------------------------------------------
// windowed-sinc interpolation, one warp per evaluation (periodic.rs:29-87)
// y has `y_len` entries of which the first `y_store` are stored (the rest read as zero: the
// reference zero-extends the lag function to 2N, periodic.rs:411).
// -------------------------------------------------------------------------------------------
__device__ __forceinline__ double y_at(const double* __restrict__ y, long long idx, long long y_store) {
    return idx < y_store ? __ldg(y + idx) : 0.0;
}

__device__ double sinc_interp_warp(const double* __restrict__ y, long long y_len, long long y_store, long long offset,
                                   long long nx, double x, long long max_depth, int lane) {
    const double fl = floor(x);
    const long long nl = (fl > 0.0) ? (long long)fl : 0;  // `x.floor() as usize` saturates negative / NaN to 0
    const long long nr = nl + 1;
    const double phil = x - (double)nl;
    const double phir = 1. - phil;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    auto at = [&](long long idx) -> double {  // an out-of-range index panics in the reference
        return (idx < 0 || idx >= y_len) ? qnan : y_at(y, idx, y_store);
    };
    if (nx < 1) return qnan;
    if (x > (double)nx) return at(offset + nx - 1);
    if (x < 0.) return y_at(y, 0, y_store);
    if (fabs(x - (double)nl) < 1.0e-10) return at(offset + nl);
    if (fabs(x - (double)nr) < 1.0e-10) return at(offset + nr);
    if ((offset + nr) < max_depth) max_depth = (offset + nr) < 0 ? 0 : offset + nr;           // :46-52
    if ((offset + nl + max_depth) >= nx) max_depth = nx - offset + nl - 1;                    // :55-57
    // sin(π(φ+n)) = (−1)ⁿ sin(πφ); sin(πφr) = sin(π(1−φl)) = sin(πφl)
    const double s0 = sinpi(phil);
    const double inv_l = 1.0 / (phil + (double)max_depth), inv_r = 1.0 / (phir + (double)max_depth);
    double accl = 0.0, accr = 0.0;
    for (long long nn = lane; nn <= max_depth; nn += 32) {
        const double sgn = (nn & 1) ? -1.0 : 1.0;
        {   // "left": φl pairs with y[offset+nr−n], clamped at 0
            long long idx = offset + nr - nn;
            if (idx < 0) idx = 0;
            const double t = phil + (double)nn;
            const double second = 0.5 + 0.5 * cospi(t * inv_l);
            accl = fma(at(idx) * sgn, second / t, accl);
        }
        {   // "right": φr pairs with y[offset+nl+n], clamped to [0, len−1]
            long long idx = offset + nl + nn;
            if (idx < 0) idx = 0;
            if (idx >= y_len) idx = y_len - 1;
            const double t = phir + (double)nn;
            const double second = 0.5 + 0.5 * cospi(t * inv_r);
            accr = fma(y_at(y, idx, y_store) * sgn, second / t, accr);
        }
    }
    double acc = accl + accr;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) acc += vbx_shfl_xor(acc, m);
    return acc * (s0 * (1.0 / kPi));
}

// periodic.rs:103-188 brent_maximize — uniform across the warp; f = +interpolate_sinc (is_max) or −.
__device__ double brent_warp(const double* __restrict__ y, long long y_len, long long y_store, long long offset, long long nx,
                             long long depth, bool is_max, double a, double b, double tol, double* fx_out, int lane) {
    const double golden = 1. - 0.6180339887498948482045868343656381177203091798057628621;
    const double EPS = 2.220446049250313e-16;
    const double sqrt_epsilon = 1.4901161193847656e-08;
    auto f = [&](double t) -> double {
        const double out = sinc_interp_warp(y, y_len, y_store, offset, nx, t, depth, lane);
        return is_max ? out : -out;
    };
    double v = a + golden * (b - a);
    double fv = f(v);
    double x = v, w = v, fx = fv, fw = fv;
    for (int iter = 1; iter <= 60; ++iter) {
        const double range = b - a;
        const double middle_range = (a + b) * 0.5;
        const double tol_act = sqrt_epsilon * fabs(x) + tol / 3.;
        if (fabs(x - middle_range) + range * 0.5 <= 2. * tol_act) break;
        double new_step = (x < middle_range) ? golden * (b - x) : golden * (a - x);
        if (fabs(x - w) >= tol_act) {
            const double t = (x - w) * (fx - fv);
            double q = (x - v) * (fx - fw);
            double p = (x - v) * q - (x - w) * t;
            q = 2. * q - t;
            if (q > 0.) p = -p; else q = -q;
            if (fabs(p) < fabs(new_step * q) && p > q * (a - x + 2. * tol_act) && p < q * (b - x - 2. * tol_act))
                new_step = p / q;
        }
        if (fabs(new_step) < tol_act) new_step = (new_step > 0.) ? tol_act : -tol_act;
        const double t = x + new_step;
        const double ft = f(t);
        if (ft <= fx) {
            if (t < x) b = x; else a = x;
            v = w; w = x; x = t;
            fv = fw; fw = fx; fx = ft;
        } else {
            if (t < x) a = t; else b = t;
            if (ft <= fw || fabs(w - x) < EPS) {
                v = w; w = t;
                fv = fw; fw = ft;
            } else if (ft <= fv || fabs(v - x) < EPS || fabs(v - w) < EPS) {
                v = t;
                fv = ft;
            }
        }
    }
    *fx_out = fx;
    return x;
}

// periodic.rs:192-230 improve_extremum
__device__ void improve_extremum_warp(const double* __restrict__ y, long long y_len, long long y_store, long long offset,
                                      long long nx, double ixmid, int interp, long long depth, bool is_max, double* xmid,
                                      double* ymid, int lane) {
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    auto at = [&](long long idx) -> double { return (idx < 0 || idx >= y_len) ? qnan : y_at(y, idx, y_store); };
    if (ixmid == 0.) { *xmid = 0.; *ymid = at(0); return; }
    if (ixmid >= (double)nx) { *xmid = (double)nx; *ymid = at(nx - 1); return; }
    if (interp == 0) { *xmid = 0.; *ymid = at(0); return; }
    if (interp == 1) {
        const double fl = floor(ixmid);
        const long long k = fl > 0.0 ? (long long)fl : 0;
        const double d = at(k + 1) - at(k - 1);
        const double mid = at(k);
        const double dy = 0.5 * d, d2y = 2.0 * mid - d;
        *xmid = ixmid + dy / d2y;
        *ymid = mid + 0.5 * dy * dy / d2y;
        return;
    }
    double fx = 0.;
    *xmid = brent_warp(y, y_len, y_store, offset, nx, depth, is_max, ixmid - 1., ixmid + 1., 1e-10, &fx, lane);
    *ymid = fx;
}

__device__ __forceinline__ double rcp_pos(double x) {  // 1/x for normal positive x: MUFU seed + one third-order step
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);   // seed error, <= 1e-6 relative (tools/cuda/rcp_test.cu)
    return fma(r, fma(e, e, e), r);     // r·(1 + e + e²): error e³, i.e. below one ulp
}
// (A single Newton step would leave 1e-12 relative error and that already moves some weak candidates' Brent paths by
// > 0.1 Hz in tests/test_gpu_pitch.py; the third-order step costs the same three DFMAs as one-and-a-half Newton steps.)

// K7: Brent over the windowed-sinc interpolant, one work-list entry per slot of LS lanes, 32 / LS slots per warp.
//
// Lane ℓ of a slot owns the terms n ≡ ℓ (mod LS) of both sides of interpolate_sinc's sum, so that per term
//   * (−1)ⁿ is a per-lane constant (LS is even),
//   * the Hann factor ½ + ½cos(π(φ+n)/(φ+D)) advances by a three-term recurrence in cos LS·δ, δ = π/(φ+D),
//   * the two sides share one reciprocal: y_l·h_l/t_l + y_r·h_r/t_r = (y_l·h_l·t_r + y_r·h_r·t_l)/(t_l·t_r).
// Brent's state is replicated in the lanes of a slot (identical arithmetic ⇒ identical values); the only cross-lane
// traffic is the shuffle that sums the partial sums.  Brent needs a different number of evaluations for every candidate
// (about 12 to 40), so every slot draws its next candidate from the tile's sorted order (a shared-memory cursor) as soon
// as it finishes: the warp stays in lockstep only over single evaluations of the interpolant.
__global__ void __launch_bounds__(128, 1) pitch_refine8q_kernel(const PitchParams P) {
    // Every evaluation of the interpolant pays ~300 instructions of setup (three sincospi, two reciprocals, the Brent
    // update) whatever the slot width, so narrow slots amortise it best: 8 lanes 5.70e6 frames/s on C4, 4 lanes 6.85e6,
    // 2 lanes 7.06e6 (results identical: a slot's arithmetic is its own).  Tiles larger than 256 entries were slower for
    // every width: a tile's ~10 lag-function rows stay in L1, 40 rows do not.
    constexpr int LS = 2;       // lanes per slot
    constexpr int TILE = 256;   // work-list entries per tile
    constexpr int SLOT_MASK = 32 - LS;  // lane & SLOT_MASK = the slot's first lane
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, li = lane & (LS - 1);
    const long long total = (long long)*P.counter;
    const int N = P.n;
    // A CTA takes tiles of TILE consecutive work-list entries (about ten frames) and walks each tile in order of
    // the start abscissa, i.e. of the interpolation depth D: the slots of a warp then run term loops of nearly the
    // same length (the list order — ascending lag inside a frame — leaves 19 % of the lanes of the term loop idle, a
    // sorted tile 3 %).  Results do not depend on the grouping: every slot's arithmetic is its own.
    __shared__ float s_key[TILE];
    __shared__ unsigned short s_ord[TILE];
    __shared__ int s_next;
    __shared__ long long s_tile;
    const int offset = -P.ixmax - 1;
    const int nx = P.ixmax - offset;
    const int ylen = 2 * N;
    const double golden = 1. - 0.6180339887498948482045868343656381177203091798057628621;
    const double EPS = 2.220446049250313e-16, sqrt_epsilon = 1.4901161193847656e-08, tol = 1e-10;
    const double sgn = (li & 1) ? -1.0 : 1.0;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    unsigned work_terms = 0, work_evals = 0;  // executed term-loop iterations / evaluation rounds of this warp

    // tiles are handed out dynamically (P.counter[1]): the grid is exactly the resident CTAs and none of them idles
    // while another still has a backlog
    while (true) {
    __syncthreads();  // the previous tile's order is no longer read
    if (threadIdx.x == 0) {
        s_tile = (long long)atomicAdd(P.counter + 1, 1ULL);
        s_next = 0;
    }
    __syncthreads();
    const long long tile0 = s_tile * TILE;
    if (tile0 >= total) {
        if (P.work && lane == 0) {  // warp-uniform counts, summed over lanes
            atomicAdd(P.work + 2, 32ULL * work_terms);
            atomicAdd(P.work + 3, 32ULL * work_evals);
        }
        break;
    }
    const int tcnt = (int)min((long long)TILE, total - tile0);
    for (int i = threadIdx.x; i < tcnt; i += blockDim.x) s_key[i] = (float)P.list[tile0 + i].n;
    __syncthreads();
    for (int i = threadIdx.x; i < tcnt; i += blockDim.x) {
        const float ki = s_key[i];
        int rank = 0;
        for (int j = 0; j < tcnt; ++j) {
            const float kj = s_key[j];
            rank += (kj < ki || (kj == ki && j < i)) ? 1 : 0;
        }
        s_ord[rank] = (unsigned short)i;
    }
    __syncthreads();
    // slot state (replicated in the lanes of a slot)
    bool have = false, dry = false;     // have: a candidate is being refined; dry: the tile's queue is exhausted
    long long e = 0;
    const double* __restrict__ y = P.y;
    double rx = 0., ry = 0.;
    double a = 0., b = 0., v = 0., w = 0., x = 0., fv = 0., fw = 0., fx = 0., t = 0.;
    int iter = 0;
    auto yat = [&](int idx) -> double { return (idx >= 0 && idx < N) ? __ldg(y + idx) : 0.0; };  // zero-extended to 2N
    {
        while (true) {
            // ---- free slots draw the next candidate of the tile ---------------------------------------------------------
            const bool want = !have && !dry;
            int qi = -1;
            if (want && li == 0) qi = atomicAdd(&s_next, 1);
            qi = __shfl_sync(FULL, qi, lane & SLOT_MASK);
            if (want) {
                if (qi >= tcnt) {
                    dry = true;
                } else {
                    e = tile0 + (int)s_ord[qi];
                    const PitchCand cd = P.list[e];
                    y = P.y + (size_t)cd.frame * N;
                    const double ixmid = cd.n;
                    // improve_extremum's early returns (periodic.rs:193-194)
                    if (ixmid == 0. || ixmid >= (double)nx) {
                        if (li == 0) {
                            double ymid = (ixmid == 0.) ? yat(0) : yat(nx - 1);
                            const double xmid = ((ixmid == 0.) ? 0. : (double)nx) + (double)offset;
                            if (ymid > 1.) ymid = 1. / ymid;
                            P.refined[e] = make_double2(P.fs / xmid, ymid);
                        }
                    } else {
                        // brent_maximize(f, (ixmid−1, ixmid+1), tol = 1e-10)
                        a = ixmid - 1.; b = ixmid + 1.;
                        v = a + golden * (b - a); w = v; x = v; fv = 0.; fw = 0.; fx = 0.;
                        t = v;
                        iter = 0;  // 0: the initial evaluation is pending
                        have = true;
                    }
                }
            }
            if (!__any_sync(FULL, have)) {
                if (__all_sync(FULL, dry)) break;
                continue;
            }
            bool done = !have;
        {
            // ---- interpolate_sinc(y, offset, nx, t, 1200): per-slot setup ----------------------------------------
            const double fl = floor(t);
            const int nl = (fl > 0.0) ? (int)fmin(fl, 1.0e9) : 0;
            const int nr = nl + 1;
            const double phil = t - (double)nl, phir = 1. - phil;
            bool special = done;
            double sval = 0.;
            int D = -1;
            if (!done) {
                if (t > (double)nx) { special = true; const int i = offset + nx - 1; sval = (i < 0 || i >= ylen) ? qnan : yat(i); }
                else if (t < 0.) { special = true; sval = yat(0); }
                else if (fabs(t - (double)nl) < 1.0e-10) { special = true; const int i = offset + nl; sval = (i < 0 || i >= ylen) ? qnan : yat(i); }
                else if (fabs(t - (double)nr) < 1.0e-10) { special = true; const int i = offset + nr; sval = (i < 0 || i >= ylen) ? qnan : yat(i); }
                else {
                    int md = 1200;
                    if (offset + nr < md) md = (offset + nr < 0) ? 0 : offset + nr;
                    if (offset + nl + md >= nx) md = nx - offset + nl - 1;
                    D = md;
                }
            }
            const bool act = !special;
            const double pl = act ? phil : 0.5, pr = act ? phir : 0.5;
            const double Dd = (double)(D < 0 ? 0 : D);
            const double inv_l = rcp_pos(pl + Dd), inv_r = rcp_pos(pr + Dd);
            // two of the three slot-uniform trigonometric values share ONE sincospi call: lane 0 of the slot takes πφ
            // (→ sin πφ), lane 1 takes LS·δ_l; three shuffles hand the results to the other lane of the slot
            double su, cu;
            sincospi(li == 0 ? pl : (li == 1 ? (double)LS * inv_l : 0.0), &su, &cu);
            const int sb = lane & SLOT_MASK;
            const double s0 = __shfl_sync(FULL, su, sb);
            const double Sdl = __shfl_sync(FULL, su, sb + 1), Cdl = __shfl_sync(FULL, cu, sb + 1);
            double Sdr, Cdr;
            sincospi((double)LS * inv_r, &Sdr, &Cdr);
            double sl, cl, sr, cr;
            double tl = pl + (double)li, tr = pr + (double)li;
            sincospi(tl * inv_l, &sl, &cl);
            sincospi(tr * inv_r, &sr, &cr);
            // Hann factor h_j = ½ + ½cos(θ0 + LS·δ·j) by the three-term recurrence h_{j+1} = K·h_j − h_{j−1} + (1 − K/2),
            // K = 2cos LS·δ (error growth ~j²·ε, j <= 600), started from h_0 and h_{−1} = ½ + ½cos(θ0 − LS·δ)
            double hl = fma(0.5, cl, 0.5), hlp = fma(0.5, fma(cl, Cdl, sl * Sdl), 0.5);
            double hr = fma(0.5, cr, 0.5), hrp = fma(0.5, fma(cr, Cdr, sr * Sdr), 0.5);
            const double Kl = 2.0 * Cdl, Kr = 2.0 * Cdr, Cl = 1.0 - Cdl, Cr = 1.0 - Cdr;
            const int L = offset + nr, R = offset + nl;
            const int Dmax = __reduce_max_sync(FULL, D);
            work_terms += (unsigned)((Dmax >= 0 ? Dmax : -1) + LS) / LS;
            ++work_evals;
            double acc = 0.;
            // Left terms read y[L − n] (>= 0 because D <= L), right terms y[R + n]; beyond N the zero extension
            // contributes nothing.  When every active slot has 0 <= R and L < N (always, for candidates at positive
            // lags) the bounds collapse into one per-side depth and the loads walk two pointers.
            const bool plain = !act || (R >= 0 && L < N);
            if (__all_sync(FULL, plain)) {
                const int Dl = D, Dr = min(D, N - 1 - R);
                const double* __restrict__ ql = y + (act ? L - li : 0);
                const double* __restrict__ qr = y + (act ? R + li : 0);
                for (int n = li; n <= Dmax; n += LS) {
                    const double yl = (n <= Dl) ? __ldg(ql) : 0.0;
                    const double yr = (n <= Dr) ? __ldg(qr) : 0.0;
                    ql -= LS;
                    qr += LS;
                    const double num = fma(yl * hl, tr, (yr * hr) * tl);
                    acc = fma(num, rcp_pos(tl * tr), acc);
                    const double nhl = fma(Kl, hl, Cl - hlp), nhr = fma(Kr, hr, Cr - hrp);
                    hlp = hl; hl = nhl; hrp = hr; hr = nhr;
                    tl += (double)LS; tr += (double)LS;
                }
            } else {
                for (int n = li; n <= Dmax; n += LS) {
                    const bool on = (n <= D);
                    int il = L - n;
                    il = il < 0 ? 0 : il;
                    int ir = R + n;
                    ir = ir < 0 ? 0 : ir;
                    const double yl = (on && il < N) ? __ldg(y + il) : 0.0;
                    const double yr = (on && ir < N) ? __ldg(y + ir) : 0.0;
                    const double num = fma(yl * hl, tr, (yr * hr) * tl);
                    acc = fma(num, rcp_pos(tl * tr), acc);
                    // advance: t += LS, Hann factors one recurrence step
                    const double nhl = fma(Kl, hl, Cl - hlp), nhr = fma(Kr, hr, Cr - hrp);
                    hlp = hl; hl = nhl; hrp = hr; hr = nhr;
                    tl += (double)LS; tr += (double)LS;
                }
            }
            acc *= sgn;
            acc += __shfl_xor_sync(FULL, acc, 1);
            const double ft = special ? sval : acc * (s0 * (1.0 / kPi));
            // ---- Brent update (periodic.rs:121-186) ---------------------------------------------------------------------
            if (!done) {
                if (iter == 0) {
                    fv = ft; fx = ft; fw = ft;
                    iter = 1;
                } else {
                    if (ft <= fx) {
                        if (t < x) b = x; else a = x;
                        v = w; w = x; x = t;
                        fv = fw; fw = fx; fx = ft;
                    } else {
                        if (t < x) a = t; else b = t;
                        if (ft <= fw || fabs(w - x) < EPS) {
                            v = w; w = t;
                            fv = fw; fw = ft;
                        } else if (ft <= fv || fabs(v - x) < EPS || fabs(v - w) < EPS) {
                            v = t;
                            fv = ft;
                        }
                    }
                    ++iter;
                }
                if (iter > 60) {
                    done = true; rx = x; ry = fx;
                } else {
                    const double range = b - a, middle_range = (a + b) * 0.5;
                    const double tol_act = sqrt_epsilon * fabs(x) + tol / 3.;
                    if (fabs(x - middle_range) + range * 0.5 <= 2. * tol_act) {
                        done = true; rx = x; ry = fx;
                    } else {
                        double new_step = (x < middle_range) ? golden * (b - x) : golden * (a - x);
                        if (fabs(x - w) >= tol_act) {
                            const double tt = (x - w) * (fx - fv);
                            double q = (x - v) * (fx - fw);
                            double p = (x - v) * q - (x - w) * tt;
                            q = 2. * q - tt;
                            if (q > 0.) p = -p; else q = -q;
                            if (fabs(p) < fabs(new_step * q) && p > q * (a - x + 2. * tol_act) && p < q * (b - x - 2. * tol_act))
                                new_step = p / q;
                        }
                        if (fabs(new_step) < tol_act) new_step = (new_step > 0.) ? tol_act : -tol_act;
                        t = x + new_step;
                    }
                }
            }
        }
            if (have && done) {
                if (li == 0) {
                    double xmid = rx + (double)offset, ymid = ry;
                    if (ymid > 1.) ymid = 1. / ymid;
                    P.refined[e] = make_double2(P.fs / xmid, ymid);
                }
                have = false;
            }
        }
    }
    }
}

// K8: append the unvoiced candidate ({0, threshold}, or {0, voiceless strength} with peaks), NaN check, stable sort by strength descending (periodic.rs:452-453)
__global__ void __launch_bounds__(128) pitch_finalize_kernel(const PitchParams P, void* cand_out, int max_cand, int32_t* n_cand_out,
                                                             uint8_t* status_out, int out_f64) {
    const int lane = threadIdx.x & 31;
    const int64_t fl = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // slab-local frame
    if (fl >= P.n_frames) return;
    const int64_t f = P.frame0 + fl;
    const int2 rg = P.range[fl];
    const double2* it = P.refined + rg.x;
    const int cnt = rg.y, total = cnt + 1;
    const unsigned FULL = 0xffffffffu;
    double unvoiced = P.threshold;
    if (P.local_peak) unvoiced = voiceless_strength(P.local_peak[f], P.global_peak[f / P.seg_frames], P.threshold, P.silence);
    auto item = [&](int i) -> double2 { return i < cnt ? it[i] : make_double2(0.0, unvoiced); };
    bool has_nan = false;
    for (int i = lane; i < total; i += 32) {
        const double s = item(i).y;
        has_nan = has_nan || (s != s);
    }
    has_nan = __any_sync(FULL, has_nan);
    auto put = [&](int slot, double2 v) {
        if (slot >= max_cand) return;
        if (out_f64) reinterpret_cast<double2*>(cand_out)[(size_t)f * max_cand + slot] = v;
        else reinterpret_cast<float2*>(cand_out)[(size_t)f * max_cand + slot] = make_float2((float)v.x, (float)v.y);
    };
    for (int i = lane; i < total; i += 32) {
        const double2 me = item(i);
        int rank = i;
        if (!has_nan) {
            rank = 0;
            for (int j = 0; j < total; ++j) {
                const double sj = item(j).y;
                rank += (sj > me.y || (sj == me.y && j < i)) ? 1 : 0;
            }
        }
        put(rank, me);
    }
    for (int s = total + lane; s < max_cand; s += 32) put(s, make_double2(0.0, 0.0));
    if (lane == 0) {
        if (n_cand_out) n_cand_out[f] = total;
        // the reference's sort panics on a NaN strength (partial_cmp().unwrap(), periodic.rs:453)
        if (status_out) status_out[f] = has_nan ? VBX_ERR_PITCH : VBX_OK;
    }
}

// batched stand-alone interpolate_sinc / improve_extremum: one warp per (series, point)
__global__ void __launch_bounds__(128) sinc_points_kernel(const double* __restrict__ y, long long n_series, long long y_len,
                                                          long long offset, long long nx, const double* __restrict__ x,
                                                          long long n_points, long long max_depth, double* out) {
    const int lane = threadIdx.x & 31;
    const long long e = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= n_series * n_points) return;
    const long long s = e / n_points;
    const double v = sinc_interp_warp(y + s * y_len, y_len, y_len, offset, nx, x[e], max_depth, lane);
    if (lane == 0) out[e] = v;
}

__global__ void __launch_bounds__(128) improve_points_kernel(const double* __restrict__ y, long long n_series, long long y_len,
                                                             long long offset, long long nx, const double* __restrict__ ixmid,
                                                             long long n_points, int interp, long long depth, int is_max,
                                                             double* xmid_out, double* ymid_out) {
    const int lane = threadIdx.x & 31;
    const long long e = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (e >= n_series * n_points) return;
    const long long s = e / n_points;
    double xm, ym;
    improve_extremum_warp(y + s * y_len, y_len, y_len, offset, nx, ixmid[e], interp, depth, is_max != 0, &xm, &ym, lane);
    if (lane == 0) { xmid_out[e] = xm; ymid_out[e] = ym; }
}

template <typename T>
__global__ void __launch_bounds__(256) pitch_extract_kernel(const T* __restrict__ cand, int64_t n_frames, int max_cand, T* out) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    out[2 * f] = cand[(size_t)f * max_cand * 2];
    out[2 * f + 1] = cand[(size_t)f * max_cand * 2 + 1];
}

// -------------------------------------------------------------------------------------------
// Viterbi pitch path (opt-in extension; SURVEY §8f rank 3).  The reference declares
// PitchExtractor::new(candidates, voiced_unvoiced_cost, voicing_threshold) and documents the intent — "a path through
// these candidates that maximizes both the smoothness of the pitch contour and the strength of the pitches"
// (periodic.rs:320-335, 394-395) — but implements arg-max.  This is Boersma's (1993) path finder over the candidate
// lists vbx_pitch returns: maximise Σ_f local(f, k_f) − Σ_f transition(k_{f−1}, k_f) with
//   local      = strength                                  (unvoiced candidate: its strength = the voicing threshold)
//                − octave_cost·log2(ceiling / frequency)    (voiced candidates only)
//   transition = 0 (both unvoiced) | voiced_unvoiced_cost (one voiced) | octave_jump_cost·|log2(f1/f2)| (both voiced).
// All three costs zero ⇒ the per-frame arg-max, i.e. PitchExtractor as the reference implements it.
// One warp per utterance: lane j owns candidate j of the current frame, the previous frame's scores travel by shuffle;
// back-pointers go to a scratch [F][32] byte array; lane 0 backtracks.  Ties keep the lower index.
// -------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) pitch_viterbi_kernel(const T* __restrict__ cand, const int32_t* __restrict__ n_cand, int64_t n_segments,
                                                            int64_t seg_frames, int K, double vuc, double ojc, double oc, double ceiling,
                                                            uint8_t* __restrict__ psi, T* __restrict__ path_out, int32_t* __restrict__ index_out) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= n_segments) return;
    const int64_t f0 = u * seg_frames;
    const double NEG = -1.0e300;
    double delta = NEG, lf = 0.0;  // best score of a path ending in this lane's candidate; log2 of its frequency
    bool voiced = false;
    int kprev = 0;
    for (int64_t j = 0; j < seg_frames; ++j) {
        const int64_t f = f0 + j;
        int kc = n_cand ? n_cand[f] : K;
        kc = kc < K ? kc : K;
        kc = kc < 32 ? kc : 32;
        double freq = 0.0, strength = 0.0;
        if (lane < kc) {
            freq = (double)cand[((size_t)f * K + lane) * 2];
            strength = (double)cand[((size_t)f * K + lane) * 2 + 1];
        }
        const bool v = freq > 0.0;
        const double my_lf = v ? log2(freq) : 0.0;
        const double local = (lane < kc) ? (v ? strength - oc * (log2(ceiling) - my_lf) : strength) : NEG;
        double best = (j == 0) ? 0.0 : NEG;
        int arg = 0;
        for (int k = 0; k < kprev; ++k) {
            const double dk = __shfl_sync(FULL, delta, k);
            const double lk = __shfl_sync(FULL, lf, k);
            const bool vk = __shfl_sync(FULL, voiced ? 1 : 0, k) != 0;
            const double tr = (v && vk) ? ojc * fabs(lk - my_lf) : ((v || vk) ? vuc : 0.0);
            const double sc = dk - tr;
            if (sc > best) { best = sc; arg = k; }
        }
        delta = (lane < kc) ? best + local : NEG;
        lf = my_lf;
        voiced = v;
        kprev = kc;
        psi[(size_t)f * 32 + lane] = (uint8_t)arg;
    }
    if (seg_frames == 0) return;
    // best final state (lowest index among equals), then backtrack
    double m = delta;
    int mi = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double om = __shfl_xor_sync(FULL, m, o);
        const int oi = __shfl_xor_sync(FULL, mi, o);
        if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
    }
    __syncwarp();
    if (lane == 0) {
        int k = mi;
        for (int64_t j = seg_frames - 1; j >= 0; --j) {
            const int64_t f = f0 + j;
            if (index_out) index_out[f] = k;
            if (path_out) {
                path_out[2 * f] = cand[((size_t)f * K + k) * 2];
                path_out[2 * f + 1] = cand[((size_t)f * K + k) * 2 + 1];
            }
            k = psi[(size_t)f * 32 + k];
        }
    }
}

constexpr int kMaxPitchFrameLen = 16384;

// Peak inputs of vbx_pitch_with_peaks: silence > 0 turns them on; a null local / global array is computed on the device.
struct PitchPeaks {
    double silence = 0.0;
    const double* local = nullptr;   // [F]
    const double* global = nullptr;  // [n_segments]
};

template <typename TIn>
int launch_pitch(vbx_ctx* ctx, const vbx_frames* fr, double fs, double threshold, double fmin, double fmax, int max_cand,
                 void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int out_dtype, double* lag_out, const PitchPeaks& peaks) {
    const int n = fr->frame_len;
    const double* win = nullptr;
    const double* lagwin = nullptr;
    int st = vbx_get_window(ctx, fr->window, n, &win, fr->dtype);
    if (st != VBX_OK) return st;
    st = vbx_get_window(ctx, VBX_WINDOW_HANN_LAG, n, &lagwin);
    if (st != VBX_OK) return st;

    PitchParams P;
    memset(&P, 0, sizeof(P));
    P.base = fr->base; P.win = win; P.lagwin = lagwin;
    P.stride = fr->frame_stride;
    P.seg_frames = vbx_frames_per_segment(fr);
    P.seg_stride = fr->frames_per_segment > 0 ? fr->segment_stride : 0;
    P.n = n; P.n16 = (n + 15) & ~15;
    P.G = P.n16 / 16;
    P.lpf = (P.G + 1) / 2;
    P.ixmax = n / 2;
    P.fs = fs; P.fmin = fmin; P.fmax = fmax; P.threshold = threshold;
    P.work = vbx_work_ptr(ctx);
    int T = 0;
    for (int p = 0; p < P.lpf; ++p) {
        const int gA = p, gB = P.G - 1 - p;
        auto steps = [&](int g) { const int len = n - 16 * g; return len > 0 ? (len + 7) / 8 : 0; };
        const int t = steps(gA) + (gB > gA ? steps(gB) : 0);
        if (t > T) T = t;
    }
    P.T = T;
    // frame buffer: f64 with 2 pad doubles per 16 (xs_words counts doubles)
    P.xs_words = ((P.n16 + 48) * 9) / 8;
    // frames per CTA: fill ~160 threads, bounded by shared memory (<= 56 KB so that 4 CTAs fit an SM)
    int fpc = 160 / P.lpf;
    if (fpc < 1) fpc = 1;
    const size_t frame_bytes = (size_t)P.xs_words * sizeof(double);
    while (fpc > 1 && fpc * frame_bytes > 56 * 1024) --fpc;
    P.fpc = fpc;
    int threads = ((fpc * P.lpf + 31) / 32) * 32;
    if (threads < 64) threads = 64;
    const size_t smem = fpc * frame_bytes;
    VBX_REQUIRE(ctx, smem <= ctx->smem_optin && threads <= 512, "frame_len %d does not fit the pitch kernel", n);
    void (*lag_kernel)(const PitchParams) = threads <= 160   ? pitch_lag64_kernel<TIn, 160>
                                            : threads <= 256 ? pitch_lag64_kernel<TIn, 256>
                                                             : pitch_lag64_kernel<TIn, 512>;
    VBX_CUDA(ctx, cudaFuncSetAttribute(lag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    // scratch per frame: y [N] f64 + worst-case candidate capacity (every other lag below N/2 a maximum)
    const int cap = P.ixmax / 2 + 1;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t per_frame = (size_t)n * 8 + (size_t)cap * (sizeof(PitchCand) + sizeof(double2)) + sizeof(int2);
    size_t budget = (size_t)2 << 30;
    if (const char* e = getenv("VBX_PITCH_SLAB_MB")) budget = (size_t)atoll(e) << 20;
    int64_t slab = (int64_t)(budget / per_frame);
    if (slab < 1) slab = 1;
    if (slab > fr->n_frames) slab = fr->n_frames;
    const size_t y_bytes = al((size_t)slab * n * 8), list_bytes = al((size_t)slab * cap * sizeof(PitchCand)),
                 ref_bytes = al((size_t)slab * cap * sizeof(double2)), range_bytes = al((size_t)slab * sizeof(int2));
    // peaks the caller did not pass are computed once for the whole batch (the finalize kernel of every slab reads them)
    const bool with_peaks = peaks.silence > 0.0;
    const int64_t n_segs = fr->n_frames / P.seg_frames;
    const size_t local_bytes = (with_peaks && !peaks.local) ? al((size_t)fr->n_frames * sizeof(double)) : 0;
    const size_t global_bytes = (with_peaks && !peaks.global) ? al((size_t)n_segs * sizeof(double)) : 0;
    st = vbx_arena_reserve(ctx, y_bytes + list_bytes + ref_bytes + range_bytes + 256 + local_bytes + global_bytes);
    if (st != VBX_OK) return st;
    char* ptr = (char*)ctx->arena;
    P.y = (double*)ptr; ptr += y_bytes;
    P.list = (PitchCand*)ptr; ptr += list_bytes;
    P.refined = (double2*)ptr; ptr += ref_bytes;
    P.range = (int2*)ptr; ptr += range_bytes;
    P.counter = (unsigned long long*)ptr; ptr += 256;
    VBX_REQUIRE(ctx, (int64_t)slab * cap < 0x7fffffffLL, "pitch slab too large");
    if (with_peaks) {
        double* local = local_bytes ? (double*)ptr : nullptr;
        double* global = global_bytes ? (double*)(ptr + local_bytes) : nullptr;
        st = vbx_launch_frame_peaks(ctx, fr, local, global);
        if (st != VBX_OK) return st;
        P.local_peak = peaks.local ? peaks.local : local;
        P.global_peak = peaks.global ? peaks.global : global;
        P.silence = peaks.silence;
    }

    for (int64_t f0 = 0; f0 < fr->n_frames; f0 += slab) {
        P.frame0 = f0;
        P.n_frames = (fr->n_frames - f0 < slab) ? fr->n_frames - f0 : slab;
        VBX_CUDA(ctx, cudaMemsetAsync(P.counter, 0, 2 * sizeof(unsigned long long), ctx->stream));
        const int64_t grid = (P.n_frames + fpc - 1) / fpc;
        VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
        lag_kernel<<<(unsigned)grid, threads, smem, ctx->stream>>>(P);
        VBX_CHECK_LAUNCH(ctx, "pitch_lag64_kernel");
        if (lag_out) {  // vbx_pitch_lag_function: hand the lag function out and stop here
            VBX_CUDA(ctx, cudaMemcpyAsync(lag_out + (size_t)f0 * n, P.y, (size_t)P.n_frames * n * sizeof(double), cudaMemcpyDeviceToDevice,
                                          ctx->stream));
            continue;
        }
        static const int resident = [] {  // CTAs of the refinement kernel that fit one SM (computed once, thread-safely)
            int r = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&r, pitch_refine8q_kernel, 128, 0) != cudaSuccess || r < 1) {
                cudaGetLastError();
                r = 4;
            }
            return r;
        }();
        pitch_refine8q_kernel<<<ctx->sm_count * resident, 128, 0, ctx->stream>>>(P);
        VBX_CHECK_LAUNCH(ctx, "pitch_refine8q_kernel");
        pitch_finalize_kernel<<<(unsigned)((P.n_frames + 3) / 4), 128, 0, ctx->stream>>>(P, cand_out, max_cand, n_cand_out,
                                                                                        status_out, out_dtype == VBX_F64);
        VBX_CHECK_LAUNCH(ctx, "pitch_finalize_kernel");
    }
    return VBX_OK;
}

int pitch_check(vbx_ctx* ctx, const vbx_frames* fr, int max_cand, const void* cand_out, int out_dtype) {
    int st = vbx_check_frames(ctx, fr, /*allow_f64=*/true);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, out_dtype == VBX_F32 || out_dtype == VBX_F64, "out_dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, max_cand >= 1, "max_candidates must be >= 1 (the unvoiced candidate always exists)");
    VBX_REQUIRE(ctx, fr->frame_len >= 2, "frame_len must be >= 2");
    VBX_REQUIRE(ctx, fr->frame_len <= kMaxPitchFrameLen, "frame_len > %d is not supported by the pitch path", kMaxPitchFrameLen);
    VBX_REQUIRE(ctx, fr->n_frames == 0 || cand_out != nullptr, "cand_out is NULL");
    return VBX_OK;
}

// The sample dtype picks the instantiation; every pitch entry point launches through here.
int launch_pitch_any(vbx_ctx* ctx, const vbx_frames* fr, double fs, double threshold, double fmin, double fmax, int max_cand,
                     void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int out_dtype, double* lag_out, const PitchPeaks& peaks) {
    cudaSetDevice(ctx->device);
    vbx_frames pv;  // the planar equivalent of an interleaved view
    const int st = vbx_planarize(ctx, fr, &pv);
    if (st != VBX_OK) return st;
    fr = &pv;
    if (fr->dtype == VBX_MULAW8)
        return launch_pitch<vbx_mulaw8>(ctx, fr, fs, threshold, fmin, fmax, max_cand, cand_out, n_cand_out, status_out, out_dtype,
                                        lag_out, peaks);
    if (fr->dtype == VBX_ALAW8)
        return launch_pitch<vbx_alaw8>(ctx, fr, fs, threshold, fmin, fmax, max_cand, cand_out, n_cand_out, status_out, out_dtype,
                                       lag_out, peaks);
    if (fr->dtype == VBX_I16)
        return launch_pitch<int16_t>(ctx, fr, fs, threshold, fmin, fmax, max_cand, cand_out, n_cand_out, status_out, out_dtype, lag_out,
                                     peaks);
    if (fr->dtype == VBX_F64)  // f64 samples (a frame the caller windowed in f64, as the reference's callers do)
        return launch_pitch<double>(ctx, fr, fs, threshold, fmin, fmax, max_cand, cand_out, n_cand_out, status_out, out_dtype, lag_out,
                                    peaks);
    return launch_pitch<float>(ctx, fr, fs, threshold, fmin, fmax, max_cand, cand_out, n_cand_out, status_out, out_dtype, lag_out, peaks);
}

}  // namespace

extern "C" {

int vbx_pitch(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold, double min_hz, double max_hz,
              int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int32_t out_dtype) {
    return vbx_pitch_with_peaks(ctx, frames, sample_rate, threshold, 0.0, nullptr, nullptr, min_hz, max_hz, max_candidates, cand_out,
                                n_cand_out, status_out, out_dtype);
}

// vbx_pitch with the reference's local_peak / global_peak honoured (periodic.rs:357; Boersma 1993): the unvoiced candidate's
// strength is voiceless_strength(local peak of the frame, global peak of its segment) instead of the threshold.
// silence_threshold == 0 is vbx_pitch itself (no peaks are read or computed).
int vbx_pitch_with_peaks(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold, double silence_threshold,
                         const double* local_peaks, const double* global_peaks, double min_hz, double max_hz, int32_t max_candidates,
                         void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = pitch_check(ctx, frames, max_candidates, cand_out, out_dtype);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, silence_threshold >= 0.0, "silence_threshold must be >= 0");
    if (frames->n_frames == 0) return VBX_OK;
    PitchPeaks pk;
    if (silence_threshold > 0.0) {
        pk.silence = silence_threshold;
        pk.local = local_peaks;
        pk.global = global_peaks;
    }
    return launch_pitch_any(ctx, frames, sample_rate, threshold, min_hz, max_hz, max_candidates, cand_out, n_cand_out, status_out,
                            out_dtype, nullptr, pk);
}

// The host pipeline cuts a segmented view into whole segments, so every chunk computes its segments' global peaks itself.  It
// cuts a single-segment view into frame ranges, and the channels of an interleaved recording into time ranges, so there the
// global peak of every segment is taken here, on the host, over its whole channel before the pipeline starts.  Caller-supplied
// peaks are uploaded once and every chunk reads its rows (a time chunk gathers its [U][J'] block of local peaks first).
int vbx_pitch_with_peaks_host(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold, double silence_threshold,
                              const double* local_peaks, const double* global_peaks, double min_hz, double max_hz,
                              int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int32_t out_dtype) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = pitch_check(ctx, frames, max_candidates, cand_out, out_dtype);
    if (st != VBX_OK) return st;
    VBX_REQUIRE(ctx, silence_threshold >= 0.0, "silence_threshold must be >= 0");
    if (frames->n_frames == 0) return VBX_OK;
    cudaSetDevice(ctx->device);
    const bool with_peaks = silence_threshold > 0.0;
    const bool segmented = frames->frames_per_segment > 0;
    const bool by_time = vbx_chunk_by_time(frames);
    const int64_t F = frames->n_frames, J = vbx_frames_per_segment(frames), n_segs = F / J;
    std::vector<double> whole;
    const double* global_src = with_peaks ? global_peaks : nullptr;
    if (with_peaks && !global_peaks && (!segmented || by_time)) {
        for (int64_t u = 0; u < n_segs; ++u) whole.push_back(vbx_host_peak(frames, u));
        global_src = whole.data();
    }
    const double* local_src = with_peaks ? local_peaks : nullptr;
    const size_t n_local = local_src ? (size_t)F : 0, n_global = global_src ? (size_t)n_segs : 0;
    const size_t n_chunk_local = by_time ? n_local : 0;  // a time chunk's local peaks, gathered from the [U][J] rows
    double* dev = nullptr;
    if (n_local + n_global > 0) {
        VBX_CUDA(ctx, cudaMalloc(&dev, (n_local + n_global + n_chunk_local) * sizeof(double)));
        cudaError_t e = cudaSuccess;
        if (n_local) e = cudaMemcpyAsync(dev, local_src, n_local * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess && n_global)
            e = cudaMemcpyAsync(dev + n_local, global_src, n_global * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) {
            cudaStreamSynchronize(ctx->stream);
            cudaFree(dev);
            return vbx_fail(ctx, VBX_ERR_CUDA, "peak upload failed: %s", cudaGetErrorString(e));
        }
    }
    const double* d_local = n_local ? dev : nullptr;
    const double* d_global = n_global ? dev + n_local : nullptr;
    const size_t pair = (out_dtype == VBX_F64) ? 16 : 8;
    vbx_host_out outs[3] = {{cand_out, (size_t)max_candidates * pair, nullptr}, {n_cand_out, 4, nullptr}, {status_out, 1, nullptr}};
    // chunked H2D / kernels / D2H pipeline (vbx_pipeline.cuh); output rows are indexed from the chunk's first frame
    const int rc = vbx_run_chunked(ctx, frames, outs, 3, [&](const vbx_frames* dfr, int64_t f0, int64_t u0, vbx_host_out* o) -> int {
        const double* chunk_local = d_local ? d_local + f0 : nullptr;
        if (d_local && by_time) {  // rows u*J + f0 .. of every segment u -> [U][J'] (the compute stream runs chunks in order)
            double* dst = dev + n_local + n_global;
            const int64_t jc = dfr->frames_per_segment;
            VBX_CUDA(ctx, cudaMemcpy2DAsync(dst, (size_t)jc * sizeof(double), d_local + f0, (size_t)J * sizeof(double),
                                            (size_t)jc * sizeof(double), (size_t)n_segs, cudaMemcpyDeviceToDevice, ctx->stream));
            chunk_local = dst;
        }
        return vbx_pitch_with_peaks(ctx, dfr, sample_rate, threshold, silence_threshold, chunk_local,
                                    d_global ? d_global + u0 : nullptr, min_hz, max_hz, max_candidates, o[0].dev, (int32_t*)o[1].dev,
                                    (uint8_t*)o[2].dev, out_dtype);
    }, 0, (size_t)96 << 20);  // compute-bound: the copies hide behind the kernels anyway, larger chunks mean fewer kernel tails
    if (dev) cudaFree(dev);  // the pipeline has drained the stream
    return rc;
}

// periodic.rs:403-408: the lag function `self_lag` the candidates are read from — autocorrelate(N), normalize, divide by the
// lag window — for every frame: lag_out [F][N] f64 (the reference then zero-extends it to 2N, :411).
int vbx_pitch_lag_function(vbx_ctx* ctx, const vbx_frames* frames, double* lag_out) {
    if (!ctx) return VBX_ERR_BADARG;
    int st = pitch_check(ctx, frames, 1, lag_out, VBX_F64);
    if (st != VBX_OK) return st;
    if (frames->n_frames == 0) return VBX_OK;
    return launch_pitch_any(ctx, frames, 1.0, 0.0, 0.0, 0.0, 1, nullptr, nullptr, nullptr, VBX_F64, lag_out, PitchPeaks());
}

int vbx_pitch_host(vbx_ctx* ctx, const vbx_frames* frames, double sample_rate, double threshold, double min_hz, double max_hz,
                   int32_t max_candidates, void* cand_out, int32_t* n_cand_out, uint8_t* status_out, int32_t out_dtype) {
    return vbx_pitch_with_peaks_host(ctx, frames, sample_rate, threshold, 0.0, nullptr, nullptr, min_hz, max_hz, max_candidates,
                                     cand_out, n_cand_out, status_out, out_dtype);
}

int vbx_pitch_extract(vbx_ctx* ctx, const void* cand, int32_t dtype, int64_t n_frames, int32_t max_candidates, void* out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_frames >= 0 && max_candidates >= 1, "bad sizes");
    if (n_frames == 0) return VBX_OK;
    VBX_REQUIRE(ctx, cand && out, "cand / out is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_frames + 255) / 256;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many frames for one launch");
    if (dtype == VBX_F64)
        pitch_extract_kernel<double><<<(unsigned)grid, 256, 0, ctx->stream>>>((const double*)cand, n_frames, max_candidates, (double*)out);
    else
        pitch_extract_kernel<float><<<(unsigned)grid, 256, 0, ctx->stream>>>((const float*)cand, n_frames, max_candidates, (float*)out);
    VBX_CHECK_LAUNCH(ctx, "pitch_extract_kernel");
    return VBX_OK;
}

int vbx_pitch_viterbi(vbx_ctx* ctx, const void* cand, int32_t dtype, const int32_t* n_cand, int64_t n_segments,
                      int64_t frames_per_segment, int32_t max_candidates, double voiced_unvoiced_cost, double octave_jump_cost,
                      double octave_cost, double ceiling_hz, void* path_out, int32_t* index_out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, dtype == VBX_F32 || dtype == VBX_F64, "dtype must be VBX_F32 or VBX_F64");
    VBX_REQUIRE(ctx, n_segments >= 0 && frames_per_segment >= 0, "negative counts");
    VBX_REQUIRE(ctx, max_candidates >= 1, "max_candidates must be >= 1");
    VBX_REQUIRE(ctx, ceiling_hz > 0.0, "ceiling_hz must be > 0");
    const int64_t F = n_segments * frames_per_segment;
    if (F == 0) return VBX_OK;
    VBX_REQUIRE(ctx, cand != nullptr && (path_out || index_out), "cand / outputs are NULL");
    cudaSetDevice(ctx->device);
    int st = vbx_arena_reserve(ctx, (size_t)F * 32);
    if (st != VBX_OK) return st;
    const int64_t grid = (n_segments + 3) / 4;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many segments for one launch");
    if (dtype == VBX_F64)
        pitch_viterbi_kernel<double><<<(unsigned)grid, 128, 0, ctx->stream>>>((const double*)cand, n_cand, n_segments, frames_per_segment,
                                                                           max_candidates, voiced_unvoiced_cost, octave_jump_cost, octave_cost,
                                                                           ceiling_hz, (uint8_t*)ctx->arena, (double*)path_out, index_out);
    else
        pitch_viterbi_kernel<float><<<(unsigned)grid, 128, 0, ctx->stream>>>((const float*)cand, n_cand, n_segments, frames_per_segment,
                                                                          max_candidates, voiced_unvoiced_cost, octave_jump_cost, octave_cost,
                                                                          ceiling_hz, (uint8_t*)ctx->arena, (float*)path_out, index_out);
    VBX_CHECK_LAUNCH(ctx, "pitch_viterbi_kernel");
    return VBX_OK;
}

int vbx_interpolate_sinc(vbx_ctx* ctx, const double* y, int64_t n_series, int64_t y_len, int64_t offset, int64_t nx,
                         const double* x, int64_t n_points, int64_t max_depth, double* out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, n_series >= 0 && n_points >= 0 && y_len >= 1 && max_depth >= 0, "bad sizes");
    if (n_series == 0 || n_points == 0) return VBX_OK;
    VBX_REQUIRE(ctx, y && x && out, "y / x / out is NULL");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_series * n_points + 3) / 4;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many points for one launch");
    sinc_points_kernel<<<(unsigned)grid, 128, 0, ctx->stream>>>(y, n_series, y_len, offset, nx, x, n_points, max_depth, out);
    VBX_CHECK_LAUNCH(ctx, "sinc_points_kernel");
    return VBX_OK;
}

int vbx_improve_extremum(vbx_ctx* ctx, const double* y, int64_t n_series, int64_t y_len, int64_t offset, int64_t nx,
                         const double* ixmid, int64_t n_points, int32_t interpolation, int64_t sinc_depth, int32_t is_max,
                         double* xmid_out, double* ymid_out) {
    if (!ctx) return VBX_ERR_BADARG;
    VBX_REQUIRE(ctx, n_series >= 0 && n_points >= 0 && y_len >= 1 && sinc_depth >= 0, "bad sizes");
    VBX_REQUIRE(ctx, interpolation >= 0 && interpolation <= 2, "interpolation must be 0 (None), 1 (Parabolic) or 2 (Sinc)");
    if (n_series == 0 || n_points == 0) return VBX_OK;
    VBX_REQUIRE(ctx, y && ixmid && xmid_out && ymid_out, "NULL pointer");
    cudaSetDevice(ctx->device);
    const int64_t grid = (n_series * n_points + 3) / 4;
    VBX_REQUIRE(ctx, grid <= 0x7fffffffLL, "too many points for one launch");
    improve_points_kernel<<<(unsigned)grid, 128, 0, ctx->stream>>>(y, n_series, y_len, offset, nx, ixmid, n_points, interpolation,
                                                                   sinc_depth, is_max, xmid_out, ymid_out);
    VBX_CHECK_LAUNCH(ctx, "improve_points_kernel");
    return VBX_OK;
}

}  // extern "C"
