// vbx_pitch_lag64.cuh — the all-lag autocorrelation of the pitch path in fp64 (periodic.rs:279-288 with L = N lags,
// then :403-439).  Included inside the anonymous namespace of vbx_pitch.cu after PitchParams.
//
// A lane owns a 16-lag group and walks the frame in 8-sample steps, group g paired with group G−1−g on the same lane so
// every lane runs the same number of steps.  The windowed samples stay the exact f64 products x·w the reference forms and
// every lag product is one DFMA into a single f64 accumulator per lag, summed in ascending i like the reference's fold.
// What is left against the oracle is the fused-multiply-add rounding (≈ 1e-16·r[0]); an fp32 sweep leaves ≈ 3e-8·r[0]
// in the lag function, which Brent on a flat, mirrored interpolant amplifies into > 0.1 Hz on 0.3 % of the weak
// (below-threshold) list entries (DESIGN.md §K6).
//
// Shared memory: the frame as doubles with 2 pad doubles per 16 (chunk k of 8 doubles starts at 8k + 2·(k >> 1)), so
// the lanes of a quarter-warp — consecutive lag groups, 16 doubles apart — read their 16-byte pieces from 8 different
// bank groups.  The 24-sample window of a lane (b0, b1, b2: three chunks of 8) rotates by renaming: the step loop is
// unrolled three times, there are no register moves.  Per step and lane: 128 DFMA, 8 LDS.128.
struct D8 {
    double2 a, b, c, d;
};

__device__ __forceinline__ int dchunk_addr(int k) { return 8 * k + 2 * (k >> 1); }   // in doubles
__device__ __forceinline__ int dword_addr(int w) { return w + 2 * (w >> 4); }

__device__ __forceinline__ void d8_load(const double* xs, int k, D8& v) {
    const double2* p = reinterpret_cast<const double2*>(xs + dchunk_addr(k));
    v.a = p[0];
    v.b = p[1];
    v.c = p[2];
    v.d = p[3];
}

// acc[j] += Σ_ii a[ii]·w[ii + j], w = the 24 samples (lo, mid, hi)
__device__ __forceinline__ void lag_step64(double (&acc)[16], const D8& A, const D8& lo, const D8& mid, const D8& hi) {
    const double a[8] = {A.a.x, A.a.y, A.b.x, A.b.y, A.c.x, A.c.y, A.d.x, A.d.y};
    const double w[24] = {lo.a.x,  lo.a.y,  lo.b.x,  lo.b.y,  lo.c.x,  lo.c.y,  lo.d.x,  lo.d.y,  mid.a.x, mid.a.y, mid.b.x, mid.b.y,
                          mid.c.x, mid.c.y, mid.d.x, mid.d.y, hi.a.x,  hi.a.y,  hi.b.x,  hi.b.y,  hi.c.x,  hi.c.y,  hi.d.x,  hi.d.y};
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) acc[jj] = fma(a[ii], w[ii + jj], acc[jj]);
    }
}

// CTA-size class MAXT, the smallest that holds a CTA's fpc·lpf lanes (launch_pitch picks it from the frame length):
//   160: frame lengths up to 5 120 samples, four CTAs per SM (96 registers);
//   256: up to 8 192, one CTA per SM (108 registers);
//   512: up to 16 384, the longest frame vbx_pitch accepts, one CTA per SM (106 registers).
template <typename TIn, int MAXT>
__global__ void __launch_bounds__(MAXT, MAXT == 160 ? 4 : 1) pitch_lag64_kernel(const PitchParams P) {
    extern __shared__ __align__(16) double xd_all[];
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int n = P.n;
    const int64_t f_first = (int64_t)blockIdx.x * P.fpc;                  // slab-local frame index
    const int nf = (int)min((int64_t)P.fpc, P.n_frames - f_first);

    // ---- stage: xs[q][dword_addr(i)] = x[i]·w[i] (exact f64 product of an fp32 sample and the f64 window), zeros beyond N
    const int span = P.n16 + 48;
    for (int q = 0; q < nf; ++q) {
        const int64_t f = P.frame0 + f_first + q;
        const int64_t seg = f / P.seg_frames;
        const TIn* __restrict__ x = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride + (f - seg * P.seg_frames) * P.stride;
        double* xs = xd_all + (size_t)q * P.xs_words;
        for (int i = tid; i < span; i += nthreads) {
            double v = 0.0;
            if (i < n) v = vbx_load_sample_d<TIn>(x + i) * __ldg(P.win + i);
            xs[dword_addr(i)] = v;
        }
    }
    __syncthreads();

    // ---- lag sweep ------------------------------------------------------------------------------------------
    const int q = tid / P.lpf, p = tid - q * P.lpf;
    if (q < nf) {
        const double* xs = xd_all + (size_t)q * P.xs_words;
        double* yrow = P.y + (size_t)(f_first + q) * n;
        const int gA = p, gB = P.G - 1 - p;
        const int nA = lag_steps(n, gA), nB = (gB > gA) ? lag_steps(n, gB) : 0;
        const double x0 = xs[0];
        double acc[16];
        D8 b0, b1, b2;
        int g = gA, left = nA, c = 0, cstep = 1, phase = 0;
        const int zero_chunk = (P.n16 + 16) >> 3;  // a chunk of zeros (doubles n16+16 .. n16+23)
        auto reset = [&]() {
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[j] = 0.0;
        };
        auto store_group = [&]() {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int lag = 16 * g + j;
                if (lag < n) {
                    double r = acc[j];
                    // r_ref[lag] = x0 + Σ_{i>=1} (periodic.rs:284): remove the i = 0 product, add the seed
                    if (x0 != 0.0) r = r - x0 * xs[dword_addr(lag)] + x0;
                    yrow[lag] = r;
                }
            }
        };
        reset();
        if (left == 0) phase = 2;
        // One step with the window registers in the roles (lo, mid, hi = the chunk loaded in this step).  A lane whose
        // group is finished stores it and starts its second group (or idles on the zero chunk) inside the same loop, so
        // all lanes of the CTA run the same number of steps.
#define VBX_LAG64_STEP(LO, MID, HI)                                                        \
    {                                                                                      \
        if (left == 0 && phase < 2) {                                                      \
            store_group();                                                                 \
            if (phase == 0 && nB > 0) {                                                    \
                phase = 1; g = gB; left = nB; c = 0;                                       \
                reset();                                                                   \
                d8_load(xs, 2 * g, LO);                                                    \
                d8_load(xs, 2 * g + 1, MID);                                               \
            } else {                                                                       \
                phase = 2;                                                                 \
            }                                                                              \
        }                                                                                  \
        if (phase == 2) { c = zero_chunk; cstep = 0; g = 0; left = 0x3fffffff; }           \
        D8 av;                                                                             \
        d8_load(xs, c, av);                                                                \
        d8_load(xs, c + 2 * g + 2, HI);                                                    \
        lag_step64(acc, av, LO, MID, HI);                                                  \
        c += cstep;                                                                        \
        --left;                                                                            \
    }
        d8_load(xs, c + 2 * g, b0);
        d8_load(xs, c + 2 * g + 1, b1);
        for (int s = 0; s < P.T; s += 3) {
            VBX_LAG64_STEP(b0, b1, b2)
            VBX_LAG64_STEP(b1, b2, b0)
            VBX_LAG64_STEP(b2, b0, b1)
        }
#undef VBX_LAG64_STEP
        if (phase < 2 && left <= 0) store_group();
    }
    __syncthreads();
    pitch_lag_post(P, reinterpret_cast<unsigned char*>(xd_all), (size_t)P.xs_words * sizeof(double), f_first, nf);
}
