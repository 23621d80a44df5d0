// vbx_lpc16.cuh — the fused window → fp64 autocorrelation → Levinson kernel for 16-sample-aligned framings
// (frame length and hop multiples of 16, at most 16 lags: the C2 shape, 400/160/13).  Included inside the
// anonymous namespace of vbx_lpc.cu after LpcParams / levinson / lpc_finish.
//
// Same arithmetic as lpc_fused_kernel (window multiply and lag products in fp64, the x[0]-seeded fold of
// periodic.rs:279-288), different walk: two lanes per frame, each consumes whole chunks of 16 samples with a
// 16-slot register ring, so that
//   * samples arrive as 4 LDS.128 and window values as 8 LDS.128 per chunk (0.75 loads per sample instead of 2),
//   * there is no tail chunk, no pad word inside a chunk (pads are 4 words after every `sv` samples and
//     sv % 16 == 0) and no separate history loop: the lane of the second half starts one or two chunks early
//     and only fills its ring from those pre-roll chunks (window multiply, no lag products).
// The two halves of a frame live in different warps (even warps: first chunks of 32 frames, odd warps: the
// rest), so the pre-roll is warp-uniform; the halves meet in shared memory.  The 8 lanes of a quarter-warp (one
// LDS.128 wavefront) hold 8 consecutive frames, whose chunk addresses differ by sv + 4 words = an odd number of
// 16-byte bank groups: conflict-free.

constexpr int kChunk = 16;

template <typename TIn>
__device__ __forceinline__ void stage_span16(const LpcParams& P, const TIn* __restrict__ base, int64_t j0, int Gc, float* s_span) {
    const int tid = threadIdx.x, nthreads = P.threads;
    const int n = P.n, sv = P.sv, pad = P.pad;
    if (P.stride <= (int64_t)n) {
        const TIn* src = base + j0 * P.stride;
        const int total = (Gc - 1) * sv + n;
        const unsigned magic = P.sv_magic;
        auto phys = [&](int s_) -> int { return s_ + pad * (int)__umulhi((unsigned)s_, magic); };
        int done = 0;
        if (sizeof(TIn) == 4 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            const float4* src4 = reinterpret_cast<const float4*>(src);
            const int n4 = total >> 2;  // total % 16 == 0
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
                    if (v < n4) *reinterpret_cast<float4*>(s_span + phys(4 * v)) = a[u];
                }
            }
            done = n4 << 2;
        }
        if (sizeof(TIn) == 2 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            // int16 PCM: 16-byte loads of 8 samples (never straddling a pad: sv % 8 == 0)
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
                        float4* dst = reinterpret_cast<float4*>(s_span + phys(8 * v));
                        dst[0] = make_float4((float)(short)(a[u].x & 0xffffu), (float)(short)(a[u].x >> 16),
                                             (float)(short)(a[u].y & 0xffffu), (float)(short)(a[u].y >> 16));
                        dst[1] = make_float4((float)(short)(a[u].z & 0xffffu), (float)(short)(a[u].z >> 16),
                                             (float)(short)(a[u].w & 0xffffu), (float)(short)(a[u].w >> 16));
                    }
                }
            }
            done = n8 << 3;
        }
        if constexpr (vbx_g711<TIn>::value) {
            if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
                // G.711: 16-byte loads of 16 codes, decoded as they land (never straddling a pad: sv % 16 == 0)
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
                            float4* dst = reinterpret_cast<float4*>(s_span + phys(16 * v));
#pragma unroll
                            for (int e = 0; e < 4; ++e) dst[e] = make_float4(x[4 * e], x[4 * e + 1], x[4 * e + 2], x[4 * e + 3]);
                        }
                    }
                }
                done = n16 << 4;
            }
        }
        for (int s0 = done + tid; s0 < total; s0 += 8 * nthreads) {  // unaligned base pointer
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
        // gapped frames: each frame's n samples land in consecutive blocks of sv == n words (+ pad)
        const int warp = tid >> 5, lane = tid & 31;
        for (int g = warp; g < Gc; g += nthreads / 32) {
            const TIn* src = base + (j0 + g) * P.stride;
            for (int j = lane; j < n; j += 32) s_span[g * (sv + pad) + j] = vbx_load_sample<TIn>(src + j);
        }
    }
}

template <int L, typename TIn>
__global__ void __maxnreg__(96) lpc_fused16_kernel(const LpcParams P) {
    static_assert(L >= 2 && L <= kChunk, "ring of 16 slots holds at most 16 lags");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_win = reinterpret_cast<double*>(smem_raw);                 // [n], n % 16 == 0
    float* s_span = reinterpret_cast<float*>(s_win + P.n);               // padded span
    double* s_out = reinterpret_cast<double*>(s_span);                   // staging, reuses the span after a barrier

    const int tid = threadIdx.x;
    const int G = P.frames_per_cta;
    const int n = P.n, sv = P.sv, pad = P.pad;
    // Frames of the batch are numbered through the segments (utterances).  With P.straddle a CTA takes G consecutive
    // frames of the BATCH — when they cross into the next segment its span is staged as two pieces (nA frames of this
    // segment, nB of the next) — so only the batch's last CTA is partial; otherwise every segment gets its own CTAs.
    int64_t seg, j0, g0;
    int Gc, nA;
    if (P.straddle) {
        g0 = (int64_t)blockIdx.x * G;
        Gc = (int)min((int64_t)G, P.n_frames - g0);
        seg = g0 / P.seg_frames;
        j0 = g0 - seg * P.seg_frames;
        nA = (int)min((int64_t)Gc, P.seg_frames - j0);
    } else {
        seg = blockIdx.x / P.ctas_per_seg;
        j0 = (int64_t)(blockIdx.x - seg * P.ctas_per_seg) * G;
        g0 = seg * P.seg_frames + j0;
        Gc = (int)min((int64_t)G, P.seg_frames - j0);
        nA = Gc;
    }
    const int nB = Gc - nA;
    // second piece: right after the first piece's padded span, 16-byte aligned
    const int totalA = (nA - 1) * sv + n;
    const int offB = (totalA + pad * ((totalA - 1) / sv) + 3) & ~3;
    const TIn* __restrict__ base = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride;

    for (int i = tid; i < n; i += P.threads) s_win[i] = __ldg(P.win + i);
    stage_span16<TIn>(P, base, j0, nA, s_span);
    if (nB > 0) stage_span16<TIn>(P, base + P.seg_stride, 0, nB, s_span + offB);
    __syncthreads();

    // warp → (32 frames, half): even warps walk the first chunks of their 32 frames and odd warps the rest, so the
    // pre-roll below is warp-uniform
    const int warp = tid >> 5, lane = tid & 31;
    const int q = warp & 1;
    const int g = (warp >> 1) * 32 + lane;
    double acc[L], h[kChunk];
#pragma unroll
    for (int j = 0; j < L; ++j) acc[j] = 0.0;
#pragma unroll
    for (int j = 0; j < kChunk; ++j) h[j] = 0.0;
    if (g < Gc) {
        const int C = n / kChunk;                               // chunks per frame
        const int nch = (C + 2) >> 1;                           // chunk passes per lane: ceil((C + 1) / 2)
        const int pre = q ? 2 * nch - C : 0;                    // pre-roll passes of the second half (1 or 2): ring fill only
        const int cpb = sv / kChunk;                            // chunks between pad words
        const int c = q ? C - nch : 0;
        const int blk = c / cpb;
        int left = cpb - (c - blk * cpb);
        const float* sp = s_span + (g < nA ? g * (sv + pad) : offB + (g - nA) * (sv + pad)) + c * kChunk + pad * blk;
        const double* wp = s_win + c * kChunk;
        int it = 0;
        for (; it < pre; ++it) {
#pragma unroll
            for (int v = 0; v < kChunk / 4; ++v) {
                const float4 t = reinterpret_cast<const float4*>(sp)[v];
                const double2 wa = reinterpret_cast<const double2*>(wp)[2 * v], wb = reinterpret_cast<const double2*>(wp)[2 * v + 1];
                h[4 * v] = (double)t.x * wa.x;
                h[4 * v + 1] = (double)t.y * wa.y;
                h[4 * v + 2] = (double)t.z * wb.x;
                h[4 * v + 3] = (double)t.w * wb.y;
            }
            sp += kChunk;
            wp += kChunk;
            if (--left == 0) { sp += pad; left = cpb; }
        }
        for (; it < nch; ++it) {
            float xf[kChunk];
#pragma unroll
            for (int v = 0; v < kChunk / 4; ++v) {
                const float4 t = reinterpret_cast<const float4*>(sp)[v];
                xf[4 * v] = t.x;
                xf[4 * v + 1] = t.y;
                xf[4 * v + 2] = t.z;
                xf[4 * v + 3] = t.w;
            }
#pragma unroll
            for (int u = 0; u < kChunk; u += 2) {
                const double2 w2 = reinterpret_cast<const double2*>(wp)[u >> 1];
                const double xa = (double)xf[u] * w2.x;
                h[u] = xa;
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(xa, h[(u - lag) & (kChunk - 1)], acc[lag]);
                const double xb = (double)xf[u + 1] * w2.y;
                h[u + 1] = xb;
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(xb, h[(u + 1 - lag) & (kChunk - 1)], acc[lag]);
            }
            sp += kChunk;
            wp += kChunk;
            if (--left == 0) { sp += pad; left = cpb; }
            if (it == 0) {
                // reference quirk (periodic.rs:284): the fold is seeded with x[0] and skips the i = 0 product, so
                // r[lag] = true_r[lag] − x0·x[lag] + x0; after the first chunk h[j] = xw[j].  (A second-half lane
                // never gets here: its pre-roll is at least one pass.)
                const double x0 = h[0];
#pragma unroll
                for (int lag = 0; lag < L; ++lag) acc[lag] = fma(x0, 1.0 - h[lag], acc[lag]);
            }
        }
    }
    // second halves park their sums in shared memory (the span is dead after the barrier); first halves add them
    __syncthreads();
    double* s_r = s_out;  // [G][L], same layout lpc_finish uses
    if (q == 1 && g < Gc) {
#pragma unroll
        for (int lag = 0; lag < L; ++lag) s_r[g * L + lag] = acc[lag];
    }
    __syncthreads();
    if (q == 0 && g < Gc) {
#pragma unroll
        for (int lag = 0; lag < L; ++lag) acc[lag] += s_r[g * L + lag];
    }
    lpc_finish<L>(P, acc, g < Gc && q == 0, g, Gc, g0, s_out);
}
