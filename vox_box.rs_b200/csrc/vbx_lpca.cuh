// vbx_lpca.cuh — the fused window → fp64 autocorrelation → Levinson kernel for ANY overlapped or packed framing with at
// most 13 lags (the C3 shape: 1102 / 441 / 13, where neither the frame length nor the hop is a multiple of 16).  Included
// inside the anonymous namespace of vbx_lpc.cu after LpcParams / levinson / lpc_finish and vbx_lpc16.cuh.
//
// It is the 16-sample-chunk walk of lpc_fused16_kernel (4 LDS.128 of samples + 8 LDS.128 of window pairs per 16 samples,
// a 16-slot register ring, no per-sample bookkeeping) made independent of the framing by ALIGNING EVERY FRAME DOWN:
//   * the CTA stages the contiguous span of its G frames from the 16-byte-aligned address at or below the span start, so
//     frame g begins at shared-memory word m + g·hop with some alignment a = (m + g·hop) mod 4;
//   * the lane treats its frame as starting at the aligned word m + g·hop − a with length N + a, padded to C = ⌈(N+3)/16⌉
//     chunks; the a leading and the trailing positions carry window weight ZERO, so they add exactly 0 to every lag sum;
//   * the shifted window tables are two rows in shared memory, E = [0, 0, w…, 0…] and O = [0, 0, 0, w…, 0…]: alignment 0
//     reads E + 2, 2 reads E, 1 reads O + 2, 3 reads O — every row start is 16-byte aligned for the LDS.128 of doubles.
// 0·x is 0 only for finite x: the staging pass looks at every sample it copies, and a CTA that saw an Inf / NaN runs the
// chunks that contain zero-weight positions through a select instead (the reference never touches those samples).
//
// A frame is split over K lanes by chunks (part q = chunks [⌊qC/K⌋, ⌊(q+1)C/K⌋)); a lane of a later part first fills its
// ring from the chunk before its range (window multiply only, no lag products).  Lane layout: tid = q·G + g, so the 8
// lanes of a quarter-warp hold 8 consecutive frames of one part: their 16-byte chunk pieces sit hop words apart, which for
// odd hop/4 patterns (441: 110.25 pieces) fall into 8 different bank groups.  The parts of a frame meet in shared memory
// (fixed order: deterministic), Levinson and the write-out are lpc_finish's.  G = 32, K = 8 (256 threads, ≈ 77 KB: 2 CTAs
// = 16 warps per SM) for the C3 shape; VBX_LPCA_PLAN="G:K" overrides.
constexpr int kLpcaMaxLags = 13;  // a + lag <= 3 + 12 = 15: the x[0]-seed fix-up reads ring slots a … a + L − 1 of chunk 0

struct LpcaExtra {
    const double* tabs;  // [2][wt] device: rows E and O
    int wt;              // row length in doubles (C·16 + 4)
    int chunks;          // C
    int span_floats;     // shared-memory floats reserved for the span
};

template <bool MASKED>
__device__ __forceinline__ void lpca_ring_fill(double (&h)[kChunk], const float* sp, const double* wp, int pos0, int lo, int hi) {
#pragma unroll
    for (int v = 0; v < kChunk / 4; ++v) {
        const float4 t = reinterpret_cast<const float4*>(sp)[v];
        const double2 wa = reinterpret_cast<const double2*>(wp)[2 * v], wb = reinterpret_cast<const double2*>(wp)[2 * v + 1];
        const float xf[4] = {t.x, t.y, t.z, t.w};
        const double ww[4] = {wa.x, wa.y, wb.x, wb.y};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            double xn = (double)xf[e] * ww[e];
            if (MASKED) {
                const int pos = pos0 + 4 * v + e;
                xn = (pos >= lo && pos < hi) ? xn : 0.0;
            }
            h[4 * v + e] = xn;
        }
    }
}

template <int L, bool MASKED>
__device__ __forceinline__ void lpca_chunk(double (&acc)[L], double (&h)[kChunk], const float* sp, const double* wp, int pos0, int lo, int hi) {
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
        double xa = (double)xf[u] * w2.x;
        if (MASKED) xa = (pos0 + u >= lo && pos0 + u < hi) ? xa : 0.0;
        h[u] = xa;
#pragma unroll
        for (int lag = 0; lag < L; ++lag) acc[lag] = fma(xa, h[(u - lag) & (kChunk - 1)], acc[lag]);
        double xb = (double)xf[u + 1] * w2.y;
        if (MASKED) xb = (pos0 + u + 1 >= lo && pos0 + u + 1 < hi) ? xb : 0.0;
        h[u + 1] = xb;
#pragma unroll
        for (int lag = 0; lag < L; ++lag) acc[lag] = fma(xb, h[(u + 1 - lag) & (kChunk - 1)], acc[lag]);
    }
}

template <int L, typename TIn>
__global__ void __launch_bounds__(256) lpc_fuseda_kernel(const LpcParams P, const LpcaExtra X) {
    static_assert(L >= 2 && L <= kLpcaMaxLags, "the seed fix-up needs a + lag <= 15");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_tab = reinterpret_cast<double*>(smem_raw);                   // [2][wt]
    float* s_span = reinterpret_cast<float*>(s_tab + 2 * X.wt);             // aligned span (16-byte aligned: wt is even)
    double* s_out = reinterpret_cast<double*>(s_span);                     // staging, reuses the span after a barrier

    const int tid = threadIdx.x, nthreads = P.threads;
    const int G = P.frames_per_cta, K = P.k;
    const int n = P.n, sv = P.sv;
    const int64_t seg = blockIdx.x / P.ctas_per_seg;
    const int64_t j0 = (int64_t)(blockIdx.x - seg * P.ctas_per_seg) * G;   // first frame of this CTA inside its segment
    const int64_t g0 = seg * P.seg_frames + j0;                            // ... and in the batch (output row)
    const int Gc = (int)min((int64_t)G, P.seg_frames - j0);
    const TIn* __restrict__ src = reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride + j0 * P.stride;
    constexpr int A = 16 / (int)sizeof(TIn);                               // samples per 16-byte load (4, 8 or 16)
    const int mis = (int)((reinterpret_cast<uintptr_t>(src) / sizeof(TIn)) & (A - 1));
    const TIn* __restrict__ src_al = src - mis;                            // 16-byte aligned

    // ---- stage the window rows and the span (word s of the span = sample src_al[s]; zeros outside the real samples) --------
    {
        const double2* t2 = reinterpret_cast<const double2*>(X.tabs);
        double2* d2 = reinterpret_cast<double2*>(s_tab);
        for (int i = tid; i < X.wt; i += nthreads) d2[i] = __ldg(t2 + i);   // 2·wt doubles = wt double2
    }
    const int first = mis, last = mis + (Gc - 1) * sv + n;                  // real samples are words [first, last)
    const int total = X.span_floats;                                        // multiple of max(A, 8)
    bool bad = false;
    if (sizeof(TIn) == 4) {
        const int nv = total >> 2;
        for (int v0 = tid; v0 < nv; v0 += 8 * nthreads) {
            float4 a[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int v = v0 + u * nthreads, s = 4 * v;
                a[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (v < nv) {
                    if (s >= first && s + 4 <= last) {
                        a[u] = __ldg(reinterpret_cast<const float4*>(src_al) + v);
                    } else {  // a vector that straddles the ends of the real samples: element-wise, zeros outside
                        if (s + 0 >= first && s + 0 < last) a[u].x = vbx_load_sample<TIn>(src_al + s + 0);
                        if (s + 1 >= first && s + 1 < last) a[u].y = vbx_load_sample<TIn>(src_al + s + 1);
                        if (s + 2 >= first && s + 2 < last) a[u].z = vbx_load_sample<TIn>(src_al + s + 2);
                        if (s + 3 >= first && s + 3 < last) a[u].w = vbx_load_sample<TIn>(src_al + s + 3);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int v = v0 + u * nthreads;
                if (v < nv) {
                    reinterpret_cast<float4*>(s_span)[v] = a[u];
                    const unsigned e0 = __float_as_uint(a[u].x), e1 = __float_as_uint(a[u].y), e2 = __float_as_uint(a[u].z),
                                   e3 = __float_as_uint(a[u].w);
                    const unsigned m = 0x7f800000u;
                    bad = bad || ((e0 & m) == m) || ((e1 & m) == m) || ((e2 & m) == m) || ((e3 & m) == m);
                }
            }
        }
    } else if constexpr (vbx_g711<TIn>::value) {
        // G.711: 16-byte loads of 16 codes, decoded as they land (always finite); two loads in flight per thread hold as many
        // samples as the four of int16 (four spill registers at 10 / 11 lags)
        const int nv = total >> 4;
        for (int v0 = tid; v0 < nv; v0 += 2 * nthreads) {
            uint4 a[2];
            bool whole[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int v = v0 + u * nthreads, s = 16 * v;
                whole[u] = (v < nv) && (s >= first && s + 16 <= last);
                if (whole[u]) a[u] = __ldg(reinterpret_cast<const uint4*>(src_al) + v);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int v = v0 + u * nthreads, s = 16 * v;
                if (v >= nv) continue;
                float e[16];
                if (whole[u]) {
                    vbx_decode16<TIn>(a[u], e);
                } else {
#pragma unroll
                    for (int k = 0; k < 16; ++k) e[k] = (s + k >= first && s + k < last) ? vbx_load_sample<TIn>(src_al + s + k) : 0.f;
                }
                float4* dst = reinterpret_cast<float4*>(s_span + s);
#pragma unroll
                for (int k = 0; k < 4; ++k) dst[k] = make_float4(e[4 * k], e[4 * k + 1], e[4 * k + 2], e[4 * k + 3]);
            }
        }
    } else {
        // int16 PCM: 16-byte loads of 8 samples (always finite)
        const int nv = total >> 3;
        for (int v0 = tid; v0 < nv; v0 += 4 * nthreads) {
            uint4 a[4];
            bool whole[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int v = v0 + u * nthreads, s = 8 * v;
                whole[u] = (v < nv) && (s >= first && s + 8 <= last);
                if (whole[u]) a[u] = __ldg(reinterpret_cast<const uint4*>(src_al) + v);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int v = v0 + u * nthreads, s = 8 * v;
                if (v >= nv) continue;
                float4* dst = reinterpret_cast<float4*>(s_span + s);
                if (whole[u]) {
                    dst[0] = make_float4((float)(short)(a[u].x & 0xffffu), (float)(short)(a[u].x >> 16),
                                         (float)(short)(a[u].y & 0xffffu), (float)(short)(a[u].y >> 16));
                    dst[1] = make_float4((float)(short)(a[u].z & 0xffffu), (float)(short)(a[u].z >> 16),
                                         (float)(short)(a[u].w & 0xffffu), (float)(short)(a[u].w >> 16));
                } else {
                    float e[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) e[k] = (s + k >= first && s + k < last) ? vbx_load_sample<TIn>(src_al + s + k) : 0.f;
                    dst[0] = make_float4(e[0], e[1], e[2], e[3]);
                    dst[1] = make_float4(e[4], e[5], e[6], e[7]);
                }
            }
        }
    }
    const bool guard = __syncthreads_or(bad) != 0;  // the staging barrier also tells every thread whether anybody saw an Inf / NaN

    // ---- per-lane partial autocorrelation over the lane's chunks ----------------------------------------------------------
    const int q = tid / G, g = tid - q * G;   // part, frame
    double acc[L], h[kChunk];
#pragma unroll
    for (int j = 0; j < L; ++j) acc[j] = 0.0;
#pragma unroll
    for (int j = 0; j < kChunk; ++j) h[j] = 0.0;
    if (g < Gc && q < K) {
        const int C = X.chunks;
        const int fstart = mis + g * sv;      // the frame's first sample (span word)
        const int a = fstart & 3;             // its alignment: the walk starts a words earlier
        const int c_lo = (q * C) / K, c_hi = ((q + 1) * C) / K;
        const int lo = a, hi = a + n;         // positions of the aligned walk that belong to the frame
        int c = c_lo > 0 ? c_lo - 1 : 0;
        const float* sp = s_span + (fstart - a) + c * kChunk;
        const double* wp = s_tab + ((a & 1) ? X.wt : 0) + ((a & 2) ? 0 : 2) + c * kChunk;
        if (c_lo > 0) {  // pre-roll: the chunk before the lane's range fills the ring (window multiply, no lag products)
            if (guard) lpca_ring_fill<true>(h, sp, wp, c * kChunk, lo, hi);
            else lpca_ring_fill<false>(h, sp, wp, c * kChunk, lo, hi);
            sp += kChunk;
            wp += kChunk;
            ++c;
        }
        for (; c < c_hi; ++c) {
            // chunks that hold zero-weight positions take the select only when a non-finite sample is around
            if (guard && (c * kChunk < lo || (c + 1) * kChunk > hi)) lpca_chunk<L, true>(acc, h, sp, wp, c * kChunk, lo, hi);
            else lpca_chunk<L, false>(acc, h, sp, wp, c * kChunk, lo, hi);
            sp += kChunk;
            wp += kChunk;
            if (c == 0) {
                // reference quirk (periodic.rs:284): the fold is seeded with x[0] and skips the i = 0 product, so
                // r[lag] = true_r[lag] + x0·(1 − x[lag]); after chunk 0 ring slot a + k holds the windowed sample k
#define VBX_LPCA_SEED(AA)                                                                      \
    {                                                                                          \
        const double x0 = h[AA];                                                               \
        _Pragma("unroll") for (int lag = 0; lag < L; ++lag) acc[lag] = fma(x0, 1.0 - h[AA + lag], acc[lag]); \
    }
                if (a == 0) VBX_LPCA_SEED(0)
                else if (a == 1) VBX_LPCA_SEED(1)
                else if (a == 2) VBX_LPCA_SEED(2)
                else VBX_LPCA_SEED(3)
#undef VBX_LPCA_SEED
            }
        }
    }
    // ---- the parts of a frame meet in shared memory (the span is dead after the barrier), summed in part order --------------
    __syncthreads();
    double* s_part = s_out + (size_t)G * (3 * L - 1);  // [K − 1][G][L], behind lpc_finish's staging
    if (q > 0 && q < K && g < Gc) {
#pragma unroll
        for (int lag = 0; lag < L; ++lag) s_part[((size_t)(q - 1) * G + g) * L + lag] = acc[lag];
    }
    __syncthreads();
    if (q == 0 && g < Gc) {
        for (int qq = 1; qq < K; ++qq) {
#pragma unroll
            for (int lag = 0; lag < L; ++lag) acc[lag] += s_part[((size_t)(qq - 1) * G + g) * L + lag];
        }
    }
    lpc_finish<L>(P, acc, q == 0 && g < Gc, g, Gc, g0, s_out);
}

// Plan for lpc_fuseda_kernel.  Returns false when the shape is not its (gapped frames, too many lags, too long a frame).
bool plan_fuseda(const vbx_ctx* ctx, int n, int64_t stride, int L, size_t in_size, LpcParams* P, LpcaExtra* X, size_t* smem_bytes) {
    if (L < 2 || L > kLpcaMaxLags || stride > (int64_t)n) return false;
    const int sv = (int)stride;
    const int C = (n + 3 + kChunk - 1) / kChunk;
    int G = 32, K = 8;
    if (const char* e = getenv("VBX_LPCA_PLAN")) {
        int a = 0, b = 0;
        if (sscanf(e, "%d:%d", &a, &b) == 2 && a >= 8 && a <= 64 && a % 8 == 0 && b >= 1 && b <= 16 && a * b <= 256 && (a * b) % 32 == 0) {
            G = a;
            K = b;
        }
    }
    while (K > 1 && C / K < 2) K >>= 1;  // every part at least two chunks
    if ((G * K) % 32 != 0) return false;
    const int A = 16 / (int)in_size;  // samples per 16-byte load: the staging pass copies whole loads
    const int64_t span = (int64_t)(A - 1) + (int64_t)(G - 1) * sv + (int64_t)C * kChunk + 3;
    const int64_t round = A > 8 ? A : 8;
    const int span_floats = (int)((span + round - 1) & ~(round - 1));
    const int wt = C * kChunk + 4;
    const size_t stage_bytes = (size_t)G * ((3 * L - 1) + (size_t)(K - 1) * L) * sizeof(double);
    size_t span_bytes = (size_t)span_floats * sizeof(float);
    const size_t bytes = (size_t)2 * wt * sizeof(double) + (span_bytes > stage_bytes ? span_bytes : stage_bytes);
    if (bytes > ctx->smem_optin || span > (1 << 24)) return false;
    P->k = K;
    P->threads = G * K;
    P->frames_per_cta = G;
    P->part = 0;
    P->span_words = span_floats;
    P->sv = sv;
    P->pad = 0;
    P->sv_magic = 0;
    X->wt = wt;
    X->chunks = C;
    X->span_floats = span_floats;
    *smem_bytes = bytes;
    return true;
}

// =====================================================================================================================
// lpc_fusedp_kernel — the same aligned-down walk as a PERSISTENT, warp-specialised CTA (one per SM) fed by TMA.
//
// The one-shot kernel above spends 40 % of its time outside the DFMA loop: every CTA stages its span (global → registers →
// shared memory, then a barrier), computes, and then seven of its eight warps wait at a barrier while one half-warp runs
// Levinson (ncu, profiles/r2_lpca_v1_full.txt: fp64 pipe 59 %, stall_barrier 18 %, stall_long_sb 10 %).  Here the three
// phases of consecutive tiles (32 frames each) overlap inside one CTA that lives for the whole launch:
//   warp 0        producer: one cp.async.bulk (TMA, global → shared, completion counted on an mbarrier) per tile into a
//                 two-deep ring of span buffers; its lanes zero-fill the few words behind the real samples;
//   warps 1 … K   compute: warp q walks part q of the tile's 32 frames (lane = frame) exactly as lpc_fuseda_kernel does and
//                 parks its L partial sums in a two-deep ring of part buffers;
//   warp K + 1    epilogue: lane = frame; adds the K parts in part order, runs Levinson in registers and writes r / ac / kc
//                 through a small staging area with coalesced stores — while the compute warps are already on the next tile.
// Hand-offs are mbarriers (full / empty for spans, pfull / pempty for parts); there is no __syncthreads() after start-up.
// The window rows are loaded once per CTA instead of once per 32 frames.  A lane whose lag-0 sum comes out non-finite
// (an Inf / NaN sample next to or inside its frame) redoes its part with the zero-weight positions selected to 0, so the
// reference's semantics hold without anybody inspecting the samples the TMA moved.  fp32 samples only (the TMA cannot
// convert PCM); int16 input keeps the one-shot kernel.
// =====================================================================================================================
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok = 0;
    const unsigned addr = smem_u32(bar);
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(addr), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

constexpr int kLpcpFrames = 32;  // frames per tile = lanes of a warp

template <int L>
__global__ void __launch_bounds__(320, 1) lpc_fusedp_kernel(const LpcParams P, const LpcaExtra X, const int n_tiles, unsigned* tile_counter) {
    static_assert(L >= 2 && L <= kLpcaMaxLags, "the seed fix-up needs a + lag <= 15");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int G = kLpcpFrames;
    const int K = P.k;
    double* s_tab = reinterpret_cast<double*>(smem_raw);                                   // [2][wt]
    float* s_span0 = reinterpret_cast<float*>(s_tab + 2 * X.wt);                            // [2][span_floats]
    double* s_part0 = reinterpret_cast<double*>(s_span0 + 2 * (size_t)X.span_floats);       // [2][K][L][G]
    double* s_stage = s_part0 + 2 * (size_t)K * L * G;                                      // [G][3L − 1]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(s_stage + (size_t)G * (3 * L - 1));
    unsigned long long *full = bars, *empty = bars + 2, *pfull = bars + 4, *pempty = bars + 6;
    // Tiles are handed out dynamically (a global counter the producer draws from): a CTA that shares its SM with another
    // kernel's CTAs (the tracker on vbx_find_formants' side stream) simply takes fewer.  The tile index travels with the
    // buffers: s_tile[s] next to span buffer s (−1 = no more tiles), s_ptile[ps] next to part buffer ps.
    int* s_tile = reinterpret_cast<int*>(bars + 8);
    int* s_ptile = s_tile + 2;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = P.n, sv = P.sv;
    if (tid == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(full + s, 33);    // the producer's expect_tx arrive + its 32 lanes after the tail fill
            mbar_init(empty + s, K);    // one elected lane per compute warp
            mbar_init(pfull + s, K);
            mbar_init(pempty + s, 1);   // the epilogue warp's elected lane
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {
        const double2* t2 = reinterpret_cast<const double2*>(X.tabs);
        double2* d2 = reinterpret_cast<double2*>(s_tab);
        for (int i = tid; i < X.wt; i += blockDim.x) d2[i] = __ldg(t2 + i);
    }
    __syncthreads();

    auto tile_src = [&](int t, int& Gc, int64_t& g0) -> const float* {
        const int64_t seg = t / P.ctas_per_seg;
        const int64_t j0 = (int64_t)(t - seg * P.ctas_per_seg) * G;
        g0 = seg * P.seg_frames + j0;
        Gc = (int)min((int64_t)G, P.seg_frames - j0);
        return reinterpret_cast<const float*>(P.base) + seg * P.seg_stride + j0 * P.stride;
    };

    if (warp == 0) {
        // ------------------------------------------------------------------ producer
        for (int it = 0;; ++it) {
            const int s = it & 1;
            mbar_wait(empty + s, ((it >> 1) & 1) ^ 1);
            int t = 0;
            if (lane == 0) t = (int)atomicAdd(tile_counter, 1u);
            t = __shfl_sync(0xffffffffu, t, 0);
            if (t >= n_tiles) {
                if (lane == 0) {
                    s_tile[s] = -1;
                    mbar_arrive(full + s);
                }
                mbar_arrive(full + s);
                break;
            }
            int Gc;
            int64_t g0;
            const float* src = tile_src(t, Gc, g0);
            const int mis = (int)((reinterpret_cast<uintptr_t>(src) >> 2) & 3);
            const float* src_al = src - mis;
            const int last = mis + (Gc - 1) * sv + n;      // words [mis, last) are this tile's samples; [0, mis) exist too
            const int last_al = last & ~3;
            float* dst = s_span0 + (size_t)s * X.span_floats;
            if (lane == 0) {
                s_tile[s] = t;
                if (last_al > 0) {
                    mbar_arrive_expect_tx(full + s, (unsigned)last_al * 4u);
                    tma_bulk_g2s(dst, src_al, (unsigned)last_al * 4u, full + s);
                } else {
                    mbar_arrive(full + s);
                }
            }
            // the ≤ 3 samples behind the last whole 16-byte piece, then zeros as far as the last frame's aligned walk reaches
            const int zend = min(X.span_floats, (last + (X.chunks * kChunk - n) + 3 + 7) & ~7);
            for (int w = last_al + lane; w < zend; w += 32) dst[w] = (w < last) ? __ldg(src_al + w) : 0.f;
            mbar_arrive(full + s);
        }
    } else if (warp <= K) {
        // ------------------------------------------------------------------ compute: part q of 32 frames
        const int q = warp - 1, g = lane;
        const int C = X.chunks;
        const int c_lo = (q * C) / K, c_hi = ((q + 1) * C) / K;
        for (int it = 0;; ++it) {
            const int s = it & 1;
            mbar_wait(full + s, (it >> 1) & 1);
            const int t = s_tile[s];
            const int ps = it & 1;
            if (t < 0) {  // no more tiles: pass the word on to the epilogue warp and leave
                if (q == 0) {
                    mbar_wait(pempty + ps, ((it >> 1) & 1) ^ 1);
                    if (lane == 0) s_ptile[ps] = -1;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(pfull + ps);
                break;
            }
            int Gc;
            int64_t g0;
            const float* src = tile_src(t, Gc, g0);
            const int mis = (int)((reinterpret_cast<uintptr_t>(src) >> 2) & 3);
            const float* span = s_span0 + (size_t)s * X.span_floats;
            double acc[L], h[kChunk];
            const int fstart = mis + g * sv;
            const int a = fstart & 3;
            const int lo = a, hi = a + n;
            for (int pass = 0; pass < 2; ++pass) {
                const bool guard = (pass == 1);
#pragma unroll
                for (int j = 0; j < L; ++j) acc[j] = 0.0;
#pragma unroll
                for (int j = 0; j < kChunk; ++j) h[j] = 0.0;
                if (g < Gc) {
                    int c = c_lo > 0 ? c_lo - 1 : 0;
                    const float* sp = span + (fstart - a) + c * kChunk;
                    const double* wp = s_tab + ((a & 1) ? X.wt : 0) + ((a & 2) ? 0 : 2) + c * kChunk;
                    if (c_lo > 0) {
                        if (guard) lpca_ring_fill<true>(h, sp, wp, c * kChunk, lo, hi);
                        else lpca_ring_fill<false>(h, sp, wp, c * kChunk, lo, hi);
                        sp += kChunk;
                        wp += kChunk;
                        ++c;
                    }
                    for (; c < c_hi; ++c) {
                        if (guard && (c * kChunk < lo || (c + 1) * kChunk > hi)) lpca_chunk<L, true>(acc, h, sp, wp, c * kChunk, lo, hi);
                        else lpca_chunk<L, false>(acc, h, sp, wp, c * kChunk, lo, hi);
                        sp += kChunk;
                        wp += kChunk;
                        if (c == 0) {
#define VBX_LPCA_SEED(AA)                                                                      \
    {                                                                                          \
        const double x0 = h[AA];                                                               \
        _Pragma("unroll") for (int lag = 0; lag < L; ++lag) acc[lag] = fma(x0, 1.0 - h[AA + lag], acc[lag]); \
    }
                            if (a == 0) VBX_LPCA_SEED(0)
                            else if (a == 1) VBX_LPCA_SEED(1)
                            else if (a == 2) VBX_LPCA_SEED(2)
                            else VBX_LPCA_SEED(3)
#undef VBX_LPCA_SEED
                        }
                    }
                }
                // a non-finite lag-0 sum: an Inf / NaN sample inside the frame (then the redo gives the same) or in a
                // zero-weight position next to it (then the redo is the reference's value)
                if (fabs(acc[0]) <= 1.7976931348623157e308) break;
            }
            mbar_wait(pempty + ps, ((it >> 1) & 1) ^ 1);
            double* part = s_part0 + ((size_t)ps * K + q) * L * G;
#pragma unroll
            for (int lag = 0; lag < L; ++lag) part[lag * G + g] = acc[lag];
            if (q == 0 && lane == 0) s_ptile[ps] = t;
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(pfull + ps);
                mbar_arrive(empty + s);
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue: lane = frame
        const int g = lane;
        for (int it = 0;; ++it) {
            const int ps = it & 1;
            mbar_wait(pfull + ps, (it >> 1) & 1);
            const int t = s_ptile[ps];
            if (t < 0) break;
            int Gc;
            int64_t g0;
            (void)tile_src(t, Gc, g0);
            double r[L], ac[L], kc[L - 1];
            const double* part = s_part0 + (size_t)ps * K * L * G;
#pragma unroll
            for (int lag = 0; lag < L; ++lag) r[lag] = part[lag * G + g];
            for (int qq = 1; qq < K; ++qq) {
#pragma unroll
                for (int lag = 0; lag < L; ++lag) r[lag] += part[((size_t)qq * L + lag) * G + g];
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(pempty + ps);
            if (P.do_levinson && g < Gc) levinson<L - 1>(r, ac, kc);
            double* s_r = s_stage;
            double* s_ac = s_r + G * L;
            double* s_kc = s_ac + G * L;
            if (g < Gc) {
#pragma unroll
                for (int lag = 0; lag < L; ++lag) s_r[g * L + lag] = r[lag];
                if (P.do_levinson) {
#pragma unroll
                    for (int lag = 0; lag < L; ++lag) s_ac[g * L + lag] = ac[lag];
#pragma unroll
                    for (int j = 0; j < L - 1; ++j) s_kc[g * (L - 1) + j] = kc[j];
                }
            }
            __syncwarp();
            auto store = [&](void* out, const double* src_s, int per_frame) {
                if (!out) return;
                const int total = Gc * per_frame;
                const int64_t off = g0 * per_frame;
                if (P.out_f64) {
                    double* o = reinterpret_cast<double*>(out) + off;
                    for (int idx = lane; idx < total; idx += 32) o[idx] = src_s[idx];
                } else {
                    float* o = reinterpret_cast<float*>(out) + off;
                    for (int idx = lane; idx < total; idx += 32) o[idx] = (float)src_s[idx];
                }
            };
            store(P.r_out, s_r, L);
            if (P.do_levinson) {
                store(P.ac_out, s_ac, L);
                store(P.kc_out, s_kc, L - 1);
            }
            __syncwarp();
        }
    }
}

// Plan for lpc_fusedp_kernel: fp32 samples, overlapped or packed frames, <= 13 lags, enough tiles to keep every SM's CTA busy.
bool plan_fusedp(const vbx_ctx* ctx, const vbx_frames* fr, int L, LpcParams* P, LpcaExtra* X, size_t* smem_bytes) {
    const int n = fr->frame_len;
    if (fr->dtype != VBX_F32 || L < 2 || L > kLpcaMaxLags || fr->frame_stride > (int64_t)n) return false;
    if (const char* e = getenv("VBX_LPCP"))
        if (atoi(e) == 0) return false;
    if ((reinterpret_cast<uintptr_t>(fr->base) & 3) != 0) return false;
    const int sv = (int)fr->frame_stride;
    const int C = (n + 3 + kChunk - 1) / kChunk;
    int K = 8;
    if (const char* e = getenv("VBX_LPCP_K")) K = atoi(e);
    if (K < 1 || K > 8) return false;
    while (K > 1 && C / K < 2) K >>= 1;
    const int G = kLpcpFrames;
    const int64_t span = 3 + (int64_t)(G - 1) * sv + (int64_t)C * kChunk + 3;
    const int span_floats = (int)((span + 7) & ~(int64_t)7);
    const int wt = C * kChunk + 4;
    const size_t bytes = (size_t)2 * wt * sizeof(double) + (size_t)2 * span_floats * sizeof(float) +
                         ((size_t)2 * K * L * G + (size_t)G * (3 * L - 1)) * sizeof(double) + 8 * sizeof(unsigned long long) + 4 * sizeof(int);
    if (bytes > ctx->smem_optin || (size_t)span_floats * 4 >= (1u << 20)) return false;  // mbarrier tx-count range
    const int64_t J = vbx_frames_per_segment(fr);
    const int64_t ctas_per_seg = (J + G - 1) / G;
    const int64_t tiles = (fr->n_frames / J) * ctas_per_seg;
    if (tiles < 2 * (int64_t)ctx->sm_count || tiles > 0x7fffffffLL) return false;
    P->k = K;
    P->threads = 32 * (K + 2);
    P->frames_per_cta = G;
    P->part = 0;
    P->span_words = span_floats;
    P->sv = sv;
    P->pad = 0;
    P->sv_magic = 0;
    X->wt = wt;
    X->chunks = C;
    X->span_floats = span_floats;
    *smem_bytes = bytes;
    return true;
}
