// vbx_mfcc_lane5.cuh — MFCC for 400-sample frames (25 ms at 16 kHz, the C5 shape): FIVE LANES PER FRAME, six frames per warp.
//
// mfcc_warp_kernel (vbx_mfcc_fast.cuh) spreads the (frame, butterfly) pairs of every pass over the 32 lanes: flexible, but
// every item pays div/mod index arithmetic, a padded-index computation per element and a twiddle fetch — 810 of its 1 496
// warp instructions per frame are integer / control and only 433 are fp64 (profiles/r1_mfcc_final_full.txt).  Here a frame
// belongs to five lanes (lane = 5·q + s, q = frame of the group, s = sub-lane; lanes 30 and 31 idle), and the transform is
// laid out so that every shared-memory address is `per-lane base + compile-time constant`:
//
//   The real frame is packed as z[n] = x[2n]·w[2n] + i·x[2n+1]·w[2n+1], n < 200, and transformed IN PLACE by
//   decimation-in-frequency passes of radix 8, 5, 5 (k = kA + 8·kB + 40·kC):
//     pass A  butterfly n1 (< 25): inputs z[n1 + 25t] straight from global memory (windowed in fp64), radix 8, output u times
//             W200^(n1·u) to slot 25u + n1.  (In this pass alone a lane owns a POSITION n1 = lane and walks three of the group's
//             frames with its seven twiddles in registers; everywhere else lane = 5·q + s works on frame q.)
//     pass B  inside every 25-block b (= kA) butterfly j = s: inputs 25b + s + 5t, radix 5, output kB times W25^(s·kB) (the four
//             twiddles live in registers), stored TRANSPOSED to 25b + 5s + col(b, kB) (four blocks in flight, __syncwarp between
//             their loads and stores);
//     pass C  butterfly (kA, kB = s): inputs 25kA + 5j + col, radix 5, no twiddle — and its five outputs Z[kA + 8s + 40kC] stay in
//             registers: the partner bins 200 − k are exactly the outputs of butterfly (8 − kA, 4 − s) in reverse order, so one lane
//             runs both butterflies and untangles the ten bins (X_k = E − i·W400^k·O) without another trip through shared memory,
//             writing (|X|², |X|) back into the slots it read.  Blocks 5..7 store their columns mirrored (col = 4 − kB), so the
//             partner's loads are `base + s` too.  The ten butterflies of blocks 0 and 4 (self-paired blocks) form a fourth unit per
//             lane whose slots come from a small table; lane 4's holds the two self-paired butterflies (bins 0 / Nyquist and 100).
//   Band sums: the M + 1 intervals between the filter-bank's bin edges are dealt to the five lanes by the host (longest first, to
//   the least loaded lane); a lane reads its bins in ascending order through a bin → slot table: both sums in the reference's order
//   (spectrum.rs:421-435, quirks as in vbx_mfcc.cu).  log10 / clamp and the DCT rows are split over the five lanes as well.
//
// The frame buffers are 205 elements apart, so the 30 lanes of a `base + s` access touch 30 consecutive 16-byte bank groups:
// conflict free (tools/mfcc_lane5_emulation.py checks the index maps against numpy and counts wavefronts).
// One persistent CTA of 8 warps per SM (48 frames in flight, 208 KB of shared memory), no CTA barrier after the tables are staged.
#pragma once

// included from inside vbx_mfcc.cu's anonymous namespace (cxt<>, mk, caddf, csubf, cmulf, mulnegi, mfcc_fast::bfly)

namespace mfcc_lane5 {

constexpr int MC = 200, N = 400, FS = 205, FW = 6, LPF = 5, WARPS = 16, PAIRS = WARPS / 2;
constexpr int kMaxItems = 132;  // intervals (num_coeffs + 1 <= 129)
constexpr int kMaxRounds = (kMaxItems + 9) / 10 + 1;
constexpr int kMaxProg = N + 6 * kMaxItems;  // words of one twin's band-sum program (padding included)
constexpr unsigned kMask = 0x3fffffffu;  // the 30 working lanes

// host-built tables (one device copy per MfccTables entry)
struct Tables {
    double2 twA[7 * 25];     // [u − 1][n1]  W200^(n1·u)
    double2 twB[4 * 5];      // [kB − 1][s]  W25^(s·kB)
    double2 twU[3 * 5 * 5];  // [kA − 1][kC][s]  ½·W400^(kA + 8s + 40kC)      (units 1..3)
    double2 twU4[6 * 5];     // [op][s]  ½·W400^k of the fourth unit's pair operations
    unsigned short u4base[2 * 5];   // [c | c'][s]  slot of input j = 0 of the fourth unit's two butterflies (input j at + 5j)
    unsigned short u4slot[12 * 5];  // [2·op | 2·op + 1][s]  slots of X_k and X_{200−k}
    // Band-sum programs of the ten twins v = 5h + s (h = which warp of the pair).  The intervals between the filter bank's bin
    // edges are sorted by length and dealt five at a time to the two warps in turn: ROUND r of warp h is five intervals of about
    // the same length, one per lane, each padded to the round's longest (round_len[h][r]) with entries that read the frame
    // buffer's zero slot with weight 0 — so the whole warp runs the same trip counts.  prog[v]: per round a header word (the
    // interval j, or kIdle) and round_len words, the BYTE offsets of the bins' slots in ascending bin order; pw[v]: the bins'
    // (rising weight, falling-slope weight) in the same order.
    int n_rounds[2];
    int round_len[2][kMaxRounds];
    int prog_len, pw_len;    // longest program / weight list: the row lengths of the shared-memory copies
    unsigned prog[2 * LPF][kMaxProg];
    double2 pw[2 * LPF][kMaxProg];
};
constexpr unsigned kIdle = 0xffffu;
constexpr int kZeroSlot = MC + 1;   // a pad slot that always holds (0, 0)

struct Params {
    const void* base;
    const double* win;    // [N]
    const double* dct;    // [n_keep][num_coeffs]
    const Tables* t;
    void* out;
    void* energies_out;
    int64_t n_frames, stride, seg_frames, seg_stride;
    int num_coeffs, n_keep, prog_len, pw_len;
    int out_f64;
};

typedef cxt<double> C;

template <typename TIn> struct RawPair;
template <> struct RawPair<float> { typedef float2 type; };
template <> struct RawPair<int16_t> { typedef short2 type; };
template <> struct RawPair<vbx_mulaw8> { typedef float2 type; };
template <> struct RawPair<vbx_alaw8> { typedef float2 type; };
template <typename TIn> __device__ __forceinline__ typename RawPair<TIn>::type load_raw(const TIn* p) {
    if constexpr (vbx_g711<TIn>::value) {  // one 2-byte load of a code pair, decoded
        const uchar2 c = __ldg(reinterpret_cast<const uchar2*>(p));
        return make_float2(vbx_decode8<TIn>(c.x), vbx_decode8<TIn>(c.y));
    } else {
        return __ldg(reinterpret_cast<const typename RawPair<TIn>::type*>(p));
    }
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// untangle one pair: za = Z_k, zb = Z_{200−k}, wh = ½·W400^k  →  (|X_k|², |X_k|), (|X_{200−k}|², |X_{200−k}|)
__device__ __forceinline__ void pair_op(const C za, const C zb, const C wh, C& pa, C& pb) {
    const double sx = za.x + zb.x, dy = za.y - zb.y, dx = za.x - zb.x, sy = za.y + zb.y;
    const double tx = wh.x * dx - wh.y * sy, ty = wh.x * sy + wh.y * dx;   // T = W·O (O = ½(dx, sy))
    const double xr = fma(0.5, sx, ty), xi = fma(0.5, dy, -tx);           // X_k = E − iT, E = ½(sx, dy)
    const double yr = fma(0.5, sx, -ty), yi = fma(-0.5, dy, -tx);         // X_{200−k} = conj(E) − i·conj(T)
    const double pwa = xr * xr + xi * xi, pwb = yr * yr + yi * yi;
    pa = mk<double>(pwa, sqrt(pwa));
    pb = mk<double>(pwb, sqrt(pwb));
}

__constant__ double kLogC[10] = {1.0 / 21.0, 1.0 / 19.0, 1.0 / 17.0, 1.0 / 15.0, 1.0 / 13.0, 1.0 / 11.0, 1.0 / 9.0, 1.0 / 7.0, 1.0 / 5.0, 1.0 / 3.0};
// log10 for the band energies: exponent split + atanh series (|t| <= 0.172, nine terms), ~35 instructions against libm's ~110;
// max relative error 4.2e-16 against a long-double reference (libm: 2.2e-16) on 2e7 arguments incl. the neighbourhood of 1, where
// the 1e-10 clamp of spectrum.rs:434 makes the RELATIVE accuracy matter.  Zero, subnormal, negative, Inf and NaN take libm.
__device__ __forceinline__ double band_log10(double x) {
    const int hi = __double2hiint(x);
    if ((unsigned)(hi - 0x00100000) >= 0x7fe00000u) return log10(x);
    int e = (hi >> 20) - 1023;
    int mh = (hi & 0x000fffff) | 0x3ff00000;             // mantissa in [1, 2)
    if (mh > 0x3ff6a09e) { mh -= 0x00100000; e += 1; }   // ... in [0.707, 1.414)
    const double m = __hiloint2double(mh, __double2loint(x));
    const double num = m - 1.0, den = m + 1.0;           // m − 1 is exact
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(den));
    r = fma(fma(-den, r, 1.0), r, r);
    r = fma(fma(-den, r, 1.0), r, r);
    double t = num * r;
    t = fma(fma(-den, t, num), r, t);                    // t = (m − 1) / (m + 1)
    const double t2 = t * t;
    double p = kLogC[0];
#pragma unroll
    for (int i = 1; i < 10; ++i) p = fma(p, t2, kLogC[i]);   // coefficients as constant-bank operands
    const double tt = t + t;
    const double lnm = fma(t2 * p, tt, tt);              // ln m = 2t (1 + t²/3 + t⁴/5 + ...)
    const double ed = (double)e;
    // log10 2 = hi + lo with 21 trailing zero bits in hi: e·hi is exact
    return fma(ed, 0x1.3441350800000p-2, fma(ed, 0x1.f79fef311f12bp-34, lnm * 0.43429448190325182765));
}

__device__ __forceinline__ constexpr int colof(int b, int kB) { return (b >= 5) ? 4 - kB : kB; }

struct Smem {
    // element offsets (in bytes) of the CTA-wide tables and the per-warp areas; computed identically on host and device
    int md, es;                 // padded row lengths of the cosine table / the per-frame energy row (doubles, even)
    size_t win, twA, twU, twU4, u4, prog, pw, dct, warp0, warp_bytes, total;
    __host__ __device__ Smem(int M, int K, int PL, int PWL) {
        md = (M + 2) & ~1;
        es = (2 * M + 2) & ~1;
        while ((es & 15) != 6) es += 2;   // rows of consecutive frames 12 banks apart: the five lanes' 8-byte accesses of two frames do not collide
        size_t o = 0;
        win = o;  o += (size_t)MC * 16;
        twA = o;  o += 7 * 25 * 16;
        twU = o;  o += 75 * 16;
        twU4 = o; o += 30 * 16;
        pw = o;   o += (size_t)2 * LPF * PWL * 16;
        dct = o;  o += (size_t)K * md * 8;
        o = (o + 15) & ~(size_t)15;
        prog = o; o += (size_t)2 * LPF * PL * 4;
        u4 = o;   o += (10 + 60) * 2;
        o = (o + 15) & ~(size_t)15;
        warp0 = o;
        warp_bytes = (size_t)FW * FS * 16 + (size_t)FW * es * 8;
        warp_bytes = (warp_bytes + 15) & ~(size_t)15;
        total = warp0 + (size_t)PAIRS * warp_bytes;
    }
};

template <typename TIn>
__global__ void __launch_bounds__(WARPS * 32, 1) mfcc_lane5_kernel(const Params P) {
    extern __shared__ __align__(16) unsigned char l5_smem[];
    const int M = P.num_coeffs, K = P.n_keep;
    const int PL = P.prog_len, PWL = P.pw_len;
    const Smem L(M, K, PL, PWL);
    const double2* s_win = reinterpret_cast<const double2*>(l5_smem + L.win);
    C* s_twA = reinterpret_cast<C*>(l5_smem + L.twA);
    C* s_twU = reinterpret_cast<C*>(l5_smem + L.twU);
    C* s_twU4 = reinterpret_cast<C*>(l5_smem + L.twU4);
    double2* s_pw = reinterpret_cast<double2*>(l5_smem + L.pw);
    double* s_dct = reinterpret_cast<double*>(l5_smem + L.dct);
    unsigned* s_prog = reinterpret_cast<unsigned*>(l5_smem + L.prog);
    unsigned short* s_u4 = reinterpret_cast<unsigned short*>(l5_smem + L.u4);   // [10] bases, then [60] slots
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    {
        const Tables* __restrict__ T = P.t;
        const double2* w2g = reinterpret_cast<const double2*>(P.win);
        double2* sw = reinterpret_cast<double2*>(l5_smem + L.win);
        for (int i = threadIdx.x; i < MC; i += blockDim.x) sw[i] = __ldg(w2g + i);
        for (int i = threadIdx.x; i < 175; i += blockDim.x) { const double2 w = __ldg(T->twA + i); s_twA[i] = mk<double>(w.x, w.y); }
        for (int i = threadIdx.x; i < 75; i += blockDim.x) { const double2 w = __ldg(T->twU + i); s_twU[i] = mk<double>(w.x, w.y); }
        for (int i = threadIdx.x; i < 30; i += blockDim.x) { const double2 w = __ldg(T->twU4 + i); s_twU4[i] = mk<double>(w.x, w.y); }
        for (int i = threadIdx.x; i < 2 * LPF * PL; i += blockDim.x) s_prog[i] = __ldg(&T->prog[i / PL][i % PL]);
        for (int i = threadIdx.x; i < 2 * LPF * PWL; i += blockDim.x) s_pw[i] = __ldg(&T->pw[i / PWL][i % PWL]);
        for (int i = threadIdx.x; i < K * L.md; i += blockDim.x) {
            const int k = i / L.md, m = i - k * L.md;
            s_dct[i] = (m < M) ? __ldg(P.dct + (size_t)k * M + m) : 0.0;
        }
        for (int i = threadIdx.x; i < 10; i += blockDim.x) s_u4[i] = T->u4base[i];
        for (int i = threadIdx.x; i < 60; i += blockDim.x) s_u4[10 + i] = T->u4slot[i];
    }
    __syncthreads();
    if (lane >= FW * LPF) return;  // lanes 30, 31: no CTA-wide barrier below (the pair barriers count warps)
    // Two warps share a group of six frames: each of the 30 lanes of one warp has a twin in the other, and the twins split every
    // phase's work list (h = which half).  The frames' residency in shared memory is what limits the SM to 48 frames; splitting
    // them over twice the warps doubles the latency hiding at the same footprint.  Named barrier 1 + pair orders the phases.
    const int pair = warp >> 1, h = warp & 1;
    const int q = lane / LPF, s = lane - q * LPF, v10 = h * LPF + s;
    auto pair_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(pair + 1) : "memory"); };
    C* const fb = reinterpret_cast<C*>(l5_smem + L.warp0 + (size_t)pair * L.warp_bytes) + q * FS;   // this frame's 200 (+5) slots
    double* const e_row = reinterpret_cast<double*>(l5_smem + L.warp0 + (size_t)pair * L.warp_bytes + (size_t)FW * FS * 16) + q * L.es;
    // pass-B twiddles W25^(s·kB), kB = 1..4, stay in registers
    C twB[4];
#pragma unroll
    for (int kB = 1; kB <= 4; ++kB) { const double2 w = __ldg(P.t->twB + (kB - 1) * 5 + s); twB[kB - 1] = mk<double>(w.x, w.y); }
    const int n_rounds = P.t->n_rounds[h];
    const int* __restrict__ round_len = P.t->round_len[h];
    if (v10 == 0) fb[kZeroSlot] = mk<double>(0.0, 0.0);   // never written again: the pad slots are nobody's output
    const unsigned* const prog = s_prog + v10 * PL;
    const double2* const pw = s_pw + v10 * PWL;

    const int64_t n_groups = (P.n_frames + FW - 1) / FW;
    const int64_t g_step = (int64_t)gridDim.x * PAIRS;
    // frame of this lane in group g: pointer to its first sample; lanes of a ragged last group shadow the last frame (no global stores)
    auto frame_of = [&](int64_t g, int64_t& f, bool& valid) -> const TIn* {
        const int64_t f_raw = g * FW + q;
        valid = f_raw < P.n_frames;
        f = valid ? f_raw : P.n_frames - 1;
        const int64_t seg = f / P.seg_frames;
        return reinterpret_cast<const TIn*>(P.base) + seg * P.seg_stride + (f - seg * P.seg_frames) * P.stride;
    };
    int64_t g = (int64_t)blockIdx.x * PAIRS + pair;
    int64_t f = 0;
    bool valid = false;
    const TIn* __restrict__ x = (g < n_groups) ? frame_of(g, f, valid) : nullptr;
    for (; g < n_groups; g += g_step) {
        // the next group's samples on their way into L2 while this one is transformed: the ten twins of a frame cover its 1 600 bytes
        int64_t f_next = 0;
        bool valid_next = false;
        const TIn* x_next = nullptr;
        if (g + g_step < n_groups) {
            x_next = frame_of(g + g_step, f_next, valid_next);
            const char* pf = reinterpret_cast<const char*>(x_next + 40 * v10);   // this twin's 40 samples: first and last byte
            prefetch_l2(pf);
            prefetch_l2(pf + 40 * sizeof(TIn) - 4);
        }
        // ---- pass A: global → window → radix 8 → twiddle → slots 25u + n1.  In THIS pass a lane owns a butterfly position
        // n1 = lane (25 of the 30 lanes) and walks three of the group's frames (warp h: frames 3h .. 3h + 2), so the eight window
        // pairs and seven twiddles of its position are loaded once per group instead of once per frame — table operands cost
        // a lane the same shared-memory wavefronts as data, and with one frame per five lanes they were 40 % of this pass's
        // traffic (measured: the pass without its table loads ran the whole kernel 10 % faster).  The frames' sample pointers
        // come from the lanes that own the frames in every other phase (lane 5q).
        {
            unsigned long long xq[3];
#pragma unroll
            for (int qq = 0; qq < 3; ++qq) xq[qq] = __shfl_sync(kMask, (unsigned long long)reinterpret_cast<uintptr_t>(x), LPF * (3 * h + qq));
            if (lane < 25) {
                const int n1 = lane;
                C tw[7];
#pragma unroll
                for (int u = 1; u < 8; ++u) tw[u - 1] = s_twA[(u - 1) * 25 + n1];
                const double2* __restrict__ ws = s_win + n1;
                C* __restrict__ o = fb - q * FS + (3 * h) * FS + n1;   // frame 3h's buffer
#pragma unroll 1
                for (int qq = 0; qq < 3; ++qq) {
                    const TIn* __restrict__ xs = reinterpret_cast<const TIn*>(qq == 0 ? xq[0] : (qq == 1 ? xq[1] : xq[2])) + 2 * n1;
                    C v[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) {
                        const typename RawPair<TIn>::type raw = load_raw<TIn>(xs + 50 * t);
                        const double2 w = ws[25 * t];
                        v[t] = mk<double>((double)raw.x * w.x, (double)raw.y * w.y);
                    }
                    mfcc_fast::bfly<8, double>(v);
                    o[0] = v[0];
#pragma unroll
                    for (int u = 1; u < 8; ++u) o[25 * u] = cmulf(v[u], tw[u - 1]);
                    o += FS;
                }
            }
        }
        pair_sync();
        // ---- pass B: radix 5 inside every 25-block (blocks 4h .. 4h + 3, two in flight), transposed store ------------------------
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
            const int b0 = 4 * h + 2 * r;
            C* __restrict__ blk = fb + 25 * b0;
            C v[2][5];
#pragma unroll
            for (int bb = 0; bb < 2; ++bb)
#pragma unroll
                for (int t = 0; t < 5; ++t) v[bb][t] = blk[25 * bb + s + 5 * t];
#pragma unroll
            for (int bb = 0; bb < 2; ++bb) {
                mfcc_fast::bfly<5, double>(v[bb]);
#pragma unroll
                for (int kB = 1; kB < 5; ++kB) v[bb][kB] = cmulf(v[bb][kB], twB[kB - 1]);
            }
            __syncwarp(kMask);   // a block is read and written by the five lanes of ONE warp
#pragma unroll
            for (int bb = 0; bb < 2; ++bb) {
                const bool mir = (b0 + bb) >= 5;   // blocks 5..7 store their columns mirrored
                C* __restrict__ ob = blk + 25 * bb + 5 * s + (mir ? 4 : 0);
#pragma unroll
                for (int kB = 0; kB < 5; ++kB) ob[mir ? -kB : kB] = v[bb][kB];
            }
        }
        pair_sync();
        // ---- pass C + untangle: units 1, 2 (h = 0) or 3 and the table-driven fourth unit (h = 1) ---------------------------------
        // A unit's ten butterfly inputs are two whole columns of two blocks; the five lanes of the warp running it cover those
        // blocks completely, so after a __syncwarp they may store the blocks' fifty bins in ANY arrangement: bin k goes to slot
        // 25·(k mod 8) + k div 8 ("kA-major"), where consecutive bins are 25 slots = one bank group apart.
        auto unit = [&](int u) {   // butterflies (u, s) and (8 − u, 4 − s)
            const C* __restrict__ ca = fb + 25 * u + s;
            const C* __restrict__ cb = fb + 25 * (8 - u) + s;   // mirrored columns: col(8 − u, 4 − s) = s
            const C* __restrict__ tw = s_twU + (u - 1) * 25 + s;
            C A[5], B[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) { A[j] = ca[5 * j]; B[j] = cb[5 * j]; }
            __syncwarp(kMask);
            mfcc_fast::bfly<5, double>(A);
            mfcc_fast::bfly<5, double>(B);
            C* __restrict__ oa = fb + 25 * u + s;               // bin u + 8s + 40kC        → 25u + (s + 5kC)
            C* __restrict__ ob = fb + 25 * (8 - u) + 24 - s;    // bin 200 − that            → 25(8 − u) + (4 − s) + 5(4 − kC)
#pragma unroll
            for (int kC = 0; kC < 5; ++kC) {
                C pa, pb;
                pair_op(A[kC], B[4 - kC], tw[kC * 5], pa, pb);
                oa[5 * kC] = pa;
                ob[-5 * kC] = pb;
            }
        };
        if (h == 0) {
            unit(1);
            unit(2);
        } else {
            unit(3);
            // unit 4: the butterflies of blocks 0 and 4 (lane 4: the two self-paired ones)
            C* __restrict__ ca = fb + s_u4[s];
            C* __restrict__ cb = fb + s_u4[5 + s];
            C A[5], B[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) { A[j] = ca[5 * j]; B[j] = cb[5 * j]; }
            __syncwarp(kMask);
            mfcc_fast::bfly<5, double>(A);
            mfcc_fast::bfly<5, double>(B);
            const bool sg = (s == 4);
            // regular lanes pair (A[i], B[4 − i]); lane 4 pairs inside each butterfly: (A0,A0) (A1,A4) (A2,A3) (B0,B4) (B1,B3) (B2,B2)
            auto sel = [&](const C a, const C b) { return mk<double>(sg ? a.x : b.x, sg ? a.y : b.y); };
            const C p3 = sel(B[0], A[3]), p4 = sel(B[1], A[4]);
            const C q0 = sel(A[0], B[4]), q1 = sel(A[4], B[3]), q2 = sel(A[3], B[2]), q3 = sel(B[4], B[1]), q4 = sel(B[3], B[0]);
            const unsigned short* __restrict__ sl = s_u4 + 10 + s;
            C pa, pb;
            pair_op(A[0], q0, s_twU4[0 * 5 + s], pa, pb); fb[sl[0]] = pa;  fb[sl[5]] = pb;
            pair_op(A[1], q1, s_twU4[1 * 5 + s], pa, pb); fb[sl[10]] = pa; fb[sl[15]] = pb;
            pair_op(A[2], q2, s_twU4[2 * 5 + s], pa, pb); fb[sl[20]] = pa; fb[sl[25]] = pb;
            pair_op(p3, q3, s_twU4[3 * 5 + s], pa, pb);   fb[sl[30]] = pa; fb[sl[35]] = pb;
            pair_op(p4, q4, s_twU4[4 * 5 + s], pa, pb);   fb[sl[40]] = pa; fb[sl[45]] = pb;
            if (sg) {
                pair_op(B[2], B[2], s_twU4[5 * 5 + s], pa, pb);
                fb[sl[50]] = pa;
            }
        }
        pair_sync();
        // ---- band sums (spectrum.rs:421-435): interval j = rising half of band j (power) and falling half of band j − 1 (magnitude);
        // this lane's intervals: a header word (bins | j << 16), then the byte offset of every bin's slot, ascending bins
        {
            const unsigned* __restrict__ pp = prog;
            const double2* __restrict__ ww = pw;
            const unsigned char* __restrict__ fbb = reinterpret_cast<const unsigned char*>(fb);
#pragma unroll 1
            for (int r = 0; r < n_rounds; ++r) {
                const int len = __ldg(round_len + r);   // the same for the whole warp
                const unsigned j = *pp++;
                double up = 0., down = 0.;
#pragma unroll 2
                for (int c = 0; c < len; ++c) {
                    const double2 sp = *reinterpret_cast<const double2*>(fbb + pp[c]);
                    const double2 w = ww[c];
                    up = fma(sp.x, w.x, up);
                    down = fma(sp.y, w.y, down);
                }
                pp += len;
                ww += len;
                if (j < (unsigned)M) e_row[j] = up;
                if (j >= 1u && j <= (unsigned)M) e_row[M + j - 1] = down;
            }
        }
        pair_sync();
#pragma unroll 1
        for (int w = v10; w < M; w += 2 * LPF) {
            double e = band_log10(e_row[w] + e_row[M + w]);
            e = (e > 1.0e-10) ? e : 1.0e-10;  // f64::max(1e-10): NaN → 1e-10
            e_row[w] = e;
            if (P.energies_out && valid) {
                const size_t o = (size_t)f * M + w;
                if (P.out_f64) reinterpret_cast<double*>(P.energies_out)[o] = e;
                else reinterpret_cast<float*>(P.energies_out)[o] = (float)e;
            }
        }
        if (v10 == 0 && (M & 1)) e_row[M] = 0.0;   // the pad the paired loads of the DCT read (its cosine entry is 0; keep it finite)
        pair_sync();
        // ---- DCT-II ×2, first n_keep rows (spectrum.rs:391-398): rows v, v + 10 share every load of the energies; four independent
        // sums hide the DFMA latency ---------------------------------------------------------------------------------------------
#pragma unroll 1
        for (int kb = 0; kb < K; kb += 4 * LPF) {
            const int k0r = kb + v10, k1r = k0r + 2 * LPF;
            const bool has0 = k0r < K, has1 = k1r < K;
            if (!__any_sync(kMask, has0)) break;
            const bool two = __any_sync(kMask, has1);            // warp-uniform: does anybody have a second row?
            const int k0 = has0 ? k0r : 0, k1 = has1 ? k1r : k0;
            const double2* __restrict__ e2 = reinterpret_cast<const double2*>(e_row);
            const double2* __restrict__ r0 = reinterpret_cast<const double2*>(s_dct + (size_t)k0 * L.md);
            const double2* __restrict__ r1 = reinterpret_cast<const double2*>(s_dct + (size_t)k1 * L.md);
            double a0 = 0., b0 = 0., a1 = 0., b1 = 0.;
            if ((M & 3) == 0) {
                // cos(πk(2m+1)/2M) at m and M−1−m differ by the sign (−1)^k, and rows k, k + 10 have the same parity: fold the
                // energies first — half the cosine loads and products
                const double sg = (k0 & 1) ? -1.0 : 1.0;
                const int Q4 = M >> 2, H = M >> 1;
#pragma unroll 2
                for (int m = 0; m < Q4; ++m) {
                    const double2 lo = e2[m], hi = e2[H - 1 - m], c0 = r0[m];
                    const double x0 = fma(sg, hi.y, lo.x), x1 = fma(sg, hi.x, lo.y);
                    a0 = fma(x0, c0.x, a0); b0 = fma(x1, c0.y, b0);
                    if (two) {
                        const double2 c1 = r1[m];
                        a1 = fma(x0, c1.x, a1); b1 = fma(x1, c1.y, b1);
                    }
                }
            } else {
                const int H = (M + 1) >> 1;
#pragma unroll 2
                for (int m = 0; m < H; ++m) {
                    const double2 ev = e2[m], c0 = r0[m];
                    a0 = fma(ev.x, c0.x, a0); b0 = fma(ev.y, c0.y, b0);
                    if (two) {
                        const double2 c1 = r1[m];
                        a1 = fma(ev.x, c1.x, a1); b1 = fma(ev.y, c1.y, b1);
                    }
                }
            }
            if (valid) {
                auto put = [&](int k, double val) {
                    const size_t o = (size_t)f * K + k;
                    if (P.out_f64) reinterpret_cast<double*>(P.out)[o] = val;
                    else reinterpret_cast<float*>(P.out)[o] = (float)val;
                };
                if (has0) put(k0, 2. * (a0 + b0));
                if (has1) put(k1, 2. * (a1 + b1));
            }
        }
        // (no barrier here: the next group's pass A writes the frame buffers, which nobody reads after the band sums, and its
        // band sums write the energy rows three barriers from now)
        x = x_next; f = f_next; valid = valid_next;
    }
}

// ---- host: tables ------------------------------------------------------------------------------------------------------------
static inline double2 l5_w(int n, long long e, double scale) {
    const double PI = 3.14159265358979323846264338327950288;
    e %= n;
    const double ang = -2.0 * PI * (double)e / (double)n;
    return make_double2(scale * cos(ang), scale * sin(ang));
}
static inline int l5_slot(int k) {  // bin k < 200 → its slot in the kA-major spectrum layout; Nyquist (k = 200) → 200
    if (k == MC) return MC;
    return 25 * (k % 8) + k / 8;
}
// slot of INPUT j = 0 of pass C's butterfly (kA, kB): pass B's transposed store, blocks 5..7 with mirrored columns
static inline int l5_in_slot(int kA, int kB) { return 25 * kA + ((kA >= 5) ? 4 - kB : kB); }

// bins: the num_coeffs + 2 filter-bank edges
// returns false if a program does not fit its table row (the caller then keeps mfcc_warp_kernel for this parameter set)
static bool build_tables(Tables& T, const int* bins, int num_coeffs, const double* wu, const double* wd) {
    memset(&T, 0, sizeof(T));
    for (int u = 1; u < 8; ++u)
        for (int n1 = 0; n1 < 25; ++n1) T.twA[(u - 1) * 25 + n1] = l5_w(200, (long long)n1 * u, 1.0);
    for (int kB = 1; kB < 5; ++kB)
        for (int s = 0; s < 5; ++s) T.twB[(kB - 1) * 5 + s] = l5_w(25, (long long)s * kB, 1.0);
    for (int kA = 1; kA <= 3; ++kA)
        for (int kC = 0; kC < 5; ++kC)
            for (int s = 0; s < 5; ++s) T.twU[(kA - 1) * 25 + kC * 5 + s] = l5_w(N, kA + 8 * s + 40 * kC, 0.5);
    // fourth unit: lane s runs butterflies c and c' of blocks 0 and 4
    const int cA[5][2] = {{4, 0}, {4, 1}, {0, 1}, {0, 2}, {0, 0}};
    const int cB[5][2] = {{4, 4}, {4, 3}, {0, 4}, {0, 3}, {4, 2}};
    for (int s = 0; s < 5; ++s) {
        T.u4base[s] = (unsigned short)l5_in_slot(cA[s][0], cA[s][1]);
        T.u4base[5 + s] = (unsigned short)l5_in_slot(cB[s][0], cB[s][1]);
        auto kof = [](const int* c, int kC) { return c[0] + 8 * c[1] + 40 * kC; };
        int ka[6], kb[6];
        if (s < 4) {
            for (int i = 0; i < 5; ++i) { ka[i] = kof(cA[s], i); kb[i] = kof(cB[s], 4 - i); }
            ka[5] = ka[0]; kb[5] = kb[0];  // unused
        } else {
            const int a[6] = {0, 40, 80, 20, 60, 100}, b[6] = {200, 160, 120, 180, 140, 100};
            for (int i = 0; i < 6; ++i) { ka[i] = a[i]; kb[i] = b[i]; }
        }
        for (int op = 0; op < 6; ++op) {
            T.twU4[op * 5 + s] = l5_w(N, ka[op], 0.5);
            T.u4slot[(2 * op) * 5 + s] = (unsigned short)l5_slot(ka[op]);
            T.u4slot[(2 * op + 1) * 5 + s] = (unsigned short)l5_slot(kb[op]);
        }
    }
    // the intervals sorted by length, five at a time to warp 0, 1, 1, 0, 0, 1, 1, ... (see Tables).  Within a round the five lanes
    // walk five different intervals in lock step and read one spectrum slot each per step: which lane takes which interval, and
    // how many zero-slot entries are put IN FRONT of each (0..3, shifting its phase), is chosen by simulating the shared-memory
    // wavefronts of the round's steps (16-byte accesses are served per quarter warp; two lanes collide when their slots share a
    // bank group) — 120 lane orders, the shifts fixed greedily lane by lane.
    std::vector<int4> iv;
    for (int j = 0; j <= num_coeffs; ++j) iv.push_back(make_int4(j, bins[j], bins[j + 1] > bins[j] ? bins[j + 1] : bins[j], 0));
    std::stable_sort(iv.begin(), iv.end(), [](const int4& a, const int4& b) { return a.z - a.y > b.z - b.y; });
    auto slot_of_bin = [](int k) { return l5_slot(k <= MC ? k : N - k); };
    // slot read by a lane at step c: interval t shifted by d
    auto slot_at = [&](const int4& t, int d, int c) { return (c >= d && c < d + (t.z - t.y)) ? slot_of_bin(t.y + c - d) : kZeroSlot; };
    // wavefronts of one step: lanes (q, s) = 5q + s of the placed lanes (mask), slots sl[s]
    auto step_wavefronts = [&](const int* sl, unsigned mask) {
        int total = 0;
        for (int qw = 0; qw < 4; ++qw) {
            int addr[8][8], cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            for (int l = 8 * qw; l < 8 * qw + 8 && l < FW * LPF; ++l) {
                const int q = l / LPF, ss = l % LPF;
                if (!(mask & (1u << ss))) continue;
                const int e = q * FS + sl[ss], b = e & 7;
                bool seen = false;
                for (int i = 0; i < cnt[b]; ++i) seen |= (addr[b][i] == e);
                if (!seen) addr[b][cnt[b]++] = e;
            }
            int worst = 0;
            for (int b = 0; b < 8; ++b) worst = cnt[b] > worst ? cnt[b] : worst;
            total += worst;
        }
        return total;
    };
    int n[2 * LPF] = {0}, nw[2 * LPF] = {0};
    T.n_rounds[0] = T.n_rounds[1] = 0;
    for (size_t first = 0, turn = 0; first < iv.size(); first += LPF, ++turn) {
        const int hh = (int)(((turn + 1) >> 1) & 1);   // warp 0, 1, 1, 0, 0, 1, 1, ...: the sorted lengths' sums stay level
        const int r = T.n_rounds[hh]++;
        int4 mem[LPF];
        for (int i = 0; i < LPF; ++i) mem[i] = (first + i < iv.size()) ? iv[first + i] : make_int4((int)kIdle, 0, 0, 0);
        const int longest = mem[0].z - mem[0].y;
        constexpr int kMaxShift = 3;
        int perm[LPF] = {0, 1, 2, 3, 4}, best_perm[LPF] = {0, 1, 2, 3, 4}, best_d[LPF] = {0, 0, 0, 0, 0};
        long best_cost = -1;
        do {
            int d[LPF] = {0, 0, 0, 0, 0};
            long cost = 0;
            unsigned mask = 0;
            for (int ss = 0; ss < LPF; ++ss) {   // place lane ss: interval mem[perm[ss]], the shift that adds the fewest wavefronts
                mask |= 1u << ss;
                long best_c = -1;
                int best_shift = 0;
                for (int sh = 0; sh <= kMaxShift; ++sh) {
                    d[ss] = sh;
                    int len = longest + kMaxShift;
                    long c_sum = 0;
                    for (int c = 0; c < len; ++c) {
                        int sl[LPF];
                        for (int l = 0; l <= ss; ++l) sl[l] = slot_at(mem[perm[l]], d[l], c);
                        c_sum += step_wavefronts(sl, mask);
                    }
                    c_sum += 8L * sh * (ss == 0 ? 1 : 0);   // a shift of every lane only lengthens the round
                    if (best_c < 0 || c_sum < best_c) { best_c = c_sum; best_shift = sh; }
                }
                d[ss] = best_shift;
                cost = best_c;
            }
            int len = 0;
            for (int ss = 0; ss < LPF; ++ss) len = std::max(len, d[ss] + (mem[perm[ss]].z - mem[perm[ss]].y));
            cost += 9L * (len - longest) - 4L * (longest + kMaxShift - len);   // a step costs ~9 more wavefronts (weights, offsets) + issue; unused tail steps cost nothing
            if (best_cost < 0 || cost < best_cost) {
                best_cost = cost;
                for (int i = 0; i < LPF; ++i) { best_perm[i] = perm[i]; best_d[i] = d[i]; }
            }
        } while (std::next_permutation(perm, perm + LPF));
        int len = 0;
        for (int ss = 0; ss < LPF; ++ss) len = std::max(len, best_d[ss] + (mem[best_perm[ss]].z - mem[best_perm[ss]].y));
        T.round_len[hh][r] = len;
        for (int ss = 0; ss < LPF; ++ss) {
            const int v = hh * LPF + ss;
            const int4 t = mem[best_perm[ss]];
            if (n[v] + len + 16 > kMaxProg) return false;
            T.prog[v][n[v]++] = (unsigned)t.x;
            for (int c = 0; c < len; ++c) {
                const bool real = c >= best_d[ss] && c < best_d[ss] + (t.z - t.y);
                const int k = t.y + c - best_d[ss];
                T.prog[v][n[v]++] = (unsigned)(real ? slot_of_bin(k) : kZeroSlot) * 16u;
                T.pw[v][nw[v]++] = real ? make_double2(wu[k], wd[k]) : make_double2(0.0, 0.0);
            }
        }
    }
    T.prog_len = 1;
    T.pw_len = 1;
    for (int v = 0; v < 2 * LPF; ++v) {
        if (n[v] > T.prog_len) T.prog_len = n[v];
        if (nw[v] > T.pw_len) T.pw_len = nw[v];
    }
    T.prog_len |= 1;                              // odd row length: the lanes' offset words in different banks
    while ((T.pw_len & 7) != 1) ++T.pw_len;       // rows one bank group apart: the lanes' weight loads do not collide
    return true;
}

}  // namespace mfcc_lane5
