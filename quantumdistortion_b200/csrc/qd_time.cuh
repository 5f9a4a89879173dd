// qd_time.cuh -- time-domain kernels of the STFT path: lookahead limiter + mix, Linkwitz-Riley
// crossover + low-band processing, elementwise distortion.
//
// Both recurrences run in float64 (SURVEY.md section 0.6), each parallelised the way its memory allows:
//   limiter   u_n = c * max(u_{n-1}, e_n)              dsp/limiter.py:62-77
//             30 ms release = a memory of ~57 000 samples: a parallel scan, associative on pairs (a, b): u -> max(a*u, b).
//             One CTA streams one clip in chunks; every thread owns KS consecutive samples, runs the recurrence over
//             them from a zero state, the per-thread aggregates are combined with warp shuffles (+ one shared-memory
//             hop across warps), and the thread re-runs its samples from its true incoming state.
//   biquad    z_{n+1} = A z_n + B x_n (DF2T state)     scipy sosfilt, dsp/crossover.py:96-97
//             pole radius 0.97: a memory of ~1 600 samples: independent tiles with a warm-up halo, one thread per tile
//             (crossover_kernel below).
#pragma once
#include "qd_common.cuh"

namespace qd {

constexpr int QD_TT = 256;          // threads per CTA
constexpr int QD_KS = 8;            // samples per thread per chunk
constexpr int QD_CHUNK = QD_TT * QD_KS;

QD_DEV int padi(int i) { return i + (i >> 5); }

struct LimiterArgs {
    const float *x;       // [batch, n] limiter input (x_post_quant)
    const float *dry;     // [batch, n] dry signal for the mix (tap_input)
    const float *low;     // optional [batch, n] processed low band (multiband recombine)
    const float *orig;    // optional [batch, n] original input (delta listen)
    float *y;             // [batch, n]
    long long n;
    int limiter_on;
    int lookahead;        // L >= 1
    double ceiling;
    double c;             // release coefficient
    float wet, dry_gain, trim;
    int apply_mix;        // 0: y = limited (stage-level entry point)
    int apply_trim;
    const float *clip_peak;   // optional [batch]: max |x| per clip from the producing spectral pass.  A clip that never
                              // exceeds the ceiling has gain exactly 1 (dsp/limiter.py:68-76): its limiter is skipped,
                              // and with an identity mix in place (x == y) the CTA has nothing to do at all.
    const int64_t *starts;    // optional ragged batch, as SpecArgsT::starts (null: clip * n, n samples each)
    const int32_t *lengths;
    int clip0;
};

// 8 consecutive samples of one clip starting at s (zero past the end); 2 x 16-byte loads when aligned
QD_DEV void load8(const float *x, long long s, long long n, bool vec, float (&v)[QD_KS]) {
    if (vec && s + QD_KS <= n) {
        const float4 lo = *reinterpret_cast<const float4 *>(x + s);
        const float4 hi = *reinterpret_cast<const float4 *>(x + s + 4);
        v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
        v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
    } else {
#pragma unroll
        for (int k = 0; k < QD_KS; ++k) v[k] = (s + k < n) ? x[s + k] : 0.0f;
    }
}

QD_DEV double limiter_e(float peak, double ceiling) {  // dsp/limiter.py:68-72
    const double p = (double)peak;
#ifdef QD_EMU
    return (p > ceiling && p > 1e-12) ? 1.0 - ceiling / p : 0.0;
#else
    // 1 - ceiling / p without the IEEE division subroutine, which was 29 % of the kernel's instructions (it runs twice
    // per sample, ncu): the peak is a float32 value, so MUFU.RCP gives 1/p to 2^-23 and two Newton steps in float64
    // square that error twice (2^-46, 2^-92: below the rounding of the steps themselves); e = fma(-ceiling, r, 1) then
    // differs from the correctly rounded 1 - ceiling / p by about 2^-52 absolute -- the same size as the rounding of the
    // reference's own two operations, and 2^-29 of the float32 step of y = float32(x (1 - u)).
    float r0;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(peak));
    double r = (double)r0;
    r = fma(fma(-p, r, 1.0), r, r);
    r = fma(fma(-p, r, 1.0), r, r);
    const double e = fma(-ceiling, r, 1.0);
    return (p > ceiling && p > 1e-12) ? e : 0.0;   // a select: the lanes with a tiny or zero peak never use r
#endif
}

// dsp/limiter.py:14-80 then dsp/pipeline.py:894-910, 1096, 1371-1375.
// Streaming structure: a thread keeps its 8 samples of the current chunk and of the next one in registers
// (the next chunk doubles as the lookahead) and prefetches the chunk after that, so no global-memory
// latency sits on the per-chunk critical path; shared buffers are double-buffered by chunk parity, which
// leaves two __syncthreads() per chunk.
__global__ void __launch_bounds__(QD_TT, 3) limiter_mix_kernel(const LimiterArgs a) {
    QD_DYN_SMEM(smem);
    const int L = a.lookahead;
    const int span = QD_CHUNK + L + 8;                // |x| kept per chunk: the chunk and its lookahead
    const int abs_stride = (padi(span) + 8 + 3) & ~3;
    const int ngroups = span / QD_KS;
    const int gmax_stride = (ngroups + 2 + 3) & ~3;
    float *s_abs0 = reinterpret_cast<float *>(smem);
    float *s_gmax0 = s_abs0 + 2 * abs_stride;
    double *s_warp0 = reinterpret_cast<double *>((reinterpret_cast<uintptr_t>(s_gmax0 + 2 * gmax_stride) + 7) & ~(uintptr_t)7);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NWARP = QD_TT / 32;
    const ClipLoc cs = clip_loc(a, (int)blockIdx.x);
    const size_t base = (size_t)cs.base;
    const long long n = cs.n;
    const float *x = a.x + base;
    const bool vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    const bool vec_out = (reinterpret_cast<uintptr_t>(a.y + base) & 15) == 0;
    const bool need_dry = a.apply_mix && a.dry_gain != 0.0f;
    const bool clip_quiet = a.clip_peak != nullptr && !((double)a.clip_peak[cs.idx] > a.ceiling);
    const bool limiter_on = a.limiter_on && !clip_quiet;
    if (!limiter_on && a.x == a.y && !need_dry && !a.low && !a.orig && (!a.apply_mix || (a.wet == 1.0f && !a.apply_trim)))
        return;   // y = float32(x * 1) in place
    const double c = a.c;
    double c_ks = 1.0;
#pragma unroll
    for (int k = 0; k < QD_KS; ++k) c_ks *= c;
    double c_32 = c_ks;  // c_ks^32
#pragma unroll
    for (int k = 0; k < 5; ++k) c_32 *= c_32;
    double lanepow = 1.0;  // c_ks^lane
    {
        double p = c_ks;
        int l = lane;
        while (l) { if (l & 1) lanepow *= p; p *= p; l >>= 1; }
    }
    double carry = 0.0;  // u at the end of the previous chunk
    const int look_threads = (L + 8 + QD_KS - 1) / QD_KS;  // threads whose next-chunk samples are lookahead
    const bool fast = limiter_on && L >= QD_KS && L + 8 <= QD_CHUNK;

    float cur[QD_KS], nxt[QD_KS], nn[QD_KS];
    load8(x, (long long)tid * QD_KS, n, vec, cur);
    load8(x, (long long)QD_CHUNK + (long long)tid * QD_KS, n, vec, nxt);
    int par = 0;
    for (long long n0 = 0; n0 < n; n0 += QD_CHUNK, par ^= 1) {
        load8(x, n0 + 2LL * QD_CHUNK + (long long)tid * QD_KS, n, vec, nn);  // lands during this chunk
        float *s_abs = s_abs0 + par * abs_stride;
        float *s_gmax = s_gmax0 + par * gmax_stride;
        double *s_warp = s_warp0 + par * (NWARP + 2);
        double u_in = 0.0;
        float peak[QD_KS];
        bool lim_active = false;
        if (limiter_on) {
            // ---- |x| of the chunk and of its lookahead into shared memory, with per-group maxima
            if (fast) {
                float m = 0.0f;
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) {
                    const float v = fabsf(cur[k]);
                    s_abs[padi(tid * QD_KS + k)] = v;
                    m = fmaxf(m, v);
                }
                s_gmax[tid] = m;
                if (tid < look_threads) {
                    float m2 = 0.0f;
#pragma unroll
                    for (int k = 0; k < QD_KS; ++k) {
                        const float v = fabsf(nxt[k]);
                        s_abs[padi(QD_CHUNK + tid * QD_KS + k)] = v;
                        m2 = fmaxf(m2, v);
                    }
                    s_gmax[QD_TT + tid] = m2;
                }
                __syncthreads();
            } else {  // very short or very long lookahead: generic staging from global memory
                for (int i = tid; i < span; i += QD_TT) {
                    const long long s = n0 + i;
                    s_abs[padi(i)] = s < n ? fabsf(x[s]) : 0.0f;
                }
                __syncthreads();
                for (int g = tid; g < ngroups; g += QD_TT) {
                    float m = 0.0f;
#pragma unroll
                    for (int k = 0; k < QD_KS; ++k) m = fmaxf(m, s_abs[padi(g * QD_KS + k)]);
                    s_gmax[g] = m;
                }
                __syncthreads();
            }
            // ---- forward-window maxima of this thread's KS samples
            if (L >= QD_KS) {
                const int q = L / QD_KS, rem = L % QD_KS;
                float mc = 0.0f;  // groups tid+1 .. tid+q-1 lie inside every window
                for (int g = tid + 1; g < tid + q; ++g) mc = fmaxf(mc, s_gmax[g]);
                float suf = 0.0f;
                float sufv[QD_KS];
#pragma unroll
                for (int k = QD_KS - 1; k >= 0; --k) { suf = fmaxf(suf, fabsf(cur[k])); sufv[k] = suf; }
                // prefix maxima over the two groups after the common ones: pab[j] = max of their first j samples
                float pab[2 * QD_KS + 1];
                pab[0] = 0.0f;
#pragma unroll
                for (int k = 0; k < 2 * QD_KS; ++k) pab[k + 1] = fmaxf(pab[k], s_abs[padi((tid + q) * QD_KS + k)]);
#pragma unroll
                for (int r = 0; r < QD_KS; ++r) {
                    // window [8t+r, 8t+r+L): tail of own group, common groups, first r+rem samples after them
                    float tailmax = 0.0f;
#pragma unroll
                    for (int j = 0; j < 2 * QD_KS; ++j) tailmax = (j == r + rem) ? pab[j] : tailmax;  // static indices only
                    peak[r] = fmaxf(fmaxf(sufv[r], mc), tailmax);
                }
            } else {
#pragma unroll
                for (int r = 0; r < QD_KS; ++r) {
                    float m = 0.0f;
                    for (int k = 0; k < L; ++k) m = fmaxf(m, s_abs[padi(tid * QD_KS + r + k)]);
                    peak[r] = m;
                }
            }
            // ---- nothing above the ceiling in this chunk and no release in progress: the gain is exactly 1
            //      (dsp/limiter.py:68-76 leaves g = 1 - (1 - 1) * c = 1), so the float64 scan is skipped.
            float pk = 0.0f;
#pragma unroll
            for (int k = 0; k < QD_KS; ++k) pk = fmaxf(pk, peak[k]);
            // a release tail below 2^-54 no longer changes g = 1 - u in float64: treat it as finished
            const int engaged = __syncthreads_or((double)pk > a.ceiling && pk > 1e-12f) || carry > 5e-17;
            if (!engaged) {
                carry = 0.0;
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) peak[k] = 0.0f;  // e = 0 everywhere, u stays 0
            } else {
            // ---- local aggregate (from the chunk carry for thread 0), then scan across the CTA
            double u = (tid == 0) ? carry : 0.0;
#pragma unroll
            for (int k = 0; k < QD_KS; ++k) u = c * fmax(u, limiter_e(peak[k], a.ceiling));
            double b = u;
            double apow = c_ks;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double o = __shfl_up_sync(QD_FULL, b, d);
                if (lane >= d) b = fmax(apow * o, b);
                apow *= apow;
            }
            if (lane == 31) s_warp[warp] = b;
            double excl = __shfl_up_sync(QD_FULL, b, 1);
            if (lane == 0) excl = 0.0;
            __syncthreads();
            double acc = 0.0, wprev = 0.0;  // aggregates of the warps before this one / of all warps
#pragma unroll
            for (int w = 0; w < NWARP; ++w) {
                if (w == warp) wprev = acc;
                acc = fmax(c_32 * acc, s_warp[w]);
            }
            u_in = (tid == 0) ? carry : fmax(lanepow * wprev, excl);
            carry = acc;  // inclusive value of the last thread = state entering the next chunk
            }
            lim_active = engaged != 0;
        }
        // ---- apply: y = float32(x * g), mix, trim, recombine, delta
        const long long s0 = n0 + (long long)tid * QD_KS;
        float out[QD_KS];
        double u = u_in;
#pragma unroll
        for (int k = 0; k < QD_KS; ++k) {
            float w = cur[k];
            if (lim_active) {
                u = c * fmax(u, limiter_e(peak[k], a.ceiling));  // 0 <= u < 1, so the reference's clip is a no-op
                w = (float)((double)cur[k] * (1.0 - u));
            }
            out[k] = w;
        }
        if (a.apply_mix) {
            float t[QD_KS];
            if (need_dry) {
                load8(a.dry + base, s0, n, vec && ((reinterpret_cast<uintptr_t>(a.dry + base) & 15) == 0), t);
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) out[k] = __fadd_rn(__fmul_rn(a.wet, out[k]), __fmul_rn(a.dry_gain, t[k]));
            } else {
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) out[k] = __fadd_rn(__fmul_rn(a.wet, out[k]), 0.0f);  // (1-dw) * dry = 0
            }
            if (a.apply_trim) {
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) out[k] = __fmul_rn(out[k], a.trim);
            }
            if (a.low) {
                load8(a.low + base, s0, n, vec && ((reinterpret_cast<uintptr_t>(a.low + base) & 15) == 0), t);
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) out[k] = __fadd_rn(t[k], out[k]);
            }
            if (a.orig) {
                load8(a.orig + base, s0, n, vec && ((reinterpret_cast<uintptr_t>(a.orig + base) & 15) == 0), t);
#pragma unroll
                for (int k = 0; k < QD_KS; ++k) out[k] = __fsub_rn(t[k], out[k]);
            }
        }
        float *yo = a.y + base;
        if (vec_out && s0 + QD_KS <= n) {
            *reinterpret_cast<float4 *>(yo + s0) = make_float4(out[0], out[1], out[2], out[3]);
            *reinterpret_cast<float4 *>(yo + s0 + 4) = make_float4(out[4], out[5], out[6], out[7]);
        } else {
#pragma unroll
            for (int k = 0; k < QD_KS; ++k)
                if (s0 + k < n) yo[s0 + k] = out[k];
        }
#pragma unroll
        for (int k = 0; k < QD_KS; ++k) { cur[k] = nxt[k]; nxt[k] = nn[k]; }
    }
}

// ---------------------------------------------------------------- crossover
struct CrossoverArgs {
    const float *x;       // [batch, n]
    float *low;           // [batch, n]
    float *high;          // [batch, n]
    long long n;
    double co[4][6];      // sections lp1, lp2, hp1, hp2 as (b0 b1 b2 1 a1 a2)
    int tile;             // output samples per thread (multiple of 32), see crossover_kernel
    int halo;             // warm-up samples before a tile (multiple of 32), from the pole radius
    int low_delay;        // samples the low band is delayed by (dsp/pipeline.py:389-396)
    int process_low;      // 1: saturate / blend / trim the low band (dsp/pipeline.py:1063-1073)
    float low_gain;
    double low_norm;
    float mono_a, mono_b;
    int apply_mono;
    float low_trim;
    int apply_low_trim;
    const int64_t *starts;    // optional ragged batch, as SpecArgsT::starts; n is then the longest clip (grid size)
    const int32_t *lengths;
    int clip0;
};

QD_DEV float low_process(float v, const CrossoverArgs &a) {
    // dsp/saturation.py:44-54: float32 gain, float32 tanh(3x), float64 division by tanh(3)
    const float t = tanhf(__fmul_rn(3.0f, __fmul_rn(v, a.low_gain)));
    float r = (float)((double)t * a.low_norm);
    if (a.apply_mono) r = __fadd_rn(__fmul_rn(a.mono_a, r), __fmul_rn(a.mono_b, r));
    if (a.apply_low_trim) r = __fmul_rn(r, a.low_trim);
    return r;
}

// Linkwitz-Riley split (dsp/crossover.py:71-118): four DF2T sections (LP, LP | HP, HP) run SEQUENTIALLY by one thread
// over its own tile of one clip, in float64, in scipy's operation order.  What makes the tiles independent is the
// filters' memory: the poles of a crossover at f_c have radius r = exp(-pi sqrt(2) f_c / sr) (0.9726 at 300 Hz / 48 kHz),
// so a state started from zero `halo` samples before the tile differs from the true state by the decayed zero-input
// response, below 1e-15 of the signal for halo = 44 / (1 - r) (host: qd_host::fill_crossover) -- under the rounding of
// the float64 recurrence itself, and nine orders below the float32 the band is stored in.  Samples before the clip are
// zeros, which IS the true initial state, so the first tile needs no special case.  No scan, no block barrier: a warp
// stages 32 samples of its 32 tiles through shared memory (coalesced 128-byte rows both ways), each lane filters its
// own row.  Algorithmic HBM bytes: 4 read + 8 written per sample (the halo re-reads hit L2).
constexpr int QD_XO_WARPS = 4;
QD_DEV void xo_section(const double *co, double xin, double &z0, double &z1, double &o) {
    // DF2T, scipy's recurrence (o = b0 x + z0; z0 = b1 x - a1 o + z1; z1 = b2 x - a2 o) in five fused operations
    o = fma(co[0], xin, z0);
    z0 = fma(-co[4], o, fma(co[1], xin, z1));
    z1 = fma(-co[5], o, co[2] * xin);
}

__global__ void __launch_bounds__(32 * QD_XO_WARPS) crossover_kernel(const CrossoverArgs a) {
    __shared__ float s_lo[QD_XO_WARPS][32][33];   // input row, overwritten by the low band
    __shared__ float s_hi[QD_XO_WARPS][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ClipLoc cs = clip_loc(a, (int)blockIdx.y);
    const size_t base = (size_t)cs.base;
    const long long n = cs.n;
    const float *x = a.x + base;
    float *low = a.low + base, *high = a.high + base;
    const long long n_tiles = (n + a.tile - 1) / a.tile;
    const long long tile0 = ((long long)blockIdx.x * QD_XO_WARPS + warp) * 32;   // the warp's first tile; lane l owns tile0 + l
    if (blockIdx.x == 0 && a.low_delay > 0) {   // head of the delayed low band: the processed zero input
        const float z = a.process_low ? low_process(0.0f, a) : 0.0f;
        for (long long i = threadIdx.x; i < a.low_delay && i < n; i += 32 * QD_XO_WARPS) low[i] = z;
    }
    if (tile0 >= n_tiles) return;
    float (*rl)[33] = s_lo[warp];
    float (*rh)[33] = s_hi[warp];
    const int rows = (int)(n_tiles - tile0 < 32 ? n_tiles - tile0 : 32);
    double st[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
    const int steps = (a.halo + a.tile) / 32;
    const long long s_first = tile0 * a.tile - a.halo;     // sample index of row 0, step 0, column 0
    // row r of a step = 32 consecutive samples of tile tile0 + r: one 128-byte row per warp load.  The rows of step
    // j + 1 are fetched into registers while step j is filtered, so no global latency sits between the steps.
    // A step whose 32 rows all lie inside the clip (nearly all of them) takes the path without per-element bounds tests.
    float nxt[32];
    auto fetch = [&](int j) {
        const long long s0 = s_first + 32LL * j;                  // row 0, column 0 of this step
        if (rows == 32 && s0 >= 0 && s0 + 31LL * a.tile + 32 <= n) {
            const float *p = x + s0 + lane;
#pragma unroll
            for (int r = 0; r < 32; ++r) nxt[r] = __ldg(p + (size_t)r * a.tile);
        } else {
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const long long sidx = s0 + (long long)r * a.tile + lane;
                nxt[r] = (r < rows && sidx >= 0 && sidx < n) ? x[sidx] : 0.0f;
            }
        }
    };
    fetch(0);
    for (int j = 0; j < steps; ++j) {
#pragma unroll
        for (int r = 0; r < 32; ++r) rl[r][lane] = nxt[r];
        __syncwarp();
        if (j + 1 < steps) fetch(j + 1);
        const bool emit = 32 * j >= a.halo;   // the warm-up steps only advance the filter states
        // ---- filter the own row
        if (lane < rows) {
            if (emit) {
#pragma unroll 4
                for (int k = 0; k < 32; ++k) {
                    const double xin = (double)rl[lane][k];
                    double l1, l2, h1, h2;
                    xo_section(a.co[0], xin, st[0][0], st[0][1], l1);
                    xo_section(a.co[1], l1, st[1][0], st[1][1], l2);
                    xo_section(a.co[2], xin, st[2][0], st[2][1], h1);
                    xo_section(a.co[3], h1, st[3][0], st[3][1], h2);
                    const float lf = (float)l2;
                    rl[lane][k] = a.process_low ? low_process(lf, a) : lf;
                    rh[lane][k] = (float)h2;
                }
            } else {
#pragma unroll 4
                for (int k = 0; k < 32; ++k) {
                    const double xin = (double)rl[lane][k];
                    double l1, l2, h1, h2;
                    xo_section(a.co[0], xin, st[0][0], st[0][1], l1);
                    xo_section(a.co[1], l1, st[1][0], st[1][1], l2);
                    xo_section(a.co[2], xin, st[2][0], st[2][1], h1);
                    xo_section(a.co[3], h1, st[3][0], st[3][1], h2);
                }
            }
        }
        __syncwarp();
        // ---- store
        if (emit) {
            const long long s0 = s_first + 32LL * j;
            if (rows == 32 && s0 + 31LL * a.tile + 32 + a.low_delay <= n) {
                float *ph = high + s0 + lane, *pl = low + s0 + lane + a.low_delay;
#pragma unroll 8
                for (int r = 0; r < 32; ++r) {
                    ph[(size_t)r * a.tile] = rh[r][lane];
                    pl[(size_t)r * a.tile] = rl[r][lane];
                }
            } else {
                for (int r = 0; r < rows; ++r) {
                    const long long sidx = s0 + (long long)r * a.tile + lane;
                    if (sidx < n) {
                        high[sidx] = rh[r][lane];
                        if (sidx + a.low_delay < n) low[sidx + a.low_delay] = rl[r][lane];
                    }
                }
            }
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------- elementwise
__global__ void distort_kernel(const float *__restrict__ x, float *__restrict__ y, long long count, int mode,
                               double fold, double bias, float tg, float tn) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        const float v = x[i];
        float r;
        if (mode == 0) {   // float64 like the reference, one rounding to float32 (see epilogue_apply)
            double t = ((double)v + bias) * fold;
            if (t > 1.0) t = 2.0 - t;
            if (t < -1.0) t = -2.0 - t;  // sequential masks, dsp/distortion.py:44-53
            r = (float)fmin(fmax(t, -1.0), 1.0);
        } else {
            r = tanhf(tg * v) * tn;
        }
        y[i] = r;
    }
}

__global__ void add_kernel(const float *__restrict__ a, const float *__restrict__ b, float *__restrict__ y,
                           long long count) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        y[i] = __fadd_rn(a[i], b[i]);
}

}  // namespace qd
