// qd_spec.cuh -- one spectral pass of the STFT path as a single kernel:
//
//   frame -> Hann window -> real FFT -> [spectral FX] -> scale-snap quantizer (gather form,
//   5-tap smear, 3-tap smoothing) -> Hermitian inverse FFT -> Hann window -> overlap-add ->
//   1/sum(w^2) -> float32 -> [wavefold | soft-tube]
//
// Replaces, per pass, the reference's
//   stft_mono                               dsp/stft_utils.py:11-97
//   _apply_spectral_quantization_to_stft    dsp/pipeline.py:228-342
//   quantize_spectrum / _apply_smear_numba  dsp/quantizer.py:343-529, 253-340
//   istft_mono                              dsp/stft_utils.py:100-234
//   apply_distortion                        dsp/distortion.py:18-114 (fused epilogue)
//
// Execution model (B200): one WARP owns one frame.  The n_fft-point real FFT is an
// (n_fft/2)-point complex FFT held in the warp's private shared-memory buffer; each lane
// runs whole radix-R DFTs (R up to 32) in registers, so n_fft = 2048 needs two passes
// (32 x 32) and a single shared-memory exchange per direction, with only __syncwarp()
// between passes.  The NW warps of a CTA take NW consecutive frames; a CTA-wide step then
// overlap-adds them in frame order (deterministic, no atomics) and streams finished hops
// to HBM.  A CTA walks a tile of consecutive hops of one clip, carrying the 3-hop OLA
// tail in shared memory.  Nothing is a dense contraction, so tensor cores are not used.
#pragma once
#include "qd_common.cuh"

namespace qd {

// ---------------------------------------------------------------- FFT configuration
template <class T, int NC> struct FftCfg;
template <class T> struct FftCfg<T, 256>  { static constexpr int R1 = 8,  R2 = 8,  R3 = 4;  };
template <class T> struct FftCfg<T, 512>  { static constexpr int R1 = 8,  R2 = 8,  R3 = 8;  };
template <> struct FftCfg<float, 1024>    { static constexpr int R1 = 32, R2 = 32, R3 = 1;  };
template <> struct FftCfg<double, 1024>   { static constexpr int R1 = 16, R2 = 8,  R3 = 8;  };  // 32 double2 would spill
template <class T> struct FftCfg<T, 2048> { static constexpr int R1 = 16, R2 = 16, R3 = 8;  };
template <class T> struct FftCfg<T, 4096> { static constexpr int R1 = 16, R2 = 16, R3 = 16; };

// one pad slot per 32 complex values keeps the stride-32 accesses of the 32x32 plan
// conflict-free (stride 33); slot 32 is never produced by pidx() and holds the Nyquist bin.
QD_DEV int pidx(int a) { return a + (a >> 5); }
constexpr int QD_NYQ_SLOT = 32;
template <int NC> __host__ __device__ constexpr int buf_slots() { return NC + NC / 32; }

// position of spectrum bin k (0..NC) inside the warp buffer after the in-place DIF passes
template <class T, int NC>
QD_DEV int spos(int k) {
    using C = FftCfg<T, NC>;
    if (k >= NC) return QD_NYQ_SLOT;
    const unsigned uk = (unsigned)k;
    if constexpr (C::R1 == 32 && NC == 1024) return (int)(33u * (uk & 31u) + (uk >> 5));
    const unsigned k1 = uk & (unsigned)(C::R1 - 1);
    const unsigned k2 = (uk / (unsigned)C::R1) & (unsigned)(C::R2 - 1);
    const unsigned k3 = uk / (unsigned)(C::R1 * C::R2);
    return pidx((int)(k1 * (unsigned)(NC / C::R1) + k2 * (unsigned)(NC / (C::R1 * C::R2)) + k3));
}
// the same for a bin known to be below NC (no Nyquist test)
template <class T, int NC>
QD_DEV int spos_lt(int k) {
    using C = FftCfg<T, NC>;
    const unsigned uk = (unsigned)k;
    if constexpr (C::R1 == 32 && NC == 1024) return (int)(33u * (uk & 31u) + (uk >> 5));
    else return spos<T, NC>(k);
}

// position of bin 32*row + lane.  For the 32x32 plan this is 33*lane + row for every bin including the
// Nyquist bin (row 32, lane 0 -> slot 32), so row loops advance by one slot per row.
template <class T, int NC>
QD_DEV int rpos(int lane, int row) {
    if constexpr (FftCfg<T, NC>::R1 == 32 && NC == 1024) return 33 * lane + row;
    else return spos<T, NC>(32 * row + lane);
}
// position of the mirror bin NC - (32*row + lane), row < NC/64
template <class T, int NC>
QD_DEV int mpos(int lane, int row) {
    if constexpr (FftCfg<T, NC>::R1 == 32 && NC == 1024) return lane == 0 ? 32 - row : 33 * (32 - lane) + 31 - row;
    else return spos<T, NC>(NC - (32 * row + lane));
}

// ---------------------------------------------------------------- device-side tables
// Gather tables of the quantizer.  A destination bin d receives, from the target at bin d+e-2 (e = 0..4):
//   tap[e] * H_slot   (smear, tap[e] = snap*smear*kernel[4-e])   and, for its own target (e = 2), base[slot] * H_slot
// where H_slot = (sum over the slot's sources) / ksum_slot and base[slot] = snap*(1-smear)*ksum_slot; ksum is 1
// except for targets whose 5-tap window is clipped at the spectrum edges (dsp/quantizer.py:311-330).
struct QuantDev {
    int n_slots;                    // distinct target bins
    int n_src;
    int row_limit;                  // rows >= row_limit hold no source and no bin that can receive energy
    const uint32_t *src_tab;        // [n_src] tail<<31 | off<<26 | slot<<13 | source bin, grouped by slot
    const uint32_t *row_active;     // [rows] bit l: bin 32*row+l gives its energy away
    const uint16_t *slot_of_bin;    // [32*rows + 4]: entry d+2 = slot whose target is bin d, else n_slots (reads 0)
    const float *slot_invk;         // [n_slots + 1]  1 / ksum_slot
    const float *slot_base;         // [n_slots + 1]  snap*(1-smear)*ksum_slot (0 for the sentinel)
    float tap[5];                   // see above
    float keep_active;              // 1 - snap
    int smoothing;                  // dsp/quantizer.py:523
};

// spectral FX of the high band (dsp/pipeline.py:64-141, dsp/spectral_fx.py:198-390); host-resolved numbers
struct FxDev {
    int mode;               // qd_fx_mode (0 = none)
    float a, b, c;          // see qd_params.fx_a / fx_b / fx_c
    double step;            // bitcrush step (dB or linear) in double for the rounding decision
    const void *table;      // int16 source bins (scramble) or float32 jitter in [-1,1) (dispersal), or null
    int table_frames;       // frames per pass in the table
    int table_per_clip;     // 0: shared by all clips
    int pass;               // 0 / 1: which quantised pass of the render this launch is
    int clip_offset;        // row of the batch's clip 0 in the per-clip table (a host-pipe chunk's first clip)
};

template <class T>
struct SpecArgsT {
    const float *x;        // [batch, n] input clips
    float *y;              // [batch, n] output (after the epilogue)
    float *tap;            // optional [batch, n]: iSTFT output before the epilogue
    float *clip_peak;      // optional [batch]: max |y| per clip (atomicMax on the bit pattern; caller zeroes it).
                           // The limiter skips a clip whose peak never exceeds the ceiling: its gain is exactly 1.
    int n;                 // samples per clip; ragged batch: the longest clip
    int batch;             // clips in this launch (a CTA may hold several clip groups)
    int n_frames;          // T = 1 + n / hop of a uniform batch (the kernels derive each clip's own from its length)
    // ragged batch (null = uniform clips at clip * n): clip c of the launch is starts[clip0 + c] - starts[0] samples
    // into x / y / tap and has lengths[clip0 + c] samples.  Launch splits advance clip0, not the pointers (clip_loc).
    const int64_t *starts;
    const int32_t *lengths;
    int clip0;
    int tile_blocks;       // output hops per CTA tile
    int quant;             // run the quantizer (else pure STFT -> iSTFT)
    int epilogue;          // 0 none, 1 wavefold, 2 tube
    double fold, bias;     // wavefold in float64 like dsp/distortion.py:37-58 ...
    int fold_exact_f32;    // ... unless bias == 0 and fold is a power of two: float32 arithmetic is exact then
    float tube_gain, tube_norm;
    const V2<T> *wtab;     // [2 NC/R1] Hann window factors (-0.5 cos A, 0.5 sin A) per first-pass butterfly (host builder)
    const V2<T> *tw1;      // access-ordered twiddles of pass 1 / pass 2 (see host builder)
    const V2<T> *tw2;
    const V2<T> *wsplit;   // [NC/2+1] V_k = -i/2 exp(-2 pi i k / n_fft)
    const T *invw;         // [16][hop]: 1/max(sum_{sl=a..b} w^2[sl*hop+c], 1e-10) at [(a*4+b)*hop + c]
    QuantDev q;
    FxDev fx;
    const T *frozen;       // optional [batch][BUF]: |X| of frame 0 by buffer position (spectral freeze)
    // formant shift (dsp/spectral_fx.py:116-195), FX kernels; null = off
    const int16_t *formant_idx;   // [NC+1] floor(k / ratio) clamped to NC        (np.interp segment, host float64)
    const float *formant_frac;    // [NC+1] k / ratio - floor(k / ratio), 0 when clamped
    int formant_order;            // lifter order (30)
};
using SpecArgs = SpecArgsT<float>;

// ---------------------------------------------------------------- FFT passes (warp level)
template <class T, int NC, int M, int R, bool TW>
QD_DEV void fwd_pass(V2<T> *buf, const V2<T> *tw, int lane) {
    constexpr int S = M / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = 0; i < NB; ++i) {
        const int u = lane + 32 * i;
        const int a0 = (u / S) * M + (u % S);
        V2<T> v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = buf[pidx(a0 + q * S)];
        dft_reg<R, -1, T>(v);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int k = qd_bitrev(r, LG);
            V2<T> t = v[r];
            if (TW && k > 0) t = cmul(t, tw[(i * R + k) * 32 + lane]);
            buf[pidx(a0 + k * S)] = t;
        }
    }
    __syncwarp();
}

template <class T, int NC, int M, int R, bool TW>
QD_DEV void inv_pass(V2<T> *buf, const V2<T> *tw, int lane) {
    constexpr int S = M / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = 0; i < NB; ++i) {
        const int u = lane + 32 * i;
        const int a0 = (u / S) * M + (u % S);
        V2<T> v[R];
#pragma unroll
        for (int k = 0; k < R; ++k) {
            V2<T> t = buf[pidx(a0 + k * S)];
            if (TW && k > 0) t = cmulc(t, tw[(i * R + k) * 32 + lane]);
            v[k] = t;
        }
        dft_reg<R, +1, T>(v);
#pragma unroll
        for (int r = 0; r < R; ++r) buf[pidx(a0 + qd_bitrev(r, LG) * S)] = v[r];
    }
    __syncwarp();
}

// Hann window of the sample pair q of a first-pass butterfly: 0.5 - 0.5 cos(A + 2 pi q / R) by angle addition from the
// butterfly's (-0.5 cos A, 0.5 sin A) pairs (wtab, see the host builder); q is a compile-time constant after unrolling
template <class T, int R>
QD_DEV V2<T> hann_pair(V2<T> wc, V2<T> ws, int q) {
    const int k = q * (32 / R);   // angle in 32nds of a turn
    if (k == 0) return padd(splat((T)0.5), wc);
    if (k == 8) return padd(splat((T)0.5), ws);
    if (k == 16) return psub(splat((T)0.5), wc);
    if (k == 24) return psub(splat((T)0.5), ws);
    return pfma(splat((T)qd_cos32(k)), wc, pfma(splat((T)qd_sin32(k)), ws, splat((T)0.5)));
}

// Twiddles exp(-2 pi i j k / NC), k = 1..R-1, of a first-pass butterfly: only the powers of two are read from the table,
// the others are products w_k = w_{k - lowbit(k)} w_{lowbit(k)} (at most log2(R) - 1 multiplications deep), because the
// pass is bound by shared-memory wavefronts, not by arithmetic.  `cur[j]` = latest w whose index has >= j trailing zeros.
template <int K> struct KConst { static constexpr int value = K; };
template <bool B> struct KBool { static constexpr bool value = B; };
template <class T, int R, int K, class F>
QD_DEV void twiddle_step(const V2<T> (&pw)[qd_log2(R)], V2<T> (&cur)[qd_log2(R) + 1], F &body) {
    if constexpr (K < R) {
        constexpr int z = qd_ctz(K);
        V2<T> w;
        if constexpr (K == (1 << z)) w = pw[z];
        else w = cmul(cur[z + 1], pw[z]);
#pragma unroll
        for (int j = 0; j <= z; ++j) cur[j] = w;
        body(KConst<K>{}, w);
        twiddle_step<T, R, K + 1, F>(pw, cur, body);
    }
}
template <class T, int R, class F>
QD_DEV void twiddle_walk(const V2<T> *twp, F &&body) {   // twp = &tw[(i * R) * 32 + lane]
    constexpr int LG = qd_log2(R);
    V2<T> pw[LG], cur[LG + 1];
#pragma unroll
    for (int z = 0; z < LG; ++z) pw[z] = twp[(1 << z) * 32];
#pragma unroll
    for (int z = 0; z <= LG; ++z) cur[z] = mk2<T>((T)1, (T)0);
    twiddle_step<T, R, 1, F>(pw, cur, body);
}

// first forward pass: reads the frame from the staging buffer, applies the analysis window
template <class T, int NC, int R>
QD_DEV void fwd_first(V2<T> *buf, const float2 *frame, const V2<T> *wtab, const V2<T> *tw, int lane) {
    constexpr int S = NC / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = 0; i < NB; ++i) {
        const int a0 = lane + 32 * i;
        const V2<T> wc = wtab[2 * a0], ws = wtab[2 * a0 + 1];
        V2<T> v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) {
            const float2 s = frame[a0 + q * S];
            v[q] = pmul(mk2<T>((T)s.x, (T)s.y), hann_pair<T, R>(wc, ws, q));
        }
        dft_reg<R, -1, T>(v);
        buf[pidx(a0)] = v[0];
        twiddle_walk<T, R>(tw + (i * R) * 32 + lane,
                           [&](auto kc, V2<T> w) {
                               constexpr int k = decltype(kc)::value;
                               buf[pidx(a0 + k * S)] = cmul(v[qd_bitrev(k, LG)], w);
                           });
    }
    __syncwarp();
}

// first forward pass of a sequence that already sits in the warp buffer (pidx layout), no window: the forward real
// FFT of the liftered cepstrum (formant shift)
template <class T, int NC, int R>
QD_DEV void fwd_first_buf(V2<T> *buf, const V2<T> *tw, int lane) {
    constexpr int S = NC / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = 0; i < NB; ++i) {
        const int a0 = lane + 32 * i;
        V2<T> v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = buf[pidx(a0 + q * S)];
        dft_reg<R, -1, T>(v);
        buf[pidx(a0)] = v[0];
        twiddle_walk<T, R>(tw + (i * R) * 32 + lane,
                           [&](auto kc, V2<T> w) {
                               constexpr int k = decltype(kc)::value;
                               buf[pidx(a0 + k * S)] = cmul(v[qd_bitrev(k, LG)], w);
                           });
    }
    __syncwarp();
}

// last inverse pass: synthesis window (the 1/n_fft of the inverse FFT is folded into the host's 1/sum(w^2) table),
// leaves the time-domain frame in buf.  WIN = false: no window (inverse real FFT of the log spectrum, formant shift)
template <class T, int NC, int R, bool WIN = true>
QD_DEV void inv_last(V2<T> *buf, const V2<T> *wtab, const V2<T> *tw, int lane) {
    constexpr int S = NC / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = 0; i < NB; ++i) {
        const int a0 = lane + 32 * i;
        V2<T> v[R];
        v[0] = buf[pidx(a0)];
        twiddle_walk<T, R>(tw + (i * R) * 32 + lane, [&](auto kc, V2<T> w) {
            constexpr int k = decltype(kc)::value;
            v[k] = cmulc(buf[pidx(a0 + k * S)], w);
        });
        dft_reg<R, +1, T>(v);
        if constexpr (WIN) {
            const V2<T> wc = wtab[2 * a0], ws = wtab[2 * a0 + 1];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int q = qd_bitrev(r, LG);
                buf[pidx(a0 + q * S)] = pmul(v[r], hann_pair<T, R>(wc, ws, q));
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r) buf[pidx(a0 + qd_bitrev(r, LG) * S)] = v[r];
        }
    }
    __syncwarp();
}

// the forward passes AFTER fwd_first (which the kernel calls itself, to release the staging buffer early)
template <class T, int NC>
QD_DEV void fft_forward(V2<T> *buf, const float2 *frame, const SpecArgsT<T> &a, const V2<T> *wtab,
                        const V2<T> *tw1, const V2<T> *tw2, int lane) {
    using C = FftCfg<T, NC>;
    if constexpr (C::R3 > 1) {
        fwd_pass<T, NC, NC / C::R1, C::R2, true>(buf, tw2, lane);
        fwd_pass<T, NC, C::R3, C::R3, false>(buf, nullptr, lane);
    } else {
        fwd_pass<T, NC, NC / C::R1, C::R2, false>(buf, nullptr, lane);
    }
    (void)a;
}

template <class T, int NC, bool WIN = true>
QD_DEV void fft_inverse(V2<T> *buf, const V2<T> *wtab, const V2<T> *tw1, const V2<T> *tw2, int lane) {
    using C = FftCfg<T, NC>;
    if constexpr (C::R3 > 1) {
        inv_pass<T, NC, C::R3, C::R3, false>(buf, nullptr, lane);
        inv_pass<T, NC, NC / C::R1, C::R2, true>(buf, tw2, lane);
    } else {
        inv_pass<T, NC, NC / C::R1, C::R2, false>(buf, nullptr, lane);
    }
    inv_last<T, NC, C::R1, WIN>(buf, wtab, tw1, lane);
}

// ---------------------------------------------------------------- real <-> complex packing
// Z = FFT_NC(x[2n] + i x[2n+1])  ->  X[k], k = 0..NC   (in place, Nyquist in the pad slot)
//   E = Z[k] + conj Z[NC-k],  T = V_k (Z[k] - conj Z[NC-k]),  V_k = W_N^k / (2i)   (host table)
//   X[k] = E/2 + T,  X[NC-k] = conj(E/2 - T)
template <class T, int NC>
QD_DEV void real_split(V2<T> *buf, const V2<T> *wsplit, int lane) {
#pragma unroll 4
    for (int row = 0; row < NC / 64; ++row) {
        const int k = lane + 32 * row;
        if (k == 0) {
            const V2<T> z0 = buf[0];
            buf[0] = mk2<T>(z0.x + z0.y, 0.0f);
            buf[QD_NYQ_SLOT] = mk2<T>(z0.x - z0.y, 0.0f);
            const int pm = spos<T, NC>(NC / 2);
            buf[pm] = cconj(buf[pm]);
        } else {
            const int pa = rpos<T, NC>(lane, row), pb = mpos<T, NC>(lane, row);
            const V2<T> za = buf[pa], zb = cconj(buf[pb]);
            const V2<T> e = cadd(za, zb);
            const V2<T> t = cmul(csub(za, zb), wsplit[k]);
            buf[pa] = pfma(e, splat((T)0.5), t);
            buf[pb] = cconj(pfma(e, splat((T)0.5), mk2<T>(-t.x, -t.y)));
        }
    }
    __syncwarp();
}

// X'[k] (only Re of DC / Nyquist used, like pocketfft c2r) -> Z' with z = IFFT_NC(Z') * 1/(2 NC)
//   E2 = X'[k] + conj X'[NC-k],  T2 = X'[k] - conj X'[NC-k],  i O2 = i conj(W_N^k) T2 = 2 conj(V_k) T2
//   Z'[k] = E2 + i O2,  Z'[NC-k] = conj(E2 - i O2)
template <class T, int NC>
QD_DEV void real_merge(V2<T> *buf, const V2<T> *wsplit, int lane) {
#pragma unroll 4
    for (int row = 0; row < NC / 64; ++row) {
        const int k = lane + 32 * row;
        if (k == 0) {
            const T a = buf[0].x, b = buf[QD_NYQ_SLOT].x;
            buf[0] = mk2<T>(a + b, a - b);
            const int pm = spos<T, NC>(NC / 2);
            const V2<T> xm = buf[pm];
            buf[pm] = mk2<T>(2.0f * xm.x, -2.0f * xm.y);
        } else {
            const int pa = rpos<T, NC>(lane, row), pb = mpos<T, NC>(lane, row);
            const V2<T> xa = buf[pa], xb = cconj(buf[pb]);
            const V2<T> e = cadd(xa, xb);
            const V2<T> h = cmulc(csub(xa, xb), wsplit[k]);             // i O2 / 2
            buf[pa] = pfma(h, splat((T)2), e);                          // E2 + i O2
            buf[pb] = cconj(pfma(h, splat((T)-2), e));                  // conj(E2 - i O2)
        }
    }
    __syncwarp();
}

// ---------------------------------------------------------------- quantizer (one frame, one warp)
// Gather form of dsp/quantizer.py:424-527 (SURVEY.md appendix A.2):
//   G_t = sum_{i -> t} |X_i|,  P_t = sum_{i -> t} X_i           (sources in ascending order)
//   tE_d = sum_e coef[d][e] G_{t(d,e)},  PS_d = sum_e coef[d][e] P_{t(d,e)}
//   new_d = |X_d| keep_d + tE_d ;  phasor_d = PS_d/|PS_d| if tE_d > 0 else X_d/|X_d|
//   out_d = smooth(new)_d * phasor_d      with [1/4,1/2,1/4], edges replicated
// 1/sqrt(x) as a single MUFU.RSQ (2 ulp); callers guard x against zero / denormals
QD_DEV float rsqrt_fast(float x) {
#ifdef QD_EMU
    return 1.0f / std::sqrt(x);
#else
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}
// float64: CUDA's rsqrt() (one MUFU seed + Newton steps, 1 ulp) instead of a square root followed by an IEEE division,
// which together were 10 % of the float64 kernels' instructions (ncu, n_fft 8192)
QD_DEV double rsqrt_fast(double x) {
#ifdef QD_EMU
    return 1.0 / std::sqrt(x);
#else
    return rsqrt(x);
#endif
}
// log2 / exp2 as single MUFU operations for the log-domain bitcrush: absolute error of lg2.approx ~1e-6 near the values
// that matter (decisions closer than 2e-4 to a rounding boundary are re-made in double), relative error of ex2.approx 2e-7
QD_DEV float log2_fast(float x) {
#ifdef QD_EMU
    return std::log2(x);
#else
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}
QD_DEV double log2_fast(double x) { return log2(x); }
QD_DEV float exp2_fast(float x) {
#ifdef QD_EMU
    return std::exp2(x);
#else
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}
QD_DEV double exp2_fast(double x) { return exp2(x); }
QD_DEV void sincos_fast(float a, float *s, float *c) {
#ifdef QD_EMU
    qd_sincos(a, s, c);
#else
    __sincosf(a, s, c);
#endif
}
QD_DEV void sincos_fast(double a, double *s, double *c) { qd_sincos(a, s, c); }
constexpr float QD_TINY2 = 1e-30f;  // |X|^2 below this is treated as an exact zero (|X| < 1e-15)

// magnitude and unit phasor of one bin (np.angle(0) = 0 -> phasor 1)
template <class T>
QD_DEV void mag_phasor(V2<T> xv, T &m, V2<T> &u) {
    const T m2 = xv.x * xv.x + xv.y * xv.y;
    const bool ok = m2 > QD_TINY2;
    const T r = rsqrt_fast(m2);
    m = ok ? m2 * r : 0.0f;
    u = ok ? pmul(xv, splat(r)) : mk2<T>(1.0f, 0.0f);
}

// [1/4,1/2,1/4] smoothing of row `cur` with two shuffles: lane 31 lends its previous-row value to lane 0,
// lane 0 lends its next-row value to lane 31 (nobody else needs those two lanes' own m_cur as a neighbour
// on that side).
// the same with the lane tests hoisted by the caller (is31 / is0) and no edge handling
template <class T>
QD_DEV T smooth_mid(T m_prev, T m_cur, T m_next, bool is0, bool is31, int lane_m1, int lane_p1) {
    const T left = __shfl_sync(QD_FULL, is31 ? m_prev : m_cur, lane_m1);
    const T right = __shfl_sync(QD_FULL, is0 ? m_next : m_cur, lane_p1);
    return 0.5f * m_cur + 0.25f * (left + right);
}
template <class T>
QD_DEV T smooth_row(T m_prev, T m_cur, T m_next, int lane, bool first_bin, bool last_bin) {
    T left = __shfl_sync(QD_FULL, lane == 31 ? m_prev : m_cur, (lane + 31) & 31);
    T right = __shfl_sync(QD_FULL, lane == 0 ? m_next : m_cur, (lane + 1) & 31);
    if (first_bin) left = m_cur;   // scipy convolve1d mode="nearest"
    if (last_bin) right = m_cur;
    return 0.5f * m_cur + 0.25f * (left + right);
}

// one bin of a row that may give energy away (active) or receive it (affected): new magnitude and phasor
template <class T>
QD_DEV T warp_max(T v) {
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) v = qd_max(v, __shfl_xor_sync(QD_FULL, v, d));
    return v;
}
template <class T>
QD_DEV T warp_sum(T v) {
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(QD_FULL, v, d);
    return v;
}

// Formant shift of one frame (dsp/spectral_fx.py:116-195) on the magnitude plane `mags`; `scr` is a second
// warp-private buffer.  The spectral envelope is the low-quefrency part of the real cepstrum:
//   L = log(max(m, 1e-12));  c = irfft(L);  c *= lifter (|q| < order);  env = Re rfft(c)
// and, because rfft(irfft(L)) = L, the reference's fine structure rfft(c (1 - lifter)) is L - env, so
//   m' = max(m, 1e-12) exp(env_shifted - env),  env_shifted[k] = np.interp(k / ratio, bins, env)
// followed by the energy renormalisation sqrt(sum m^2 / sum m'^2).  The two FFTs are the warp's own n_fft-point
// real FFT (merge + inverse passes, forward passes + split) without the Hann window; the interpolation segment and
// fraction of every bin come from the host (float64, so the segment index is the reference's).
template <class T, int NC>
QD_DEV void formant_frame(T *mags, V2<T> *scr, const SpecArgsT<T> &a, const V2<T> *tw1, const V2<T> *wsplit, int lane) {
    constexpr int NBINS = NC + 1;
    constexpr int ROWS = (NBINS + 31) / 32;
    T e0 = 0.0f;
    for (int row = 0; row < ROWS; ++row) {
        if (row < ROWS - 1 || lane == 0) {
            const int p = rpos<T, NC>(lane, row);
            const T m = mags[p];
            e0 += m * m;
            scr[p] = mk2<T>(log2_fast(qd_max(m, (T)1e-12)) * (T)0.6931471805599453, (T)0);   // ln m by MUFU.LG2
        }
    }
    __syncwarp();
    real_merge<T, NC>(scr, wsplit, lane);
    fft_inverse<T, NC, false>(scr, nullptr, tw1, a.tw2, lane);       // scr[pidx(j)] = n_fft * (c[2j], c[2j+1])
    {
        const int n = 2 * NC;
        const int order = a.formant_order < NC ? a.formant_order : NC;   // min(lifter_order, len // 2)
        const T inv_n = (T)1 / (T)n;
        for (int j = lane; j < NC; j += 32) {                             // lifter[:order] = lifter[-order+1:] = 1
            const V2<T> v = scr[pidx(j)];
            const int q0 = 2 * j, q1 = 2 * j + 1;
            scr[pidx(j)] = mk2<T>((q0 < order || q0 > n - order) ? v.x * inv_n : (T)0,
                                  (q1 < order || q1 > n - order) ? v.y * inv_n : (T)0);
        }
    }
    __syncwarp();
    fwd_first_buf<T, NC, FftCfg<T, NC>::R1>(scr, tw1, lane);
    fft_forward<T, NC>(scr, nullptr, a, nullptr, tw1, a.tw2, lane);
    real_split<T, NC>(scr, wsplit, lane);                             // Re scr[pos(k)] = env[k]
    T e1 = 0.0f;
    for (int row = 0; row < ROWS; ++row) {
        if (row < ROWS - 1 || lane == 0) {
            const int p = rpos<T, NC>(lane, row);
            const int k = 32 * row + lane;
            const int j = (int)__ldg(a.formant_idx + k);
            const T fr = (T)__ldg(a.formant_frac + k);
            const T f0 = scr[spos<T, NC>(j)].x;
            const T f1 = scr[spos<T, NC>(j < NC ? j + 1 : NC)].x;
            const T es = (f1 - f0) * fr + f0;                             // np.interp: slope * (x - xp[j]) + fp[j]
            const T m = qd_max(mags[p], (T)1e-12) * exp2_fast((es - scr[p].x) * (T)1.4426950408889634);   // MUFU.EX2
            mags[p] = m;
            e1 += m * m;
        }
    }
    e0 = warp_sum(e0);
    e1 = warp_sum(e1);
    if (e1 > (T)1e-12) {
        const T sc = sqrt(e0 / e1);
        for (int row = 0; row < ROWS; ++row)
            if (row < ROWS - 1 || lane == 0) mags[rpos<T, NC>(lane, row)] *= sc;
    }
    __syncwarp();
}

// Spectral FX on one frame (high band only).  On entry buf holds X; on exit buf holds the unit phasors and
// mags[pos] the (processed) magnitudes, both indexed by buffer position, so that a bin whose magnitude
// becomes 0 keeps its phase for the smoothing that follows (SURVEY.md section 0.5).
template <class T, int NC>
QD_DEV void fx_frame(V2<T> *buf, T *mags, const FxDev &fx, int lane, long long tab_base, const T *frozen,
                     V2<T> *scr, const SpecArgsT<T> &a, const V2<T> *tw1, const V2<T> *wsplit) {
    constexpr int NBINS = NC + 1;
    constexpr int ROWS = (NBINS + 31) / 32;
    T mx = 0.0f, sm = 0.0f;
    // On entry buf holds the packed FFT output Z.  One paired sweep (bin k and its mirror NC - k, like the plain
    // quantizer) forms X[k] = E/2 + V_k (Z[k] - conj Z[NC-k]) and X[NC-k] in registers and leaves the unit phasors in
    // buf and the magnitudes in the plane -- no separate real_split sweep.  DC / Nyquist fall out of the same formula
    // (Z[NC] = Z[0], V_0 = -i/2); the Nyquist phasor goes to the pad slot.
    {
        constexpr int HR = NC / 64;
#pragma unroll 2
        for (int i = 0; i < HR; ++i) {
            const int k = 32 * i + lane;
            const int pa = rpos<T, NC>(lane, i);
            const int pb = k == 0 ? QD_NYQ_SLOT : mpos<T, NC>(lane, i);
            const V2<T> za = buf[pa], zb = cconj(buf[k == 0 ? pa : pb]);
            const V2<T> e = cadd(za, zb);
            const V2<T> t = cmul(csub(za, zb), wsplit[k]);
            T ml, mh;
            V2<T> ul, uh;
            mag_phasor<T>(pfma(e, splat((T)0.5), t), ml, ul);
            mag_phasor<T>(cconj(pfma(e, splat((T)0.5), mk2<T>(-t.x, -t.y))), mh, uh);
            if (frozen) { ml = frozen[pa]; mh = frozen[pb]; }  // dsp/pipeline.py:285-287, 303-304: first-frame magnitudes, own phases
            buf[pa] = ul; buf[pb] = uh;
            mags[pa] = ml; mags[pb] = mh;
            mx = qd_max(mx, qd_max(ml, mh));
            sm += ml + mh;
        }
        if (lane == 0) {   // the walks meet at bin NC/2: X[NC/2] = conj Z[NC/2]
            const int pm = spos<T, NC>(NC / 2);
            T m;
            V2<T> u;
            mag_phasor<T>(cconj(buf[pm]), m, u);
            if (frozen) m = frozen[pm];
            buf[pm] = u;
            mags[pm] = m;
            mx = qd_max(mx, m);
            sm += m;
        }
    }
    __syncwarp();
    {
        if (a.formant_idx) {   // dsp/pipeline.py:306-310: after the freeze, before the FX
            formant_frame<T, NC>(mags, scr, a, tw1, wsplit, lane);
            mx = 0.0f;
            sm = 0.0f;
            for (int row = 0; row < ROWS; ++row) {
                if (row < ROWS - 1 || lane == 0) {
                    const T m = mags[rpos<T, NC>(lane, row)];
                    mx = qd_max(mx, m);
                    sm += m;
                }
            }
        }
    }
    mx = warp_max(mx);  // max / sum of the magnitudes BEFORE the effect (dsp/pipeline.py:90,105; spectral_fx.py:387)
    if (fx.mode == 1 || fx.mode == 2) {
        // bitcrush (dsp/spectral_fx.py:198-260); np.round is half-to-even = rint
        const T thr = fx.c > 0.0f ? fx.c : fx.b * mx;
        const bool has_step = fx.step > 0.0, log_mode = fx.mode == 1;
        const T q_scale = (T)(6.020599913279624 / fx.step);          // 20 log10(m) / step_db = log2(m) * q_scale
        const T e_scale = (T)(fx.step * 0.16609640474436813);        // 10^(q step_db / 20) = 2^(q * e_scale)
#pragma unroll 2
        for (int row = 0; row < ROWS; ++row) {
            if (row < ROWS - 1 || lane == 0) {
                const int p = rpos<T, NC>(lane, row);
                T m = mags[p];
                if (has_step) {
                    if (log_mode) {
                        const T mm = qd_max(m, 1e-12f);
                        const T q = log2_fast(mm) * q_scale;
                        T rq = qd_rint(q);
                        // close to a rounding boundary: decide in double.  The float32 evaluation of q is good to ~1e-5
                        // (log2f 1 ulp of |log2 m| <= 40, one multiply), so a band of 2e-4 is ample; a wider one sends
                        // most warps down the float64 log10 (a lane in the band is enough)
                        if (qd_abs(qd_abs(q - rq) - 0.5f) < 2e-4f)
                            rq = (T)rint(20.0 * log10((double)mm) / fx.step);
                        m = exp2_fast(rq * e_scale);
                    } else {
                        m = qd_max((T)(rint((double)m / fx.step) * fx.step), 0.0f);
                    }
                }
                if (thr > 0.0f && m < thr) m = 0.0f;
                mags[p] = m;
            }
        }
    } else if (fx.mode == 3) {
        // phase dispersal (dsp/spectral_fx.py:263-323)
        const T thresh = fx.c >= 0.0f ? fx.c : 0.01f * mx;
        const T inv_mx = 1.0f / (mx + 1e-12f);
        const float *jit = reinterpret_cast<const float *>(fx.table);
        for (int row = 0; row < ROWS; ++row) {
            if (row < ROWS - 1 || lane == 0) {
                const int p = rpos<T, NC>(lane, row);
                const T m = mags[p];
                if (!(thresh > 0.0f) || m > thresh) {
                    T rot = fx.a * (m * inv_mx);
                    if (jit) rot += (T)__ldg(jit + tab_base + 32 * row + lane) * (T)fx.b;
                    T sn, cs;
                    sincos_fast(rot, &sn, &cs);   // |rot| <= 1.2 pi: the MUFU pair is good to ~1e-6 there
                    const V2<T> u = buf[p];
                    buf[p] = mk2<T>(u.x * cs - u.y * sn, u.x * sn + u.y * cs);
                }
            }
        }
    } else if (fx.mode == 4 || fx.mode == 5) {
        // bin scramble (dsp/spectral_fx.py:326-390): gather through the host-replayed index table
        sm = warp_sum(sm);
        const int16_t *idx = reinterpret_cast<const int16_t *>(fx.table);
        if constexpr (ROWS <= 33) {   // n_fft <= 2048: the whole frame fits the row registers
            T val[ROWS];
            T s2 = 0.0f;
#pragma unroll
            for (int row = 0; row < ROWS; ++row) {
                val[row] = 0.0f;
                if (row < ROWS - 1 || lane == 0) {
                    const int src = idx ? (int)__ldg(idx + tab_base + 32 * row + lane) : 32 * row + lane;
                    val[row] = mags[spos<T, NC>(src)];
                    s2 += val[row];
                }
            }
            s2 = warp_sum(s2);
            const T scale = sm / (s2 + 1e-12f);
            __syncwarp();
#pragma unroll
            for (int row = 0; row < ROWS; ++row)
                if (row < ROWS - 1 || lane == 0) mags[rpos<T, NC>(lane, row)] = val[row] * scale;
        } else {
            // longer frames: tiles of CH rows.  A tile's sources lie within `half` bins of it (half <= 32 CH, checked
            // by the host), so tile c-1 may be overwritten once tile c has been gathered; the energy rescale needs the
            // sum over the whole frame and runs as a second sweep (same product m[idx] * scale as the reference).
            constexpr int CH = sizeof(T) == 4 ? 32 : 16;
            constexpr int NCH = (ROWS + CH - 1) / CH;
            T prev[CH], cur[CH];
            T s2 = 0.0f;
#pragma unroll 1
            for (int c = 0; c <= NCH; ++c) {
                if (c < NCH) {
#pragma unroll
                    for (int r = 0; r < CH; ++r) {
                        const int row = c * CH + r;
                        cur[r] = 0.0f;
                        if (row < ROWS - 1 || (row == ROWS - 1 && lane == 0)) {
                            const int src = idx ? (int)__ldg(idx + tab_base + 32 * row + lane) : 32 * row + lane;
                            cur[r] = mags[spos<T, NC>(src)];
                            s2 += cur[r];
                        }
                    }
                }
                __syncwarp();   // every lane has gathered tile c before tile c-1 is overwritten
                if (c > 0) {
#pragma unroll
                    for (int r = 0; r < CH; ++r) {
                        const int row = (c - 1) * CH + r;
                        if (row < ROWS - 1 || (row == ROWS - 1 && lane == 0)) mags[rpos<T, NC>(lane, row)] = prev[r];
                    }
                }
#pragma unroll
                for (int r = 0; r < CH; ++r) prev[r] = cur[r];
            }
            s2 = warp_sum(s2);
            const T scale = sm / (s2 + 1e-12f);
            __syncwarp();
            for (int row = 0; row < ROWS; ++row)
                if (row < ROWS - 1 || lane == 0) mags[rpos<T, NC>(lane, row)] *= scale;
        }
    }
    __syncwarp();
}

// table read: read-only global path, or a plain load when the table was copied into shared memory
template <bool TS, class T>
QD_DEV T tld(const T *p) {
    if constexpr (TS) return *p;
    else return __ldg(p);
}

// one step of the segmented warp scan of Q1: add the values shuffled up by d when the lane has at least d
// same-slot sources below it (one ISETP + three predicated FADD)
template <class T>
QD_DEV void seg_scan_step(T &g, V2<T> &p, int off, int d) {
    const T go = __shfl_up_sync(QD_FULL, g, d);
    const T pxo = __shfl_up_sync(QD_FULL, p.x, d);
    const T pyo = __shfl_up_sync(QD_FULL, p.y, d);
#ifdef QD_EMU
    if (off >= d) { g += go; p.x += pxo; p.y += pyo; }
#else
    if constexpr (sizeof(T) == 4) {
        asm("{\n\t.reg .pred q;\n\tsetp.ge.s32 q, %6, %7;\n\t@q add.f32 %0, %0, %3;\n\t@q add.f32 %1, %1, %4;\n\t@q add.f32 %2, %2, %5;\n\t}"
            : "+f"(g), "+f"(p.x), "+f"(p.y) : "f"(go), "f"(pxo), "f"(pyo), "r"(off), "r"(d));
    } else {
        if (off >= d) { g += go; p.x += pxo; p.y += pyo; }
    }
#endif
}

// ---------------------------------------------------------------- quantizer fused with the real split / merge
// The spectral pass is bound by shared-memory wavefronts, so the quantizer does not run real_split / real_merge as
// separate sweeps over the warp buffer: the plain (no-FX) variant reads the packed-FFT output Z[k], Z[NC-k]
// as a pair, forms X[k] and X[NC-k] in registers, quantizes both, and writes Z'[k], Z'[NC-k] back -- one read
// and one write of the buffer instead of three.  A lane walks bin k = 32 i + lane upwards (low side) and its
// mirror NC - k downwards (high side); both sides keep the rolling three-row window of the smoothing, and
// the two walks meet at bin NC/2.

// X[k] for any k in 0..NC straight from Z (Q1 sources).  DC / Nyquist come out of the same formula because
// Z[NC] = Z[0] and V_0 = -i/2.
template <class T, int NC>
QD_DEV V2<T> split_bin(const V2<T> *buf, const V2<T> *wsplit, int k) {
    const bool hi = 2 * k > NC;
    const int kk = hi ? NC - k : k;
    const V2<T> za = buf[spos_lt<T, NC>(kk)];
    const V2<T> zb = cconj(buf[spos_lt<T, NC>((NC - kk) & (NC - 1))]);
    const V2<T> t = cmul(csub(za, zb), wsplit[kk]);
    const V2<T> e = cadd(za, zb);
    return hi ? cconj(pfma(e, splat((T)0.5), mk2<T>(-t.x, -t.y))) : pfma(e, splat((T)0.5), t);
}

// quantizer arithmetic of bin d (any lane / row mapping): magnitude after giving away / receiving energy, and
// the phasor of the arriving sum when energy arrived
template <class T, bool TS>
QD_DEV void quant_apply(T m, V2<T> &u, T &nm, int d, const T *slotG, const V2<T> *slotP, const QuantDev &q) {
    nm = ((tld<TS>(q.row_active + (d >> 5)) >> (d & 31)) & 1u) ? m * (T)q.keep_active : m;
    const uint16_t *sb = q.slot_of_bin + d;
    T te = (T)0;
    V2<T> ps = mk2<T>((T)0, (T)0);
#pragma unroll
    for (int e = 0; e < 5; ++e) {
        const int s = tld<TS>(sb + e);
        T c = (T)q.tap[e];
        if (e == 2) c += (T)tld<TS>(q.slot_base + s);
        te += c * slotG[s];
        ps = pfma(splat(c), slotP[s], ps);
    }
    nm += te;
    if (te > (T)0) {
        const T p2 = ps.x * ps.x + ps.y * ps.y;
        const bool ok = p2 > (T)QD_TINY2;
        const T r = rsqrt_fast(p2);
        u = ok ? pmul(ps, splat(r)) : mk2<T>((T)1, (T)0);
    }
}

// FX = true: buf holds the unit phasors of X and `mags` the (processed) magnitudes, both by buffer position with the
// Nyquist bin in the pad slot (fx_frame): the walk loads them instead of splitting Z, the Hermitian merge is the same.
template <class T, int NC, bool TS, bool FX = false>
QD_DEV void quantize_frame_fused(V2<T> *buf, const T *mags, T *slotG, V2<T> *slotP, const QuantDev &q, const V2<T> *wsplit, int lane) {
    // Q1: per-target gathers (see quantize_frame), the source bins split on the fly
    for (int s = lane; s <= q.n_slots; s += 32) {
        slotG[s] = 0.0f;
        slotP[s] = mk2<T>(0.0f, 0.0f);
    }
    __syncwarp();
#pragma unroll 1
    for (int i0 = 0; i0 < q.n_src; i0 += 32) {
        const int i = i0 + lane;
        uint32_t e = 0u;
        T g = 0.0f;
        V2<T> p = mk2<T>(0.0f, 0.0f);
        if (i < q.n_src) {
            e = tld<TS>(q.src_tab + i);
            if constexpr (FX) {
                const int pos = spos<T, NC>((int)(e & 0x1fffu));
                g = mags[pos];
                p = pmul(buf[pos], splat(g));
            } else {
                p = split_bin<T, NC>(buf, wsplit, (int)(e & 0x1fffu));
                const T m2 = p.x * p.x + p.y * p.y;
                g = m2 > QD_TINY2 ? m2 * rsqrt_fast(m2) : 0.0f;
            }
        }
        const int off = (int)((e >> 26) & 31u);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) seg_scan_step<T>(g, p, off, d);
        if (e >> 31) {
            const int sid = (int)((e >> 13) & 0x1fffu);
            slotG[sid] += g;
            slotP[sid] = padd(slotP[sid], p);
        }
        __syncwarp();
    }
    for (int sl = lane; sl < q.n_slots; sl += 32) {
        const T ik = (T)tld<TS>(q.slot_invk + sl);
        slotG[sl] *= ik;
        slotP[sl] = pmul(slotP[sl], splat(ik));
    }
    __syncwarp();

    // Q3: paired walk.  l* = low side (bins ascending), h* = high side (bins descending); *p/*c/*n = previous,
    // current, next row of the rolling smoothing window; the pair of iteration i-1 is finished in iteration i.
    constexpr int HR = NC / 64;
    const bool smooth = q.smoothing != 0;
    T lp = 0.0f, lc = 0.0f, ln = 0.0f, hp = 0.0f, hc = 0.0f, hn = 0.0f;
    V2<T> luc = mk2<T>(1.0f, 0.0f), lun = luc, huc = luc, hun = luc, vc = luc, vn = luc;
    int pac = 0, pbc = 0;
    const bool is0 = lane == 0, is31 = lane == 31;
    const int lane_m1 = (lane + 31) & 31, lane_p1 = (lane + 1) & 31;
    // `edge`: the pair being finished is iteration 0, whose lane 0 holds the two spectrum edges (DC, Nyquist)
    auto emit = [&](bool edge) {
        T ol = lc, oh = hc;
        if (smooth) {
            if (edge) {
                ol = smooth_row<T>(lp, lc, ln, lane, is0, false);
                oh = smooth_row<T>(hp, hc, hn, lane, is0, false);
            } else {
                ol = smooth_mid<T>(lp, lc, ln, is0, is31, lane_m1, lane_p1);
                oh = smooth_mid<T>(hp, hc, hn, is0, is31, lane_m1, lane_p1);
            }
        }
        V2<T> xa = pmul(luc, splat(ol));
        V2<T> xb = cconj(pmul(huc, splat(oh)));
        if (edge && is0) { xa.y = 0.0f; xb.y = 0.0f; }   // only Re of DC / Nyquist (pocketfft c2r)
        // Hermitian merge (see real_merge): Z'[k] = E2 + i O2, Z'[NC-k] = conj(E2 - i O2)
        const V2<T> e2 = cadd(xa, xb);
        const V2<T> h = cmulc(csub(xa, xb), vc);
        buf[pac] = pfma(h, splat((T)2), e2);
        buf[pbc] = cconj(pfma(h, splat((T)-2), e2));
    };
#pragma unroll 2
    for (int i = 0; i < HR; ++i) {
        const int k = 32 * i + lane;
        const int pa = rpos<T, NC>(lane, i);
        const int pb = k == 0 ? pa : mpos<T, NC>(lane, i);   // Z[NC] = Z[0]
        vn = wsplit[k];
        T ml, mh;
        if constexpr (FX) {
            const int pbr = k == 0 ? QD_NYQ_SLOT : pb;        // the Nyquist phasor / magnitude live in the pad slot
            lun = buf[pa]; ml = mags[pa];
            hun = buf[pbr]; mh = mags[pbr];
        } else {
            const V2<T> za = buf[pa], zb = cconj(buf[pb]);
            const V2<T> e = cadd(za, zb);
            const V2<T> t = cmul(csub(za, zb), vn);
            const V2<T> xl = pfma(e, splat((T)0.5), t);                            // X[k]
            const V2<T> xh = cconj(pfma(e, splat((T)0.5), mk2<T>(-t.x, -t.y)));    // X[NC-k]
            mag_phasor<T>(xl, ml, lun);
            mag_phasor<T>(xh, mh, hun);
        }
        if (i < q.row_limit) quant_apply<T, TS>(ml, lun, ln, k, slotG, slotP, q);
        else ln = ml;
        if (NC - 32 * i - 31 < 32 * q.row_limit) quant_apply<T, TS>(mh, hun, hn, NC - k, slotG, slotP, q);
        else hn = mh;
        if (i > 1) emit(false);
        else if (i == 1) emit(true);
        lp = lc; lc = ln; luc = lun;
        hp = hc; hc = hn; huc = hun;
        vc = vn; pac = pa; pbc = pb;
    }
    // the two walks meet at bin NC/2 (lane 0)
    {
        const int pm = spos<T, NC>(NC / 2);
        T mm = 0.0f;
        V2<T> um = mk2<T>(1.0f, 0.0f);
        if (lane == 0) {
            T m0;
            if constexpr (FX) { um = buf[pm]; m0 = mags[pm]; }
            else mag_phasor<T>(cconj(buf[pm]), m0, um);
            if ((NC / 64) < q.row_limit) quant_apply<T, TS>(m0, um, mm, NC / 2, slotG, slotP, q);
            else mm = m0;
        }
        ln = mm; hn = mm;
        emit(HR == 1);
        const T left = __shfl_sync(QD_FULL, lc, 31);    // bin NC/2 - 1
        const T right = __shfl_sync(QD_FULL, hc, 31);   // bin NC/2 + 1
        if (lane == 0) {
            const T om = smooth ? 0.5f * mm + 0.25f * (left + right) : mm;
            buf[pm] = mk2<T>(2.0f * om * um.x, -2.0f * om * um.y);
        }
    }
    __syncwarp();
}

// ---------------------------------------------------------------- the kernel
// NG independent groups of NW warps share one CTA (and its tables); each group streams its own clip and
// synchronises only with itself (named barrier), so one group's overlap-add step overlaps the other's FFTs.
// SA ("stage aliased"): the one-warp float64 formant variant of n_fft 8192 does not fit 227 KB with a staging buffer
// of its own, so the samples are staged in the warp's formant scratch buffer (dead until the frame's FFT is done;
// no prefetch of the next batch).
template <class T, int NC, int NW, int NG = 1, bool SA = false>
struct SpecSmem {
    static constexpr int HOP = NC / 2;                       // n_fft / 4 samples
    static constexpr int BUF = buf_slots<NC>();               // V2<T> per warp buffer
    static constexpr int STAGE = (NW + 3) * HOP;              // floats
    static constexpr int TAIL = 3 * HOP;                      // floats
    static_assert(!SA || (NW == 1 && NG == 1 && (size_t)STAGE * sizeof(float) <= (size_t)BUF * sizeof(V2<T>)), "stage alias");
    static constexpr size_t off_buf = 0;
    static constexpr size_t off_stage = off_buf + (size_t)NW * BUF * sizeof(V2<T>);
    static constexpr size_t off_tail = off_stage + (SA ? 0 : (size_t)STAGE * sizeof(float));
    static constexpr size_t off_flags = off_tail + (size_t)TAIL * sizeof(T);
    static constexpr size_t off_slot = off_flags + 64 * sizeof(int);
    // per-warp gather scratch: G[cap] floats then P[cap] V2<T>, cap even so P stays 8-byte aligned
    __host__ __device__ static int slot_cap(int n_slots) { return (n_slots + 2) & ~1; }
    __host__ __device__ static size_t off_tables(int n_slots) {
        return (off_slot + (size_t)NW * (size_t)slot_cap(n_slots) * 3 * sizeof(T) + 15) & ~(size_t)15;
    }
    // shared-memory copies of the hot tables (TS kernels): window, pass-1 twiddles, split twiddles,
    // then the quantizer tables (gather list, row masks, affected-bin entries)
    __host__ __device__ static size_t table_bytes(int n_src, int n_slots) {
        const int rows = (NC + 1 + 31) / 32;
        size_t b = (size_t)(NC + NC + NC / 2 + 2) * sizeof(V2<T>);
        b += ((size_t)n_src * 4 + 15) & ~(size_t)15;                   // src_tab
        b += ((size_t)rows * 4 + 15) & ~(size_t)15;                    // row_active
        b += ((size_t)(32 * rows + 4) * 2 + 15) & ~(size_t)15;         // slot_of_bin
        b += 2 * (((size_t)(n_slots + 1) * 4 + 15) & ~(size_t)15);     // slot_invk, slot_base
        return b + 64;
    }
    // layout: NG x [warp buffers | staging | OLA tail | flags | gather scratch], tables, FX magnitude planes
    __host__ __device__ static size_t group_bytes(int n_slots) { return off_tables(n_slots); }
    static size_t bytes(int n_slots, bool tables_in_smem = false, int n_src = 0, int /*unused*/ = 0, bool fx = false,
                        bool formant = false) {
        // FX kernels append one magnitude plane (BUF values of T) per warp, the formant shift a scratch buffer
        return NG * group_bytes(n_slots) + (tables_in_smem ? table_bytes(n_src, n_slots) : 16) +
               (fx ? (size_t)NG * NW * BUF * sizeof(T) : 0) + (formant ? (size_t)NG * NW * BUF * sizeof(V2<T>) : 0);
    }
};

// wavefold / tube on the float32 iSTFT sample (dsp/distortion.py:18-90)
// EF ("epilogue float"): the caller guarantees that the epilogue is none or a wavefold that is exact in float32 (no
// bias, power-of-two gain -- the reference defaults); no tanh either.  The float64 branch below is only a dozen instructions, but the overlap-add loop
// around it is unrolled NW + 3 times in the headline kernel, whose code already fills the instruction cache: with the
// branch compiled in, that kernel ran 3 % slower even though the branch was never taken (measured, A/B on one box).
template <bool EF>
QD_DEV float epilogue_apply(float v, int mode, double fold, double bias, int exact_f32, float tg, float tn) {
    if (mode == 1) {
        // dsp/distortion.py:37-58 computes in float64 and rounds to float32 once; the negative fold is tested on the
        // already folded value (:44-56).  (x + bias) * fold reaches several units before it is folded back, so float32
        // arithmetic would carry the rounding error of the large intermediate (~2e-7) into the small result -- and the
        // second spectral pass amplifies its input error.  With bias == 0 and fold a power of two float32 is exact.
        if constexpr (!EF) {
            if (!exact_f32) {
                double y = ((double)v + bias) * fold;
                if (y > 1.0) y = 2.0 - y;
                if (y < -1.0) y = -2.0 - y;
                return (float)fmin(fmax(y, -1.0), 1.0);
            }
        }
        float y = v * (float)fold;
        if (y > 1.0f) y = 2.0f - y;
        if (y < -1.0f) y = -2.0f - y;
        return fminf(fmaxf(y, -1.0f), 1.0f);
    }
    if constexpr (!EF) {
        if (mode == 2) return tanhf(tg * v) * tn;
    }
    return v;
}

// barrier among the 32*NW threads of one clip group (barrier 0 stays the CTA-wide __syncthreads)
template <int NG, int COUNT>
QD_DEV void group_sync(int g) {
    if constexpr (NG == 1) {
        __syncthreads();
    } else {
#ifdef QD_EMU
        qd_emu::named_barrier(g + 1, COUNT);
#else
        asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "n"(COUNT) : "memory");
#endif
    }
}

template <class T, int NC, int NW, bool TS = false, bool FX = false, int NG = 1, bool SA = false, bool EF = false>
__global__ void __launch_bounds__(32 * NW * NG)
spec_pass_kernel(const SpecArgsT<T> a) {
    using L = SpecSmem<T, NC, NW, NG, SA>;
    constexpr int HOP = L::HOP;
    constexpr int HP = HOP / 2;              // V2<T> pairs per hop
    constexpr int HPP = HP + HP / 32;        // the same span inside a padded warp buffer
    QD_DYN_SMEM(smem);
    constexpr int nthreads = 32 * NW;        // threads of one clip group
    const int grp = NG == 1 ? 0 : (int)threadIdx.x / nthreads;
    const int tid = NG == 1 ? (int)threadIdx.x : (int)threadIdx.x % nthreads;
    const int lane = tid & 31, warp = tid >> 5;
    unsigned char *gs = smem + (size_t)grp * L::group_bytes(a.q.n_slots);   // this group's private region
    unsigned char *tables_base = smem + (size_t)NG * L::group_bytes(a.q.n_slots);
    V2<T> *bufs = reinterpret_cast<V2<T> *>(gs + L::off_buf);
    float *stage = reinterpret_cast<float *>(gs + L::off_stage);
    if constexpr (SA)   // the formant scratch buffer of the (only) warp, see SpecSmem
        stage = reinterpret_cast<float *>(tables_base + 16 + (size_t)NG * NW * L::BUF * sizeof(T));
    V2<T> *tail = reinterpret_cast<V2<T> *>(gs + L::off_tail);
    V2<T> *buf = bufs + (size_t)warp * L::BUF;
    const int slot_cap = (a.q.n_slots + 2) & ~1;
    T *slotG = reinterpret_cast<T *>(gs + L::off_slot) + (size_t)warp * slot_cap * 3;
    V2<T> *slotP = reinterpret_cast<V2<T> *>(slotG + slot_cap);

    const int clip = (int)blockIdx.y * NG + grp;
    bool group_live = clip < a.batch;   // the last CTA may carry an empty group
    const ClipLoc cs = clip_loc(a, group_live ? clip : 0);
    const int idx = a.clip0 + clip;     // = cs.idx once the empty group has left; per-clip arrays are indexed by it
    const long long fx_row = a.fx.table_per_clip ? a.fx.clip_offset + idx : 0;
    const T *frozen = a.frozen ? a.frozen + (size_t)idx * L::BUF : nullptr;
    const int n = (int)cs.n;
    const float *x = a.x + cs.base;
    float *y = a.y + cs.base;
    float *tap = a.tap ? a.tap + cs.base : nullptr;
    // 8-byte vector stores need an even clip length and 8-byte aligned rows; 16-byte staging loads an aligned clip start
    const bool vec2 = ((n & 1) == 0) && ((reinterpret_cast<uintptr_t>(y) & 7) == 0) &&
                      (!tap || (reinterpret_cast<uintptr_t>(tap) & 7) == 0);
    const bool vec4 = (reinterpret_cast<uintptr_t>(x) & 15) == 0;

    // output hop-blocks (of the zero-padded timeline) this CTA owns: [j0, j1); block 2 <-> sample 0
    const int j_end = 2 + (n + HOP - 1) / HOP;
    const int j0 = 2 + blockIdx.x * a.tile_blocks;
    const int j1 = min(j0 + a.tile_blocks, j_end);
    // a group past its clip's end has nothing to do.  With NG = 2 the groups of a CTA may belong to clips of different
    // lengths, and the table fill below needs the whole CTA: such a group leaves with the empty group, after the last
    // CTA-wide barrier; the CTA returns here only when neither group has work.
    if constexpr (NG == 1) {
        if (j0 >= j1) return;
    } else {
        group_live = group_live && j0 < j1;
        if (!__syncthreads_or(group_live)) return;
    }
    const int t_first = j0 - 3;  // first frame that touches block j0 (may be < 0: skipped)
    const int n_frames = 1 + n / HOP;

    for (int i = tid; i < 3 * HP; i += nthreads) tail[i] = mk2<T>(0.0f, 0.0f);

    // TMA staging: the samples of the NEXT batch of frames are fetched by one cp.async.bulk while this batch
    // is still in its quantizer / inverse FFT; `full` (mbarrier, transaction bytes) says when they have landed,
    // `consumed` counts the warps that are done reading the staging buffer of the current batch.
    uint64_t *full = reinterpret_cast<uint64_t *>(gs + L::off_flags);
    int *consumed = reinterpret_cast<int *>(gs + L::off_flags + 8);
    if (tid == 0) {
        mbar_init(full, 1);
        *consumed = 0;
    }
    uint32_t full_parity = 0;
    bool tma_pending = false;
    constexpr uint32_t STAGE_BYTES = (uint32_t)(L::STAGE * sizeof(float));
    __syncthreads();

    // hot tables: read through L1/L2, or (TS) copied once per CTA into shared memory
    const V2<T> *wtab = a.wtab, *tw1 = a.tw1, *wsplit = a.wsplit;
    QuantDev qq = a.q;
    if constexpr (TS) {
        const int ctid = threadIdx.x, cthreads = nthreads * NG;   // the whole CTA fills the shared tables
        V2<T> *t_w = reinterpret_cast<V2<T> *>(tables_base);
        V2<T> *t_tw = t_w + NC;
        V2<T> *t_ws = t_tw + NC;
        for (int i = ctid; i < NC; i += cthreads) t_tw[i] = a.tw1[i];
        for (int i = ctid; i < 2 * (NC / FftCfg<T, NC>::R1); i += cthreads) t_w[i] = a.wtab[i];
        for (int i = ctid; i <= NC / 2; i += cthreads) t_ws[i] = a.wsplit[i];
        wtab = t_w; tw1 = t_tw; wsplit = t_ws;
        if (a.quant) {
            constexpr int ROWS = (NC + 1 + 31) / 32;
            unsigned char *qb = reinterpret_cast<unsigned char *>(t_ws + NC / 2 + 2);
            uint32_t *s_src = reinterpret_cast<uint32_t *>(qb);
            qb += ((size_t)a.q.n_src * 4 + 15) & ~(size_t)15;
            uint32_t *s_ra = reinterpret_cast<uint32_t *>(qb);
            qb += ((size_t)ROWS * 4 + 15) & ~(size_t)15;
            uint16_t *s_sb = reinterpret_cast<uint16_t *>(qb);
            qb += ((size_t)(32 * ROWS + 4) * 2 + 15) & ~(size_t)15;
            float *s_ik = reinterpret_cast<float *>(qb);
            qb += ((size_t)(a.q.n_slots + 1) * 4 + 15) & ~(size_t)15;
            float *s_bs = reinterpret_cast<float *>(qb);
            for (int i = ctid; i < a.q.n_src; i += cthreads) s_src[i] = a.q.src_tab[i];
            for (int i = ctid; i < ROWS; i += cthreads) s_ra[i] = a.q.row_active[i];
            for (int i = ctid; i < 32 * ROWS + 4; i += cthreads) s_sb[i] = a.q.slot_of_bin[i];
            for (int i = ctid; i <= a.q.n_slots; i += cthreads) { s_ik[i] = a.q.slot_invk[i]; s_bs[i] = a.q.slot_base[i]; }
            qq.src_tab = s_src; qq.row_active = s_ra; qq.slot_of_bin = s_sb; qq.slot_invk = s_ik; qq.slot_base = s_bs;
        }
        __syncthreads();
    }
    if (!group_live) return;   // after the last CTA-wide barrier; the other group only uses its named barrier

    float out_peak = 0.0f;   // max |y| this thread stored
    for (int tb = t_first; tb < j1; tb += NW) {
        // ---- stage the samples of frames tb .. tb+NW-1 (zero outside the clip)
        const long long s0 = (long long)tb * HOP - NC;  // clip index of staging[0]
        const long long s0n = s0 + (long long)NW * HOP;  // the same for the next batch
        const bool next_by_tma = !SA && vec4 && (tb + NW < j1) && s0n >= 0 && s0n + L::STAGE <= n;
        if (tma_pending) {
            mbar_wait(full, full_parity);  // bulk copy issued during the previous batch
            full_parity ^= 1u;
        } else {
            if (vec4 && s0 >= 0 && s0 + L::STAGE <= n) {
                const float4 *src = reinterpret_cast<const float4 *>(x + s0);
                float4 *dst = reinterpret_cast<float4 *>(stage);
#pragma unroll 4
                for (int i = tid; i < L::STAGE / 4; i += nthreads) dst[i] = src[i];
            } else {
                for (int i = tid; i < L::STAGE; i += nthreads) {
                    const long long s = s0 + i;
                    stage[i] = (s >= 0 && s < n) ? x[s] : 0.0f;
                }
            }
            group_sync<NG, 32 * NW>(grp);
        }
        tma_pending = next_by_tma;
        // ---- one frame per warp (a frame outside the clip contributes zeros)
        const int t = tb + warp;
        const bool live = t >= 0 && t < n_frames;
        if (live) {
            const float2 *frame = reinterpret_cast<const float2 *>(stage + warp * HOP);
            fwd_first<T, NC, FftCfg<T, NC>::R1>(buf, frame, wtab, tw1, lane);
        }
        // this warp no longer needs the staging buffer; the last warp to say so starts the next bulk copy
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(consumed, 1) == NW - 1) {
                *consumed = 0;
                if (next_by_tma) {
                    mbar_expect_tx(full, STAGE_BYTES);
                    bulk_g2s(stage, x + s0n, STAGE_BYTES, full);
                }
            }
        }
        if (live) {
            fft_forward<T, NC>(buf, nullptr, a, wtab, tw1, a.tw2, lane);
            if (!a.quant) real_split<T, NC>(buf, wsplit, lane);
            if (a.quant) {
                if constexpr (FX) {
                    // magnitude planes (and the formant scratch buffers) follow the shared tables
                    unsigned char *planes = tables_base + (TS ? L::table_bytes(a.q.n_src, a.q.n_slots) : 16);
                    T *mags = reinterpret_cast<T *>(planes) + (size_t)(grp * NW + warp) * L::BUF;
                    const int tf = t < a.fx.table_frames ? t : a.fx.table_frames - 1;
                    const long long tab_base =
                        ((fx_row * 2 + a.fx.pass) * a.fx.table_frames + tf) * (NC + 1);
                    V2<T> *scr = reinterpret_cast<V2<T> *>(planes + (size_t)NG * NW * L::BUF * sizeof(T)) +
                                 (size_t)(grp * NW + warp) * L::BUF;   // only there when the formant shift is on
                    fx_frame<T, NC>(buf, mags, a.fx, lane, tab_base,
                                    frozen, scr, a, tw1, wsplit);
                    quantize_frame_fused<T, NC, TS, true>(buf, mags, slotG, slotP, qq, wsplit, lane);
                } else {
                    quantize_frame_fused<T, NC, TS, false>(buf, nullptr, slotG, slotP, qq, wsplit, lane);
                }
            }
            if (!a.quant) real_merge<T, NC>(buf, wsplit, lane);
            fft_inverse<T, NC>(buf, wtab, tw1, a.tw2, lane);
        } else {
            for (int i = lane; i < L::BUF; i += 32) buf[i] = mk2<T>(0.0f, 0.0f);
        }
        group_sync<NG, 32 * NW>(grp);
        // ---- overlap-add in frame order; blocks tb .. tb+NW-1 are now complete.  A thread owns one
        //      column of sample pairs: slice sl of warp w's frame sits at bufs[w][sl*HPP + pidx(c)].
        //      The hop loop is unrolled only in the EF kernel (small epilogue): elsewhere NW + 3 copies of the store path
        //      cost more instruction-cache misses than the loop overhead they save.
        for (int c = tid; c < HP; c += nthreads) {
            const int pc = pidx(c);
            // one output hop of this thread's column; FAST = float32-only epilogue, 8-byte stores, no tap
            auto hop = [&](int h, auto fast_tag) {
                constexpr bool FAST = decltype(fast_tag)::value;
                V2<T> v = (h < 3) ? tail[h * HP + c] : mk2<T>(0.0f, 0.0f);   // partial sums carried from the last batch
                const int w0 = h - 3 > 0 ? h - 3 : 0, w1 = h < NW - 1 ? h : NW - 1;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int w = w0 + k;
                    if (w <= w1) v = padd(v, bufs[(size_t)w * L::BUF + (h - w) * HPP + pc]);
                }
                if (h >= NW) {
                    tail[(h - NW) * HP + c] = v;  // partial sums of the next three blocks (slot h - NW < h: already read)
                    return;
                }
                const int j = tb + h;
                if (j < j0 || j >= j1) return;
                const long long nidx = (long long)(j - 2) * HOP + 2 * c;
                if (nidx >= n) return;
                // frames covering block j: slices sl = j - t with t in [max(0,j-3), min(j,T-1)]
                const int sl_a = j - n_frames + 1 > 0 ? j - n_frames + 1 : 0;
                const int sl_b = j < 3 ? j : 3;
                V2<T> inv = mk2<T>(0.0f, 0.0f);
                if (sl_a <= sl_b) inv = __ldg(reinterpret_cast<const V2<T> *>(a.invw + (sl_a * 4 + sl_b) * HOP) + c);
                const V2<T> vi = pmul(v, inv);
                const float2 o = make_float2((float)vi.x, (float)vi.y);  // float32 like istft_mono
                const float2 r = make_float2(epilogue_apply<FAST>(o.x, a.epilogue, a.fold, a.bias, a.fold_exact_f32, a.tube_gain, a.tube_norm),
                                             epilogue_apply<FAST>(o.y, a.epilogue, a.fold, a.bias, a.fold_exact_f32, a.tube_gain, a.tube_norm));
                if (FAST || vec2) {  // nidx is even and n is even, so nidx + 1 < n
                    if (!FAST && tap) *reinterpret_cast<float2 *>(tap + nidx) = o;
                    *reinterpret_cast<float2 *>(y + nidx) = r;
                    out_peak = fmaxf(out_peak, fmaxf(fabsf(r.x), fabsf(r.y)));
                } else {
                    if (tap) tap[nidx] = o.x;
                    y[nidx] = r.x;
                    out_peak = fmaxf(out_peak, fabsf(r.x));
                    if (nidx + 1 < n) {
                        if (tap) tap[nidx + 1] = o.y;
                        y[nidx + 1] = r.y;
                        out_peak = fmaxf(out_peak, fabsf(r.y));
                    }
                }
            };
            // The kernel's code fills the instruction cache, so only the EF kernel unrolls the hop loop, and only with
            // the compact hop (no tanh, no float64, no scalar stores, no tap: the reference defaults on aligned clips);
            // every other case runs the general hop in a rolled loop -- NW + 3 copies of it cost more in instruction
            // fetch than the loop overhead they save (measured: 60.1 -> 56.2 ms per render of 4096 clips).
            if (EF && vec2 && !tap) {
#pragma unroll
                for (int h = 0; h < NW + 3; ++h) hop(h, KBool<EF>{});
            } else {
#pragma unroll 1
                for (int h = 0; h < NW + 3; ++h) hop(h, KBool<false>{});
            }
        }
        group_sync<NG, 32 * NW>(grp);
    }
    if (a.clip_peak) {   // non-negative floats order like their bit patterns
        out_peak = warp_max(out_peak);
        if (lane == 0) atomicMax(reinterpret_cast<unsigned *>(a.clip_peak) + idx, __float_as_uint(out_peak));
    }
}

// |X| of frame 0 of every clip, by buffer position (input of the spectral-freeze variant of the pass).
// One warp per clip; frame 0 = n_fft/2 zeros of centre padding followed by the first n_fft/2 samples.
template <class T, int NC>
__global__ void __launch_bounds__(32)
freeze_mag_kernel(const SpecArgsT<T> a, T *out) {
    constexpr int BUF = buf_slots<NC>();
    QD_DYN_SMEM(smem);
    V2<T> *buf = reinterpret_cast<V2<T> *>(smem);
    float *stage = reinterpret_cast<float *>(smem + (size_t)BUF * sizeof(V2<T>));
    const int lane = threadIdx.x;
    const ClipLoc cs = clip_loc(a, (int)blockIdx.x);
    const float *x = a.x + cs.base;
    for (int i = lane; i < 2 * NC; i += 32) {
        const long long s = (long long)i - NC;
        stage[i] = (s >= 0 && s < cs.n) ? x[s] : 0.0f;
    }
    __syncwarp();
    fwd_first<T, NC, FftCfg<T, NC>::R1>(buf, reinterpret_cast<const float2 *>(stage), a.wtab, a.tw1, lane);
    fft_forward<T, NC>(buf, nullptr, a, a.wtab, a.tw1, a.tw2, lane);
    real_split<T, NC>(buf, a.wsplit, lane);
    T *o = out + (size_t)cs.idx * BUF;
    for (int p = lane; p < BUF; p += 32) {
        const V2<T> v = buf[p];
        const T m2 = v.x * v.x + v.y * v.y;
        o[p] = m2 > (T)QD_TINY2 ? m2 * rsqrt_fast(m2) : (T)0;
    }
}

}  // namespace qd
