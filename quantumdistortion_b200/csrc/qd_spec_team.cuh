// qd_spec_team.cuh -- the spectral pass for the three-pass FFT plans (every n_fft but 2048 in float32, every n_fft in
// float64): a TEAM of CW warps owns one frame, and the frame buffers are XOR-swizzled instead of padded.
//
// qd_spec.cuh gives every frame to one warp, whose private buffer holds the frame's spectrum.  At n_fft 4096 / 8192 that
// buffer is 17 / 34 KB (float32) or 68 KB (float64, n_fft 8192), so only 8 / 4 / 2 warps fit one SM and the pass is bound
// by latency, not by any pipe (ncu: 31 % / 19 % issue-active).  Here the frames keep their buffers but CW warps share the
// work on each of them, which multiplies the resident warps by CW at the same shared-memory footprint:
//   * FFT passes: the butterflies of one pass are independent, warp w takes butterfly groups w, w + CW, ...; a named
//     barrier of the team's 32 CW threads stands where the one-warp version has __syncwarp();
//   * quantizer gather (Q1): every target slot belongs to ONE warp of the team (host schedule, build_team_gather): a
//     warp walks its own 32-aligned gather list, so slot sums are race free and their summation order is fixed;
//   * quantizer walk (Q3): warp w owns a range of rows of the paired walk; the magnitudes of the two rows that border its
//     range are computed first, by the neighbour's rule, before any warp overwrites the buffer (barrier), so the
//     3-tap smoothing sees the same window as the one-warp walk;
//   * staging, overlap-add, epilogue and the HBM side are those of spec_pass_kernel (one clip per CTA).
// The short three-pass plans (n_fft 512 / 1024) run it with CW = 1: the one-warp schedule, for the swizzled layout alone
// (the 33/32 padding of qd_spec.cuh is conflict-free only for the 32 x 32 plan of n_fft 2048; see tpos below).
// Same arithmetic per bin as qd_spec.cuh (the helpers are shared); only the association of the Q1 partial sums differs
// (chunks of 32 sources are counted from the start of each warp's list).  Plain variant only (no spectral FX).
#pragma once
#include "qd_spec.cuh"

namespace qd {

constexpr int QD_TEAM_MAX = 8;

// gather lists of the team kernel: warp w of a team reads src_tab[begin[w] .. begin[w + 1]) (multiples of 32;
// entries like QuantDev::src_tab, padding entries are 0: no tail bit, nothing is stored)
struct TeamGather {
    const uint32_t *src_tab;
    int begin[QD_TEAM_MAX + 1];
};

template <int CW>
QD_DEV void team_sync(int team) {
    if constexpr (CW == 1) {
        __syncwarp();
    } else {
#ifdef QD_EMU
        qd_emu::named_barrier(team + 1, 32 * CW);
#else
        asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "n"(32 * CW) : "memory");
#endif
    }
}

// ---------------------------------------------------------------- buffer layout: XOR swizzle instead of the 33/32 padding
// The padding of qd_spec.cuh is conflict-free for the 32 x 32 plan only.  The three-pass plans touch the buffer in four
// patterns -- per half-warp (8-byte elements) or quarter-warp (16-byte elements) the lanes differ in
//   first / last pass, overlap-add : the lowest index bits,
//   middle pass (stride S2)        : the lowest bits below S2 and the bits from M2 upwards,
//   third pass (stride 1 per lane) : the bits from R3 upwards,
//   rows of the walk (bin k)       : the bits from NC / R1 upwards (k mod R1 is the slowest digit of the position)
// and element a sits at  a ^ low(a),  low = a GF(2)-linear image of the higher index bits (for the long frames
// ((a >> S1) & M1) ^ ((a >> S2) & M2)) that folds exactly those bits onto the bank bits, so that each pattern is a
// bijection onto the 16 (8) banks.  Bits above the bank bits are untouched: the map is a
// permutation of [0, NC), and it is linear over XOR, so pos(a0 + q S) = pos(a0) ^ pos(q S) with a compile-time second term
// whenever a0 and q S occupy different bits (they do in every pass).
// low(a): what is XORed onto the bank bits; a function of index bits above the bank bits only.
template <class T, int NC> struct TeamSwz;
template <> struct TeamSwz<float, 2048>  { static __host__ __device__ constexpr int low(int a) { return ((a >> 4) & 15) ^ ((a >> 8) & 7); } };
template <> struct TeamSwz<float, 4096>  { static __host__ __device__ constexpr int low(int a) { return ((a >> 4) & 15) ^ ((a >> 8) & 15); } };
template <> struct TeamSwz<double, 2048> { static __host__ __device__ constexpr int low(int a) { return ((a >> 3) & 7) ^ ((a >> 7) & 7); } };
template <> struct TeamSwz<double, 4096> { static __host__ __device__ constexpr int low(int a) { return ((a >> 4) & 7) ^ ((a >> 8) & 7); } };
// the short frames (one warp per frame, CW = 1) have three-pass plans too: 8 x 8 x 8 (n_fft 1024) and 8 x 8 x 4 (n_fft 512).
// Half-warp patterns of 8 x 8 x 8: {a0..a3}, {a0,a1,a2,a6}, {a3..a6}, rows {a6,a7,a8,a3};
// of 8 x 8 x 4: {a0..a3}, {a0,a1,a5,a6}, {a2..a5}, rows {a5,a6,a7,a2}.  Bank images of the higher bits (b3 b2 b1 b0):
template <> struct TeamSwz<float, 512> {   // a4 -> 0001, a5 -> 0010, a6 -> 1100, a7 -> 0001, a8 -> 0010
    static __host__ __device__ constexpr int low(int a) { return ((a >> 4) & 3) ^ (((a >> 6) & 1) * 12) ^ ((a >> 7) & 3); }
};
template <> struct TeamSwz<float, 256> {   // a4 -> 0010, a5 -> 0101, a6 -> 1000, a7 -> 0010
    static __host__ __device__ constexpr int low(int a) { return (((a >> 4) & 1) << 1) ^ (((a >> 5) & 1) * 5) ^ (((a >> 6) & 1) << 3) ^ (((a >> 7) & 1) << 1); }
};
template <> struct TeamSwz<double, 1024> { static __host__ __device__ constexpr int low(int a) { return ((a >> 3) & 7) ^ ((a >> 6) & 7); } };   // 16 x 8 x 8
template <> struct TeamSwz<double, 512> { static __host__ __device__ constexpr int low(int a) { return ((a >> 3) & 7) ^ ((a >> 6) & 7); } };
template <> struct TeamSwz<double, 256> { static __host__ __device__ constexpr int low(int a) { return ((a >> 3) & 7) ^ ((a >> 6) & 3); } };
template <class T, int NC>
QD_DEV constexpr int tpos(int a) { return a ^ TeamSwz<T, NC>::low(a); }
// position of spectrum bin k (0 <= k < NC) after the in-place DIF passes (digit order of qd::spos)
template <class T, int NC>
QD_DEV int tspos(int k) {
    using C = FftCfg<T, NC>;
    const unsigned uk = (unsigned)k;
    const unsigned k1 = uk & (unsigned)(C::R1 - 1);
    const unsigned k2 = (uk / (unsigned)C::R1) & (unsigned)(C::R2 - 1);
    const unsigned k3 = uk / (unsigned)(C::R1 * C::R2);
    return tpos<T, NC>((int)(k1 * (unsigned)(NC / C::R1) + k2 * (unsigned)(NC / (C::R1 * C::R2)) + k3));
}

// ---------------------------------------------------------------- FFT passes, butterfly groups dealt to the team's warps
template <class T, int NC, int R, int CW>
QD_DEV void t_fwd_first(V2<T> *buf, const float2 *frame, const V2<T> *wtab, const V2<T> *tw, int lane, int wsub, int team) {
    constexpr int S = NC / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = wsub; i < NB; i += CW) {
        const int a0 = lane + 32 * i;
        const V2<T> wc = __ldg(wtab + 2 * a0), ws = __ldg(wtab + 2 * a0 + 1);
        V2<T> v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) {
            const float2 s = frame[a0 + q * S];
            v[q] = pmul(mk2<T>((T)s.x, (T)s.y), hann_pair<T, R>(wc, ws, q));
        }
        dft_reg<R, -1, T>(v);
        const int p0 = tpos<T, NC>(a0);
        buf[p0] = v[0];
        twiddle_walk<T, R>(tw + (i * R) * 32 + lane,
                           [&](auto kc, V2<T> w) {
                               constexpr int k = decltype(kc)::value;
                               buf[p0 ^ tpos<T, NC>(k * S)] = cmul(v[qd_bitrev(k, LG)], w);
                           });
    }
}

// first forward pass of a sequence that already sits in the buffer (swizzled positions), no window
template <class T, int NC, int R, int CW>
QD_DEV void t_fwd_first_buf(V2<T> *buf, const V2<T> *tw, int lane, int wsub) {
    constexpr int S = NC / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = wsub; i < NB; i += CW) {
        const int p0 = tpos<T, NC>(lane + 32 * i);
        V2<T> v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = buf[p0 ^ tpos<T, NC>(q * S)];
        dft_reg<R, -1, T>(v);
        buf[p0] = v[0];
        twiddle_walk<T, R>(tw + (i * R) * 32 + lane,
                           [&](auto kc, V2<T> w) {
                               constexpr int k = decltype(kc)::value;
                               buf[p0 ^ tpos<T, NC>(k * S)] = cmul(v[qd_bitrev(k, LG)], w);
                           });
    }
}

template <class T, int NC, int M, int R, bool TW, int CW>
QD_DEV void t_fwd_pass(V2<T> *buf, const V2<T> *tw, int lane, int wsub) {
    constexpr int S = M / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = wsub; i < NB; i += CW) {
        const int u = lane + 32 * i;
        const int p0 = tpos<T, NC>((u / S) * M + (u % S));
        V2<T> v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = buf[p0 ^ tpos<T, NC>(q * S)];
        dft_reg<R, -1, T>(v);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int k = qd_bitrev(r, LG);
            V2<T> t = v[r];
            if (TW && k > 0) t = cmul(t, __ldg(tw + (i * R + k) * 32 + lane));
            buf[p0 ^ tpos<T, NC>(k * S)] = t;
        }
    }
}

template <class T, int NC, int M, int R, bool TW, int CW>
QD_DEV void t_inv_pass(V2<T> *buf, const V2<T> *tw, int lane, int wsub) {
    constexpr int S = M / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = wsub; i < NB; i += CW) {
        const int u = lane + 32 * i;
        const int p0 = tpos<T, NC>((u / S) * M + (u % S));
        V2<T> v[R];
#pragma unroll
        for (int k = 0; k < R; ++k) {
            V2<T> t = buf[p0 ^ tpos<T, NC>(k * S)];
            if (TW && k > 0) t = cmulc(t, __ldg(tw + (i * R + k) * 32 + lane));
            v[k] = t;
        }
        dft_reg<R, +1, T>(v);
#pragma unroll
        for (int r = 0; r < R; ++r) buf[p0 ^ tpos<T, NC>(qd_bitrev(r, LG) * S)] = v[r];
    }
}

template <class T, int NC, int R, int CW>
QD_DEV void t_inv_last(V2<T> *buf, const V2<T> *wtab, const V2<T> *tw, int lane, int wsub) {
    constexpr int S = NC / R;
    constexpr int NB = NC / R / 32;
    constexpr int LG = qd_log2(R);
#pragma unroll 1
    for (int i = wsub; i < NB; i += CW) {
        const int a0 = lane + 32 * i;
        V2<T> v[R];
        const int p0 = tpos<T, NC>(a0);
        v[0] = buf[p0];
        twiddle_walk<T, R>(tw + (i * R) * 32 + lane, [&](auto kc, V2<T> w) {
            constexpr int k = decltype(kc)::value;
            v[k] = cmulc(buf[p0 ^ tpos<T, NC>(k * S)], w);
        });
        dft_reg<R, +1, T>(v);
        const V2<T> wc = __ldg(wtab + 2 * a0), ws = __ldg(wtab + 2 * a0 + 1);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int q = qd_bitrev(r, LG);
            buf[p0 ^ tpos<T, NC>(q * S)] = pmul(v[r], hann_pair<T, R>(wc, ws, q));
        }
    }
}

// the forward passes after t_fwd_first / the whole inverse FFT; every pass ends at the team barrier
template <class T, int NC, int CW>
QD_DEV void t_fft_forward_rest(V2<T> *buf, const V2<T> *tw2, int lane, int wsub, int team) {
    using C = FftCfg<T, NC>;
    static_assert(C::R3 > 1, "the team kernel is built for the three-pass plans");
    t_fwd_pass<T, NC, NC / C::R1, C::R2, true, CW>(buf, tw2, lane, wsub);
    team_sync<CW>(team);
    t_fwd_pass<T, NC, C::R3, C::R3, false, CW>(buf, nullptr, lane, wsub);
    team_sync<CW>(team);
}

template <class T, int NC, int CW>
QD_DEV void t_fft_inverse(V2<T> *buf, const V2<T> *wtab, const V2<T> *tw1, const V2<T> *tw2, int lane, int wsub, int team) {
    using C = FftCfg<T, NC>;
    t_inv_pass<T, NC, C::R3, C::R3, false, CW>(buf, nullptr, lane, wsub);
    team_sync<CW>(team);
    t_inv_pass<T, NC, NC / C::R1, C::R2, true, CW>(buf, tw2, lane, wsub);
    team_sync<CW>(team);
    t_inv_last<T, NC, C::R1, CW>(buf, wtab, tw1, lane, wsub);
    // the caller's CTA-wide barrier before the overlap-add closes this pass
}

// real split / merge (quantizer off): the (k, NC - k) pairs are independent, rows dealt to the warps
template <class T, int NC, int CW>
QD_DEV void t_split_merge(V2<T> *buf, const V2<T> *wsplit, int lane, int wsub) {
    // real_merge(real_split(Z)) on one pair: X[k] = E/2 + T, X[NC-k] = conj(E/2 - T), then Z'[k] = E2 + i O2, ...
#pragma unroll 1
    for (int row = wsub; row < NC / 64; row += CW) {
        const int k = lane + 32 * row;
        if (k == 0) {
            const V2<T> z0 = buf[0];                          // tspos(0) = 0
            const T a = z0.x + z0.y, b = z0.x - z0.y;       // X[0], X[NC] (real)
            buf[0] = mk2<T>(a + b, a - b);
            const int pm = tspos<T, NC>(NC / 2);
            const V2<T> xm = cconj(buf[pm]);
            buf[pm] = mk2<T>(2.0f * xm.x, -2.0f * xm.y);
        } else {
            const int pa = tspos<T, NC>(k), pb = tspos<T, NC>(NC - k);
            const V2<T> w = __ldg(wsplit + k);
            const V2<T> za = buf[pa], zb = cconj(buf[pb]);
            const V2<T> e = cadd(za, zb);
            const V2<T> t = cmul(csub(za, zb), w);
            const V2<T> xa = pfma(e, splat((T)0.5), t);
            const V2<T> xb = pfma(e, splat((T)0.5), mk2<T>(-t.x, -t.y));   // conj of X[NC-k]
            const V2<T> e2 = cadd(xa, xb);
            const V2<T> h = cmulc(csub(xa, xb), w);
            buf[pa] = pfma(h, splat((T)2), e2);
            buf[pb] = cconj(pfma(h, splat((T)-2), e2));
        }
    }
}

// ---------------------------------------------------------------- quantizer, one frame, CW warps
template <class T, int NC, int CW>
QD_DEV void quantize_frame_team(V2<T> *buf, T *slotG, V2<T> *slotP, const QuantDev &q, const TeamGather &tg,
                                const V2<T> *wsplit, int lane, int wsub, int team) {
    const int tlane = wsub * 32 + lane;
    for (int s = tlane; s <= q.n_slots; s += 32 * CW) {
        slotG[s] = 0.0f;
        slotP[s] = mk2<T>(0.0f, 0.0f);
    }
    team_sync<CW>(team);
    // Q1: this warp's slots only (see TeamGather)
#pragma unroll 1
    for (int i0 = tg.begin[wsub]; i0 < tg.begin[wsub + 1]; i0 += 32) {
        const uint32_t e = __ldg(tg.src_tab + i0 + lane);
        V2<T> p;
        {   // X[k] straight from the packed spectrum (qd::split_bin with this kernel's positions)
            const int k = (int)(e & 0x1fffu);
            const bool hi = 2 * k > NC;
            const int kk = hi ? NC - k : k;
            const V2<T> za = buf[tspos<T, NC>(kk)];
            const V2<T> zb = cconj(buf[tspos<T, NC>((NC - kk) & (NC - 1))]);
            const V2<T> t = cmul(csub(za, zb), __ldg(wsplit + kk));
            const V2<T> ee = cadd(za, zb);
            p = hi ? cconj(pfma(ee, splat((T)0.5), mk2<T>(-t.x, -t.y))) : pfma(ee, splat((T)0.5), t);
        }
        const T m2 = p.x * p.x + p.y * p.y;
        T g = m2 > QD_TINY2 ? m2 * rsqrt_fast(m2) : 0.0f;
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
    team_sync<CW>(team);
    for (int sl = tlane; sl < q.n_slots; sl += 32 * CW) {
        const T ik = (T)__ldg(q.slot_invk + sl);
        slotG[sl] *= ik;
        slotP[sl] = pmul(slotP[sl], splat(ik));
    }
    team_sync<CW>(team);

    // Q3: rows [ra, rb) of the paired walk belong to this warp
    constexpr int HR = NC / 64;
    static_assert(HR % CW == 0, "rows per warp");
    constexpr int RPW = HR / CW;
    const int ra = wsub * RPW, rb = ra + RPW;
    const bool smooth = q.smoothing != 0;
    const bool is0 = lane == 0, is31 = lane == 31;
    const int lane_m1 = (lane + 31) & 31, lane_p1 = (lane + 1) & 31;
    // X[k], X[NC-k] of row i from the packed spectrum, magnitudes after the quantizer (ml, mh) and phasors
    auto row = [&](int i, T &nl, T &nh, V2<T> &ul, V2<T> &uh, V2<T> &v, int &pa, int &pb) {
        const int k = 32 * i + lane;
        pa = tspos<T, NC>(k);
        pb = k == 0 ? pa : tspos<T, NC>(NC - k);   // Z[NC] = Z[0]
        v = __ldg(wsplit + k);
        const V2<T> za = buf[pa], zb = cconj(buf[pb]);
        const V2<T> e = cadd(za, zb);
        const V2<T> t = cmul(csub(za, zb), v);
        T ml, mh;
        mag_phasor<T>(pfma(e, splat((T)0.5), t), ml, ul);
        mag_phasor<T>(cconj(pfma(e, splat((T)0.5), mk2<T>(-t.x, -t.y))), mh, uh);
        if (i < q.row_limit) quant_apply<T, false>(ml, ul, nl, k, slotG, slotP, q);
        else nl = ml;
        if (NC - 32 * i - 31 < 32 * q.row_limit) quant_apply<T, false>(mh, uh, nh, NC - k, slotG, slotP, q);
        else nh = mh;
    };
    // the rows that border the range, before anybody writes (their phasors are not needed)
    T pre_l = 0.0f, pre_h = 0.0f, post_l = 0.0f, post_h = 0.0f;
    {
        V2<T> u0, u1, v;
        int p0, p1;
        if (ra > 0) row(ra - 1, pre_l, pre_h, u0, u1, v, p0, p1);
        if (rb < HR) row(rb, post_l, post_h, u0, u1, v, p0, p1);
    }
    // the two walks meet at bin NC/2 (lane 0 of the last warp)
    const int pm = tspos<T, NC>(NC / 2);
    T mm = 0.0f;
    V2<T> um = mk2<T>(1.0f, 0.0f);
    if (rb == HR && lane == 0) {
        T m0;
        mag_phasor<T>(cconj(buf[pm]), m0, um);
        if ((NC / 64) < q.row_limit) quant_apply<T, false>(m0, um, mm, NC / 2, slotG, slotP, q);
        else mm = m0;
    }
    team_sync<CW>(team);

    T lp = 0.0f, lc = pre_l, ln = 0.0f, hp = 0.0f, hc = pre_h, hn = 0.0f;
    V2<T> luc = mk2<T>(1.0f, 0.0f), lun = luc, huc = luc, hun = luc, vc = luc, vn = luc;
    int pac = 0, pbc = 0;
    auto emit = [&](bool edge) {   // finishes the pair (luc, huc) at (pac, pbc) with the window (p, c, n)
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
        const V2<T> e2 = cadd(xa, xb);
        const V2<T> h = cmulc(csub(xa, xb), vc);
        buf[pac] = pfma(h, splat((T)2), e2);
        buf[pbc] = cconj(pfma(h, splat((T)-2), e2));
    };
#pragma unroll 1
    for (int i = ra; i < rb; ++i) {
        int pa, pb;
        row(i, ln, hn, lun, hun, vn, pa, pb);
        if (i > ra) emit(i == 1);
        lp = lc; lc = ln; luc = lun;
        hp = hc; hc = hn; huc = hun;
        vc = vn; pac = pa; pbc = pb;
    }
    if (rb < HR) {
        ln = post_l; hn = post_h;
        emit(rb == 1);
    } else {
        ln = mm; hn = mm;
        emit(HR == 1);
        const T left = __shfl_sync(QD_FULL, lc, 31);    // bin NC/2 - 1
        const T right = __shfl_sync(QD_FULL, hc, 31);   // bin NC/2 + 1
        if (lane == 0) {
            const T om = smooth ? 0.5f * mm + 0.25f * (left + right) : mm;
            buf[pm] = mk2<T>(2.0f * om * um.x, -2.0f * om * um.y);
        }
    }
    team_sync<CW>(team);
}

// ---------------------------------------------------------------- the kernel: NF frames per batch, CW warps per frame
template <class T, int NC, int NF, int CW>
__global__ void __launch_bounds__(32 * NF * CW)
spec_pass_team_kernel(const SpecArgsT<T> a, const TeamGather tg) {
    using L = SpecSmem<T, NC, NF, 1, false>;
    using C = FftCfg<T, NC>;
    constexpr int HOP = L::HOP;
    constexpr int HP = HOP / 2;
    constexpr int nthreads = 32 * NF * CW;
    static_assert(CW == 1 || NF <= 15, "one named barrier per team");
    QD_DYN_SMEM(smem);
    const int tid = (int)threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int team = warp / CW, wsub = warp % CW;
    V2<T> *bufs = reinterpret_cast<V2<T> *>(smem + L::off_buf);
    float *stage = reinterpret_cast<float *>(smem + L::off_stage);
    V2<T> *tail = reinterpret_cast<V2<T> *>(smem + L::off_tail);
    V2<T> *buf = bufs + (size_t)team * L::BUF;
    const int slot_cap = (a.q.n_slots + 2) & ~1;
    T *slotG = reinterpret_cast<T *>(smem + L::off_slot) + (size_t)team * slot_cap * 3;
    V2<T> *slotP = reinterpret_cast<V2<T> *>(slotG + slot_cap);

    const ClipLoc cs = clip_loc(a, (int)blockIdx.y);   // one clip per CTA: the early return below is uniform
    const int n = (int)cs.n;
    const float *x = a.x + cs.base;
    float *y = a.y + cs.base;
    float *tap = a.tap ? a.tap + cs.base : nullptr;
    const bool vec2 = ((n & 1) == 0) && ((reinterpret_cast<uintptr_t>(y) & 7) == 0) &&
                      (!tap || (reinterpret_cast<uintptr_t>(tap) & 7) == 0);
    const bool vec4 = (reinterpret_cast<uintptr_t>(x) & 15) == 0;

    const int j_end = 2 + (n + HOP - 1) / HOP;
    const int j0 = 2 + blockIdx.x * a.tile_blocks;
    const int j1 = min(j0 + a.tile_blocks, j_end);
    if (j0 >= j1) return;
    const int t_first = j0 - 3;
    const int n_frames = 1 + n / HOP;

    for (int i = tid; i < 3 * HP; i += nthreads) tail[i] = mk2<T>(0.0f, 0.0f);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + L::off_flags);
    int *consumed = reinterpret_cast<int *>(smem + L::off_flags + 8);
    if (tid == 0) {
        mbar_init(full, 1);
        *consumed = 0;
    }
    uint32_t full_parity = 0;
    bool tma_pending = false;
    constexpr uint32_t STAGE_BYTES = (uint32_t)(L::STAGE * sizeof(float));
    __syncthreads();

    float out_peak = 0.0f;
    for (int tb = t_first; tb < j1; tb += NF) {
        // ---- stage the samples of frames tb .. tb+NF-1 (see spec_pass_kernel)
        const long long s0 = (long long)tb * HOP - NC;
        const long long s0n = s0 + (long long)NF * HOP;
        const bool next_by_tma = vec4 && (tb + NF < j1) && s0n >= 0 && s0n + L::STAGE <= n;
        if (tma_pending) {
            mbar_wait(full, full_parity);
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
            __syncthreads();
        }
        tma_pending = next_by_tma;
        const int t = tb + team;
        const bool live = t >= 0 && t < n_frames;   // uniform over the team
        if (live) {
            const float2 *frame = reinterpret_cast<const float2 *>(stage + team * HOP);
            t_fwd_first<T, NC, C::R1, CW>(buf, frame, a.wtab, a.tw1, lane, wsub, team);
        }
        __syncwarp();   // every lane of this warp has read its samples
        // the last warp of the CTA to leave the staging buffer starts the next bulk copy
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(consumed, 1) == NF * CW - 1) {
                *consumed = 0;
                if (next_by_tma) {
                    mbar_expect_tx(full, STAGE_BYTES);
                    bulk_g2s(stage, x + s0n, STAGE_BYTES, full);
                }
            }
        }
        if (live) {
            team_sync<CW>(team);
            t_fft_forward_rest<T, NC, CW>(buf, a.tw2, lane, wsub, team);
            if (a.quant) {
                quantize_frame_team<T, NC, CW>(buf, slotG, slotP, a.q, tg, a.wsplit, lane, wsub, team);
            } else {
                t_split_merge<T, NC, CW>(buf, a.wsplit, lane, wsub);
                team_sync<CW>(team);
            }
            t_fft_inverse<T, NC, CW>(buf, a.wtab, a.tw1, a.tw2, lane, wsub, team);
        } else {
            for (int i = wsub * 32 + lane; i < L::BUF; i += 32 * CW) buf[i] = mk2<T>(0.0f, 0.0f);
        }
        __syncthreads();
        // ---- overlap-add in frame order (spec_pass_kernel's general hop, rolled)
        for (int c = tid; c < HP; c += nthreads) {
#pragma unroll 1
            for (int h = 0; h < NF + 3; ++h) {
                V2<T> v = (h < 3) ? tail[h * HP + c] : mk2<T>(0.0f, 0.0f);
                const int w0 = h - 3 > 0 ? h - 3 : 0, w1 = h < NF - 1 ? h : NF - 1;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int w = w0 + k;
                    if (w <= w1) v = padd(v, bufs[(size_t)w * L::BUF + tpos<T, NC>((h - w) * HP + c)]);
                }
                if (h >= NF) {
                    tail[(h - NF) * HP + c] = v;
                    continue;
                }
                const int j = tb + h;
                if (j < j0 || j >= j1) continue;
                const long long nidx = (long long)(j - 2) * HOP + 2 * c;
                if (nidx >= n) continue;
                const int sl_a = j - n_frames + 1 > 0 ? j - n_frames + 1 : 0;
                const int sl_b = j < 3 ? j : 3;
                V2<T> inv = mk2<T>(0.0f, 0.0f);
                if (sl_a <= sl_b) inv = __ldg(reinterpret_cast<const V2<T> *>(a.invw + (sl_a * 4 + sl_b) * HOP) + c);
                const V2<T> vi = pmul(v, inv);
                const float2 o = make_float2((float)vi.x, (float)vi.y);
                const float2 r = make_float2(epilogue_apply(o.x, a.epilogue, a.fold, a.bias, a.fold_exact_f32, a.tube_gain, a.tube_norm),
                                             epilogue_apply(o.y, a.epilogue, a.fold, a.bias, a.fold_exact_f32, a.tube_gain, a.tube_norm));
                if (vec2) {
                    if (tap) *reinterpret_cast<float2 *>(tap + nidx) = o;
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
            }
        }
        __syncthreads();
    }
    if (a.clip_peak) {
        out_peak = warp_max(out_peak);
        if (lane == 0) atomicMax(reinterpret_cast<unsigned *>(a.clip_peak) + cs.idx, __float_as_uint(out_peak));
    }
}

}  // namespace qd
