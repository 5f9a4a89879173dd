// qd_peaks.cuh -- strongest STFT bins per frame, the device half of the scale-alignment metric
//
// Replaces the per-frame part of avg_cents_offset_from_scale (dsp/analyses.py:53-142):
//   S = stft_mono(x)  (dsp/stft_utils.py:11-97, same framing as the render)        :90-96
//   per frame: bins in descending |S|, stop below min_db, skip bin 0 (freq <= 0),
//   keep the first topn                                                              :106-135
// The cents offset of a bin depends only on its frequency and the key/scale, so the host keeps a float64
// table cents[bin] (quantumdistortion_b200/analyses.py) and this kernel only has to name the bins.
//
// One warp owns one frame (the FFT passes of qd_spec.cuh); each lane keeps the best K of its bins, then K
// rounds of a warp-wide argmax pop the winners in order.
#pragma once
#include "qd_spec.cuh"

namespace qd {

constexpr int QD_PEAKS_MAX = 8;

template <class T>
struct PeaksArgsT {
    const float *x;       // [batch, n]
    int16_t *bins;        // [batch, n_frames, topn]: bin index, -1 = no (further) bin above the threshold
    int n, n_frames, topn;
    int clip0;            // clip of blockIdx.y == 0 (launch splits advance it, see for_each_launch)
    T min_mag2;           // (10^(min_db/20))^2
    const V2<T> *wtab, *tw1, *tw2, *wsplit;
};

template <class T, int NC>
__global__ void __launch_bounds__(256)
peaks_kernel(const PeaksArgsT<T> a) {
    constexpr int BUF = buf_slots<NC>();
    constexpr int ROWS = (NC + 1 + 31) / 32;
    QD_DYN_SMEM(smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const size_t per_warp = (size_t)BUF * sizeof(V2<T>) + (size_t)2 * NC * sizeof(float);
    V2<T> *buf = reinterpret_cast<V2<T> *>(smem + (size_t)warp * per_warp);
    float *stage = reinterpret_cast<float *>(smem + (size_t)warp * per_warp + (size_t)BUF * sizeof(V2<T>));
    const int clip = a.clip0 + (int)blockIdx.y;
    const int t = blockIdx.x * nw + warp;
    if (t >= a.n_frames) return;
    const float *x = a.x + (size_t)clip * a.n;
    const long long s0 = (long long)t * (NC / 2) - NC;   // centre padding of n_fft/2 (dsp/stft_utils.py:59-62)
    for (int i = lane; i < 2 * NC; i += 32) {
        const long long s = s0 + i;
        stage[i] = (s >= 0 && s < a.n) ? x[s] : 0.0f;
    }
    __syncwarp();
    SpecArgsT<T> sa{};
    sa.tw2 = a.tw2;
    fwd_first<T, NC, FftCfg<T, NC>::R1>(buf, reinterpret_cast<const float2 *>(stage), a.wtab, a.tw1, lane);
    fft_forward<T, NC>(buf, nullptr, sa, a.wtab, a.tw1, a.tw2, lane);
    real_split<T, NC>(buf, a.wsplit, lane);
    // local best-K (descending) of this lane's bins; bin 0 never counts (freq <= 0, dsp/analyses.py:116-118)
    T bv[QD_PEAKS_MAX];
    int bi[QD_PEAKS_MAX];
#pragma unroll
    for (int j = 0; j < QD_PEAKS_MAX; ++j) { bv[j] = (T)-1; bi[j] = -1; }
    for (int row = 0; row < ROWS; ++row) {
        const int k = 32 * row + lane;
        if (k == 0 || k > NC) continue;
        const V2<T> v = buf[rpos<T, NC>(lane, row)];
        T m2 = v.x * v.x + v.y * v.y;
        int idx = k;
        if (!(m2 >= a.min_mag2)) continue;           // below min_db: never selected (:113-114)
#pragma unroll
        for (int j = 0; j < QD_PEAKS_MAX; ++j) {      // insertion into the sorted list (ties: lower bin first)
            if (m2 > bv[j]) {
                const T tv = bv[j]; const int ti = bi[j];
                bv[j] = m2; bi[j] = idx;
                m2 = tv; idx = ti;
            }
        }
    }
    int16_t *out = a.bins + ((size_t)clip * a.n_frames + t) * a.topn;
    for (int r = 0; r < a.topn; ++r) {
        T best = bv[0];
        int bidx = bi[0] >= 0 ? bi[0] : 0x7fffffff;
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            const T ov = __shfl_xor_sync(QD_FULL, best, d);
            const int oi = __shfl_xor_sync(QD_FULL, bidx, d);
            if (ov > best || (ov == best && oi < bidx)) { best = ov; bidx = oi; }
        }
        const bool any = best >= (T)0;
        if (any && bi[0] == bidx) {                  // the winner pops its head
#pragma unroll
            for (int j = 0; j < QD_PEAKS_MAX - 1; ++j) { bv[j] = bv[j + 1]; bi[j] = bi[j + 1]; }
            bv[QD_PEAKS_MAX - 1] = (T)-1; bi[QD_PEAKS_MAX - 1] = -1;
        }
        if (lane == 0) out[r] = any ? (int16_t)bidx : (int16_t)-1;
    }
}

}  // namespace qd
