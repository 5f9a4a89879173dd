// qd_autotune.cuh -- the reference's default mode "autotune_v1" (dsp/autotune.py, dsp/pipeline.py:537-601):
//
//   zero-phase band split (sosfiltfilt x4)  ->  YIN pitch track on the detector band  ->  note-hold state machine
//   ->  per-sample ratio track  ->  granular two-tap pitch shifter  ->  envelope-followed sub oscillator  ->  mix
//
// Where the reference is a per-sample Python loop, the kernels keep its operation order and precision (explicit
// round-to-nearest intrinsics where an FMA would change a float32 result; NumPy's NEP-50 scalar typing followed operation
// by operation).  The IIR sweeps are blocked affine scans in float64, YIN's difference function is one running float64
// prefix per lag shared by all frames, the shifter read-out, oscillator and mix run wide; only the delay-tap accumulation,
// the envelope follower and the note-hold state machine stay sequential per clip (one lane, warp-staged tiles).
// The detector is float64 like the reference because the shifter integrates 1 - ratio: the pitch has to match to ~1e-9
// for the output to stay inside the 1e-4 parity bound.
#pragma once
#include <type_traits>

#include "qd_spec.cuh"
#include "qd_spec_team.cuh"
#include "qd_time.cuh"
#include "qd_yin.cuh"

namespace qd {

struct AtFilter {         // one zero-phase 4th-order Butterworth (two second-order sections), dsp/autotune.py:88-100
    int on;               // 0: cutoff <= 0 -> identity (astype float32)
    double sos[2][6];
    double zi[2][2];      // scipy.signal.sosfilt_zi
};

constexpr int AT_EDGE = 15;   // sosfiltfilt default padlen = 3 * ntaps, ntaps = 5

// ---------------------------------------------------------------- zero-phase filter
// scipy.signal.sosfiltfilt(sos, x_float32).astype(float32): odd extension by 15 samples formed in float32, forward sweep
// from the state zi * ext[0], backward sweep from zi * y[-1], float64 in between (oracle/qd_autotune.py
// sosfiltfilt_restated).  `scratch` holds the forward result: [jobs][batch][n + 30] doubles.
struct AtFiltArgs {
    const float *x[2];    // input per job, packed like the batch
    float *y[2];          // output per job
    AtFilter f[2];
    int jobs;
    double *scratch;      // clip i of job j at j * scratch_job + base_i + 2 AT_EDGE i (uniform: [job][batch][n + 30])
    long long scratch_job;
    long long n;
    const int64_t *starts;
    const int32_t *lengths;
    int clip0;
};

// tile / CTA shape of the warp-staged sequential kernels below (delay taps, envelope follower): all lanes move a tile of
// AT_TS samples (coalesced), lane 0 runs the dependent chain over it out of shared memory
constexpr int AT_TS = 512;    // samples per tile
constexpr int AT_FW = 4;      // warps per CTA

// Zero-phase filter, segment-parallel like the crossover (qd_time.cuh): one thread filters one tile of one (clip, job)
// sequentially in float64 -- the two DF2T sections in scipy's recurrence -- after a warm-up of `halo` samples
// from a zero state.  The poles of these Butterworth designs have radius r < 1, so after halo = 44 / (1 - r) samples the
// zero-started state equals the true one to below 1e-15 (the host derives halo per filter from its poles: 160 samples
// at 5 kHz, about 12 000 at the detector's 71.5 Hz high-pass); the first tile starts from scipy's exact initial state
// zi * x_ext[0] instead.  Two launches per filter bank: the forward sweep over the odd-extended input writes float64 into
// `scratch`, the backward sweep reads it reversed and writes float32.  A warp stages 32 samples of its 32 tiles through
// shared memory (coalesced rows both ways); no scan, no block barrier.  41 -> ~10 ms per 1024 clips for the four filters.
struct AtFiltSegArgs {
    AtFiltArgs base;
    int tile[2], halo[2];   // per job, multiples of 32, tile >= 2 * halo; the tile before at_filt_tile
};

constexpr int AT_SW = 4;    // warps per CTA

// A low cutoff has a long warm-up and few tiles per clip: while a clip of m extended samples does not fill one warp,
// halve the tile (down to the warm-up length): twice the threads and a shorter dependent chain per thread.  Chosen per
// clip, because the warm-up start points depend on the tile: a clip gets the tile (and the rounding) it gets alone.
__host__ __device__ inline int at_filt_tile(int tile, int halo, long long m) {
    while (tile / 2 >= (halo > 4096 ? halo : 4096) && (m + tile - 1) / tile < 32) tile /= 2;
    return tile;
}

template <bool BWD>
__global__ void __launch_bounds__(32 * AT_SW) at_filt_seg_kernel(const AtFiltSegArgs q) {
    const AtFiltArgs &a = q.base;
    __shared__ double s_row[AT_SW][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int job = blockIdx.z;
    const ClipLoc c = clip_loc(a, blockIdx.y);
    const long long n = c.n;
    if (n <= AT_EDGE) return;   // not rendered: the odd extension needs more than AT_EDGE samples
    const float *__restrict__ x = a.x[job] + c.base;
    float *__restrict__ y = a.y[job] + c.base;
    const AtFilter &f = a.f[job];
    if (!f.on) {   // identity (astype float32): copied once, by the forward launch
        if (!BWD)
            for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) y[i] = x[i];
        return;
    }
    const long long m = n + 2 * AT_EDGE;
    double *__restrict__ s = a.scratch + job * a.scratch_job + c.base + 2LL * AT_EDGE * c.idx;
    const int halo = q.halo[job], tile = at_filt_tile(q.tile[job], halo, m);
    const long long n_tiles = (m + tile - 1) / tile;
    const long long tile0 = ((long long)blockIdx.x * AT_SW + warp) * 32;
    if (tile0 >= n_tiles) return;
    const int rows = (int)(n_tiles - tile0 < 32 ? n_tiles - tile0 : 32);
    // position p runs in processing order: forward p = index into the extended sequence, backward p <-> index m - 1 - p.
    // The forward input is the odd extension by AT_EDGE samples, formed in float32 like scipy does for a float32 input.
    const float x_first = BWD ? 0.0f : x[0], x_last = BWD ? 0.0f : x[n - 1];
    using Raw = typename std::conditional<BWD, double, float>::type;   // what a fetch leaves in registers
    double (*row)[33] = s_row[warp];
    const long long p_first = tile0 * tile - halo;          // row 0, step 0, column 0
    const long long p_own = p_first + (long long)lane * tile;
    double st[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    const int steps = (halo + tile) / 32;
    // A fetch only LOADS (32 independent loads, raw values and two edge masks kept in registers); whatever consumes the
    // values -- the float32 edge arithmetic, the conversion to float64 -- happens one step later, when the rows go to
    // shared memory.  Consuming them inside the fetch made every step wait for DRAM (forward sweep: 26 -> 6 ms).
    Raw nxt[32];
    unsigned m_ok = 0u, m_left = 0u, m_right = 0u;         // bit r: row r holds a sample / a left- / right-edge sample
    bool nxt_plain = false;                                // the fetched step lies wholly inside the clip: no masks needed
    // A step is "plain" when all 32 rows of the warp exist and every position of the step lies in [lo, hi): then a row is
    // one pointer plus r * tile, and the bookkeeping below (64-bit positions, edge masks, selects: three quarters of the
    // kernel's instructions before this path existed) is skipped.  Forward loads and backward stores need the interior of
    // the odd extension, backward loads and forward stores only the extended range itself.
    const bool full = rows == 32;
    auto plain = [&](int j, long long lo, long long hi) {
        const long long p0 = p_first + 32LL * j;
        return full && p0 >= lo && p0 + 31LL * tile + 31 < hi;
    };
    auto fetch = [&](int j) {
        nxt_plain = BWD ? plain(j, 0, m) : plain(j, AT_EDGE, n + AT_EDGE);
        if (nxt_plain) {
            const long long p = p_first + 32LL * j + lane;
            if (BWD) {
                const double *src = s + (m - 1 - p);
#pragma unroll
                for (int r = 0; r < 32; ++r) nxt[r] = (Raw)src[-(long long)r * tile];
            } else {
                const float *src = x + (p - AT_EDGE);
#pragma unroll
                for (int r = 0; r < 32; ++r) nxt[r] = (Raw)src[(long long)r * tile];
            }
            return;
        }
        m_ok = 0u; m_left = 0u; m_right = 0u;
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const long long p = p_first + (long long)r * tile + 32LL * j + lane;
            const bool ok = r < rows && p >= 0 && p < m;
            m_ok |= (unsigned)ok << r;
            if (BWD) {
                nxt[r] = (Raw)s[ok ? m - 1 - p : 0];         // always a valid address: nothing here waits for the load
            } else {
                const bool left = ok && p < AT_EDGE, right = ok && p >= n + AT_EDGE;
                const long long idx = !ok ? 0 : left ? AT_EDGE - p : right ? 2 * n + AT_EDGE - 2 - p : p - AT_EDGE;
                nxt[r] = (Raw)x[idx];
                m_left |= (unsigned)left << r;
                m_right |= (unsigned)right << r;
            }
        }
    };
    if (tile0 + lane == 0) {                                // the very first tile starts from scipy's steady state
        double v0;
        if (BWD) v0 = s[m - 1];
        else v0 = (double)__fsub_rn(__fmul_rn(2.0f, x_first), x[AT_EDGE]);   // x_ext[0]
        st[0][0] = f.zi[0][0] * v0; st[0][1] = f.zi[0][1] * v0;
        st[1][0] = f.zi[1][0] * v0; st[1][1] = f.zi[1][1] * v0;
    }
    fetch(0);
    for (int j = 0; j < steps; ++j) {
        if (nxt_plain) {
#pragma unroll
            for (int r = 0; r < 32; ++r) row[r][lane] = (double)nxt[r];
        } else {
#pragma unroll
            for (int r = 0; r < 32; ++r) {
                const bool ok = (m_ok >> r) & 1u;
                if (BWD) {
                    row[r][lane] = ok ? (double)nxt[r] : 0.0;
                } else {   // odd extension in float32: 2 x[0] - x[AT_EDGE - p] on the left, 2 x[n-1] - x[mirror] on the right
                    const float v = (float)nxt[r];
                    const bool l = (m_left >> r) & 1u, rt = (m_right >> r) & 1u;
                    row[r][lane] = !ok ? 0.0 : (double)((l || rt) ? __fsub_rn(__fmul_rn(2.0f, l ? x_first : x_last), v) : v);
                }
            }
        }
        __syncwarp();
        if (j + 1 < steps) fetch(j + 1);
        const long long p_step = p_own + 32LL * j;          // steps are 32-aligned: a step lies wholly before or after p = 0
        if (lane < rows && p_step >= 0) {
#pragma unroll 4
            for (int k = 0; k < 32; ++k) {
                double v = row[lane][k];
#pragma unroll
                for (int sec = 0; sec < 2; ++sec) {
                    const double *co = f.sos[sec];
                    const double o = co[0] * v + st[sec][0];
                    st[sec][0] = co[1] * v - co[4] * o + st[sec][1];
                    st[sec][1] = co[2] * v - co[5] * o;
                    v = o;
                }
                row[lane][k] = v;
            }
        }
        __syncwarp();
        if (32 * j >= halo) {
            if (BWD ? plain(j, AT_EDGE, n + AT_EDGE) : plain(j, 0, m)) {
                const long long p = p_first + 32LL * j + lane;
                if (!BWD) {
                    double *dst = s + p;
#pragma unroll
                    for (int r = 0; r < 32; ++r) dst[(long long)r * tile] = row[r][lane];
                } else {
                    float *dst = y + (m - 1 - p - AT_EDGE);
#pragma unroll
                    for (int r = 0; r < 32; ++r) dst[-(long long)r * tile] = (float)row[r][lane];
                }
            } else {
#pragma unroll 8
                for (int r = 0; r < rows; ++r) {
                    const long long p = p_first + (long long)r * tile + 32LL * j + lane;
                    if (p < m) {
                        if (!BWD) {
                            s[p] = row[r][lane];
                        } else {
                            const long long i = m - 1 - p;
                            if (i >= AT_EDGE && i < n + AT_EDGE) y[i - AT_EDGE] = (float)row[r][lane];
                        }
                    }
                }
            }
        }
        __syncwarp();
    }
}

// body = (audio - sub - air) in float32 (dsp/autotune.py:112)
__global__ void at_body_kernel(const float *__restrict__ x, const float *__restrict__ sub, const float *__restrict__ air,
                               float *__restrict__ body, long long count) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        body[i] = __fsub_rn(__fsub_rn(x[i], sub[i]), air[i]);
}

// ---------------------------------------------------------------- detector (dsp/autotune.py:217-236)
// rms and spectral flatness (symmetric Hann, float32 warp FFT) per frame here, YIN (float64) by the sliding kernels below.
struct AtDetArgs {
    const float *det;        // detector side chain, packed like the batch
    double *feat;            // [frame rows, 4] (at_row0): rms, flatness, pitch, confidence
    long long n;
    const int64_t *starts;
    const int32_t *lengths;
    int clip0, batch;
    int frame_size, hop;
    int min_tau, max_tau;
    double sr, min_freq, max_freq, threshold;
    const float *hann;       // [frame_size] np.hanning (symmetric), float32
    const float2 *tw1, *tw2, *wsplit;   // float32 FFT tables of n_fft = frame_size
};

// rms, spectral flatness and the silence flag with one WARP per frame:
// the lanes load the frame once, accumulate the sums and write the Hann-windowed samples straight into the warp's FFT
// buffer.  feat = (rms, flatness, 1 or 0 for "not silent", 0).
constexpr int AT_SW_STATS = 12;   // frames (warps) per CTA: 12 x 16.9 KB of FFT buffers = 203 KB, one CTA per SM
template <int NC>
__global__ void __launch_bounds__(32 * AT_SW_STATS) at_frame_stats_kernel(const AtDetArgs a, long long total_frames) {
    constexpr int FS = 2 * NC;
    constexpr int BUF = buf_slots<NC>();
    QD_DYN_SMEM(smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long fr = (long long)blockIdx.x * AT_SW_STATS + warp;
    if (fr >= total_frames) return;
    float2 *buf = reinterpret_cast<float2 *>(smem) + (size_t)warp * BUF;
    // the clip that owns frame row fr: uniform rows are clip-major; a ragged batch searches its row starts (at_row0)
    int ci;
    if (a.starts) {
        int lo = 0, hi = a.batch - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if ((long long)(a.starts[mid] - a.starts[0]) / a.hop + mid <= fr) lo = mid; else hi = mid - 1;
        }
        ci = lo;
    } else {
        ci = (int)(fr / at_rows(a.n, a.hop));
    }
    const ClipLoc c = clip_loc(a, ci);
    const long long frame = fr - at_row0(a.starts != nullptr, c, a.n, a.hop);
    if (frame >= at_rows(c.n, a.hop)) return;            // a row between two clips
    const long long n = c.n;
    const float *x = a.det + c.base;
    const long long start = frame * a.hop;
    float sq = 0.0f, mx = 0.0f;
    for (int j = lane; j < NC; j += 32) {
        const long long s0 = start + 2 * j;
        const float v0 = s0 < n ? x[s0] : 0.0f, v1 = s0 + 1 < n ? x[s0 + 1] : 0.0f;
        sq += v0 * v0 + v1 * v1;
        mx = fmaxf(mx, fmaxf(fabsf(v0), fabsf(v1)));
        buf[tpos<float, NC>(j)] = make_float2(v0 * a.hann[2 * j], v1 * a.hann[2 * j + 1]);
    }
    sq = warp_sum(sq);
    mx = warp_max(mx);
    __syncwarp();
    // the three-pass FFT on the swizzled buffer layout of qd_spec_team.cuh (one warp per frame: CW = 1); on the padded
    // layout this kernel was bound by shared-memory bank conflicts (LSU data pipe 82 %)
    t_fwd_first_buf<float, NC, FftCfg<float, NC>::R1, 1>(buf, a.tw1, lane, 0);
    __syncwarp();
    t_fft_forward_rest<float, NC, 1>(buf, a.tw2, lane, 0, 0);
    // |X| + 1e-8 and its logarithm with the fast float32 units (rsqrt, lg2: ~1e-6 relative, like the float32 FFT that
    // produced X; the flatness is only compared with a threshold); a lane adds its bins in float32, the lanes'
    // partial sums are added in float64.  X[k] and X[NC-k] come out of the packed spectrum pair by pair (real split).
    float lgf = 0.0f, arf = 0.0f;
    auto add_bin = [&](float re, float im) {
        const float p2 = fmaf(re, re, im * im);
        const float m = (p2 > 0.0f ? p2 * rsqrtf(p2) : 0.0f) + 1e-8f;
        lgf += __log2f(m);
        arf += m;
    };
#pragma unroll 2
    for (int row = 0; row < NC / 64; ++row) {
        const int k = 32 * row + lane;
        if (k == 0) {
            const float2 z0 = buf[0];
            add_bin(z0.x + z0.y, 0.0f);                                   // DC
            add_bin(z0.x - z0.y, 0.0f);                                   // Nyquist
            const float2 zm = buf[tspos<float, NC>(NC / 2)];
            add_bin(zm.x, zm.y);                                          // |X[NC/2]| = |conj Z[NC/2]|
        } else {
            const float2 za = buf[tspos<float, NC>(k)], zb = cconj(buf[tspos<float, NC>(NC - k)]);
            const float2 e = cadd(za, zb);
            const float2 t = cmul(csub(za, zb), __ldg(a.wsplit + k));
            const float2 xa = pfma(e, splat(0.5f), t), xb = pfma(e, splat(0.5f), make_float2(-t.x, -t.y));
            add_bin(xa.x, xa.y);
            add_bin(xb.x, xb.y);
        }
    }
    const double lg = warp_sum((double)lgf) * 0.693147180559945309417, ar = warp_sum((double)arf);
    if (lane == 0) {
        const double geo = exp(lg / (double)(NC + 1)), ari = ar / (double)(NC + 1);
        double *o = a.feat + (size_t)fr * 4;
        o[0] = (double)sqrtf(sq / (float)FS);
        o[1] = ari <= 1e-8 ? 1.0 : geo / ari;
        o[2] = (!((double)mx < 1e-6) && a.max_tau > a.min_tau) ? 1.0 : 0.0;
        o[3] = 0.0;
    }
}

// ---------------------------------------------------------------- YIN: the difference function lives in qd_yin.cuh

// cumulative-mean normalisation and pick (dsp/autotune.py:162-197), one warp per frame
__global__ void __launch_bounds__(256) at_yin_pick_kernel(const AtYinArgs a) {
    QD_DYN_SMEM(smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long fr = (long long)blockIdx.x * 8 + warp;        // frame index over the whole batch
    if (fr >= a.total_frames) return;
    double *cm = reinterpret_cast<double *>(smem) + (size_t)warp * a.stride;
    double *ft = a.feat + (size_t)fr * 4;
    const double *d = a.diff + (size_t)fr * a.stride;
    // running sum over tau by warp scans of 32 lags
    double run = 0.0;
    for (int t0 = 1; t0 <= a.max_tau; t0 += 32) {
        const int t = t0 + lane;
        const double v = t <= a.max_tau ? d[t] : 0.0;
        double inc = v;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const double o = __shfl_up_sync(QD_FULL, inc, sft);
            if (lane >= sft) inc += o;
        }
        const double rs = run + inc;                               // running_sum including lag t
        if (t <= a.max_tau) cm[t] = rs > 0.0 ? v * (double)t / rs : 1.0;
        run += __shfl_sync(QD_FULL, inc, 31);
    }
    __syncwarp();
    // the first lag below the threshold: 32 lags per step, the lowest set bit of the ballot
    int first = -1;
    const bool wanted = ft[2] != 0.0 && a.max_tau > a.min_tau;
    if (wanted) {
        for (int t0 = a.min_tau; t0 <= a.max_tau && first < 0; t0 += 32) {
            const int t = t0 + lane;
            const unsigned hit = __ballot_sync(QD_FULL, t <= a.max_tau && cm[t] < a.threshold);
            if (hit) first = t0 + __ffs(hit) - 1;
        }
    }
    if (lane == 0) {
        double pitch = 0.0, conf = 0.0;
        if (wanted) {
            int est = -1;
            if (first >= 0) {
                int t = first;
                while (t + 1 <= a.max_tau && cm[t + 1] < cm[t]) ++t;
                est = t;
            }
            if (est >= 0) {
                double better = (double)est;
                if (a.min_tau < est && est < a.max_tau) {
                    const double s0 = cm[est - 1], s1 = cm[est], s2 = cm[est + 1];
                    const double den = 2.0 * (s0 - 2.0 * s1 + s2);
                    if (fabs(den) > 1e-12) better = (double)est + (s0 - s2) / den;
                }
                const double p = better > 0.0 ? a.sr / better : 0.0;
                if (!(p < a.min_freq || p > a.max_freq)) {
                    pitch = p;
                    conf = fmin(fmax(1.0 - cm[est], 0.0), 1.0);
                }
            }
        }
        ft[2] = pitch;
        ft[3] = conf;
    }
}

// ---------------------------------------------------------------- note-hold state machine, one thread per clip
struct AtHoldArgs {
    const double *feat;      // [frame rows, 4]
    double *ratio;           // [frame rows]
    long long n, total_frames;   // total_frames: frame rows of the batch
    const int64_t *starts;
    const int32_t *lengths;
    int clip0, batch, hop;
    int root_pc, n_intervals;
    int intervals[8];
    double strength, rms_thr, flat_thr, conf_thr, change_cents;
    int confirm_frames, release_frames;
};

QD_DEV double at_pymod(double v, double w) {   // Python's float %, w > 0
    double m = fmod(v, w);
    if (m != 0.0 && m < 0.0) m += w;
    return m;
}

QD_DEV double at_nearest_scale_freq(double freq, const AtHoldArgs &a) {   // dsp/autotune.py:65-85
    if (freq <= 0.0) return freq;
    const double midi = 69.0 + 12.0 * log2(freq / 440.0);
    const double in_oct = at_pymod(at_pymod(midi - (double)a.root_pc, 12.0) + 12.0, 12.0);
    const double base = midi - in_oct;
    double best = rint(midi), best_d = INFINITY;
    for (int o = -1; o <= 1; ++o)
        for (int k = 0; k < a.n_intervals; ++k) {
            const double cand = base + (double)a.intervals[k] + (double)o * 12.0;
            const double d = fabs(midi - cand);
            if (d < best_d) { best_d = d; best = cand; }
        }
    return 440.0 * exp2((best - 69.0) / 12.0);
}

// The target note of a voiced frame depends on that frame alone: one thread per frame leaves it in ratio[] (0 = unvoiced),
// so the sequential kernel below only runs the state machine.
__global__ void at_target_kernel(const AtHoldArgs a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.total_frames) return;                     // (rows between the clips of a ragged batch are never read)
    const double *f = a.feat + (size_t)i * 4;
    const double rms = f[0], flat = f[1], p = f[2], conf = f[3];
    const bool voiced = p > 0.0 && rms >= a.rms_thr && flat <= a.flat_thr && conf >= a.conf_thr;
    a.ratio[i] = voiced ? at_nearest_scale_freq(p, a) : 0.0;
}

// note-hold state machine (dsp/autotune.py:236-285), one thread per clip; ratio[] holds the targets on entry
__global__ void at_hold_kernel(const AtHoldArgs a) {
    const int clip = blockIdx.x * blockDim.x + threadIdx.x;
    if (clip >= a.batch) return;
    const ClipLoc c = clip_loc(a, clip);
    const int frames = (int)at_rows(c.n, a.hop);
    if (frames == 0) return;
    const long long r0 = at_row0(a.starts != nullptr, c, a.n, a.hop);
    const double *f = a.feat + r0 * 4;
    double *out = a.ratio + r0;
    double held = 0.0, cand = 0.0, last = 1.0;
    int cand_n = 0, rel = a.release_frames + 1;
    double tgt_n = out[0], p_n = f[2];                   // the next frame's inputs are loaded one step ahead
    for (int i = 0; i < frames; ++i) {
        const double tgt = tgt_n, p = p_n;
        if (i + 1 < frames) { tgt_n = out[i + 1]; p_n = f[4 * (i + 1) + 2]; }
        const bool voiced = tgt > 0.0;                   // the target of a voiced frame is a positive frequency
        double r;
        if (voiced) {
            if (held <= 0.0) {
                held = tgt; cand = 0.0; cand_n = 0;
            } else {
                const double dc = fabs(1200.0 * log2(fmax(tgt, 1e-6) / fmax(held, 1e-6)));
                if (dc >= a.change_cents) {
                    const double cd = cand > 0.0 ? fabs(1200.0 * log2(fmax(tgt, 1e-6) / fmax(cand, 1e-6))) : INFINITY;
                    if (cand > 0.0 && cd < 20.0) ++cand_n;
                    else { cand = tgt; cand_n = 1; }
                    if (cand_n >= a.confirm_frames) { held = cand; cand = 0.0; cand_n = 0; }
                } else {
                    cand = 0.0; cand_n = 0;
                }
            }
            r = fmin(fmax(1.0 + a.strength * ((held / p) - 1.0), 0.5), 2.0);
            rel = 0;
            last = r;
        } else {
            ++rel;
            if (held > 0.0 && rel <= a.release_frames) {
                r = last;
            } else {
                held = 0.0; cand = 0.0; cand_n = 0;
                r = 1.0; last = 1.0;
            }
        }
        out[i] = r;
    }
}

// np.interp(arange(n), centers, ratio) as float32 (dsp/autotune.py:293-294): centers[k] = min(n-1, k*hop + fs/2)
QD_DEV float at_ratio_at(const double *ratio, int frames, long long n, int hop, int half, long long s) {
    const double x = (double)s;
    auto cen = [&](int k) -> double { const long long c = (long long)k * hop + half; return (double)(c < n - 1 ? c : n - 1); };
    if (x < cen(0)) return (float)ratio[0];
    if (x > cen(frames - 1)) return (float)ratio[frames - 1];
    // largest j with centers[j] <= x (duplicates at the end resolve to the last one)
    long long j = (s - half) / hop;
    if (j < 0) j = 0;
    if (j > frames - 1) j = frames - 1;
    while (j + 1 <= frames - 1 && cen((int)j + 1) <= x) ++j;
    while (j > 0 && cen((int)j) > x) --j;
    if (j == frames - 1) return (float)ratio[j];
    const double x0 = cen((int)j), x1 = cen((int)j + 1);
    if (x0 == x) return (float)ratio[j];
    const double slope = (ratio[j + 1] - ratio[j]) / (x1 - x0);
    return (float)__dadd_rn(__dmul_rn(slope, x - x0), ratio[j]);   // NumPy: multiply, then add
}

// ---------------------------------------------------------------- granular shifter
// Pass 1 (one thread per clip): the two delay taps, exactly the reference's sequential float64 accumulation with wraps
// (dsp/autotune.py:327-337), plus the np.allclose(ratio, 1, atol=1e-3) early-out flag.  Pass 2 (wide): read-out.
struct AtShiftArgs {
    const float *body;       // packed like the batch
    const double *ratio;     // [frame rows]
    long long *tile_sum;     // [tile rows] (at_row0, unit AT_TS) slope sums per tile, then the tap at every tile start
    float *ratio_track;      // optional, packed like the batch
    int *flat_flag;          // [batch] 1: ratio track allclose to 1 -> output = body
    float *out;              // corrected body, packed like the batch
    long long n;
    const int64_t *starts;
    const int32_t *lengths;
    int clip0, hop, half;
    int max_delay, buf_size;
};

// the np.interp segment that contains sample s: r(i) = (i == x0) ? y0 : slope * (i - x0) + y0 for every i of the segment
struct AtSeg { double x0, y0, slope; };
QD_DEV AtSeg at_segment_at(const double *ratio, int frames, long long n, int hop, int half, long long s) {
    const double x = (double)s;
    auto cen = [&](int k) -> double { const long long c = (long long)k * hop + half; return (double)(c < n - 1 ? c : n - 1); };
    if (x < cen(0)) return AtSeg{-1.0, ratio[0], 0.0};
    long long j = (s - half) / hop;
    if (j < 0) j = 0;
    if (j > frames - 1) j = frames - 1;
    while (j + 1 <= frames - 1 && cen((int)j + 1) <= x) ++j;
    while (j > 0 && cen((int)j) > x) --j;
    if (j == frames - 1) return AtSeg{cen((int)j), ratio[j], 0.0};
    const double x0 = cen((int)j), x1 = cen((int)j + 1);
    return AtSeg{x0, ratio[j], (ratio[j + 1] - ratio[j]) / (x1 - x0)};
}

// The tap accumulation is exact integer arithmetic in disguise: the per-sample slope 1 - ratio (ratio a float32 in
// [0.5, 2]) is a multiple of 2^-24 with |slope| <= 1, the taps start at multiples of 2^-24 and stay below max_delay, so
// every float64 addition and every wrap of the reference's loop (dsp/autotune.py:327-337) is exact.  In units of 2^-24 the
// taps are T_n = (T_0 + sum_{k<=n} S_k) mod M -- an int64 prefix sum, associative and bit-exact, so it runs as a scan in
// three launches, and the taps themselves never go to memory:
//   at_tap_sums_kernel  one warp per 512-sample tile: the tile's sum of slopes (and whether its ratio track is flat)
//   at_tap_scan_kernel  one warp per clip: exclusive scan of the tile sums (mod M) = the tap at every tile start
//   at_shift_kernel     one warp per tile: slopes again, warp scan + tile start = the taps of its samples, then the read-out
constexpr int AT_SPL = AT_TS / 32;   // samples per lane and tile
constexpr int AT_TW = 8;             // tiles (warps) per CTA

// the ratio track at sample i (np.interp of the per-frame ratios, float32) and its slope 1 - ratio in units of 2^-24
struct AtTileCtx {
    AtSeg sg;                // the np.interp segment of the whole tile (aligned tiles only)
    bool aligned;
    double r_last;
    long long n;             // the clip's samples and frames
    int frames;
};
QD_DEV long long at_slope(const AtShiftArgs &a, const double *__restrict__ ratio, const AtTileCtx &c, long long i, float *r_out) {
    float r;
    if (!c.aligned) r = at_ratio_at(ratio, c.frames, c.n, a.hop, a.half, i);
    else if (i == c.n - 1) r = (float)c.r_last;                 // the last sample sits on the (repeated) last centre
    else if ((double)i == c.sg.x0) r = (float)c.sg.y0;
    else r = (float)__dadd_rn(__dmul_rn(c.sg.slope, (double)i - c.sg.x0), c.sg.y0);
    *r_out = r;
    return (long long)((1.0 - (double)fminf(fmaxf(r, 0.5f), 2.0f)) * (double)(1ll << 24));   // exact: a multiple of 2^-24
}
QD_DEV AtTileCtx at_tile_ctx(const AtShiftArgs &a, const double *__restrict__ ratio, long long n, long long i0) {
    const int frames = (int)at_rows(n, a.hop);
    AtTileCtx c{AtSeg{0.0, 1.0, 0.0}, false, ratio[frames - 1], n, frames};
    c.aligned = (a.hop % AT_TS) == 0 && (a.half % AT_TS) == 0 && (a.max_delay % 4) == 0;
    if (c.aligned) c.sg = at_segment_at(ratio, frames, n, a.hop, a.half, i0);
    return c;
}

// (a tile holds no frame centre strictly inside when hop and frame_size / 2 are multiples of the tile: 512 | 512, 2048)
__global__ void __launch_bounds__(32 * AT_TW) at_tap_sums_kernel(const AtShiftArgs a) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ClipLoc c = clip_loc(a, blockIdx.y);
    const long long tile = (long long)blockIdx.x * AT_TW + warp;
    if (tile >= at_rows(c.n, AT_TS)) return;
    const bool rg = a.starts != nullptr;
    const double *__restrict__ ratio = a.ratio + at_row0(rg, c, a.n, a.hop);
    float *__restrict__ rt = a.ratio_track ? a.ratio_track + c.base : nullptr;
    const AtTileCtx cx = at_tile_ctx(a, ratio, c.n, tile * AT_TS);
    bool flat = true;
    long long run = 0;
#pragma unroll 4
    for (int k = 0; k < AT_SPL; ++k) {
        const long long i = tile * AT_TS + (long long)lane * AT_SPL + k;
        if (i < c.n) {
            float r;
            run += at_slope(a, ratio, cx, i, &r);
            if (rt) rt[i] = r;
            if (!(fabs((double)r - 1.0) <= 1e-3 + 1e-5)) flat = false;   // np.allclose(r, 1.0, atol=1e-3)
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) run += __shfl_xor_sync(QD_FULL, run, d);
    flat = __all_sync(QD_FULL, flat);
    if (lane == 0) {
        a.tile_sum[at_row0(rg, c, a.n, AT_TS) + tile] = run;
        if (!flat) a.flat_flag[c.idx] = 1;               // zeroed before the launch: "some tile is not flat" until the scan
    }
}

// tile_sum -> tap 0 at the start of every tile (in [0, M)); flat_flag -> 1 when no tile of the clip raised it
__global__ void __launch_bounds__(32) at_tap_scan_kernel(const AtShiftArgs a) {
    const int lane = threadIdx.x;
    const ClipLoc c = clip_loc(a, blockIdx.x);
    const long long tiles = at_rows(c.n, AT_TS);
    long long *ts = a.tile_sum + at_row0(a.starts != nullptr, c, a.n, AT_TS);
    const long long M = (long long)a.max_delay << 24;
    long long carry = M / 4;                             // tap 0 starts at 0.25 * max_delay
    for (long long t0 = 0; t0 < tiles; t0 += 32) {
        const long long t = t0 + lane;
        const long long v = t < tiles ? ts[t] : 0;
        long long inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long o = __shfl_up_sync(QD_FULL, inc, d);
            if (lane >= d) inc += o;
        }
        long long start = carry + (inc - v);             // 32 tiles move a tap by at most 2^38 units: a few wraps
        while (start < 0) start += M;
        while (start >= M) start -= M;
        if (t < tiles) ts[t] = start;
        carry += __shfl_sync(QD_FULL, inc, 31);
        while (carry < 0) carry += M;
        while (carry >= M) carry -= M;
    }
    if (lane == 0) a.flat_flag[c.idx] = a.flat_flag[c.idx] ? 0 : 1;   // from "some tile is not flat" to "the clip is flat"
}

// read-out with the latency trim folded in: out = raw[lat:] ++ zeros(lat) unless the early-out copied the body
// (dsp/autotune.py:339-358); sample i of the shifter lands at out[i - lat].  A lane computes its 16 consecutive samples and
// the warp writes the tile through shared memory (stride 17: no bank conflicts either way) in coalesced rows.
__global__ void __launch_bounds__(32 * AT_TW) at_shift_kernel(const AtShiftArgs a) {
    __shared__ float s_out[AT_TW][AT_TS + AT_TS / 16];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ClipLoc c = clip_loc(a, blockIdx.y);
    const long long n = c.n;
    const long long tile = (long long)blockIdx.x * AT_TW + warp;
    if (tile >= at_rows(n, AT_TS)) return;
    const long long i0 = tile * AT_TS;
    const float *__restrict__ x = a.body + c.base;
    float *__restrict__ out = a.out + c.base;
    if (a.flat_flag[c.idx] != 0) {
        for (long long i = i0 + lane; i < i0 + AT_TS && i < n; i += 32) out[i] = x[i];
        return;
    }
    const long long lat = n > a.max_delay / 2 ? a.max_delay / 2 : 0;
    const bool rg = a.starts != nullptr;
    const double *__restrict__ ratio = a.ratio + at_row0(rg, c, a.n, a.hop);
    const long long unit = 1ll << 24;
    const long long M = (long long)a.max_delay * unit, half_m = M / 2;   // the second tap runs half a grain behind
    const AtTileCtx cx = at_tile_ctx(a, ratio, n, i0);
    long long run = 0;                                   // the lane's 16 slopes: summed here, walked again below
#pragma unroll 4
    for (int k = 0; k < AT_SPL; ++k) {
        const long long i = i0 + (long long)lane * AT_SPL + k;
        float r;
        if (i < n) run += at_slope(a, ratio, cx, i, &r);
    }
    long long incl = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long o = __shfl_up_sync(QD_FULL, incl, d);
        if (lane >= d) incl += o;
    }
    long long tap = a.tile_sum[at_row0(rg, c, a.n, AT_TS) + tile] + (incl - run);   // tap 0 before the lane's first sample, unwrapped
    const double md = (double)a.max_delay, size = (double)a.buf_size;
    const int mask = a.buf_size - 1;
    float *so = s_out[warp];
#pragma unroll 1
    for (int k = 0; k < AT_SPL; ++k) {
        const long long i = i0 + (long long)lane * AT_SPL + k;
        float val = 0.0f;
        if (i < n) {
            float r;
            tap += at_slope(a, ratio, cx, i, &r);        // |tap| stays below M + 2^34: a few wraps at most
        }
        if (i < n && i >= lat) {
            long long t0 = tap;
            while (t0 < 0) t0 += M;
            while (t0 >= M) t0 -= M;
            long long t1 = t0 + half_m;
            if (t1 >= M) t1 -= M;
            const int w = (int)(i & mask);
            double mixed = 0.0, wsum = 0.0;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const double d = (double)(t == 0 ? t0 : t1) * (1.0 / (double)unit);
                const double phase = d / md;
                const double weight = 0.5 * (1.0 - cos(2.0 * 3.141592653589793 * phase));
                // (w - d) + size lies in (size / 2, 2 size): Python's float % is one exact conditional subtraction here
                const double wd = ((double)w - d) + size;
                const double rp = wd >= size ? wd - size : wd;
                const int b = ((int)rp) & mask;
                const int nx = (b + 1) & mask;
                const double fr = rp - (double)(int)rp;
                const long long j0 = i - ((w - b) & mask), j1 = i - ((w - nx) & mask);
                const float s0 = j0 >= 0 ? x[j0] : 0.0f, s1 = j1 >= 0 ? x[j1] : 0.0f;
                const float smp = __fadd_rn(__fmul_rn(s0, (float)(1.0 - fr)), __fmul_rn(s1, (float)fr));   // float32 (NEP 50)
                mixed += (double)smp * weight;
                wsum += weight;
            }
            val = wsum > 1e-6 ? (float)(mixed / wsum) : 0.0f;
        }
        so[lane * (AT_SPL + 1) + k] = val;
    }
    __syncwarp();
    for (int j = lane; j < AT_TS; j += 32) {
        const long long i = i0 + j;
        if (i >= n) break;
        if (i >= n - lat) out[i] = 0.0f;               // the tail that no shifted sample reaches
        if (i >= lat) out[i - lat] = so[j + j / AT_SPL];
    }
}

// ---------------------------------------------------------------- sub layer and final mix
struct AtMixArgs {
    const float *x, *sub, *air, *corrected;   // packed like the batch, as are env, sub_layer and y
    float *env;              // scratch
    float *env_max;          // [batch]
    float *sub_layer;        // optional
    float *y;                // autotune output
    long long n;
    long long seg_min;       // clips of at least seg_min samples take at_env_seg_kernel, shorter ones at_env_kernel
    const int64_t *starts;
    const int32_t *lengths;
    int clip0, batch;
    int sub_enabled;         // cfg.sub_enabled
    int layer_on;            // sub_enabled and sub_level > 0 and freq > 0
    float att, rel;          // float32(exp(-1/(ms*sr/1000)))
    float level, preserve, air_mix;
    float phase_k, sr_f;     // float32(2 pi f), float32(sr): phase = f32(f32(k * i) / sr)
};

// envelope follower, float32 sequential per clip (dsp/autotune.py:363-377 with NEP-50 scalar types)
__global__ void __launch_bounds__(32 * AT_FW) at_env_kernel(const AtMixArgs a) {
    __shared__ float s_io[AT_FW][AT_TS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int clip = blockIdx.x * AT_FW + warp;
    if (clip >= a.batch) return;
    const ClipLoc c = clip_loc(a, clip);
    if (c.n >= a.seg_min) return;
    const long long n = c.n;
    const float *__restrict__ x = a.x + c.base;
    float *__restrict__ env = a.env + c.base;
    float *io = s_io[warp];
    constexpr int PER = AT_TS / 32;
    float nxt[PER];
    float cur = 0.0f, top = 0.0f;
#pragma unroll
    for (int k = 0; k < PER; ++k) io[lane + 32 * k] = lane + 32 * k < n ? x[lane + 32 * k] : 0.0f;
    __syncwarp();
    for (long long i0 = 0; i0 < n; i0 += AT_TS) {
        const bool more = i0 + AT_TS < n;
        if (more) {
#pragma unroll
            for (int k = 0; k < PER; ++k) { const long long i = i0 + AT_TS + lane + 32 * k; nxt[k] = i < n ? x[i] : 0.0f; }
        }
        const int cnt = (int)(n - i0 < AT_TS ? n - i0 : AT_TS);
        if (lane == 0) {
            for (int k = 0; k < cnt; ++k) {
                const float s = fabsf(io[k]);
                const float c = s > cur ? a.att : a.rel;
                cur = __fadd_rn(s, __fmul_rn(c, __fsub_rn(cur, s)));
                io[k] = cur;
                top = fmaxf(top, cur);
            }
        }
        __syncwarp();
        for (int k = lane; k < cnt; k += 32) env[i0 + k] = io[k];
        __syncwarp();
        if (more) {
#pragma unroll
            for (int k = 0; k < PER; ++k) io[lane + 32 * k] = nxt[k];
        }
        __syncwarp();
    }
    if (lane == 0) a.env_max[c.idx] = top;
}

// The same follower, segment-parallel: both branches of the recurrence pull `cur` towards |x| by a factor of at least
// 1 - max(att, rel), so two runs over the same input that start from different states approach each other by that factor
// per sample whichever branches they take.  One thread follows one tile of `tile` samples after a warm-up of `halo`
// samples from zero (host: max(att, rel)^halo < 1e-10, far below a float32 ulp); a warp stages 32 samples of its 32 tiles
// through shared memory like the zero-phase filters.  The clip maximum is an atomicMax on the float bits (env >= 0);
// env_max must be zeroed before the launch.
__global__ void __launch_bounds__(32 * AT_SW) at_env_seg_kernel(const AtMixArgs a, int tile, int halo) {
    __shared__ float s_row[AT_SW][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ClipLoc c = clip_loc(a, blockIdx.y);
    const long long n = c.n;
    if (n < a.seg_min) return;
    const float *__restrict__ x = a.x + c.base;
    float *__restrict__ env = a.env + c.base;
    const long long n_tiles = (n + tile - 1) / tile;
    const long long tile0 = ((long long)blockIdx.x * AT_SW + warp) * 32;
    if (tile0 >= n_tiles) return;
    const int rows = (int)(n_tiles - tile0 < 32 ? n_tiles - tile0 : 32);
    float (*row)[33] = s_row[warp];
    const long long p_first = tile0 * tile - halo;          // row 0, step 0, column 0
    const long long p_own = p_first + (long long)lane * tile;
    const int steps = (halo + tile) / 32;
    float nxt[32];
    auto plain = [&](int j) {                               // all 32 rows exist and the whole step lies inside the clip
        const long long p0 = p_first + 32LL * j;
        return rows == 32 && p0 >= 0 && p0 + 31LL * tile + 31 < n;
    };
    auto fetch = [&](int j) {                               // loads only: the values are consumed one step later
        if (plain(j)) {
            const float *src = x + (p_first + 32LL * j + lane);
#pragma unroll
            for (int r = 0; r < 32; ++r) nxt[r] = src[(long long)r * tile];
            return;
        }
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const long long p = p_first + (long long)r * tile + 32LL * j + lane;
            nxt[r] = x[(r < rows && p >= 0 && p < n) ? p : 0];
        }
    };
    float cur = 0.0f, top = 0.0f;
    fetch(0);
    for (int j = 0; j < steps; ++j) {
#pragma unroll
        for (int r = 0; r < 32; ++r) row[r][lane] = nxt[r];
        __syncwarp();
        if (j + 1 < steps) fetch(j + 1);
        const long long p_step = p_own + 32LL * j;          // steps are 32-aligned: a step lies wholly before or after p = 0
        const bool own = 32 * j >= halo;                    // past the warm-up: these samples are the tile's output
        if (lane < rows && p_step >= 0 && p_step < n) {
#pragma unroll 8
            for (int k = 0; k < 32; ++k) {
                const float s = fabsf(row[lane][k]);
                const float c = s > cur ? a.att : a.rel;
                cur = __fadd_rn(s, __fmul_rn(c, __fsub_rn(cur, s)));
                if (own) {
                    row[lane][k] = cur;
                    if (p_step + k < n) top = fmaxf(top, cur);
                }
            }
        }
        __syncwarp();
        if (own) {
            if (plain(j)) {
                float *dst = env + (p_first + 32LL * j + lane);
#pragma unroll
                for (int r = 0; r < 32; ++r) dst[(long long)r * tile] = row[r][lane];
            } else {
#pragma unroll 8
                for (int r = 0; r < rows; ++r) {
                    const long long p = p_first + (long long)r * tile + 32LL * j + lane;
                    if (p < n) env[p] = row[r][lane];
                }
            }
        }
        __syncwarp();
    }
    top = warp_max(top);
    if (lane == 0) atomicMax(reinterpret_cast<int *>(a.env_max + c.idx), __float_as_int(top));
}

__global__ void at_mix_kernel(const AtMixArgs a) {
    const ClipLoc c = clip_loc(a, blockIdx.y);
    const long long base = c.base;
    const float top = a.layer_on ? a.env_max[c.idx] : 0.0f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < c.n; i += (long long)gridDim.x * blockDim.x) {
        float layer = 0.0f;
        if (a.layer_on) {
            float e = a.env[base + i];
            if ((double)top > 1e-6) e = __fdiv_rn(e, top);
            const float phase = __fdiv_rn(__fmul_rn(a.phase_k, (float)i), a.sr_f);
            layer = __fmul_rn(__fmul_rn(a.level, e), sinf(phase));
        }
        if (a.sub_layer) a.sub_layer[base + i] = layer;
        const float sub = a.sub[base + i];
        const float low = a.sub_enabled ? __fadd_rn(__fmul_rn(a.preserve, sub), layer) : sub;
        a.y[base + i] = __fadd_rn(__fadd_rn(low, a.corrected[base + i]), __fmul_rn(a.air_mix, a.air[base + i]));
    }
}

}  // namespace qd
