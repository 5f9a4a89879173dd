// qd_api.cu -- C ABI of libqd_b200.so (see include/qd_b200.h).  sm_100a only; no CPU fallback.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <map>
#include <mutex>
#include <tuple>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/qd_b200.h"
#include "qd_err.hpp"
#include "qd_host_tables.hpp"
#include "qd_host_time.hpp"
#include "qd_spec_launch.hpp"
#include "qd_spec_team_launch.hpp"
#include "qd_peaks.cuh"
#include "qd_autotune.cuh"
#include "qd_time.cuh"

#ifndef QD_NW_1024
#define QD_NW_1024 16
#endif

namespace {

using qd_err::ensure_dyn_smem;
using qd_err::fail;
using qd_launch::launch_spec_t;

template <class T>
cudaError_t upload(const std::vector<T> &h, T **d) {
    *d = nullptr;
    const size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
    cudaError_t e = cudaMalloc((void **)d, bytes);
    if (e != cudaSuccess) return e;
    if (!h.empty()) e = cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
}

struct HostPipe {   // resources of qd_render_host* (qd_host_pipe.inc)
    int64_t cap = 0;         // samples per device buffer (the longest chunk's packed span)
    int64_t cap_clips = 0;   // clips per chunk the workspace is sized for
    int64_t *d_starts = nullptr;   // ragged calls: the caller's starts / lengths, uploaded once per call
    int32_t *d_lengths = nullptr;
    int64_t d_clips = 0;
    float *dx[2] = {nullptr, nullptr};
    float *dy[2] = {nullptr, nullptr};
    int16_t *dxr[2] = {nullptr, nullptr};   // PCM16 transport: raw input / output chunks on the device
    int16_t *dyr[2] = {nullptr, nullptr};
    void *pin_in[3] = {nullptr, nullptr, nullptr};    // pinned staging rings for pageable callers
    void *pin_out[3] = {nullptr, nullptr, nullptr};
    void *ws = nullptr;
    size_t ws_bytes = 0;
    cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_run[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    cudaEvent_t ev_ring_in[3] = {nullptr, nullptr, nullptr}, ev_ring_out[3] = {nullptr, nullptr, nullptr};
};

}  // namespace

struct qd_plan {
    qd_params p;
    int nc = 0, hop = 0, n_frames = 0, nw = 0;
    bool has_quant = false;
    std::vector<void *> owned;  // device allocations
    qd::SpecArgsT<float> spec{};     // table pointers filled once (float32 FFT)
    qd::SpecArgsT<double> spec64{};  // the same for the float64 parity path
    bool f64 = false;
    bool ts = false;           // float32 n_fft 2048: tables fit the shared-memory kernel variant
    bool ts_fx = false;        // the same for the 12-warp FX variant (no formant scratch)
    size_t spec_smem = 0;      // dynamic shared memory of the pass kernel in use
    const void *fx_table = nullptr;
    int64_t fx_tables = 0;
    HostPipe pipe;
    int sm_count = 148;
    qd::TeamGather team_tg{};  // gather lists of the team kernel (long frames, plain passes); team_nf = 0: not used
    int team_nf = 0, team_cw = 0;
    size_t team_smem = 0;
    // optional per-kernel device timing (qd_plan_enable_timing)
    bool timing = false;
    struct Stamp { cudaEvent_t a, b; int cls; };
    std::vector<Stamp> stamps;
    std::vector<cudaEvent_t> free_events;
    double t_ms[QD_KERNEL_CLASSES] = {0, 0, 0, 0};
    int64_t t_launches[QD_KERNEL_CLASSES] = {0, 0, 0, 0};
};

namespace {
// How the clips of one render sit in their buffers: uniform (starts == null: clip c at c * n_samples) or a ragged batch
// (device arrays, offsets relative to starts[0]).  span = packed extent in samples; max_n = the longest clip.
struct Packing {
    const int64_t *starts = nullptr;
    const int32_t *lengths = nullptr;
    int64_t span = 0;
    int max_n = 0;
    int64_t clip_offset = 0;   // row of clip 0 in a per-clip FX table (qd_render_host: the chunk's first clip)
};
// intermediates of a render ([x_dist], [low], [high]) use the packing of x, each padded to 256 bytes
size_t padded_span(int64_t span) { return ((size_t)span + 63) & ~(size_t)63; }

struct TimeScope {  // brackets the launches of one kernel class with events on the launch stream
    qd_plan *pl; cudaStream_t st; int cls; cudaEvent_t a = nullptr, b = nullptr;
    static cudaEvent_t get(qd_plan *p) {
        cudaEvent_t e = nullptr;
        if (!p->free_events.empty()) { e = p->free_events.back(); p->free_events.pop_back(); }
        else cudaEventCreate(&e);
        return e;
    }
    TimeScope(qd_plan *p, cudaStream_t s, int c) : pl(p), st(s), cls(c) {
        if (pl->timing) { a = get(pl); b = get(pl); cudaEventRecord(a, st); }
    }
    ~TimeScope() {
        if (pl->timing) { cudaEventRecord(b, st); pl->stamps.push_back({a, b, cls}); }
    }
};
}  // namespace

namespace {

// ---- kernel selection.  float32: n_fft 2048 (the headline size) runs 16 warps per CTA with its tables in
//      shared memory (falls back to 8 warps + L1 tables when they do not fit); float64 (parity path) and the
//      FX variants read tables through L1.  Must stay in sync with the switch in dispatch_spec().
template <class T> int pick_nw(int nc, bool fx, bool formant = false) {
    if (sizeof(T) == 4 && formant) return nc <= 1024 ? 8 : nc == 2048 ? 4 : 1;   // scratch buffer per warp
    // n_fft 8192: one warp (182 KB); n_fft 2048: six warps beside their magnitude planes, four with the formant scratch
    if (sizeof(T) == 8 && fx) return nc <= 512 ? 8 : nc == 1024 ? (formant ? 4 : 6) : nc == 2048 ? 2 : 1;
    if (sizeof(T) == 8) return nc <= 1024 ? 8 : nc == 2048 ? 4 : 2;
    if (fx) return nc == 1024 ? 12 : nc < 1024 ? 8 : nc == 2048 ? 4 : 2;   // what fits beside the FX magnitude planes
    return nc == 1024 ? QD_NW_1024 : nc < 1024 ? 8 : 4;  // 16 = two independent groups of 8 warps per CTA
}

template <class T, int NC, int NW>
size_t smem_of(int n_slots, bool ts, int n_src, int formant, bool fx) {
    return qd::SpecSmem<T, NC, NW>::bytes(n_slots, ts, n_src, 0, fx, formant != 0);
}

template <class T>
size_t spec_smem_bytes(int nc, int nw, bool ts, int n_slots, int n_src, int formant, bool fx) {
    const int fm = formant;
    switch (nc) {
        case 256:  return nw == 8 ? smem_of<T, 256, 8>(n_slots, false, 0, fm, fx) : 0;
        case 512:  return nw == 8 ? smem_of<T, 512, 8>(n_slots, false, 0, fm, fx) : 0;
        case 1024:
            if (nw == 16) return qd::SpecSmem<T, 1024, 8, 2>::bytes(n_slots, ts, n_src, 0, fx);
            return nw == 8 ? smem_of<T, 1024, 8>(n_slots, false, 0, fm, fx)
                 : nw == 12 ? smem_of<T, 1024, 12>(n_slots, false, 0, fm, fx)
                 : nw == 6 ? smem_of<T, 1024, 6>(n_slots, false, 0, fm, fx)
                 : nw == 4 ? smem_of<T, 1024, 4>(n_slots, false, 0, fm, fx) : 0;
        case 2048: return nw == 4 ? smem_of<T, 2048, 4>(n_slots, false, 0, fm, fx)
                        : nw == 2 ? smem_of<T, 2048, 2>(n_slots, false, 0, fm, fx) : 0;
        case 4096:
            if (nw == 1 && sizeof(T) == 8 && fm)   // float64 formant shift at n_fft 8192: samples staged in the scratch buffer
                return qd::SpecSmem<T, 4096, 1, 1, true>::bytes(n_slots, false, 0, 0, fx, true);
            return nw == 4 ? smem_of<T, 4096, 4>(n_slots, false, 0, fm, fx)
                 : nw == 2 ? smem_of<T, 4096, 2>(n_slots, false, 0, fm, fx)
                 : nw == 1 ? smem_of<T, 4096, 1>(n_slots, false, 0, fm, fx) : 0;
    }
    return 0;
}

template <class T, bool FX>
int dispatch_spec(int nc, int nw, bool ts, const qd::SpecArgsT<T> &a, int tiles, int64_t batch, cudaStream_t st) {
    switch (nc) {
        case 256:  return launch_spec_t<T, 256, 8, false, FX>(a, tiles, batch, st);
        case 512:  return launch_spec_t<T, 512, 8, false, FX>(a, tiles, batch, st);
        case 1024:
            if constexpr (sizeof(T) == 4 && !FX) {
                if (nw == 16 && ts) {
                    // no epilogue, or a wavefold that is exact in float32 (the reference defaults): the kernel whose
                    // unrolled overlap-add carries neither the float64 nor the tanh branch
                    if (a.epilogue == 0 || (a.epilogue == 1 && a.fold_exact_f32)) return launch_spec_t<T, 1024, 8, true, false, 2, false, true>(a, tiles, batch, st);
                    return launch_spec_t<T, 1024, 8, true, false, 2>(a, tiles, batch, st);
                }
            }
            if constexpr (sizeof(T) == 8 && FX) return nw == 6 ? launch_spec_t<T, 1024, 6, false, true>(a, tiles, batch, st)
                                                               : launch_spec_t<T, 1024, 4, false, true>(a, tiles, batch, st);
            else if constexpr (FX) return nw == 8 ? launch_spec_t<T, 1024, 8, false, true>(a, tiles, batch, st)
                                             : ts ? launch_spec_t<T, 1024, 12, true, true>(a, tiles, batch, st)
                                                  : launch_spec_t<T, 1024, 12, false, true>(a, tiles, batch, st);
            else return launch_spec_t<T, 1024, 8, false, false>(a, tiles, batch, st);
        case 2048:
            if constexpr (sizeof(T) == 8 && FX) return launch_spec_t<T, 2048, 2, false, true>(a, tiles, batch, st);
            else return launch_spec_t<T, 2048, 4, false, FX>(a, tiles, batch, st);
        case 4096:
            if constexpr (sizeof(T) == 8 && FX) {   // one warp per CTA; with the formant scratch the samples are staged in it
                if (a.formant_idx) return launch_spec_t<T, 4096, 1, false, true, 1, true>(a, tiles, batch, st);
                return launch_spec_t<T, 4096, 1, false, true>(a, tiles, batch, st);
            } else if constexpr (sizeof(T) == 8) return launch_spec_t<T, 4096, 2, false, false>(a, tiles, batch, st);
            else if constexpr (FX) return nw == 1 ? launch_spec_t<T, 4096, 1, false, true>(a, tiles, batch, st)
                                                  : launch_spec_t<T, 4096, 2, false, true>(a, tiles, batch, st);
            else return launch_spec_t<T, 4096, 4, false, false>(a, tiles, batch, st);
    }
    return fail(QD_ERR_UNSUPPORTED, "n_fft not supported");
}

template <class T, int NC>
int launch_freeze_t(const qd::SpecArgsT<T> &a, T *out, int64_t batch, cudaStream_t st) {
    static std::atomic<uint64_t> attr_mask{0};  // devices this instantiation was opted in on
    auto kern = qd::freeze_mag_kernel<T, NC>;
    const size_t smem = (size_t)qd::buf_slots<NC>() * sizeof(qd::V2<T>) + (size_t)2 * NC * sizeof(float) + 16;
    if (int rc_ = ensure_dyn_smem(kern, attr_mask, 227 * 1024)) return rc_;
    kern<<<(unsigned)batch, 32, smem, st>>>(a, out);
    QD_CUDA(cudaGetLastError());
    return QD_OK;
}

template <class T>
int launch_freeze(int nc, const qd::SpecArgsT<T> &a, T *out, int64_t batch, cudaStream_t st) {
    switch (nc) {
        case 256:  return launch_freeze_t<T, 256>(a, out, batch, st);
        case 512:  return launch_freeze_t<T, 512>(a, out, batch, st);
        case 1024: return launch_freeze_t<T, 1024>(a, out, batch, st);
        case 2048: return launch_freeze_t<T, 2048>(a, out, batch, st);
        case 4096: return launch_freeze_t<T, 4096>(a, out, batch, st);
    }
    return fail(QD_ERR_UNSUPPORTED, "n_fft not supported");
}

template <class T>
int launch_spec_prec(qd_plan *pl, qd::SpecArgsT<T> a, const Packing &pk, const float *src, float *dst, float *tap, int quant,
                     int epilogue, int64_t batch, cudaStream_t st, int fx_pass, float *clip_peak, void *frozen_ws) {
    a.starts = pk.starts;
    a.lengths = pk.lengths;
    a.clip0 = 0;
    a.n = pk.max_n;
    a.x = src;
    a.y = dst;
    a.tap = tap;
    a.clip_peak = clip_peak;
    if (clip_peak) QD_CUDA(cudaMemsetAsync(clip_peak, 0, (size_t)batch * sizeof(float), st));
    a.quant = quant;
    a.epilogue = epilogue;
    const bool fx = quant && (pl->p.fx_mode != QD_FX_NONE || pl->p.spectral_freeze || pl->p.formant_ratio > 0.0);
    a.fx.pass = fx_pass;
    a.fx.clip_offset = (int)pk.clip_offset;
    a.fx.table = pl->fx_table;
    // a pass that does not run the FX uses the plain kernel of the same warp count
    int nw = fx ? pl->nw : pick_nw<T>(pl->nc, false) == 16 && !pl->ts ? 8 : pick_nw<T>(pl->nc, false);
    const bool ts = fx ? pl->ts_fx : pl->ts;
    const int ng = (nw == 16) ? 2 : 1;   // clips per CTA
    // three-pass plans without FX: the team kernel (qd_spec_team.cuh; several warps per frame at n_fft >= 4096)
    const bool team = !fx && pl->team_nf > 0;
    // tiling: whole clips when the batch alone fills the GPU, else cut clips along time.  The grid covers the longest
    // clip (CTAs past a shorter clip's end exit at once); the tile is cut from the mean clip
    const int total_blocks = (pk.max_n + pl->hop - 1) / pl->hop;
    const int mean_blocks = (int)((pk.span / batch + pl->hop - 1) / pl->hop);
    const int ctas_per_sm = std::max<int>(1, (int)((227 * 1024) / ((team ? pl->team_smem : pl->spec_smem) + 1024)));
    const int64_t want = (int64_t)pl->sm_count * ctas_per_sm * 2 * ng;
    const int wpg = team ? pl->team_nf : nw / ng;  // frames per batch of one clip group
    int tile = total_blocks;
    if (batch < want) {
        const int64_t per_clip = (want + batch - 1) / batch;
        tile = (int)((mean_blocks + per_clip - 1) / per_clip);
        const int min_tile = 4 * wpg - 3;  // keeps the 3-frame halo recompute below 10 %
        if (tile < min_tile) tile = min_tile;
        tile = ((tile + 3 + wpg - 1) / wpg) * wpg - 3;  // whole batches of frames
        if (tile > total_blocks) tile = total_blocks;
    }
    if (tile < 1) tile = 1;
    a.tile_blocks = tile;
    const int tiles = (total_blocks + tile - 1) / tile;
    a.frozen = nullptr;
    if (fx && pl->p.spectral_freeze) {
        // frame-0 magnitudes of THIS pass's input (each quantised pass freezes its own first frame)
        T *frozen = reinterpret_cast<T *>(frozen_ws);
        int rc = launch_freeze<T>(pl->nc, a, frozen, batch, st);
        if (rc != QD_OK) return rc;
        a.frozen = frozen;
    }
    if (team) return qd_launch::launch_spec_team<T>(pl->nc, a, pl->team_tg, tiles, batch, st);
    if (fx) return dispatch_spec<T, true>(pl->nc, nw, ts, a, tiles, batch, st);
    return dispatch_spec<T, false>(pl->nc, nw, ts, a, tiles, batch, st);
    (void)nw;
}

// One spectral pass over [batch, n]: src -> dst (+ optional tap of the pre-epilogue signal).  frozen_ws: the render
// workspace's scratch for the frame-0 magnitudes of the spectral freeze.
int launch_spec(qd_plan *pl, const Packing &pk, const float *src, float *dst, float *tap, int quant, int epilogue,
                int64_t batch, cudaStream_t st, int fx_pass = 0, float *clip_peak = nullptr, void *frozen_ws = nullptr) {
    TimeScope ts(pl, st, QD_KERNEL_SPECTRAL);
    if (pl->f64) return launch_spec_prec<double>(pl, pl->spec64, pk, src, dst, tap, quant, epilogue, batch, st, fx_pass, clip_peak, frozen_ws);
    return launch_spec_prec<float>(pl, pl->spec, pk, src, dst, tap, quant, epilogue, batch, st, fx_pass, clip_peak, frozen_ws);
}

int launch_limiter(const qd::LimiterArgs &a, int64_t batch, cudaStream_t st) {
    static std::atomic<uint64_t> attr_mask{0};  // devices this instantiation was opted in on
    const size_t smem = qd_host::limiter_smem_bytes(a.lookahead);
    if (smem > 200 * 1024) return fail(QD_ERR_UNSUPPORTED, "limiter lookahead too long");
    if (int rc_ = ensure_dyn_smem(qd::limiter_mix_kernel, attr_mask, 200 * 1024)) return rc_;
    qd::for_each_launch(batch, 1 << 30, [&](int clip0, int nb) {   // one clip per CTA on gridDim.x
        qd::LimiterArgs c = a;
        c.clip0 = clip0;
        qd::limiter_mix_kernel<<<(unsigned)nb, qd::QD_TT, smem, st>>>(c);
    });
    QD_CUDA(cudaGetLastError());
    return QD_OK;
}

// the wavefold's (x + bias) * fold is exact in float32 when there is no bias and the gain is a power of two
int fold_exact_in_f32(double fold, double bias) {
    int e = 0;
    return bias == 0.0 && fold > 0.0 && std::frexp(fold, &e) == 0.5 && e > -100 && e < 100;
}

void launch_crossover(const qd::CrossoverArgs &c, int64_t batch, cudaStream_t st) {
    const long long n_tiles = (c.n + c.tile - 1) / c.tile;
    const unsigned gx = (unsigned)((n_tiles + 32 * qd::QD_XO_WARPS - 1) / (32 * qd::QD_XO_WARPS));
    qd::for_each_launch(batch, qd::QD_GRID_Y_MAX, [&](int clip0, int nb) {
        qd::CrossoverArgs k = c;
        k.clip0 = clip0;
        qd::crossover_kernel<<<dim3(gx, (unsigned)nb, 1), 32 * qd::QD_XO_WARPS, 0, st>>>(k);
    });
}

int ew_grid(int64_t count, int sm_count) {
    const int64_t blocks = (count + 255) / 256;
    return (int)std::min<int64_t>(blocks, (int64_t)sm_count * 16);
}

}  // namespace

namespace {
// FFT tables of the peaks kernel, built once per (device, n_fft, precision) and kept for the process lifetime
struct PeakTables { void *wtab = nullptr, *tw1 = nullptr, *tw2 = nullptr, *wsplit = nullptr; };
std::mutex g_peak_mu;
std::map<std::tuple<int, int, int>, PeakTables> g_peak_tables;

template <class T>
int peak_tables(int dev, int n_fft, PeakTables *out) {
    std::lock_guard<std::mutex> lk(g_peak_mu);
    const auto key = std::make_tuple(dev, n_fft, (int)sizeof(T));
    auto it = g_peak_tables.find(key);
    if (it == g_peak_tables.end()) {
        qd_host::SpecTablesT<T> st;
        if (!qd_host::build_spec_tables<T>(n_fft, &st)) return fail(QD_ERR_UNSUPPORTED, "n_fft must be one of 512, 1024, 2048, 4096, 8192");
        PeakTables pt;
        typename qd_host::Pair<T>::type *a = nullptr, *b = nullptr, *c = nullptr, *d = nullptr;
        QD_CUDA(upload(st.wtab, &a));
        QD_CUDA(upload(st.tw1, &b));
        QD_CUDA(upload(st.tw2, &c));
        QD_CUDA(upload(st.wsplit, &d));
        pt.wtab = a; pt.tw1 = b; pt.tw2 = c; pt.wsplit = d;
        it = g_peak_tables.emplace(key, pt).first;
    }
    *out = it->second;
    return QD_OK;
}

template <class T, int NC>
int launch_peaks_t(qd::PeaksArgsT<T> a, int64_t batch, cudaStream_t st) {
    static std::atomic<uint64_t> attr_mask{0};  // devices this instantiation was opted in on
    auto kern = qd::peaks_kernel<T, NC>;
    if (int rc_ = ensure_dyn_smem(kern, attr_mask, 227 * 1024)) return rc_;
    constexpr size_t per_warp = qd::peaks_warp_smem<T, NC>();
    constexpr int nw = qd::peaks_warps<T, NC>();
    const unsigned gx = (unsigned)((a.n_frames + nw - 1) / nw);
    qd::for_each_launch(batch, qd::QD_GRID_Y_MAX, [&](int clip0, int nb) {
        qd::PeaksArgsT<T> c = a;
        c.clip0 = clip0;
        kern<<<dim3(gx, (unsigned)nb, 1), 32 * nw, per_warp * nw, st>>>(c);
    });
    QD_CUDA(cudaGetLastError());
    return QD_OK;
}

// Uniform batches pass null starts / lengths (n = the clip length); ragged ones their device arrays (n = the longest clip).
template <class T>
int launch_peaks(const float *x, const int64_t *starts, const int32_t *lengths, int64_t batch, int n, int n_fft, int topn,
                 double min_mag, int16_t *bins, cudaStream_t st) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return fail(QD_ERR_NO_DEVICE, "no CUDA device: libqd_b200 has no CPU path"); }
    PeakTables pt;
    int rc = peak_tables<T>(dev, n_fft, &pt);
    if (rc != QD_OK) return rc;
    qd::PeaksArgsT<T> a{};
    a.x = x; a.bins = bins; a.starts = starts; a.lengths = lengths; a.n = n; a.topn = topn;
    a.n_frames = 1 + n / (n_fft / 4);
    a.min_mag2 = (T)(min_mag * min_mag);
    a.wtab = reinterpret_cast<const qd::V2<T> *>(pt.wtab);
    a.tw1 = reinterpret_cast<const qd::V2<T> *>(pt.tw1);
    a.tw2 = reinterpret_cast<const qd::V2<T> *>(pt.tw2);
    a.wsplit = reinterpret_cast<const qd::V2<T> *>(pt.wsplit);
    switch (n_fft / 2) {
        case 256:  return launch_peaks_t<T, 256>(a, batch, st);
        case 512:  return launch_peaks_t<T, 512>(a, batch, st);
        case 1024: return launch_peaks_t<T, 1024>(a, batch, st);
        case 2048: return launch_peaks_t<T, 2048>(a, batch, st);
        case 4096: return launch_peaks_t<T, 4096>(a, batch, st);
    }
    return fail(QD_ERR_UNSUPPORTED, "n_fft must be one of 512, 1024, 2048, 4096, 8192");
}
}  // namespace

extern "C" {

int qd_abi_version(void) { return QD_ABI_VERSION; }

const char *qd_last_error(void) { return qd_err::g_err.c_str(); }

int qd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        cudaDeviceProp pr;
        if (cudaGetDeviceProperties(&pr, i) == cudaSuccess && pr.major == 10) ++ok;
    }
    return ok;
}

int qd_spectral_peaks_device(const float *x, int64_t batch, int32_t n_samples, int32_t n_fft, int32_t topn,
                             double min_mag, int32_t precision, int16_t *bins, void *stream) {
    if (!x || !bins || batch < 0 || n_samples < 0) return fail(QD_ERR_INVALID_ARG, "null / negative argument");
    if (batch > INT32_MAX) return fail(QD_ERR_INVALID_ARG, "batch of more than 2^31 - 1 clips");
    if (topn < 1 || topn > qd::QD_PEAKS_MAX) return fail(QD_ERR_INVALID_ARG, "topn must be 1..8");
    if (batch == 0) return QD_OK;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (precision == QD_PRECISION_F64) return launch_peaks<double>(x, nullptr, nullptr, batch, n_samples, n_fft, topn, min_mag, bins, st);
    if (precision == QD_PRECISION_F32) return launch_peaks<float>(x, nullptr, nullptr, batch, n_samples, n_fft, topn, min_mag, bins, st);
    return fail(QD_ERR_INVALID_ARG, "bad precision");
}

int qd_spectral_peaks_device_varlen(const float *x, const int64_t *starts, const int32_t *lengths, int64_t batch,
                                    int32_t max_samples, int32_t n_fft, int32_t topn, double min_mag, int32_t precision,
                                    int16_t *bins, void *stream) {
    if (!x || !starts || !lengths || !bins || batch < 0 || max_samples < 0) return fail(QD_ERR_INVALID_ARG, "null / negative argument");
    if (batch > INT32_MAX) return fail(QD_ERR_INVALID_ARG, "batch of more than 2^31 - 1 clips");
    if (topn < 1 || topn > qd::QD_PEAKS_MAX) return fail(QD_ERR_INVALID_ARG, "topn must be 1..8");
    if (precision != QD_PRECISION_F64 && precision != QD_PRECISION_F32) return fail(QD_ERR_INVALID_ARG, "bad precision");
    if (batch == 0) return QD_OK;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (precision == QD_PRECISION_F64) return launch_peaks<double>(x, starts, lengths, batch, max_samples, n_fft, topn, min_mag, bins, st);
    return launch_peaks<float>(x, starts, lengths, batch, max_samples, n_fft, topn, min_mag, bins, st);
}

int qd_plan_create(const qd_params *params, const qd_tables *tables, qd_plan **out) {
    if (!params || !out) return fail(QD_ERR_INVALID_ARG, "null argument");
    *out = nullptr;
    if (params->struct_size != sizeof(qd_params)) return fail(QD_ERR_INVALID_ARG, "qd_params size mismatch (ABI)");
    const qd_params &p = *params;
    if (p.n_samples < 0 || p.sample_rate <= 0) return fail(QD_ERR_INVALID_ARG, "bad n_samples / sample_rate");
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return fail(QD_ERR_NO_DEVICE, "no CUDA device: libqd_b200 has no CPU path"); }
    cudaDeviceProp pr;
    QD_CUDA(cudaGetDeviceProperties(&pr, dev));
    if (pr.major != 10) return fail(QD_ERR_NO_DEVICE, "device is not sm_100 (B200)");
    qd_host::SpecTables st;
    if (!qd_host::build_spec_tables<float>(p.n_fft, &st)) return fail(QD_ERR_UNSUPPORTED, "n_fft must be one of 512, 1024, 2048, 4096, 8192");
    const bool need_quant = !p.passthrough && (p.pre_quant || p.post_quant);
    if (need_quant && !tables) return fail(QD_ERR_INVALID_ARG, "quantizer tables required");
    if (p.fx_mode < QD_FX_NONE || p.fx_mode > QD_FX_SCRAMBLE_SWAP) return fail(QD_ERR_INVALID_ARG, "bad fx_mode");
    if (p.fx_mode != QD_FX_NONE && !p.multiband) return fail(QD_ERR_INVALID_ARG, "spectral FX act on the high band of a multiband render only");
    if (p.fx_mode == QD_FX_SCRAMBLE_PICK && p.n_fft > 2048 && p.fx_a > 512.0)
        return fail(QD_ERR_UNSUPPORTED, "bin scramble at n_fft > 2048 gathers in tiles: window / 2 must be <= 512 bins");
    if (p.precision != QD_PRECISION_F32 && p.precision != QD_PRECISION_F64) return fail(QD_ERR_INVALID_ARG, "bad precision");

    qd_plan *pl = new qd_plan();
    pl->p = p;
    pl->nc = st.nc;
    pl->hop = st.hop;
    pl->n_frames = 1 + p.n_samples / st.hop;
    pl->f64 = p.precision == QD_PRECISION_F64;
    pl->sm_count = pr.multiProcessorCount;
    pl->has_quant = need_quant;
    auto keep = [&](void *d) { pl->owned.push_back(d); };
    auto bail = [&](int code, const std::string &m) { qd_plan_destroy(pl); return fail(code, m); };
#define QD_UP(vec, ptr)                                                                   \
    do {                                                                                  \
        cudaError_t e_ = upload(vec, &ptr);                                               \
        if (ptr) keep(ptr);                                                               \
        if (e_ != cudaSuccess) return bail(QD_ERR_CUDA, cudaGetErrorString(e_));          \
    } while (0)
    qd::QuantDev qdev{};
    int n_slots = 0;
    if (need_quant) {
        if (tables->n_bins != st.nc + 1) return bail(QD_ERR_INVALID_ARG, "tables->n_bins != n_fft/2+1");
        qd_host::QuantTablesH qt;
        std::string err;
        if (!qd_host::build_quant_tables(*tables, &qt, &err, pl->f64)) return bail(QD_ERR_INVALID_ARG, err);
        uint16_t *d_sb;
        uint32_t *d_ra, *d_st;
        float *d_ik, *d_bs;
        QD_UP(qt.src_tab, d_st);
        {   // long frames: the plain passes run the team kernel, which reads one gather list per warp of a team
            const qd_launch::TeamShape ts_ = pl->f64 ? qd_launch::team_shape<double>(st.nc) : qd_launch::team_shape<float>(st.nc);
            if (ts_.nf > 0) {
                std::vector<uint32_t> ttab;
                qd_host::build_team_gather(qt, ts_.cw, &ttab, pl->team_tg.begin);
                uint32_t *d_tt;
                QD_UP(ttab, d_tt);
                pl->team_tg.src_tab = d_tt;
            }
        }
        QD_UP(qt.row_active, d_ra);
        QD_UP(qt.slot_of_bin, d_sb);
        QD_UP(qt.slot_invk, d_ik);
        QD_UP(qt.slot_base, d_bs);
        qdev.n_slots = qt.n_slots;
        qdev.n_src = (int)qt.src_tab.size();
        qdev.row_limit = qt.row_limit;
        qdev.src_tab = d_st;
        qdev.row_active = d_ra;
        qdev.slot_of_bin = d_sb;
        qdev.slot_invk = d_ik;
        qdev.slot_base = d_bs;
        for (int e = 0; e < 5; ++e) qdev.tap[e] = qt.tap[e];
        qdev.keep_active = qt.keep_active;
        qdev.smoothing = p.bin_smoothing ? 1 : 0;
        n_slots = qt.n_slots;
    }
    const bool formant = need_quant && p.formant_ratio > 0.0;
    if (formant && p.formant_order < 2) return bail(QD_ERR_INVALID_ARG, "formant_order must be >= 2");
    const bool fx = need_quant && (p.fx_mode != QD_FX_NONE || p.spectral_freeze || formant);
    qd::FxDev fxd{};
    fxd.mode = (need_quant && p.fx_mode != QD_FX_NONE) ? p.fx_mode : 0;
    fxd.a = (float)p.fx_a; fxd.b = (float)p.fx_b; fxd.c = (float)p.fx_c;
    fxd.step = p.fx_a;
    fxd.table_frames = p.fx_table_frames > 0 ? p.fx_table_frames : 1;
    fxd.table_per_clip = p.fx_table_per_clip;
    // formant shift: np.interp(k / ratio, arange(n_bins), env) as segment index and fraction per bin, in float64
    // (dsp/spectral_fx.py:173-183); beyond the last bin the envelope is held (right = env[-1])
    int16_t *d_fi = nullptr;
    float *d_ff = nullptr;
    if (formant) {
        const int nb = st.nc + 1;
        std::vector<int16_t> fi((size_t)nb);
        std::vector<float> ff((size_t)nb);
        for (int k = 0; k < nb; ++k) {
            const double x = (double)k / p.formant_ratio;
            if (x >= (double)(nb - 1)) { fi[k] = (int16_t)(nb - 1); ff[k] = 0.0f; }
            else { const double fl = std::floor(x); fi[k] = (int16_t)fl; ff[k] = (float)(x - fl); }
        }
        QD_UP(fi, d_fi);
        QD_UP(ff, d_ff);
    }
    if (pl->f64) {
        qd_host::SpecTablesT<double> sd;
        qd_host::build_spec_tables<double>(p.n_fft, &sd);
        qd_host::D2 *d_wtab, *d_tw1, *d_tw2, *d_wsplit;
        double *d_invw;
        QD_UP(sd.wtab, d_wtab);
        QD_UP(sd.tw1, d_tw1);
        QD_UP(sd.tw2, d_tw2);
        QD_UP(sd.wsplit, d_wsplit);
        QD_UP(sd.invw, d_invw);
        qd::SpecArgsT<double> &a = pl->spec64;
        a.n = p.n_samples;
        a.n_frames = pl->n_frames;
        a.fold = p.fold_amount; a.bias = p.bias; a.tube_gain = p.tube_gain; a.tube_norm = p.tube_norm;
        a.fold_exact_f32 = fold_exact_in_f32(p.fold_amount, p.bias);
        a.wtab = reinterpret_cast<const double2 *>(d_wtab);
        a.tw1 = reinterpret_cast<const double2 *>(d_tw1);
        a.tw2 = reinterpret_cast<const double2 *>(d_tw2);
        a.wsplit = reinterpret_cast<const double2 *>(d_wsplit);
        a.invw = d_invw;
        a.q = qdev;
        a.fx = fxd;
        a.formant_idx = d_fi; a.formant_frac = d_ff; a.formant_order = p.formant_order;
        pl->nw = pick_nw<double>(pl->nc, fx, formant);
        if (pl->nw == 6 && spec_smem_bytes<double>(pl->nc, 6, false, n_slots, qdev.n_src, 0, fx) > 227 * 1024) pl->nw = 4;  // many target slots
        pl->ts = false;
        pl->spec_smem = spec_smem_bytes<double>(pl->nc, pl->nw, false, n_slots, qdev.n_src, formant ? 1 : 0, fx);
    } else {
        qd_host::F2 *d_wtab, *d_tw1, *d_tw2, *d_wsplit;
        float *d_invw;
        QD_UP(st.wtab, d_wtab);
        QD_UP(st.tw1, d_tw1);
        QD_UP(st.tw2, d_tw2);
        QD_UP(st.wsplit, d_wsplit);
        QD_UP(st.invw, d_invw);
        qd::SpecArgsT<float> &a = pl->spec;
        a.n = p.n_samples;
        a.n_frames = pl->n_frames;
        a.fold = p.fold_amount; a.bias = p.bias; a.tube_gain = p.tube_gain; a.tube_norm = p.tube_norm;
        a.fold_exact_f32 = fold_exact_in_f32(p.fold_amount, p.bias);
        a.wtab = reinterpret_cast<const float2 *>(d_wtab);
        a.tw1 = reinterpret_cast<const float2 *>(d_tw1);
        a.tw2 = reinterpret_cast<const float2 *>(d_tw2);
        a.wsplit = reinterpret_cast<const float2 *>(d_wsplit);
        a.invw = d_invw;
        a.q = qdev;
        a.fx = fxd;
        a.formant_idx = d_fi; a.formant_frac = d_ff; a.formant_order = p.formant_order;
        pl->nw = pick_nw<float>(pl->nc, fx, formant);
        pl->ts = (pl->nc == 1024 && pl->nw == 16);
        if (fx && pl->nc == 1024 && pl->nw == 12 && !formant)   // FX variant with its tables in shared memory, when they fit
            pl->ts_fx = qd::SpecSmem<float, 1024, 12>::bytes(n_slots, true, qdev.n_src, 0, true, false) <= 227 * 1024;
        pl->spec_smem = pl->ts_fx ? qd::SpecSmem<float, 1024, 12>::bytes(n_slots, true, qdev.n_src, 0, true, false)
                                  : spec_smem_bytes<float>(pl->nc, pl->nw, pl->ts, n_slots, qdev.n_src, formant ? 1 : 0, fx);
        if (pl->ts && pl->spec_smem > 227 * 1024) {  // tables too large for shared memory: 8 warps, tables through L1
            pl->nw = 8;
            pl->ts = false;
            pl->spec_smem = spec_smem_bytes<float>(pl->nc, 8, false, n_slots, qdev.n_src, 0, fx);
        }
    }
#undef QD_UP
    {   // long frames: plain passes on the team kernel when its CTA fits (else the one-warp-per-frame kernel above)
        const qd_launch::TeamShape ts_ = pl->f64 ? qd_launch::team_shape<double>(pl->nc) : qd_launch::team_shape<float>(pl->nc);
        const size_t tsm = pl->f64 ? qd_launch::team_smem_bytes<double>(pl->nc, n_slots) : qd_launch::team_smem_bytes<float>(pl->nc, n_slots);
        if (ts_.nf > 0 && tsm > 0 && tsm <= 227 * 1024) { pl->team_nf = ts_.nf; pl->team_cw = ts_.cw; pl->team_smem = tsm; }
    }
    if (pl->spec_smem == 0 || pl->spec_smem > 227 * 1024)
        return bail(QD_ERR_UNSUPPORTED, "shared memory need of this (n_fft, target table, precision) exceeds 227 KB");
    *out = pl;
    return QD_OK;
}

void qd_plan_destroy(qd_plan *pl) {
    if (!pl) return;
    for (void *d : pl->owned) cudaFree(d);
    for (auto &sp : pl->stamps) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    for (auto e : pl->free_events) cudaEventDestroy(e);
    HostPipe &hp = pl->pipe;
    for (int i = 0; i < 2; ++i) {
        if (hp.dx[i]) cudaFree(hp.dx[i]);
        if (hp.dy[i]) cudaFree(hp.dy[i]);
        if (hp.dxr[i]) cudaFree(hp.dxr[i]);
        if (hp.dyr[i]) cudaFree(hp.dyr[i]);
        if (hp.ev_in[i]) cudaEventDestroy(hp.ev_in[i]);
        if (hp.ev_run[i]) cudaEventDestroy(hp.ev_run[i]);
        if (hp.ev_out[i]) cudaEventDestroy(hp.ev_out[i]);
    }
    for (int i = 0; i < 3; ++i) {
        if (hp.pin_in[i]) cudaFreeHost(hp.pin_in[i]);
        if (hp.pin_out[i]) cudaFreeHost(hp.pin_out[i]);
        if (hp.ev_ring_in[i]) cudaEventDestroy(hp.ev_ring_in[i]);
        if (hp.ev_ring_out[i]) cudaEventDestroy(hp.ev_ring_out[i]);
    }
    if (hp.ws) cudaFree(hp.ws);
    if (hp.d_starts) cudaFree(hp.d_starts);
    if (hp.d_lengths) cudaFree(hp.d_lengths);
    if (hp.s_in) cudaStreamDestroy(hp.s_in);
    if (hp.s_run) cudaStreamDestroy(hp.s_run);
    if (hp.s_out) cudaStreamDestroy(hp.s_out);
    delete pl;
}

size_t qd_plan_workspace_bytes_varlen(const qd_plan *pl, int64_t batch, int64_t span_samples) {
    if (!pl || batch <= 0 || span_samples < 0) return 0;
    const size_t bufs = pl->p.multiband ? 3 : 1;  // [x_dist] (+ [low][high]), packed like x
    const size_t frozen = pl->p.spectral_freeze ? (size_t)batch * (size_t)(pl->nc + pl->nc / 32) * sizeof(double) + 256 : 0;
    return bufs * padded_span(span_samples) * sizeof(float) + 256 + frozen + (size_t)batch * sizeof(float) + 256;   // + per-clip peaks
}

size_t qd_plan_workspace_bytes(const qd_plan *pl, int64_t batch) {
    if (!pl || batch <= 0) return 0;
    return qd_plan_workspace_bytes_varlen(pl, batch, (int64_t)pl->p.n_samples * batch);
}

int qd_plan_launches_per_render(const qd_plan *pl) {
    if (!pl) return 0;
    const qd_params &p = pl->p;
    int n = 0;
    if (p.multiband) n += 1;                        // crossover
    if (p.passthrough) return n + 1 + (p.multiband ? 1 : 0);
    if (p.no_spectral) return n + 2;                // distortion, limiter + mix
    if (p.pre_quant) n += 1;                        // pass A
    if (p.post_quant || !p.pre_quant) n += 1;       // pass B (or the bare STFT->iSTFT)
    n += 1;                                         // limiter + mix
    return n;
}

int qd_plan_enable_timing(qd_plan *pl, int on) {
    if (!pl) return fail(QD_ERR_INVALID_ARG, "null plan");
    pl->timing = on != 0;
    return QD_OK;
}

int qd_plan_read_timing(qd_plan *pl, double *ms, int64_t *launches) {
    if (!pl || !ms || !launches) return fail(QD_ERR_INVALID_ARG, "null argument");
    for (auto &sp : pl->stamps) {
        QD_CUDA(cudaEventSynchronize(sp.b));
        float t = 0.0f;
        QD_CUDA(cudaEventElapsedTime(&t, sp.a, sp.b));
        pl->t_ms[sp.cls] += (double)t;
        pl->t_launches[sp.cls] += 1;
        pl->free_events.push_back(sp.a);
        pl->free_events.push_back(sp.b);
    }
    pl->stamps.clear();
    for (int i = 0; i < QD_KERNEL_CLASSES; ++i) {
        ms[i] = pl->t_ms[i];
        launches[i] = pl->t_launches[i];
        pl->t_ms[i] = 0.0;
        pl->t_launches[i] = 0;
    }
    return QD_OK;
}

int qd_plan_set_fx_table(qd_plan *pl, const void *device_table, int64_t n_tables) {
    if (!pl) return fail(QD_ERR_INVALID_ARG, "null plan");
    pl->fx_table = device_table;
    pl->fx_tables = n_tables;
    return QD_OK;
}

}  // extern "C"

namespace {
// qd_render_device and qd_render_device_varlen: one render of `batch` clips packed as `pk` says (batch, span > 0)
int render_impl(qd_plan *pl, const float *x, float *y, const Packing &pk, int64_t batch, const qd_taps *taps,
                void *workspace, size_t workspace_bytes, void *stream) {
    if (workspace_bytes < qd_plan_workspace_bytes_varlen(pl, batch, pk.span) || !workspace)
        return fail(QD_ERR_WORKSPACE, "workspace too small (see qd_plan_workspace_bytes)");
    const qd_params &p = pl->p;
    if (p.fx_mode != QD_FX_NONE && (p.pre_quant || p.post_quant) && !p.passthrough) {
        const bool needs_table = p.fx_mode == QD_FX_SCRAMBLE_PICK || p.fx_mode == QD_FX_SCRAMBLE_SWAP ||
                                 (p.fx_mode == QD_FX_PHASE_DISPERSAL && p.fx_b != 0.0);
        if (needs_table && !pl->fx_table) return fail(QD_ERR_INVALID_ARG, "FX table missing (qd_plan_set_fx_table)");
        if (needs_table && p.fx_table_per_clip && pk.clip_offset + batch > pl->fx_tables)
            return fail(QD_ERR_INVALID_ARG, "per-clip FX table shorter than the batch");
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t count = (size_t)pk.span;   // elementwise kernels and tap copies run over the packed span
    const size_t stride = padded_span(pk.span);
    float *tap_pre = taps ? taps->pre_quant : nullptr;
    float *tap_dist = taps ? taps->post_dist : nullptr;
    float *w_a = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    float *w_low = w_a + stride;
    float *w_high = w_low + stride;
    void *frozen_ws = reinterpret_cast<void *>((reinterpret_cast<uintptr_t>(w_a + (p.multiband ? 3 : 1) * stride) + 255) & ~(uintptr_t)255);
    // per-clip peak of the limiter input, written by the spectral pass that produces it (behind the freeze scratch)
    const size_t frozen_bytes = p.spectral_freeze ? (size_t)batch * (size_t)(pl->nc + pl->nc / 32) * sizeof(double) + 256 : 0;
    float *clip_peak = reinterpret_cast<float *>((reinterpret_cast<uintptr_t>(frozen_ws) + frozen_bytes + 255) & ~(uintptr_t)255);
    if (!p.limiter_on) clip_peak = nullptr;
    int rc;

    const float *src = x;   // what the single-band chain sees (dsp/pipeline.py:1076: the high band)
    const float *low = nullptr;
    if (p.multiband) {
        qd::CrossoverArgs c{};
        c.x = x; c.low = w_low; c.high = w_high; c.n = (long long)pk.max_n;
        c.starts = pk.starts; c.lengths = pk.lengths;
        qd_host::fill_crossover(c, &p.sos_low[0][0], &p.sos_high[0][0]);
        c.low_delay = p.low_delay;
        c.process_low = 1;
        c.low_gain = p.low_gain; c.low_norm = p.low_norm;
        c.mono_a = p.mono_a; c.mono_b = p.mono_b; c.apply_mono = p.apply_mono_blend;
        c.low_trim = p.low_trim_gain; c.apply_low_trim = p.apply_low_trim;
        {
            TimeScope ts(pl, st, QD_KERNEL_CROSSOVER);
            launch_crossover(c, batch, st);
        }
        QD_CUDA(cudaGetLastError());
        src = w_high;
        low = w_low;
    }

    if (p.passthrough) {  // dsp/pipeline.py:477-535: no distortion, limiter or mix
        float *dst = p.multiband ? w_a : y;
        if ((rc = launch_spec(pl, pk, src, dst, nullptr, 0, 0, batch, st)) != QD_OK) return rc;
        if (tap_pre) QD_CUDA(cudaMemcpyAsync(tap_pre, src, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
        if (p.multiband) {
            qd::add_kernel<<<ew_grid((int64_t)count, pl->sm_count), 256, 0, st>>>(low, w_a, y, (long long)count);
            QD_CUDA(cudaGetLastError());
            if (tap_dist) QD_CUDA(cudaMemcpyAsync(tap_dist, y, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
        } else if (tap_dist) {
            QD_CUDA(cudaMemcpyAsync(tap_dist, y, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        if (p.delta_listen) {
            // output = input - processed (dsp/pipeline.py:1371-1375)
            qd::LimiterArgs d{};
            d.x = y; d.y = y; d.dry = y; d.orig = x; d.n = (long long)pk.max_n; d.limiter_on = 0; d.lookahead = 1;
            d.starts = pk.starts; d.lengths = pk.lengths;
            d.wet = 1.0f; d.dry_gain = 0.0f; d.apply_mix = 1;
            if ((rc = launch_limiter(d, batch, st)) != QD_OK) return rc;
        }
        return QD_OK;
    }

    const int epi = p.distortion_mode == QD_DIST_TUBE ? 2 : 1;
    const float *x_pq = nullptr;  // limiter input
    if (p.no_spectral) {
        // dsp/pipeline.py:537-601 with the pitch stage gated off: x_pre = band (:570), distortion (:580-588), no
        // spectral post-quantisation (:591), then the common tail (_finalize_single_band_output, :180-223)
        if (tap_pre) QD_CUDA(cudaMemcpyAsync(tap_pre, src, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
        qd::distort_kernel<<<ew_grid((int64_t)count, pl->sm_count), 256, 0, st>>>(
            src, w_a, (long long)count, p.distortion_mode, p.fold_amount, p.bias, p.tube_gain, p.tube_norm);
        QD_CUDA(cudaGetLastError());
        x_pq = w_a;
        clip_peak = nullptr;   // no spectral pass measured the limiter input
    } else if (p.pre_quant) {
        // pass A: STFT -> quantize -> iSTFT (= pre_quant tap) -> distortion        (:635-721)
        if ((rc = launch_spec(pl, pk, src, w_a, tap_pre, 1, epi, batch, st, 0, p.post_quant ? nullptr : clip_peak,
                              frozen_ws)) != QD_OK) return rc;
        if (p.post_quant) {  // pass B on the distorted signal                         (:729-801)
            if ((rc = launch_spec(pl, pk, w_a, y, nullptr, 1, 0, batch, st, 1, clip_peak, frozen_ws)) != QD_OK) return rc;
            x_pq = y;
        } else {
            x_pq = w_a;       // :851-853
        }
    } else {
        // distortion only reaches the tap (SURVEY.md appendix C.1, C.2)
        if (tap_pre) QD_CUDA(cudaMemcpyAsync(tap_pre, src, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
        if (tap_dist) {
            qd::distort_kernel<<<ew_grid((int64_t)count, pl->sm_count), 256, 0, st>>>(
                src, w_a, (long long)count, p.distortion_mode, p.fold_amount, p.bias, p.tube_gain, p.tube_norm);
            QD_CUDA(cudaGetLastError());
        }
        if ((rc = launch_spec(pl, pk, src, y, nullptr, p.post_quant ? 1 : 0, 0, batch, st, 0, clip_peak, frozen_ws)) != QD_OK) return rc;
        x_pq = y;
    }
    if (tap_dist) {  // dsp/pipeline.py:916 / :1107 (low band added in multiband mode)
        if (low) {
            qd::add_kernel<<<ew_grid((int64_t)count, pl->sm_count), 256, 0, st>>>(low, w_a, tap_dist, (long long)count);
            QD_CUDA(cudaGetLastError());
        } else {
            QD_CUDA(cudaMemcpyAsync(tap_dist, w_a, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
    }
    qd::LimiterArgs l{};
    l.x = x_pq; l.dry = src; l.low = low; l.orig = p.delta_listen ? x : nullptr; l.y = y; l.n = (long long)pk.max_n;
    l.starts = pk.starts; l.lengths = pk.lengths;
    l.limiter_on = p.limiter_on; l.lookahead = p.lookahead > 0 ? p.lookahead : 1;
    l.ceiling = p.ceiling_lin; l.c = p.release_coeff;
    l.wet = p.wet; l.dry_gain = p.dry; l.trim = p.trim_gain; l.apply_trim = p.apply_trim; l.apply_mix = 1;
    l.clip_peak = clip_peak;   // written by the spectral pass that produced x_pq
    TimeScope ts(pl, st, QD_KERNEL_LIMITER);
    return launch_limiter(l, batch, st);
}
}  // namespace

extern "C" {

int qd_render_device(qd_plan *pl, const float *x, float *y, int64_t batch, const qd_taps *taps,
                     void *workspace, size_t workspace_bytes, void *stream) {
    if (!pl || !x || !y || batch < 0) return fail(QD_ERR_INVALID_ARG, "null argument");
    if (batch > INT32_MAX) return fail(QD_ERR_INVALID_ARG, "batch of more than 2^31 - 1 clips");
    if (batch == 0 || pl->p.n_samples == 0) return QD_OK;
    Packing pk;
    pk.span = (int64_t)pl->p.n_samples * batch;
    pk.max_n = pl->p.n_samples;
    return render_impl(pl, x, y, pk, batch, taps, workspace, workspace_bytes, stream);
}

int qd_render_device_varlen(qd_plan *pl, const float *x, float *y, const int64_t *starts, const int32_t *lengths,
                            int64_t batch, int64_t span_samples, int32_t max_samples, const qd_taps *taps,
                            void *workspace, size_t workspace_bytes, void *stream) {
    if (!pl || !x || !y || !starts || !lengths || batch < 0 || span_samples < 0 || max_samples < 0)
        return fail(QD_ERR_INVALID_ARG, "null / negative argument");
    if (max_samples > pl->p.n_samples) return fail(QD_ERR_INVALID_ARG, "max_samples exceeds the plan's n_samples");
    if (batch > INT32_MAX) return fail(QD_ERR_INVALID_ARG, "ragged batch of more than 2^31 - 1 clips");
    if (batch == 0 || span_samples == 0 || max_samples == 0) return QD_OK;
    Packing pk;
    pk.starts = starts;
    pk.lengths = lengths;
    pk.span = span_samples;
    pk.max_n = max_samples;
    return render_impl(pl, x, y, pk, batch, taps, workspace, workspace_bytes, stream);
}

int qd_limiter_device(const float *x, float *y, int64_t batch, int64_t n, int32_t lookahead, double ceiling_lin,
                      double release_coeff, void *stream) {
    if (!x || !y || batch < 0 || n < 0 || lookahead < 1) return fail(QD_ERR_INVALID_ARG, "bad limiter argument");
    if (batch > INT32_MAX) return fail(QD_ERR_INVALID_ARG, "batch of more than 2^31 - 1 clips");
    if (batch == 0 || n == 0) return QD_OK;
    qd::LimiterArgs a{};
    a.x = x; a.y = y; a.n = (long long)n; a.limiter_on = 1; a.lookahead = lookahead;
    a.ceiling = ceiling_lin; a.c = release_coeff; a.apply_mix = 0;
    return launch_limiter(a, batch, (cudaStream_t)stream);
}

int qd_crossover_device(const float *x, float *low, float *high, int64_t batch, int64_t n,
                        const double sos_low[2][6], const double sos_high[2][6], void *stream) {
    if (!x || !low || !high || !sos_low || !sos_high || batch < 0 || n < 0) return fail(QD_ERR_INVALID_ARG, "bad crossover argument");
    if (batch > INT32_MAX) return fail(QD_ERR_INVALID_ARG, "batch of more than 2^31 - 1 clips");
    if (batch == 0 || n == 0) return QD_OK;
    qd::CrossoverArgs c{};
    c.x = x; c.low = low; c.high = high; c.n = (long long)n;
    qd_host::fill_crossover(c, &sos_low[0][0], &sos_high[0][0]);
    launch_crossover(c, batch, (cudaStream_t)stream);
    QD_CUDA(cudaGetLastError());
    return QD_OK;
}

int qd_distort_device(const float *x, float *y, int64_t count, int32_t mode, double fold_amount, double bias,
                      float tube_gain, float tube_norm, void *stream) {
    if (!x || !y || count < 0) return fail(QD_ERR_INVALID_ARG, "bad distortion argument");
    if (mode != QD_DIST_WAVEFOLD && mode != QD_DIST_TUBE) return fail(QD_ERR_INVALID_ARG, "unsupported distortion mode");
    if (count == 0) return QD_OK;
    int sm = 148;
    qd::distort_kernel<<<ew_grid(count, sm), 256, 0, (cudaStream_t)stream>>>(x, y, (long long)count, mode, fold_amount,
                                                                               bias, tube_gain, tube_norm);
    QD_CUDA(cudaGetLastError());
    return QD_OK;
}

void *qd_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void qd_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

}  // extern "C"

#include "qd_autotune_api.inc"
#include "qd_host_pipe.inc"
