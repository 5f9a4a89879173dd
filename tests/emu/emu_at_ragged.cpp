// tests/emu/emu_at_ragged.cpp -- TEST INFRASTRUCTURE: runs the autotune_v1 kernels on the CPU through cuda_emu.h, one
// stage at a time on a given input, uniform (one clip) or a ragged batch (per-clip starts / lengths).
// tests/test_emu_ragged_autotune.py compares every clip of a packed batch with the same clip run alone,
// tests/test_emu_autotune_stages.py compares every stage with oracle/qd_autotune.py fed the same input.
//
//   emu_at_ragged yin <frame_size> <hop> <max_tau> <cols> <x.f32> <starts.i64|-> <lengths.i32|-> <diff.f64>
//   emu_at_ragged filt <sos.f64: jobs x 2 x 6> <zi.f64: jobs x 2 x 2> <x.f32> <starts|-> <lengths|-> <y.f32: jobs x span>
//   emu_at_ragged stats <hop> <min_tau> <max_tau> <det.f32> <starts|-> <lengths|-> <feat.f64: rows x 4>
//   emu_at_ragged pick <sr> <min_tau> <max_tau> <min_freq> <max_freq> <threshold> <diff.f64: rows x stride>
//                      <feat.f64: rows x 4> <feat_out.f64>
//   emu_at_ragged hold <n> <hop> <root_pc> <intervals, comma-separated> <strength> <rms_thr> <flat_thr> <conf_thr>
//                      <change_cents> <confirm> <release> <feat.f64: rows x 4> <starts|-> <lengths|-> <ratio.f64: rows>
//   emu_at_ragged shift <hop> <half> <max_delay> <buf_size> <body.f32> <starts|-> <lengths|-> <ratio.f64: rows>
//                       <corrected.f32> <ratio_track.f32> <flat.i32: batch>
//   emu_at_ragged env <att> <rel> <tile> <halo> <seg_min> <x.f32> <starts|-> <lengths|-> <env.f32> <env_max.f32: batch>
//   emu_at_ragged mix <sub_enabled> <layer_on> <att> <rel> <tile> <halo> <seg_min> <level> <preserve> <air_mix>
//                     <phase_k> <sr> <x.f32> <sub.f32> <air.f32> <corrected.f32> <starts|-> <lengths|-> <y.f32>
//                     <sub_layer.f32>
// With "-" for starts / lengths x is one clip (the uniform path); otherwise x is packed and the batch is len(starts).
// Frame rows (stats / pick / hold / shift) are laid out as the library lays them out (qd::at_row0); feat and ratio rows
// no clip owns keep their initial value.  Every mode launches the production kernels with the production block shapes
// (qd_autotune_api.inc: at_render); the filter bank takes its tiles from the poles like the library
// (qd_host::segment_tiling, qd::at_filt_tile), the frame stats the library's FFT tables and Hann window (at_tables).
// `hold` and `stats` take the clip length from `n` / the x file when uniform; `n` is ignored for a ragged batch.
#include "cuda_emu.h"

namespace qd_emu {
thread_local Block *g_blk = nullptr;
thread_local dim3 g_tid, g_bid;
}  // namespace qd_emu

#include "cuda_emu_at.h"
#include "../../quantumdistortion_b200/csrc/qd_autotune.cuh"
#include "../../quantumdistortion_b200/csrc/qd_host_time.hpp"
#include "../../quantumdistortion_b200/csrc/qd_host_tables.hpp"

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>

template <class T>
static std::vector<T> read_all(const char *path) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f) { std::cerr << "cannot open " << path << "\n"; std::exit(2); }
    const size_t bytes = (size_t)f.tellg();
    f.seekg(0);
    std::vector<T> v(bytes / sizeof(T));
    f.read(reinterpret_cast<char *>(v.data()), (std::streamsize)(v.size() * sizeof(T)));
    return v;
}
template <class T>
static void write_all(const char *path, const std::vector<T> &v) {
    std::ofstream(path, std::ios::binary).write(reinterpret_cast<const char *>(v.data()), (std::streamsize)(v.size() * sizeof(T)));
}

struct Batch {
    std::vector<float> x;
    std::vector<int64_t> starts;
    std::vector<int32_t> lengths;
    bool ragged;
    long long n_max, span;
    int batch;
};
static Batch load(const char *xp, const char *sp, const char *lp) {
    Batch b;
    b.x = read_all<float>(xp);
    b.ragged = std::string(sp) != "-";
    b.span = (long long)b.x.size();
    if (b.ragged) {
        b.starts = read_all<int64_t>(sp);
        b.lengths = read_all<int32_t>(lp);
        b.batch = (int)b.starts.size();
        b.n_max = *std::max_element(b.lengths.begin(), b.lengths.end());
    } else {
        b.batch = 1;
        b.n_max = b.span;
    }
    return b;
}
// the clips alone (no samples): uniform one clip of n samples, or a ragged batch
static Batch load_clips(long long n, const char *sp, const char *lp) {
    Batch b;
    b.ragged = std::string(sp) != "-";
    if (b.ragged) {
        b.starts = read_all<int64_t>(sp);
        b.lengths = read_all<int32_t>(lp);
        b.batch = (int)b.starts.size();
        b.n_max = *std::max_element(b.lengths.begin(), b.lengths.end());
        b.span = b.starts.back() - b.starts[0] + b.lengths.back();
    } else {
        b.batch = 1;
        b.n_max = b.span = n;
    }
    return b;
}
template <class A>
static void set_clips(A &a, const Batch &b) {
    a.n = b.n_max;
    a.starts = b.ragged ? b.starts.data() : nullptr;
    a.lengths = b.ragged ? b.lengths.data() : nullptr;
    a.clip0 = 0;
}
// rows of a per-clip table with one row per `unit` samples (at_layout)
static long long table_rows(const Batch &b, int unit) {
    return b.ragged ? b.span / unit + b.batch : qd::at_rows(b.n_max, unit);
}
static double num(const char *s) { return std::strtod(s, nullptr); }

// the envelope follower(s) as at_render chooses them: the segment kernel for clips of at least seg_min samples, one warp
// per clip for the others; env_max zeroed first
static void run_env(qd::AtMixArgs &m, const Batch &b, int tile, int halo) {
    std::fill(m.env_max, m.env_max + b.batch, 0.0f);
    if (b.n_max >= m.seg_min) {
        const long long n_tiles = (b.n_max + tile - 1) / tile;
        const unsigned gx = (unsigned)((n_tiles + 32 * qd::AT_SW - 1) / (32 * qd::AT_SW));
        qd_emu::launch(dim3(gx, b.batch, 1), dim3(32 * qd::AT_SW), 0, [&] { qd::at_env_seg_kernel(m, tile, halo); });
    }
    if (b.ragged || b.n_max < m.seg_min)
        qd_emu::launch(dim3((b.batch + qd::AT_FW - 1) / qd::AT_FW), dim3(32 * qd::AT_FW), 0, [&] { qd::at_env_kernel(m); });
}

int main(int argc, char **argv) {
    if (argc < 2) { std::cerr << "usage: see source\n"; return 2; }
    const std::string mode = argv[1];
    if (mode == "yin" && argc == 10) {
        const Batch b = load(argv[6], argv[7], argv[8]);
        qd::AtYinArgs a{};
        set_clips(a, b);
        a.frame_size = std::atoi(argv[2]); a.hop = std::atoi(argv[3]); a.max_tau = std::atoi(argv[4]);
        constexpr int L = qd::AT_YL;
        const int total_cols = (a.max_tau + L - 1) / L;
        a.lag_threads = std::min(std::min(std::atoi(argv[5]), total_cols), (int)qd::AT_YC);
        const int tblocks = (total_cols + a.lag_threads - 1) / a.lag_threads;
        a.frames = (int)qd::at_rows(a.n, a.hop);
        a.stride = (a.max_tau + 2) & ~1;
        const long long rows = b.ragged ? b.span / a.hop + b.batch : qd::at_rows(a.n, a.hop);
        std::vector<double> diff((size_t)rows * a.stride, -1.0);
        a.det = b.x.data(); a.diff = diff.data();
        const size_t smem = qd::at_yin_smem_doubles(a.hop, (tblocks - 1) * a.lag_threads, a.lag_threads) * sizeof(double) + 128;
        qd_emu::launch(dim3(tblocks, b.batch, 1), dim3(qd::AT_YT), smem, [&] { qd::at_yin_diff_kernel(a); });
        write_all(argv[9], diff);
        return 0;
    }
    if (mode == "filt" && argc == 8) {
        const std::vector<double> sos = read_all<double>(argv[2]), zi = read_all<double>(argv[3]);
        const int jobs = (int)(sos.size() / 12);
        const Batch b = load(argv[4], argv[5], argv[6]);
        qd::AtFiltSegArgs q{};
        qd::AtFiltArgs &a = q.base;
        set_clips(a, b);
        a.jobs = jobs;
        std::vector<float> y((size_t)jobs * b.span, 0.0f);
        std::vector<double> scratch((size_t)jobs * (b.span + 2 * qd::AT_EDGE * b.batch), 0.0);
        a.scratch = scratch.data();
        a.scratch_job = b.span + 2LL * qd::AT_EDGE * b.batch;
        long long tiles = 1;
        const long long m = b.n_max + 2 * qd::AT_EDGE;
        for (int j = 0; j < jobs; ++j) {
            a.f[j].on = 1;
            std::memcpy(a.f[j].sos, &sos[12 * j], sizeof(a.f[j].sos));
            std::memcpy(a.f[j].zi, &zi[4 * j], sizeof(a.f[j].zi));
            a.x[j] = b.x.data();
            a.y[j] = y.data() + (size_t)j * b.span;
            qd_host::segment_tiling(qd_host::sos_pole_radius(&a.f[j].sos[0][0], 2), &q.tile[j], &q.halo[j]);
            tiles = std::max(tiles, qd::at_rows(m, qd::at_filt_tile(q.tile[j], q.halo[j], m)));
        }
        const unsigned gx = (unsigned)((tiles + 32 * qd::AT_SW - 1) / (32 * qd::AT_SW));
        qd_emu::launch(dim3(gx, b.batch, jobs), dim3(32 * qd::AT_SW), 0, [&] { qd::at_filt_seg_kernel<false>(q); });
        qd_emu::launch(dim3(gx, b.batch, jobs), dim3(32 * qd::AT_SW), 0, [&] { qd::at_filt_seg_kernel<true>(q); });
        write_all(argv[7], y);
        return 0;
    }
    if (mode == "stats" && argc == 9) {
        const Batch b = load(argv[5], argv[6], argv[7]);
        constexpr int FS = 4096, NC = FS / 2;
        qd_host::SpecTablesT<float> st;
        if (!qd_host::build_spec_tables<float>(FS, &st)) { std::cerr << "fft tables\n"; return 2; }
        std::vector<float> hann(FS);   // np.hanning: symmetric (at_tables)
        for (int i = 0; i < FS; ++i) hann[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * (double)i / (double)(FS - 1)));
        qd::AtDetArgs d{};
        set_clips(d, b);
        d.batch = b.batch;
        d.frame_size = FS; d.hop = std::atoi(argv[2]);
        d.min_tau = std::atoi(argv[3]); d.max_tau = std::atoi(argv[4]);
        const long long rows = table_rows(b, d.hop);
        std::vector<double> feat((size_t)rows * 4, -1.0);
        d.det = b.x.data(); d.feat = feat.data(); d.hann = hann.data();
        d.tw1 = reinterpret_cast<const float2 *>(st.tw1.data());
        d.tw2 = reinterpret_cast<const float2 *>(st.tw2.data());
        d.wsplit = reinterpret_cast<const float2 *>(st.wsplit.data());
        const size_t smem = (size_t)qd::AT_SW_STATS * qd::buf_slots<NC>() * sizeof(float2) + 64;
        qd_emu::launch(dim3((unsigned)((rows + qd::AT_SW_STATS - 1) / qd::AT_SW_STATS)), dim3(32 * qd::AT_SW_STATS), smem,
                       [&] { qd::at_frame_stats_kernel<NC>(d, rows); });
        write_all(argv[8], feat);
        return 0;
    }
    if (mode == "pick" && argc == 11) {
        qd::AtYinArgs a{};
        a.sr = num(argv[2]); a.min_tau = std::atoi(argv[3]); a.max_tau = std::atoi(argv[4]);
        a.min_freq = num(argv[5]); a.max_freq = num(argv[6]); a.threshold = num(argv[7]);
        a.stride = (a.max_tau + 2) & ~1;
        std::vector<double> diff = read_all<double>(argv[8]), feat = read_all<double>(argv[9]);
        a.total_frames = (long long)(feat.size() / 4);
        if ((long long)diff.size() != a.total_frames * a.stride) { std::cerr << "diff rows\n"; return 2; }
        a.diff = diff.data(); a.feat = feat.data();
        const size_t smem = (size_t)8 * a.stride * sizeof(double) + 64;
        qd_emu::launch(dim3((unsigned)((a.total_frames + 7) / 8)), dim3(256), smem, [&] { qd::at_yin_pick_kernel(a); });
        write_all(argv[10], feat);
        return 0;
    }
    if (mode == "hold" && argc == 17) {
        const Batch b = load_clips(std::atoll(argv[2]), argv[14], argv[15]);
        qd::AtHoldArgs h{};
        set_clips(h, b);
        h.batch = b.batch; h.hop = std::atoi(argv[3]); h.root_pc = std::atoi(argv[4]);
        std::stringstream iv(argv[5]);
        for (std::string tok; std::getline(iv, tok, ',') && h.n_intervals < 8;) h.intervals[h.n_intervals++] = std::atoi(tok.c_str());
        h.strength = num(argv[6]); h.rms_thr = num(argv[7]); h.flat_thr = num(argv[8]); h.conf_thr = num(argv[9]);
        h.change_cents = num(argv[10]); h.confirm_frames = std::atoi(argv[11]); h.release_frames = std::atoi(argv[12]);
        const std::vector<double> feat = read_all<double>(argv[13]);
        h.total_frames = (long long)(feat.size() / 4);
        if (h.total_frames != table_rows(b, h.hop)) { std::cerr << "feat rows\n"; return 2; }
        std::vector<double> ratio((size_t)h.total_frames, -1.0);
        h.feat = feat.data(); h.ratio = ratio.data();
        qd_emu::launch(dim3((unsigned)((h.total_frames + 255) / 256)), dim3(256), 0, [&] { qd::at_target_kernel(h); });
        qd_emu::launch(dim3((unsigned)((b.batch + 31) / 32)), dim3(32), 0, [&] { qd::at_hold_kernel(h); });
        write_all(argv[16], ratio);
        return 0;
    }
    if (mode == "shift" && argc == 13) {
        const Batch b = load(argv[6], argv[7], argv[8]);
        qd::AtShiftArgs s{};
        set_clips(s, b);
        s.hop = std::atoi(argv[2]); s.half = std::atoi(argv[3]); s.max_delay = std::atoi(argv[4]); s.buf_size = std::atoi(argv[5]);
        const std::vector<double> ratio = read_all<double>(argv[9]);
        if ((long long)ratio.size() != table_rows(b, s.hop)) { std::cerr << "ratio rows\n"; return 2; }
        std::vector<long long> tile_sum((size_t)table_rows(b, qd::AT_TS), 0);
        std::vector<float> out((size_t)b.span, -7.0f), track((size_t)b.span, -7.0f);
        std::vector<int> flag((size_t)b.batch, 0);   // zeroed before the launch, as in at_render
        s.body = b.x.data(); s.ratio = ratio.data(); s.tile_sum = tile_sum.data();
        s.ratio_track = track.data(); s.flat_flag = flag.data(); s.out = out.data();
        const unsigned gx = (unsigned)((qd::at_rows(b.n_max, qd::AT_TS) + qd::AT_TW - 1) / qd::AT_TW);
        qd_emu::launch(dim3(gx, b.batch, 1), dim3(32 * qd::AT_TW), 0, [&] { qd::at_tap_sums_kernel(s); });
        qd_emu::launch(dim3(b.batch), dim3(32), 0, [&] { qd::at_tap_scan_kernel(s); });
        qd_emu::launch(dim3(gx, b.batch, 1), dim3(32 * qd::AT_TW), 0, [&] { qd::at_shift_kernel(s); });
        write_all(argv[10], out);
        write_all(argv[11], track);
        write_all(argv[12], flag);
        return 0;
    }
    if (mode == "env" && argc == 12) {
        const Batch b = load(argv[7], argv[8], argv[9]);
        qd::AtMixArgs m{};
        set_clips(m, b);
        m.batch = b.batch;
        m.att = (float)num(argv[2]); m.rel = (float)num(argv[3]);
        m.seg_min = std::atoll(argv[6]);
        std::vector<float> env((size_t)b.span, -7.0f), emax((size_t)b.batch, -7.0f);
        m.x = b.x.data(); m.env = env.data(); m.env_max = emax.data();
        run_env(m, b, std::atoi(argv[4]), std::atoi(argv[5]));
        write_all(argv[10], env);
        write_all(argv[11], emax);
        return 0;
    }
    if (mode == "mix" && argc == 22) {
        const Batch b = load(argv[14], argv[18], argv[19]);
        const std::vector<float> sub = read_all<float>(argv[15]), air = read_all<float>(argv[16]), corr = read_all<float>(argv[17]);
        if ((long long)sub.size() != b.span || (long long)air.size() != b.span || (long long)corr.size() != b.span) {
            std::cerr << "band sizes\n";
            return 2;
        }
        qd::AtMixArgs m{};
        set_clips(m, b);
        m.batch = b.batch;
        m.sub_enabled = std::atoi(argv[2]); m.layer_on = std::atoi(argv[3]);
        m.att = (float)num(argv[4]); m.rel = (float)num(argv[5]);
        m.seg_min = std::atoll(argv[8]);
        m.level = (float)num(argv[9]); m.preserve = (float)num(argv[10]); m.air_mix = (float)num(argv[11]);
        m.phase_k = (float)num(argv[12]); m.sr_f = (float)num(argv[13]);
        std::vector<float> env((size_t)b.span, -7.0f), emax((size_t)b.batch, -7.0f);
        std::vector<float> y((size_t)b.span, -7.0f), layer((size_t)b.span, -7.0f);
        m.x = b.x.data(); m.sub = sub.data(); m.air = air.data(); m.corrected = corr.data();
        m.env = env.data(); m.env_max = emax.data(); m.sub_layer = layer.data(); m.y = y.data();
        if (m.layer_on) run_env(m, b, std::atoi(argv[6]), std::atoi(argv[7]));
        const unsigned gx = (unsigned)std::min<long long>((b.n_max + 255) / 256, 1024);
        qd_emu::launch(dim3(gx, b.batch, 1), dim3(256), 0, [&] { qd::at_mix_kernel(m); });
        write_all(argv[20], y);
        write_all(argv[21], layer);
        return 0;
    }
    std::cerr << "usage: see source\n";
    return 2;
}
