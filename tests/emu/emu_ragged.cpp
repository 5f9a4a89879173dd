// tests/emu/emu_ragged.cpp -- TEST INFRASTRUCTURE: runs the kernels of a ragged batch (per-clip starts / lengths) on the
// CPU through cuda_emu.h, so that tests/test_emu_ragged.py can compare every clip with the same clip rendered alone.
//
//   emu_ragged [-p <clips per launch>] [-q] [-x] <mode> ...
//   emu_ragged spec <f32|f64> <n_fft> <nw> <tile_blocks> <quant> <x.f32> <starts.i64|-> <lengths.i32|-> <tb.i32> <mask.u8> <y.f32>
//       nw = 16: the two-group kernel of n_fft 2048 (NG = 2); nw >= 100: team kernel, 100 * frames + warps per frame.
//       Also writes <y>.peak: the per-clip peaks (clip_peak) and two rows no clip owns.
//   emu_ragged limiter <lookahead> <x.f32> <starts|-> <lengths|-> <y.f32>
//   emu_ragged crossover <low_delay> <sos_lp.f64> <sos_hp.f64> <tile> <halo> <x.f32> <starts|-> <lengths|-> <low.f32> <high.f32>
// With "-" for starts / lengths x is one clip (the uniform path), with "u<B>" B uniform clips of len(x) / B samples;
// otherwise x is packed and the batch is len(starts).  -p splits the batch into launches of that many clips with
// qd::for_each_launch, as the library does at its grid limits (default: one launch).  -q: the limiter reads per-clip
// peaks that mark every odd clip quiet.  -x (spec, n_fft 1024, nw 4): the FX kernel with a per-clip bin-scramble table
// (clip 0 at row 1, as in a chunk of a host render) and the spectral freeze (freeze_mag_kernel in one launch).
#include "cuda_emu.h"

namespace qd_emu {
thread_local Block *g_blk = nullptr;
thread_local dim3 g_tid, g_bid;
}  // namespace qd_emu

#include "../../quantumdistortion_b200/csrc/qd_host_tables.hpp"
#include "../../quantumdistortion_b200/csrc/qd_spec.cuh"
#include "../../quantumdistortion_b200/csrc/qd_spec_team.cuh"
#include "../../quantumdistortion_b200/csrc/qd_time.cuh"
#include "../../quantumdistortion_b200/csrc/qd_host_time.hpp"

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <fstream>
#include <iostream>
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

static int64_t g_per_launch = INT32_MAX;
static bool g_quiet_odd = false, g_fx = false;

// batch layout: uniform (B clips of len(x) / B samples) or the ragged arrays
struct Layout {
    std::vector<int64_t> starts;
    std::vector<int32_t> lengths;
    int batch = 1, max_n = 0;
    bool ragged = false;
};
static Layout layout(const char *sp, const char *lp, size_t x_size) {
    Layout l;
    if (sp[0] == '-' || sp[0] == 'u') {
        if (sp[0] == 'u') l.batch = std::atoi(sp + 1);
        l.max_n = (int)(x_size / l.batch);
        return l;
    }
    l.ragged = true;
    l.starts = read_all<int64_t>(sp);
    l.lengths = read_all<int32_t>(lp);
    l.batch = (int)l.starts.size();
    for (int32_t n : l.lengths) l.max_n = std::max(l.max_n, (int)n);
    return l;
}
template <class A>
static void apply(A &a, const Layout &l) {
    a.n = l.max_n;
    if (l.ragged) { a.starts = l.starts.data(); a.lengths = l.lengths.data(); }
}

template <class T>
static int spec(int argc, char **argv) {
    using T2 = qd::V2<T>;
    const int n_fft = std::atoi(argv[3]), nw = std::atoi(argv[4]), tile_blocks = std::atoi(argv[5]), quant = std::atoi(argv[6]);
    const std::vector<float> x = read_all<float>(argv[7]);
    const Layout l = layout(argv[8], argv[9], x.size());
    const std::vector<int32_t> tb = read_all<int32_t>(argv[10]);
    const std::vector<uint8_t> mask = read_all<uint8_t>(argv[11]);
    (void)argc;
    qd_host::SpecTablesT<T> st;
    if (!qd_host::build_spec_tables<T>(n_fft, &st)) { std::cerr << "unsupported n_fft\n"; return 2; }
    double kw[5], ks = 0;   // the 5-tap smear kernel (dsp/quantizer.py:460-465)
    for (int i = 0; i < 5; ++i) { kw[i] = std::exp(-0.5 * (i - 2) * (i - 2)); ks += kw[i]; }
    for (int i = 0; i < 5; ++i) kw[i] /= ks;
    qd_tables ht{};
    ht.n_bins = n_fft / 2 + 1;
    ht.target_bins = tb.data();
    ht.active_mask = mask.data();
    ht.snap = 0.8;
    ht.smear = 0.3;
    ht.smear_radius = 2;
    ht.smear_w = kw;
    qd_host::QuantTablesH qt;
    std::string err;
    if (!qd_host::build_quant_tables(ht, &qt, &err, sizeof(T) == 8)) { std::cerr << err << "\n"; return 2; }
    std::vector<float> y(x.size(), -777.0f);
    std::vector<float> peak((size_t)l.batch + 2, 0.0f);   // zeroed by the caller, as in launch_spec_prec
    qd::SpecArgsT<T> a{};
    a.x = x.data();
    a.y = y.data();
    a.clip_peak = peak.data();
    apply(a, l);
    a.n_frames = 1 + a.n / st.hop;
    a.tile_blocks = tile_blocks;
    a.quant = quant;
    a.epilogue = 1; a.fold = 2.0; a.bias = 0.0; a.fold_exact_f32 = 1;
    a.wtab = reinterpret_cast<const T2 *>(st.wtab.data());
    a.tw1 = reinterpret_cast<const T2 *>(st.tw1.data());
    a.tw2 = reinterpret_cast<const T2 *>(st.tw2.data());
    a.wsplit = reinterpret_cast<const T2 *>(st.wsplit.data());
    a.invw = st.invw.data();
    a.q.n_slots = qt.n_slots;
    a.q.n_src = (int)qt.src_tab.size();
    a.q.row_limit = qt.row_limit;
    a.q.src_tab = qt.src_tab.data();
    a.q.row_active = qt.row_active.data();
    a.q.slot_of_bin = qt.slot_of_bin.data();
    a.q.slot_invk = qt.slot_invk.data();
    a.q.slot_base = qt.slot_base.data();
    for (int e = 0; e < 5; ++e) a.q.tap[e] = qt.tap[e];
    a.q.keep_active = qt.keep_active;
    a.q.smoothing = 1;
    a.fx.table_frames = 1;
    const int tiles = std::max(1, ((a.n + st.hop - 1) / st.hop + tile_blocks - 1) / tile_blocks);   // the longest clip
    const int nc = n_fft / 2;
    // one launch per range of clips; clips_per_cta = NG
    auto each = [&](int clips_per_cta, auto kern) {
        qd::for_each_launch(l.batch, g_per_launch, [&](int clip0, int nb) {
            a.clip0 = clip0;
            a.batch = nb;
            kern((nb + clips_per_cta - 1) / clips_per_cta);
        });
        write_all(argv[12], y);
        write_all((std::string(argv[12]) + ".peak").c_str(), peak);
    };
    if (nw >= 100) {
        const int nf = nw / 100, cw = nw % 100;
        std::vector<uint32_t> ttab;
        qd::TeamGather tg{};
        qd_host::build_team_gather(qt, cw, &ttab, tg.begin);
        tg.src_tab = ttab.data();
#define QD_TEAMCASE(NC_, NF_, CW_)                                                                                       \
        if (nc == NC_ && nf == NF_ && cw == CW_) {                                                                       \
            each(1, [&](int rows) {                                                                                       \
                qd_emu::launch(dim3(tiles, rows, 1), dim3(32 * NF_ * CW_, 1, 1), qd::SpecSmem<T, NC_, NF_>::bytes(qt.n_slots), \
                               [&] { qd::spec_pass_team_kernel<T, NC_, NF_, CW_>(a, tg); });                                \
            });                                                                                                           \
            return 0;                                                                                                     \
        }
        QD_TEAMCASE(512, 8, 1) QD_TEAMCASE(2048, 2, 2)
        std::cerr << "no team instantiation\n";
        return 2;
    }
    if (nc == 1024 && nw == 16) {   // two clip groups per CTA, tables in shared memory (the headline kernel's shape)
        each(2, [&](int rows) {
            qd_emu::launch(dim3(tiles, rows, 1), dim3(32 * 16, 1, 1), qd::SpecSmem<T, 1024, 8, 2>::bytes(qt.n_slots, true, a.q.n_src, 0),
                           [&] { qd::spec_pass_kernel<T, 1024, 8, true, false, 2>(a); });
        });
    } else if (nc == 512 && nw == 4 && g_fx) {
        constexpr int NC = 512, BUF = qd::buf_slots<NC>();
        std::vector<int16_t> table((size_t)(l.batch + 1) * 2 * a.n_frames * (NC + 1));
        uint32_t r = 12345;   // source bins of the scramble: any bin 0 .. NC
        for (int16_t &v : table) { r = r * 1664525u + 1013904223u; v = (int16_t)((r >> 8) % (NC + 1)); }
        a.fx.mode = 4;
        a.fx.table = table.data();
        a.fx.table_frames = a.n_frames;
        a.fx.table_per_clip = 1;
        a.fx.clip_offset = 1;
        std::vector<T> frozen((size_t)l.batch * BUF);
        qd_emu::launch(dim3(l.batch), dim3(32), (size_t)BUF * sizeof(T2) + (size_t)2 * NC * sizeof(float) + 16,
                       [&] { qd::freeze_mag_kernel<T, NC>(a, frozen.data()); });
        a.frozen = frozen.data();
        each(1, [&](int rows) {
            qd_emu::launch(dim3(tiles, rows, 1), dim3(32 * 4, 1, 1), qd::SpecSmem<T, NC, 4>::bytes(qt.n_slots, false, 0, 0, true, false),
                           [&] { qd::spec_pass_kernel<T, NC, 4, false, true>(a); });
        });
    } else if (nc == 512 && nw == 4) {
        each(1, [&](int rows) {
            qd_emu::launch(dim3(tiles, rows, 1), dim3(32 * 4, 1, 1), qd::SpecSmem<T, 512, 4>::bytes(qt.n_slots),
                           [&] { qd::spec_pass_kernel<T, 512, 4>(a); });
        });
    } else {
        std::cerr << "no instantiation\n";
        return 2;
    }
    return 0;
}

int main(int argc, char **argv) {
    for (;;) {
        const std::string opt = argc > 1 ? argv[1] : "";
        const int used = opt == "-p" ? 2 : (opt == "-q" || opt == "-x") ? 1 : 0;
        if (!used) break;
        if (opt == "-p") g_per_launch = std::atoll(argv[2]);
        g_quiet_odd |= opt == "-q";
        g_fx |= opt == "-x";
        argv += used;
        argc -= used;
    }
    const std::string mode = argc > 1 ? argv[1] : "";
    if (mode == "spec" && argc == 13) return std::string(argv[2]) == "f64" ? spec<double>(argc, argv) : spec<float>(argc, argv);
    if (mode == "limiter" && argc == 7) {
        const std::vector<float> x = read_all<float>(argv[3]);
        const Layout l = layout(argv[4], argv[5], x.size());
        std::vector<float> y(x.size(), -777.0f);
        qd::LimiterArgs a{};
        a.x = x.data(); a.y = y.data();
        apply(a, l);
        a.limiter_on = 1; a.lookahead = std::atoi(argv[2]); a.ceiling = 0.5; a.c = 0.999;
        a.apply_mix = 0;
        std::vector<float> peak;   // -q: odd clips quiet (skipped, y = x), even clips loud
        if (g_quiet_odd) {
            for (int i = 0; i < l.batch; ++i) peak.push_back(i % 2 ? 0.0f : 1e9f);
            a.clip_peak = peak.data();
        }
        qd::for_each_launch(l.batch, g_per_launch, [&](int clip0, int nb) {
            a.clip0 = clip0;
            qd_emu::launch(dim3(nb), dim3(qd::QD_TT), qd_host::limiter_smem_bytes(a.lookahead), [&] { qd::limiter_mix_kernel(a); });
        });
        write_all(argv[6], y);
        return 0;
    }
    if (mode == "crossover" && argc == 12) {
        const std::vector<double> lp = read_all<double>(argv[3]), hp = read_all<double>(argv[4]);
        const std::vector<float> x = read_all<float>(argv[7]);
        const Layout l = layout(argv[8], argv[9], x.size());
        std::vector<float> lo(x.size(), -777.0f), hi(x.size(), -777.0f);
        qd::CrossoverArgs a{};
        a.x = x.data(); a.low = lo.data(); a.high = hi.data();
        apply(a, l);
        a.low_delay = std::atoi(argv[2]);
        qd_host::fill_crossover(a, lp.data(), hp.data());
        a.tile = std::atoi(argv[5]);
        a.halo = std::atoi(argv[6]);
        const long long n_tiles = (a.n + a.tile - 1) / a.tile;
        const unsigned gx = (unsigned)std::max<long long>(1, (n_tiles + 32 * qd::QD_XO_WARPS - 1) / (32 * qd::QD_XO_WARPS));
        qd::for_each_launch(l.batch, g_per_launch, [&](int clip0, int nb) {
            a.clip0 = clip0;
            qd_emu::launch(dim3(gx, nb, 1), dim3(32 * qd::QD_XO_WARPS), 0, [&] { qd::crossover_kernel(a); });
        });
        write_all(argv[10], lo);
        write_all(argv[11], hi);
        return 0;
    }
    std::cerr << "usage: see source\n";
    return 2;
}
