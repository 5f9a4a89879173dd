// tests/emu/emu_spec_ef.cpp -- TEST INFRASTRUCTURE: runs the n_fft 2048 two-group spectral pass
// (spec_pass_kernel<float, 1024, 8, TS, noFX, NG = 2>) on the CPU through cuda_emu.h, as the library launches it for a
// render without a tap: either its EF instantiation (epilogue none, or a wavefold exact in float32) or the general one.
// Used by tests/test_emu_ef_overlap_add.py to compare the two bit for bit.
//
//   emu_spec_ef <ef 0|1> <epilogue 0|1> <fold> <tile_blocks> <x.f32> <starts.i64|u<B>> <lengths.i32|-> <tb.i32> <mask.u8> <y.f32>
// u<B>: x holds B uniform clips of len(x) / B samples; otherwise x is packed and the batch is len(starts).  One quantised
// pass (snap 1.0, smear 0.1, smoothing on).  Writes <y> (every sample of x's layout; -777 where no clip wrote) and
// <y>.peak: the per-clip peaks (clip_peak) and two rows no clip owns.
#include "cuda_emu.h"

namespace qd_emu {
thread_local Block *g_blk = nullptr;
thread_local dim3 g_tid, g_bid;
}  // namespace qd_emu

#include "../../quantumdistortion_b200/csrc/qd_host_tables.hpp"
#include "../../quantumdistortion_b200/csrc/qd_spec.cuh"

#include <algorithm>
#include <cmath>
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
static void write_all(const std::string &path, const std::vector<T> &v) {
    std::ofstream(path, std::ios::binary).write(reinterpret_cast<const char *>(v.data()), (std::streamsize)(v.size() * sizeof(T)));
}

int main(int argc, char **argv) {
    if (argc != 11) { std::cerr << "usage: see source\n"; return 2; }
    using T = float;
    using T2 = qd::V2<T>;
    constexpr int N_FFT = 2048, NC = 1024, NW = 8, NG = 2;
    const int ef = std::atoi(argv[1]), epilogue = std::atoi(argv[2]), tile_blocks = std::atoi(argv[4]);
    const double fold = std::atof(argv[3]);
    const std::vector<float> x = read_all<float>(argv[5]);
    std::vector<int64_t> starts;
    std::vector<int32_t> lengths;
    int batch = 1, max_n = 0;
    if (argv[6][0] == 'u') {
        batch = std::atoi(argv[6] + 1);
        max_n = (int)(x.size() / batch);
    } else {
        starts = read_all<int64_t>(argv[6]);
        lengths = read_all<int32_t>(argv[7]);
        batch = (int)starts.size();
        for (int32_t n : lengths) max_n = std::max(max_n, (int)n);
    }
    const std::vector<int32_t> tb = read_all<int32_t>(argv[8]);
    const std::vector<uint8_t> mask = read_all<uint8_t>(argv[9]);
    qd_host::SpecTablesT<T> st;
    if (!qd_host::build_spec_tables<T>(N_FFT, &st)) { std::cerr << "unsupported n_fft\n"; return 2; }
    double kw[5], ks = 0;   // the 5-tap smear kernel (dsp/quantizer.py:460-465)
    for (int i = 0; i < 5; ++i) { kw[i] = std::exp(-0.5 * (i - 2) * (i - 2)); ks += kw[i]; }
    for (int i = 0; i < 5; ++i) kw[i] /= ks;
    qd_tables ht{};
    ht.n_bins = N_FFT / 2 + 1;
    ht.target_bins = tb.data();
    ht.active_mask = mask.data();
    ht.snap = 1.0;
    ht.smear = 0.1;
    ht.smear_radius = 2;
    ht.smear_w = kw;
    qd_host::QuantTablesH qt;
    std::string err;
    if (!qd_host::build_quant_tables(ht, &qt, &err, false)) { std::cerr << err << "\n"; return 2; }
    std::vector<float> y(x.size(), -777.0f);
    std::vector<float> peak((size_t)batch + 2, 0.0f);   // zeroed by the caller, as in launch_spec_prec
    qd::SpecArgsT<T> a{};
    a.x = x.data();
    a.y = y.data();
    a.clip_peak = peak.data();
    a.n = max_n;
    if (!starts.empty()) { a.starts = starts.data(); a.lengths = lengths.data(); }
    a.batch = batch;
    a.n_frames = 1 + a.n / st.hop;
    a.tile_blocks = tile_blocks;
    a.quant = 1;
    a.epilogue = epilogue;
    a.fold = fold; a.bias = 0.0; a.tube_gain = 1.0f; a.tube_norm = 1.0f;
    int e = 0;   // as qd_render_device decides it
    a.fold_exact_f32 = fold > 0.0 && std::frexp(fold, &e) == 0.5 && e > -100 && e < 100;
    if (ef && epilogue != 0 && !(epilogue == 1 && a.fold_exact_f32)) { std::cerr << "EF: epilogue none or an exact wavefold\n"; return 2; }
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
    for (int i = 0; i < 5; ++i) a.q.tap[i] = qt.tap[i];
    a.q.keep_active = qt.keep_active;
    a.q.smoothing = 1;
    a.fx.table_frames = 1;
    const int tiles = std::max(1, ((a.n + st.hop - 1) / st.hop + tile_blocks - 1) / tile_blocks);   // the longest clip
    const size_t smem = qd::SpecSmem<T, NC, NW, NG>::bytes(qt.n_slots, true, a.q.n_src, 0);
    const dim3 grid(tiles, (batch + NG - 1) / NG, 1), block(32 * NW * NG, 1, 1);
    if (ef) qd_emu::launch(grid, block, smem, [&] { qd::spec_pass_kernel<T, NC, NW, true, false, NG, false, true>(a); });
    else qd_emu::launch(grid, block, smem, [&] { qd::spec_pass_kernel<T, NC, NW, true, false, NG>(a); });
    write_all(argv[10], y);
    write_all(std::string(argv[10]) + ".peak", peak);
    return 0;
}
