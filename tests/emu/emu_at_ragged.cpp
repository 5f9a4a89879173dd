// tests/emu/emu_at_ragged.cpp -- TEST INFRASTRUCTURE: runs autotune_v1 kernels of a ragged batch (per-clip starts /
// lengths) on the CPU through cuda_emu.h, so that tests/test_emu_ragged_autotune.py can compare every clip with the
// same clip run alone.
//
//   emu_at_ragged yin <frame_size> <hop> <max_tau> <cols> <x.f32> <starts.i64|-> <lengths.i32|-> <diff.f64>
//   emu_at_ragged filt <sos.f64: jobs x 2 x 6> <zi.f64: jobs x 2 x 2> <x.f32> <starts|-> <lengths|-> <y.f32: jobs x span>
// With "-" for starts / lengths x is one clip (the uniform path); otherwise x is packed and the batch is len(starts).
// The filter bank takes its tiles from the poles like the library (qd_host::segment_tiling, qd::at_filt_tile).
#include "cuda_emu.h"

namespace qd_emu {
thread_local Block *g_blk = nullptr;
thread_local dim3 g_tid, g_bid;
}  // namespace qd_emu

#include "cuda_emu_at.h"
#include "../../quantumdistortion_b200/csrc/qd_autotune.cuh"
#include "../../quantumdistortion_b200/csrc/qd_host_time.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>
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
template <class A>
static void set_clips(A &a, const Batch &b) {
    a.n = b.n_max;
    a.starts = b.ragged ? b.starts.data() : nullptr;
    a.lengths = b.ragged ? b.lengths.data() : nullptr;
    a.clip0 = 0;
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
    std::cerr << "usage: see source\n";
    return 2;
}
