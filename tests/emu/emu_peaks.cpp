// tests/emu/emu_peaks.cpp -- TEST INFRASTRUCTURE: runs peaks_kernel (csrc/qd_peaks.cuh) on the CPU through cuda_emu.h,
// with the library's FFT tables and launch geometry, so that tests/test_emu_peaks.py can compare its bins with the
// oracle and every clip of a packed batch with the same clip alone.
//
//   emu_peaks [-p <clips per launch>] <f32|f64> <n_fft> <topn> <min_mag> <x.f32> <starts.i64|-|u<B>> <lengths.i32|-> <bins.i16>
// With "-" for starts / lengths x is one clip, with "u<B>" B uniform clips of len(x) / B samples; otherwise x is packed
// and the batch is len(starts).  bins gets the rows of qd_spectral_peaks_device(_varlen): B * (1 + n / hop) for a
// uniform batch, span / hop + B for a ragged one, every entry pre-filled with SENTINEL so that rows the kernel must not
// write can be checked.  -p splits the batch into launches of that many clips with qd::for_each_launch, as the library
// does at the grid limit (default: one launch).
#include "cuda_emu.h"

namespace qd_emu {
thread_local Block *g_blk = nullptr;
thread_local dim3 g_tid, g_bid;
}  // namespace qd_emu

#include "../../quantumdistortion_b200/csrc/qd_host_tables.hpp"
#include "../../quantumdistortion_b200/csrc/qd_peaks.cuh"

#include <climits>
#include <fstream>
#include <iostream>
#include <string>

static constexpr int16_t SENTINEL = 0x5a5a;

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

template <class T, int NC>
static void run(qd::PeaksArgsT<T> a, int batch, int64_t per_launch) {
    constexpr int nw = qd::peaks_warps<T, NC>();
    const unsigned gx = (unsigned)((a.n_frames + nw - 1) / nw);
    qd::for_each_launch(batch, per_launch, [&](int clip0, int nb) {
        a.clip0 = clip0;
        qd_emu::launch(dim3(gx, (unsigned)nb, 1), dim3(32 * nw), qd::peaks_warp_smem<T, NC>() * nw,
                       [&] { qd::peaks_kernel<T, NC>(a); });
    });
}

template <class T>
static int peaks(char **argv, int64_t per_launch) {
    using T2 = qd::V2<T>;
    const int n_fft = std::atoi(argv[2]), topn = std::atoi(argv[3]);
    const double min_mag = std::atof(argv[4]);
    const std::vector<float> x = read_all<float>(argv[5]);
    const char *sp = argv[6], *lp = argv[7];
    const int hop = n_fft / 4;
    std::vector<int64_t> starts;
    std::vector<int32_t> lengths;
    int batch = 1, n = 0;
    long long rows;
    if (sp[0] == '-' || sp[0] == 'u') {
        if (sp[0] == 'u') batch = std::atoi(sp + 1);
        n = (int)(x.size() / batch);
        rows = (long long)batch * (1 + n / hop);
    } else {
        starts = read_all<int64_t>(sp);
        lengths = read_all<int32_t>(lp);
        batch = (int)starts.size();
        for (int32_t l : lengths) n = std::max(n, (int)l);
        rows = (starts.back() - starts.front() + lengths.back()) / hop + batch;
    }
    qd_host::SpecTablesT<T> st;
    if (!qd_host::build_spec_tables<T>(n_fft, &st)) { std::cerr << "unsupported n_fft\n"; return 2; }
    std::vector<int16_t> bins((size_t)rows * topn, SENTINEL);
    qd::PeaksArgsT<T> a{};
    a.x = x.data();
    a.bins = bins.data();
    if (!starts.empty()) { a.starts = starts.data(); a.lengths = lengths.data(); }
    a.n = n;
    a.n_frames = 1 + n / hop;
    a.topn = topn;
    a.min_mag2 = (T)(min_mag * min_mag);
    a.wtab = reinterpret_cast<const T2 *>(st.wtab.data());
    a.tw1 = reinterpret_cast<const T2 *>(st.tw1.data());
    a.tw2 = reinterpret_cast<const T2 *>(st.tw2.data());
    a.wsplit = reinterpret_cast<const T2 *>(st.wsplit.data());
    switch (n_fft / 2) {
        case 256:  run<T, 256>(a, batch, per_launch); break;
        case 512:  run<T, 512>(a, batch, per_launch); break;
        case 1024: run<T, 1024>(a, batch, per_launch); break;
        case 2048: run<T, 2048>(a, batch, per_launch); break;
        case 4096: run<T, 4096>(a, batch, per_launch); break;
        default: std::cerr << "unsupported n_fft\n"; return 2;
    }
    std::ofstream(argv[8], std::ios::binary).write(reinterpret_cast<const char *>(bins.data()), (std::streamsize)(bins.size() * 2));
    return 0;
}

int main(int argc, char **argv) {
    int64_t per_launch = INT32_MAX;
    if (argc > 2 && std::string(argv[1]) == "-p") {
        per_launch = std::atoll(argv[2]);
        argv += 2;
        argc -= 2;
    }
    if (argc != 9) { std::cerr << "usage: see source\n"; return 2; }
    return std::string(argv[1]) == "f64" ? peaks<double>(argv, per_launch) : peaks<float>(argv, per_launch);
}
