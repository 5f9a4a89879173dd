// spectral pass for the three-pass FFT plans: teams of warps per frame on swizzled buffers (qd_spec_team.cuh) -- float32
// n_fft 512 / 1024 / 4096, float64 n_fft 2048 / 4096 / 8192
#include <atomic>

#include "qd_err.hpp"
#include "qd_spec_team_launch.hpp"

namespace qd_launch {

template <class T, int NC, int NF, int CW>
static int launch_spec_team_t(const qd::SpecArgsT<T> &a, const qd::TeamGather &tg, int tiles, int64_t batch, cudaStream_t st) {
    static std::atomic<uint64_t> attr_mask{0};  // devices this instantiation was opted in on
    auto kern = qd::spec_pass_team_kernel<T, NC, NF, CW>;
    if (int rc_ = qd_err::ensure_dyn_smem(kern, attr_mask, 227 * 1024)) return rc_;
    const size_t smem = qd::SpecSmem<T, NC, NF>::bytes(a.q.n_slots);
    if (smem > 227 * 1024) return qd_err::fail(QD_ERR_UNSUPPORTED, "shared memory need of the team kernel exceeds 227 KB");
    qd::for_each_launch(batch, qd::QD_GRID_Y_MAX, [&](int clip0, int nb) {
        qd::SpecArgsT<T> c = a;
        c.clip0 = clip0;
        c.batch = nb;
        kern<<<dim3((unsigned)tiles, (unsigned)nb, 1), 32 * NF * CW, smem, st>>>(c, tg);
    });
    QD_CUDA(cudaGetLastError());
    return QD_OK;
}

template <>
int launch_spec_team<float>(int nc, const qd::SpecArgsT<float> &a, const qd::TeamGather &tg, int tiles, int64_t batch, cudaStream_t st) {
    if (nc == 2048) return launch_spec_team_t<float, 2048, 7, 4>(a, tg, tiles, batch, st);
    if (nc == 4096) return launch_spec_team_t<float, 4096, 4, 4>(a, tg, tiles, batch, st);   // n_fft 8192 under precision="float32"
    if (nc == 512) return launch_spec_team_t<float, 512, 8, 1>(a, tg, tiles, batch, st);
    if (nc == 256) return launch_spec_team_t<float, 256, 8, 1>(a, tg, tiles, batch, st);
    return qd_err::fail(QD_ERR_UNSUPPORTED, "no float32 team kernel for this n_fft");
}

template <>
int launch_spec_team<double>(int nc, const qd::SpecArgsT<double> &a, const qd::TeamGather &tg, int tiles, int64_t batch, cudaStream_t st) {
    if (nc == 1024) return launch_spec_team_t<double, 1024, 8, 2>(a, tg, tiles, batch, st);
    if (nc == 2048) return launch_spec_team_t<double, 2048, 4, 4>(a, tg, tiles, batch, st);
    if (nc == 4096) return launch_spec_team_t<double, 4096, 2, 8>(a, tg, tiles, batch, st);
    return qd_err::fail(QD_ERR_UNSUPPORTED, "no float64 team kernel for this n_fft");
}

}  // namespace qd_launch
