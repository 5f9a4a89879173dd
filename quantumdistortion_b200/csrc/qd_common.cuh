// qd_common.cuh -- shared definitions for the sm_100a kernels of libqd_b200.so.
//
// The same headers compile two ways:
//   nvcc  -gencode arch=compute_100a,code=sm_100a   -> the product (qd_api.cu)
//   g++   -DQD_EMU (tests/emu/cuda_emu.h)            -> CPU single-stepping of the kernel
//          source for index-math tests in the GPU-less build container (test only).
#pragma once

#ifdef QD_EMU
#include "cuda_emu.h"
#define QD_SINCOSF(x, s, c) sincosf_emu((x), (s), (c))
#define QD_EXP10F(x) exp10f_emu(x)
#else
#include <cuda_runtime.h>
#include <stdint.h>
#define QD_DYN_SMEM(name) extern __shared__ __align__(128) unsigned char name[]
#define QD_SINCOSF(x, s, c) sincosf((x), (s), (c))
#define QD_EXP10F(x) exp10f(x)
#endif

#define QD_DEV __device__ __forceinline__
#define QD_FULL 0xffffffffu

namespace qd {

// ---------------------------------------------------------------- precision-generic complex helpers
// The spectral pass is written once for T = float (the fast path) and T = double (the parity path for
// ill-conditioned configurations: wide-open band mask, n_fft >= 4096).
template <class T> struct Vec2;
template <> struct Vec2<float>  { using type = float2; };
template <> struct Vec2<double> { using type = double2; };
template <class T> using V2 = typename Vec2<T>::type;
template <class T> QD_DEV V2<T> mk2(T a, T b);
template <> QD_DEV float2  mk2<float>(float a, float b)    { return make_float2(a, b); }
template <> QD_DEV double2 mk2<double>(double a, double b) { return make_double2(a, b); }

// ---------------------------------------------------------------- packed float2 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2)
// Blackwell issues one instruction for both halves of a 64-bit register pair (add/sub/mul/fma.rn.f32x2).  The
// spectral pass is issue bound, and complex data already lives in float2 pairs, so every complex add/sub
// is one FADD2 and a twiddle multiply is FMUL2 + FFMA2.  ptxas folds scalar broadcasts (`R.F32`) and half swaps
// (`.LO_HI`) of the operands into the instruction, so splat()/swap() below cost nothing.  Each half rounds
// exactly like the scalar .rn instruction.  double2 (parity path) and the host emulation use scalar code.
#ifdef QD_EMU
QD_DEV float2 padd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
QD_DEV float2 psub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
QD_DEV float2 pmul(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
QD_DEV float2 pfma(float2 a, float2 b, float2 c) { return make_float2(a.x * b.x + c.x, a.y * b.y + c.y); }
#else
QD_DEV unsigned long long f2_bits(float2 a) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y));
    return r;
}
QD_DEV float2 bits_f2(unsigned long long v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
QD_DEV float2 padd(float2 a, float2 b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
QD_DEV float2 psub(float2 a, float2 b) {
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
QD_DEV float2 pmul(float2 a, float2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
QD_DEV float2 pfma(float2 a, float2 b, float2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
    return bits_f2(r);
}
#endif
QD_DEV double2 padd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
QD_DEV double2 psub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
QD_DEV double2 pmul(double2 a, double2 b) { return make_double2(a.x * b.x, a.y * b.y); }
QD_DEV double2 pfma(double2 a, double2 b, double2 c) { return make_double2(a.x * b.x + c.x, a.y * b.y + c.y); }
QD_DEV float2  splat(float a)  { return make_float2(a, a); }
QD_DEV double2 splat(double a) { return make_double2(a, a); }
QD_DEV float2  pswap(float2 a)  { return make_float2(a.y, a.x); }
QD_DEV double2 pswap(double2 a) { return make_double2(a.y, a.x); }

#define QD_COMPLEX_OPS(T2, MK)                                                                         \
    QD_DEV T2 cadd(T2 a, T2 b) { return padd(a, b); }                                                  \
    QD_DEV T2 csub(T2 a, T2 b) { return psub(a, b); }                                                  \
    /* a * b = a * splat(b.x) + (-a.y, a.x) * b.y */                                                   \
    QD_DEV T2 cmul(T2 a, T2 b) {                                                                       \
        const T2 t = pmul(a, splat(b.x));                                                              \
        return MK(t.x - a.y * b.y, t.y + a.x * b.y);                                                   \
    }                                                                                                  \
    /* a * conj(b) */                                                                                  \
    QD_DEV T2 cmulc(T2 a, T2 b) {                                                                      \
        const T2 t = pmul(a, splat(b.x));                                                              \
        return MK(t.x + a.y * b.y, t.y - a.x * b.y);                                                   \
    }                                                                                                  \
    QD_DEV T2 cconj(T2 a) { return MK(a.x, -a.y); }
QD_COMPLEX_OPS(float2, make_float2)
QD_COMPLEX_OPS(double2, make_double2)

QD_DEV float  qd_max(float a, float b)   { return fmaxf(a, b); }
QD_DEV double qd_max(double a, double b) { return fmax(a, b); }
QD_DEV float  qd_abs(float a)  { return fabsf(a); }
QD_DEV double qd_abs(double a) { return fabs(a); }
QD_DEV float  qd_rint(float a)  { return rintf(a); }
QD_DEV double qd_rint(double a) { return rint(a); }
QD_DEV float  qd_log10(float a)  { return log10f(a); }
QD_DEV double qd_log10(double a) { return log10(a); }
QD_DEV float  qd_log2(float a)  { return log2f(a); }
QD_DEV double qd_log2(double a) { return log2(a); }
QD_DEV float  qd_log(float a)  { return logf(a); }
QD_DEV double qd_log(double a) { return log(a); }
QD_DEV float  qd_exp(float a)  { return expf(a); }
QD_DEV double qd_exp(double a) { return exp(a); }
QD_DEV float  qd_exp2(float a)  { return exp2f(a); }
QD_DEV double qd_exp2(double a) { return exp2(a); }
QD_DEV float  qd_exp10(float a)  { return QD_EXP10F(a); }
QD_DEV double qd_exp10(double a) { return pow(10.0, a); }
QD_DEV void qd_sincos(float a, float *s, float *c)    { QD_SINCOSF(a, s, c); }
QD_DEV void qd_sincos(double a, double *s, double *c) { *s = sin(a); *c = cos(a); }

// ---------------------------------------------------------------- TMA bulk copy + mbarrier (sm_90+)
// One-dimensional cp.async.bulk global -> shared, completion signalled on an mbarrier with transaction
// bytes.  The host emulation completes the copy synchronously and bumps a phase counter.
#ifdef QD_EMU
QD_DEV void mbar_init(uint64_t *bar, int) { *bar = 0; }
QD_DEV void mbar_expect_tx(uint64_t *, uint32_t) {}
QD_DEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    std::memcpy(dst, src, bytes);
    __atomic_add_fetch(bar, 1, __ATOMIC_SEQ_CST);
}
QD_DEV void mbar_wait(uint64_t *bar, uint32_t parity) {
    while ((__atomic_load_n(bar, __ATOMIC_SEQ_CST) & 1u) == parity) std::this_thread::yield();
}
#else
QD_DEV uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
QD_DEV void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // visible to the async proxy
}
QD_DEV void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
QD_DEV void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
QD_DEV void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
#endif

// cos(2*pi*k/32), k = 0..8 (quarter wave); everything else by symmetry
__host__ __device__ constexpr double qd_cos32_q(int k) {
    return k == 0 ? 1.0
         : k == 1 ? 0.98078528040323044913
         : k == 2 ? 0.92387953251128675613
         : k == 3 ? 0.83146961230254523708
         : k == 4 ? 0.70710678118654752440
         : k == 5 ? 0.55557023301960222474
         : k == 6 ? 0.38268343236508977173
         : k == 7 ? 0.19509032201612826785
                  : 0.0;
}
__host__ __device__ constexpr double qd_cos32(int k) {  // k in [0,32)
    return k <= 8 ? qd_cos32_q(k) : k <= 16 ? -qd_cos32_q(16 - k) : k <= 24 ? -qd_cos32_q(k - 16) : qd_cos32_q(32 - k);
}
__host__ __device__ constexpr double qd_sin32(int k) { return qd_cos32((k + 24) & 31); }  // sin(a) = cos(a - pi/2)

// d * exp(DIR * 2*pi*i * k/32);  k is a compile-time constant after unrolling.
template <int DIR, class T>
QD_DEV V2<T> mul_w32(V2<T> d, int k) {
    k &= 31;
    if (k == 0) return d;
    if (k == 16) return mk2<T>(-d.x, -d.y);
    if (k == 8) return DIR > 0 ? mk2<T>(-d.y, d.x) : mk2<T>(d.y, -d.x);
    if (k == 24) return DIR > 0 ? mk2<T>(d.y, -d.x) : mk2<T>(-d.y, d.x);
    const T c = (T)qd_cos32(k);
    const T s = (T)(DIR > 0 ? qd_sin32(k) : -qd_sin32(k));
    // (x c - y s, y c + x s) = d * (c, c) + swap(d) * (-s, s): FMUL2 + FFMA2
    return pfma(pswap(d), mk2<T>(-s, s), pmul(d, splat(c)));
}

__host__ __device__ constexpr int qd_log2(int r) { return r <= 1 ? 0 : 1 + qd_log2(r >> 1); }
__host__ __device__ constexpr int qd_ctz(int v) { return (v & 1) ? 0 : 1 + qd_ctz(v >> 1); }  // v > 0
__host__ __device__ constexpr int qd_bitrev(int v, int bits) {
    int o = 0;
    for (int i = 0; i < bits; ++i) o |= ((v >> i) & 1) << (bits - 1 - i);
    return o;
}

// In-register radix-2 decimation-in-frequency DFT of R points (R = 2..32), fully unrolled.
// Input natural order; on return v[r] holds output index qd_bitrev(r, log2 R).
// DIR = -1: forward (exp(-2 pi i nk/R)); DIR = +1: inverse, unnormalised.
template <int R, int DIR, class T>
QD_DEV void dft_reg(V2<T> (&v)[R]) {
#pragma unroll
    for (int half = R / 2; half >= 1; half >>= 1) {
#pragma unroll
        for (int base = 0; base < R; base += 2 * half) {
#pragma unroll
            for (int i = 0; i < half; ++i) {
                const V2<T> a = v[base + i];
                const V2<T> b = v[base + i + half];
                v[base + i] = cadd(a, b);
                if (i * (16 / half) == 8)   // (a - b) * (-/+ i) without forming a - b as a pair
                    v[base + i + half] = DIR > 0 ? mk2<T>(b.y - a.y, a.x - b.x) : mk2<T>(a.y - b.y, b.x - a.x);
                else
                    v[base + i + half] = mul_w32<DIR, T>(csub(a, b), i * (16 / half));
            }
        }
    }
}

// Clip c of a launch: its index in the batch (idx = clip0 + c), its sample offset in the packed buffers and its length.
// Uniform batches (starts == null) hold clip i at i * n, n samples each; a ragged batch reads its per-clip arrays
// starts / lengths, offsets relative to starts[0] (n is then the longest clip, which sizes the grids).  Launch splits
// (for_each_launch) advance clip0 for both kinds, so no pointer moves and per-clip arrays are indexed by idx.
struct ClipLoc { int idx; long long base, n; };
template <class A>
QD_DEV ClipLoc clip_loc(const A &a, int c) {
    const int i = a.clip0 + c;
    if (a.starts) return {i, (long long)(a.starts[i] - a.starts[0]), (long long)a.lengths[i]};
    return {i, (long long)i * a.n, (long long)a.n};
}

// Covers clips [0, batch) with launches of at most per_launch clips: fn(clip0, nb) for each.  Grids put clips on
// gridDim.y, whose limit is QD_GRID_Y_MAX; a kernel with g clips per CTA passes g * QD_GRID_Y_MAX.  Clip indices
// are int: the entry points reject batches past INT32_MAX.
constexpr int64_t QD_GRID_Y_MAX = 65535;
template <class Fn>
inline void for_each_launch(int64_t batch, int64_t per_launch, Fn &&fn) {
    for (int64_t b0 = 0; b0 < batch; b0 += per_launch) fn((int)b0, (int)(batch - b0 < per_launch ? batch - b0 : per_launch));
}

// Per-clip tables with one row per `unit` samples (detector frames: unit = hop, ceil(n / hop) frames per clip;
// delay-tap tiles: unit = AT_TS).  Uniform batches keep clip i at row i * rows(n).  Ragged batches put it at
// floor(base / unit) + i: no scan, valid for any sub-range of clips, and rows of consecutive clips cannot overlap
// because starts[i + 1] >= starts[i] + n_i.  So a ragged batch has at most span / unit + batch rows.
__host__ __device__ inline long long at_rows(long long n, int unit) { return (n + unit - 1) / unit; }
QD_DEV long long at_row0(bool ragged, const ClipLoc &c, long long n_uniform, int unit) {
    return ragged ? c.base / unit + c.idx : (long long)c.idx * at_rows(n_uniform, unit);
}

}  // namespace qd
