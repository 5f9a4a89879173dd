// qd_yin.cuh -- the YIN difference function of the autotune_v1 detector (dsp/autotune.py:130-160) by sliding sums.
//
// The mean of a frame cancels in c[j] - c[j+tau], so the difference function of frame f is a window sum over the
// (zero-extended) clip, and with the square expanded it needs ONE float64 operation per (sample, lag) pair instead of two:
//   d_f(tau) = sum_{j=s}^{p-1} (x[j] - x[j+tau])^2 = E(s, p) + E(s+tau, p+tau) - 2 R_tau(s, p),   s = f*hop, p = s + W - tau
//   E(a, b) = sum_{a <= j < b} x[j]^2  (shared by all lags),   R_tau(a, b) = sum_{a <= j < b} x[j] x[j+tau]
// (the inputs are float32, so every product is exact in float64).  Consecutive frames overlap by 7/8, so the sums are kept
// per hop block: R_tau of every block is accumulated once, V = E(block + tau) - 2 R_tau(block) of a finished block is parked
// in a ring per lag, and a frame's value is assembled from the parked blocks f .. b-1, the partial block, and prefix sums of
// squares over the current tile.  Every term is a sum over at most one frame, so nothing cancels against a clip-long
// running total (the largest term is 2 E_frame against d: relative error ~4e-16 E_frame / d).
//
// Work split (round 2, fourth version).  B200 issues 64 DFMA lanes per SM and cycle (measured: 33 TFLOP/s) and moves 128 B
// of shared memory per cycle, so a (sample, lag) pair may cost 1/64 cycle of arithmetic but an 8-byte operand costs 1/16:
// the walk has to reuse its operands from registers, and everything that is not the walk has to stay off its critical path.
//
//  * One CTA per SM works on one clip (and up to 42 * 16 lags); its twelve warps have two roles.
//  * EIGHT WALKER WARPS in two teams of four (one warp of each team per SM sub-partition, i.e. per FP64 pipe: a single
//    warp cannot keep the pipe busy through its own loads and block changes).  Team 0 walks the even hop blocks, team 1
//    the odd ones, so the two warps that share a pipe are in different phases of their blocks.  A walker thread owns
//    L = 16 consecutive lags (a "column") and one THIRD of a block's samples (the three partial sums of a lag meet in
//    shared memory once per block), and walks it 16 samples at a time: the 16 own samples are eight broadcast 16-byte loads from a
//    natural-order copy of the block, and of the 31 lagged samples x[j + tau0 .. j + tau0 + 30] fifteen are the previous
//    iteration's registers -- 16 new 8-byte loads, one per plane of the tile, which is stored de-interleaved by 16 so that
//    the lanes' stride-16 addresses are consecutive words.  24 loads and 256 DFMA per iteration.
//  * A lag's window ends somewhere inside every block.  With tau0 = 1 (mod 16) and frame size and hop multiples of 16 the
//    16 lags of a thread end in the SAME iteration, lag u after 15 - u of its samples: the thread stores S[u] from inside
//    that iteration (predicated stores, no divergence, no remainder products afterwards).
//  * FOUR HELPER WARPS run one block ahead and one block behind the walkers: they load the next block's samples (through
//    registers, fetched before the assembly starts), build its prefix sums of squares, and assemble the frames that the
//    previous block closed.  Tile, prefix sums and partial sums exist three times (two blocks being walked, one being
//    assembled and refilled); the roles meet at six mbarriers
//    (full / done per buffer): the producer side arrives, the consumer side only waits for the phase, so a walker warp
//    never waits for another walker warp.
#pragma once
#include "qd_common.cuh"

namespace qd {

struct AtYinArgs {
    const float *det;        // packed like the batch (qd_common.cuh: clip_loc)
    double *diff;            // [frame rows, stride] difference function, entry tau (frame rows: at_row0)
    double *feat;            // [frame rows, 4]; feat[2] holds 1 / 0 (frame not silent) on entry of the pick kernel
    long long n;
    long long total_frames;  // frame rows of the batch
    const int64_t *starts;   // optional ragged batch
    const int32_t *lengths;
    int clip0;
    int frames;              // ceil(n / hop), the longest clip's; the kernels derive every clip's own
    int frame_size, hop, stride;
    int min_tau, max_tau;
    int lag_threads;         // columns (of AT_YL lags) per CTA, <= AT_YC
    double sr, min_freq, max_freq, threshold;
};

constexpr int AT_YL = 16;         // lags per walker thread = samples per iteration = planes of the tile
constexpr int AT_YG = 3;          // sample groups per block: a walker owns a third of a block
constexpr int AT_YC = 42;         // columns per CTA: AT_YG * AT_YC = 126 walker threads per team
constexpr int AT_YTEAM = 128;     // threads of a walker team: four warps, one per SM sub-partition
constexpr int AT_YW = 2 * AT_YTEAM;   // two teams (warps 0-3 take the even blocks, warps 4-7 the odd ones)
constexpr int AT_YH = 128;        // helper threads (warps 8-11)
constexpr int AT_YNS = 3;         // buffers: two blocks being walked, one being assembled / refilled
constexpr int AT_YT = AT_YW + AT_YH;
constexpr int AT_YR = 9;          // ring depth: frame_size / hop + 1 blocks
enum { AT_BAR_HELP = 1 };         // named barrier of the helper warps (0 is __syncthreads)

__host__ __device__ inline int at_yin_odd(int v) { return v | 1; }
// Strides: an array [16][stride] indexed (u, t) is used with consecutive t by the walkers (conflict-free) and with u
// fastest by the helpers; with an odd stride the 32 doubles of a warp then fall on the 16 eight-byte bank slots twice each,
// the two wavefronts 256 bytes need anyway.

// shared memory in doubles: 3 x (tile, natural-order block, prefix sums, partial sums, captures), ring, scratch, lag table
__host__ __device__ inline size_t at_yin_smem_doubles(int hop, int first_col, int cols) {
    (void)first_col;    // the tile starts at the CTA's first lag: its size does not depend on where the lag range begins
    const size_t plane = (size_t)AT_YL * at_yin_odd(hop / AT_YL + cols + 1), rs = (size_t)AT_YL * at_yin_odd(cols);
    return AT_YNS * (2 * plane + 2 * hop + 8 + (AT_YG + 1) * rs) + AT_YR * rs + 48 + 2 * AT_YNS + (AT_YL * cols + 1) / 2 + 16;
}

QD_DEV void at_bar_sync(int id, int count) {
#ifdef QD_EMU
    qd_emu::named_barrier(id, count);
#else
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
#endif
}

// Shared-memory barriers with an arrival count (mbarrier): the producers arrive, the consumers only wait for the phase to
// flip, so the consumers never wait for one another.  Host emulation: completed phases in the low word, pending arrivals
// and the count above it.
#ifdef QD_EMU
QD_DEV void at_mbar_init(uint64_t *bar, int count) { *bar = ((uint64_t)count << 48) | ((uint64_t)count << 32); }
QD_DEV void at_mbar_arrive(uint64_t *bar) {
    uint64_t old = __atomic_load_n(bar, __ATOMIC_SEQ_CST), upd;
    do {
        const uint64_t count = old >> 48, pending = ((old >> 32) & 0xffff) - 1, phase = old & 0xffffffffu;
        upd = pending ? (count << 48) | (pending << 32) | phase : (count << 48) | (count << 32) | ((phase + 1) & 0xffffffffu);
    } while (!__atomic_compare_exchange_n(bar, &old, upd, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST));
}
QD_DEV void at_mbar_wait(uint64_t *bar, uint32_t parity) {
    while ((__atomic_load_n(bar, __ATOMIC_SEQ_CST) & 1u) == parity) std::this_thread::yield();
}
#else
QD_DEV void at_mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
QD_DEV void at_mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
QD_DEV void at_mbar_wait(uint64_t *bar, uint32_t parity) { mbar_wait(bar, parity); }
#endif

__global__ void __launch_bounds__(AT_YT, 1) at_yin_diff_kernel(const AtYinArgs a) {
    constexpr int L = AT_YL, G = AT_YG;
    QD_DYN_SMEM(smem);
    const int tid = threadIdx.x;
    const int cols = a.lag_threads;                     // columns of this CTA
    const int c0 = blockIdx.x * cols;                   // first column: lags tau0 .. tau0 + L cols - 1, tau0 = 1 + L c0
    const int tau0 = 1 + L * c0;
    const int W = a.frame_size, hop = a.hop;
    // A block needs its own samples [0, hop) and the lagged ones [B0, B0 + span), B0 = L c0 (relative to the block start):
    // one range when the CTA holds the first lags (c0 = 0), two when a wide lag range is split over several CTAs.  The
    // tile and its prefix sums cover the lagged range; prefix sums only ever meet as differences within one range, except
    // E(s, p) = energies of whole blocks + qa(off), which wants the own range (`qa`, natural order, used when c0 > 0).
    const int B0 = L * c0;
    const int span = hop + L * cols;
    const int Q = at_yin_odd(span / L + 1);             // plane stride of tile and prefix sums
    const int PL = L * Q;
    const int sp = at_yin_odd(cols);                    // row stride of the per-lag arrays
    const int RS = L * sp;                              // one [L][sp] array
    double *tile = reinterpret_cast<double *>(smem);    // [3][L][Q]: sample B0 + i of the block at (i % L) * Q + i / L
    double *own = tile + AT_YNS * PL;                   // [3][hop] the block's own samples in natural order
    double *qt = own + AT_YNS * hop;                    // [3][L][Q] prefix sums of squares, same layout: qt(i) = E(j0, j0 + i)
    double *qa = qt + AT_YNS * PL;                      // [3][hop + 1] prefix sums of squares of the own range (c0 > 0 only)
    double *xs = qa + AT_YNS * (hop + 8);               // [3][G][L][sp] R_tau of each third of the block
    double *xp = xs + AT_YNS * G * RS;                  // [3][cols][L] R_tau of the block up to the lag's window end
    double *ringV = xp + AT_YNS * RS;                   // [AT_YR][L][sp] E(block + tau) - 2 R_tau(block) of finished blocks
    double *wtot = ringV + (size_t)AT_YR * RS;          // [16] warp totals of the prefix sum
    double *be = wtot + 16;                             // [16] energies of the last blocks
    double *ebq = be + 16;                              // [16] ebq[q] = energy of the q blocks before the one being assembled
    uint64_t *mbar = reinterpret_cast<uint64_t *>(ebq + 16);   // full[3] (helpers -> walkers), done[3] (walkers -> helpers)
    int *lagc = reinterpret_cast<int *>(mbar + 2 * AT_YNS);      // [L * cols] per lag: off | q << 12 | group << 16 | live << 20
    const ClipLoc clip = clip_loc(a, blockIdx.y);
    const long long n = clip.n;
    const int frames = (int)at_rows(n, hop);
    const float *x = a.det + clip.base;
    double *out = a.diff + at_row0(a.starts != nullptr, clip, a.n, hop) * a.stride;
    const int blocks = frames + W / hop;
    const int n_all = hop / L;                          // iterations per block, split over the G groups as evenly as possible
    auto group_begin = [&](int g) { return g * (n_all / G) + min(g, n_all % G); };
    uint64_t *full = mbar, *done = mbar + AT_YNS;
    if (tid < AT_YNS) {
        at_mbar_init(full + tid, 1);                    // one helper thread arrives after the helpers' own barrier
        at_mbar_init(done + tid, AT_YTEAM / 32);        // one lane per warp of the team that walked the block
    }
    __syncthreads();

    if (tid < AT_YW) {
        // ================================================================ walkers: team, group g (a third of the samples), column t
        const int team = tid / AT_YTEAM, wt = tid % AT_YTEAM;
        const bool walker = wt < G * cols;
        const int g = walker ? wt / cols : 0, t = walker ? wt % cols : 0;
        const int it0 = group_begin(g), n_it = group_begin(g + 1) - it0;
        // window length of the thread's first lag: W - tau0 - L t = L - 1 (mod L); lag u ends L - 1 - u samples into
        // iteration off0 / L of the block
        const int off0 = (W - tau0 - L * t) % hop;
        const int cap = off0 / L - it0;                 // the thread's own iteration index of the capture (or out of range)
        for (int b = team; b < blocks; b += 2) {
            const int s = b % AT_YNS;
            at_mbar_wait(full + s, (b / AT_YNS) & 1);   // tile / own of block b are in buffer s (the warp waits for nobody else)
            if (walker) {
                const double *ownp = own + s * hop + L * it0;
                const double *lagp = tile + s * PL + (it0 + t);         // plane p of iteration it: lagp[p * Q + it (+ 1)]
                double *xpp = xp + s * RS + L * t;          // captures: xp[column][lag]
                double S[L], wo[L];
#pragma unroll
                for (int u = 0; u < L; ++u) S[u] = 0.0;
#pragma unroll
                for (int p = 1; p < L; ++p) wo[p] = lagp[p * Q];                 // x[j + tau0 + v], v = p - 1 < L - 1
                auto load_own = [&](int it, double (&av)[L]) {
#pragma unroll
                    for (int h = 0; h < L / 2; ++h) {
                        const double2 o2 = *reinterpret_cast<const double2 *>(ownp + L * it + 2 * h);
                        av[2 * h] = o2.x;
                        av[2 * h + 1] = o2.y;
                    }
                };
                auto load_lag = [&](int it, double (&wn)[L]) {
#pragma unroll
                    for (int p = 0; p < L; ++p) wn[p] = lagp[p * Q + it + 1];    // v = L - 1 + p
                };
                auto step = [&](int it, const double (&av)[L], const double (&wn)[L]) {
                    const bool c = it == cap;
                    if (c) xpp[L - 1] = S[L - 1];                                 // the last lag ends before the first sample
#pragma unroll
                    for (int k = 0; k < L; ++k) {
#pragma unroll
                        for (int u = 0; u < L; ++u) {
                            const int v = k + u;                                 // lagged sample x[j + k + tau0 + u]
                            S[u] = fma(av[k], v < L - 1 ? wo[v + 1] : wn[v - (L - 1)], S[u]);
                        }
                        if (k < L - 1 && c) xpp[L - 2 - k] = S[L - 2 - k];    // lag L - 2 - k ends after sample k
                    }
#pragma unroll
                    for (int p = 1; p < L; ++p) wo[p] = wn[p];
                };
                double av[L], wn[L];
#pragma unroll 2
                for (int it = 0; it < n_it; ++it) {      // two walker warps share a sub-partition: the partner covers the loads
                    load_own(it, av);
                    load_lag(it, wn);
                    step(it, av, wn);
                }
                double *xsp = xs + (size_t)(s * G + g) * RS + t;
#pragma unroll
                for (int u = 0; u < L; ++u) xsp[u * sp] = S[u];
            }
            __syncwarp();
            if ((tid & 31) == 0) at_mbar_arrive(done + s);   // this warp's partial sums of block b are in buffer s, tile s is free
        }
    } else {
        // ================================================================ helpers
        const int h = tid - AT_YW, hl = h & 31, hw = h >> 5;
        auto helper_sync = [&]() { at_bar_sync(AT_BAR_HELP, AT_YH); };
        for (int col = h; col < L * cols; col += AT_YH) {
            const int tau = tau0 + col, wlen = W - tau, off = wlen % hop;
            int gc = 0;
            while (gc + 1 < G && off / L >= group_begin(gc + 1)) ++gc;             // the third the window ends in
            lagc[col] = off | ((wlen / hop) << 12) | (gc << 16) | ((tau <= a.max_tau ? 1 : 0) << 20);
        }
        if (h < 16) be[h] = 0.0;
        // the samples of a block travel through registers: fetched before the assembly of an earlier block starts, stored
        // after it (the global-memory latency is off the helpers' critical path)
        constexpr int PF = 10, PFO = 4;                  // 10 x 128 lagged-range samples, 4 x 128 own samples; any rest directly
        float pf[PF], pfo[PFO];
        auto fetch = [&](int b) {
            const long long j0 = (long long)b * hop;
#pragma unroll
            for (int r = 0; r < PF; ++r) {
                const int i = h + r * AT_YH;
                const long long sidx = j0 + B0 + i;
                pf[r] = (i < span && sidx < n) ? x[sidx] : 0.0f;
            }
            if (c0 > 0) {
#pragma unroll
                for (int r = 0; r < PFO; ++r) {
                    const int i = h + r * AT_YH;
                    const long long sidx = j0 + i;
                    pfo[r] = (i < hop && sidx < n) ? x[sidx] : 0.0f;
                }
            }
        };
        // Prefix sums of squares of nth chunks of L samples: thread hh scans chunk hh (sample p of it at src[p * sp_ + hh * sh_]:
        // plane p, index hh of a tile, conflict-free; or own[L hh + p]), the chunk totals are scanned over the threads, and
        // every entry is written once: dst(L hh + p) = total before the chunk + its first p squares, entry L nth = the total.
        // 128 threads cover 2032 samples per round.  `be_hh`: the chunk boundary that is the end of the block (or -1).
        auto prefix = [&](const double *src, double *dst, int sp_, int sh_, int nth, int be_hh, int b) {
            double carry = 0.0;
            for (int r0 = 0, par = 0; r0 <= nth; r0 += AT_YH, par ^= 4) {
                const int hh = r0 + h;
                double sq[L], loc[L];
#pragma unroll
                for (int p = 0; p < L; ++p) {
                    const double v = hh < nth ? src[p * sp_ + hh * sh_] : 0.0;
                    sq[p] = v * v;
                }
                loc[0] = sq[0];
#pragma unroll
                for (int p = 1; p < L; ++p) loc[p] = loc[p - 1] + sq[p];
                const double run = loc[L - 1];
                double inc = run;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const double o = __shfl_up_sync(QD_FULL, inc, d);
                    if (hl >= d) inc += o;
                }
                if (hl == 31) wtot[par + hw] = inc;
                helper_sync();
                double base = carry + (inc - run);
                for (int w = 0; w < hw; ++w) base += wtot[par + w];
                for (int w = 0; w < AT_YH / 32; ++w) carry += wtot[par + w];
                if (hh <= nth) {
                    dst[hh * sh_] = base;
                    if (hh < nth) {
#pragma unroll
                        for (int p = 1; p < L; ++p) dst[p * sp_ + hh * sh_] = base + loc[p - 1];
                    }
                    if (hh == be_hh) be[b & 15] = base;                           // E(j0, j0 + hop)
                }
            }
        };
        // samples (from the registers) and prefix sums of squares of block b into buffer s
        auto produce = [&](int b, int s) {
            double *tl = tile + s * PL, *ow = own + s * hop;
#pragma unroll
            for (int r = 0; r < PF; ++r) {
                const int i = h + r * AT_YH;
                if (i < span) {
                    const double v = (double)pf[r];
                    tl[(i % L) * Q + i / L] = v;
                    if (c0 == 0 && i < hop) ow[i] = v;
                }
            }
            for (int i = h + PF * AT_YH; i < span; i += AT_YH) {
                const long long sidx = (long long)b * hop + B0 + i;
                tl[(i % L) * Q + i / L] = sidx < n ? (double)x[sidx] : 0.0;
            }
            if (c0 > 0) {
#pragma unroll
                for (int r = 0; r < PFO; ++r) {
                    const int i = h + r * AT_YH;
                    if (i < hop) ow[i] = (double)pfo[r];
                }
                for (int i = h + PFO * AT_YH; i < hop; i += AT_YH) {
                    const long long sidx = (long long)b * hop + i;
                    ow[i] = sidx < n ? (double)x[sidx] : 0.0;
                }
            }
            helper_sync();
            prefix(tl, qt + s * PL, Q, 1, span / L, c0 == 0 ? hop / L : -1, b);
            if (c0 > 0) {
                helper_sync();                                                   // the scan scratch is free again
                prefix(ow, qa + s * (hop + 8), 1, L, hop / L, hop / L, b);
            }
            helper_sync();                                                       // everything of block b is in buffer s
            if (h == 0) at_mbar_arrive(full + s);
        };
        // frames closed by block b: every lag closes exactly one frame per block (frame b - q at offset off)
        int slot_b = 0;                                                          // b % AT_YR
        auto assemble = [&](int b, int s) {
            if (h < AT_YR) {                                                     // energies of the h blocks before b, nearest first
                double e = 0.0;
                for (int i = 1; i <= h; ++i) e += be[(b - i) & 15];
                ebq[h] = e;
            }
            helper_sync();
            const double *q = qt + s * PL, *qown = qa + s * (hop + 8), *xsb = xs + (size_t)s * G * RS, *xpb = xp + s * RS;
            auto qv = [&](int i) { return q[(i % L) * Q + i / L]; };           // lagged range: entry i is sample B0 + i
            for (int col = h; col < L * cols; col += AT_YH) {
                const int lc = lagc[col];
                const int off = lc & 4095, qq = (lc >> 12) & 15, gc = (lc >> 16) & 15, tau = tau0 + col;
                const int at = (col % L) * sp + col / L;
                double r = 0.0, pu = xpb[col];               // R_tau of the whole block / up to the window's end
#pragma unroll
                for (int gg = 0; gg < G; ++gg) {
                    const double sv = xsb[gg * RS + at];
                    r += sv;
                    pu += gg < gc ? sv : 0.0;
                }
                const int f = b - qq;
                // the parked blocks f .. b - 1 (at most 8): independent loads, summed pairwise
                double rv[8];
                int slot = slot_b - qq;
                if (slot < 0) slot += AT_YR;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    rv[i] = i < qq ? ringV[slot * RS + at] : 0.0;
                    slot = slot + 1 == AT_YR ? 0 : slot + 1;
                }
                const double v = ((rv[0] + rv[1]) + (rv[2] + rv[3])) + ((rv[4] + rv[5]) + (rv[6] + rv[7]));
                const int tr = 1 + col;                                                  // tau relative to the lagged range
                const double qtau = qv(tr);
                if ((lc >> 20) && f >= 0 && f < frames) {
                    const double e1 = ebq[qq] + (c0 == 0 ? qv(off) : qown[off]);         // E(s, p)
                    const double cur = (qv(off + tr) - qtau) - 2.0 * pu;                 // the partial block: E(. + tau) - 2 R
                    out[(size_t)f * a.stride + tau] = fmax(e1 + (v + cur), 0.0);
                }
                ringV[slot_b * RS + at] = (qv(hop + tr) - qtau) - 2.0 * r;
            }
            slot_b = slot_b + 1 == AT_YR ? 0 : slot_b + 1;
            helper_sync();                                                       // ebq, qt[s], xs[s], xp[s] have been read
        };
        helper_sync();
        for (int b = 0; b < AT_YNS && b < blocks; ++b) {
            fetch(b);
            produce(b, b);
        }
        for (int b = 0, s = 0; b < blocks; ++b, s = s + 1 == AT_YNS ? 0 : s + 1) {
            const bool more = b + AT_YNS < blocks;
            if (more) fetch(b + AT_YNS);                 // lands while the walkers finish block b and its frames are assembled
            at_mbar_wait(done + s, (b / AT_YNS) & 1);    // the walkers have left block b
            assemble(b, s);
            if (more) produce(b + AT_YNS, s);
        }
    }
}

}  // namespace qd
