/*
 * include/qd_b200.h -- C ABI of libqd_b200.so (B200 / sm_100a).
 *
 * Drop-in boundary for the STFT processing path of TGALLOWAY1/QuantumDistortion.
 * The reference has no FFI of its own: its boundary is the Python callable
 *   quantum_distortion/dsp/pipeline.py:1113-1155   process_audio(audio, sr, **params)
 * and everything below it is NumPy/SciPy/Numba.  This library is what a binding for
 * that call binds (see INTEGRATION.md for the ctypes stub a maintainer would add):
 * plain C, plain pointers and sizes, no torch types.
 *
 * Division of labour (mirrors SURVEY.md section 8(b)):
 *   host (Python, quantumdistortion_b200/tables.py)  -- resolves the reference's
 *       keyword arguments into the numbers and integer tables below, in float64,
 *       with the reference's own formulas (bit-exact target bins, masks, RNG tables);
 *   this library -- runs the kernels.  No allocation and no host synchronisation
 *       inside qd_render_device(); one plan may be used from one thread at a time.
 *
 * All functions return 0 on success or a negative qd_status; qd_last_error() gives a
 * thread-local message.  All "device" pointers are CUDA device pointers on the
 * current device; `stream` is a cudaStream_t passed as void*.  The device entry
 * points take at most 2^31 - 1 clips per call (more: QD_ERR_INVALID_ARG).
 */
#ifndef QD_B200_H
#define QD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QD_ABI_VERSION 6

typedef enum qd_status {
    QD_OK = 0,
    QD_ERR_INVALID_ARG = -1,   /* bad pointer / size / enum */
    QD_ERR_UNSUPPORTED = -2,   /* e.g. n_fft not in {512,...,8192} */
    QD_ERR_CUDA = -3,          /* a CUDA call or launch failed */
    QD_ERR_WORKSPACE = -4,     /* workspace too small */
    QD_ERR_NO_DEVICE = -5      /* no sm_100 device visible: there is no CPU fallback */
} qd_status;

/* dsp/distortion.py:93-114 */
typedef enum qd_distortion_mode { QD_DIST_WAVEFOLD = 0, QD_DIST_TUBE = 1 } qd_distortion_mode;

/* dsp/pipeline.py:64-141 (one FX per render, high band only) */
typedef enum qd_fx_mode {
    QD_FX_NONE = 0,
    QD_FX_BITCRUSH_LOG = 1,      /* dsp/spectral_fx.py:248-251 */
    QD_FX_BITCRUSH_UNIFORM = 2,  /* dsp/spectral_fx.py:242-246 */
    QD_FX_PHASE_DISPERSAL = 3,   /* dsp/spectral_fx.py:263-323 */
    QD_FX_SCRAMBLE_PICK = 4,     /* dsp/spectral_fx.py:360-367 */
    QD_FX_SCRAMBLE_SWAP = 5      /* dsp/spectral_fx.py:368-381 */
} qd_fx_mode;

/*
 * Scalar parameters of one render, already resolved by the host from the reference's
 * process_audio keyword arguments (dsp/pipeline.py:1113-1155, config.py:64-130).
 */
typedef struct qd_params {
    uint32_t struct_size;        /* sizeof(qd_params), for ABI checks */
    int32_t  sample_rate;
    int32_t  n_fft;              /* dsp/pipeline.py:149 N_FFT_DEFAULT; hop = n_fft/4 */
    int32_t  n_samples;          /* samples per clip (all clips of a batch share it); longest clip for ragged renders */

    int32_t  passthrough;        /* dsp/pipeline.py:477-535 */
    int32_t  pre_quant;          /* pre_quant  and snap_strength > 0  (:635) */
    int32_t  post_quant;         /* post_quant and snap_strength > 0  (:728) */
    int32_t  bin_smoothing;      /* dsp/quantizer.py:523 */

    int32_t  distortion_mode;    /* qd_distortion_mode */
    float    tube_gain;          /* a * max(drive,0), a = 1 + 4*clip(warmth,0,1)  (:75-83) */
    float    tube_norm;          /* 1 / tanh(a)                                  (:88) */

    int32_t  limiter_on;         /* dsp/pipeline.py:882 */
    int32_t  lookahead;          /* samples, dsp/limiter.py:53 (Python round, half-even) */
    double   fold_amount;        /* dsp/distortion.py:37: the wavefold runs in float64 like the reference's */
    double   bias;               /*   ((x + bias) * fold_amount, folds, clip) and rounds to float32 once    */
    double   ceiling_lin;        /* 10^(dB/20), dsp/limiter.py:52 */
    double   release_coeff;      /* exp(-1/release_samples), dsp/limiter.py:60 */

    float    wet;                /* float32(clip(dry_wet,0,1))      dsp/pipeline.py:894-895 */
    float    dry;                /* float32(1 - clip(dry_wet,0,1)) */
    float    trim_gain;          /* float32(10^(output_trim_db/20)), applied iff apply_trim */
    int32_t  apply_trim;         /* output_trim_db != 0             (:898) */
    int32_t  delta_listen;       /* dsp/pipeline.py:1371-1375 */

    int32_t  multiband;          /* dsp/pipeline.py:1011-1110 */
    int32_t  low_delay;          /* N_FFT_DEFAULT // 2              (:1056, :380-386) */
    double   sos_low[2][6];      /* dsp/crossover.py:48-66 (scipy butter, cascaded twice) */
    double   sos_high[2][6];
    float    low_gain;           /* max(lowband_drive, 0)           dsp/saturation.py:44 */
    double   low_norm;           /* 1 / np.tanh(3.0)                dsp/saturation.py:54 */
    float    low_trim_gain;      /* float32(10^(low_trim/20)), applied iff apply_low_trim */
    int32_t  apply_low_trim;
    float    mono_a;             /* mono_strength blend, dsp/pipeline.py:1064-1070:    */
    float    mono_b;             /*   low = mono_a*l + mono_b*l  iff apply_mono_blend   */
    int32_t  apply_mono_blend;

    int32_t  fx_mode;            /* qd_fx_mode; 0 unless high band of a multiband render */
    double   fx_a;               /* bitcrush: step_db | step; dispersal: amount; scramble (random_pick): window / 2 */
    double   fx_b;               /* bitcrush: threshold factor (x frame max) or <0 = absolute in fx_c;
                                    dispersal: rand_amt */
    double   fx_c;               /* bitcrush: absolute threshold; dispersal: absolute thresh (<0: 0.01*max) */
    int32_t  fx_table_frames;    /* frames per pass in the FX random table (0 = no table) */
    int32_t  fx_table_per_clip;  /* 0: one table shared by every clip; 1: [batch] tables */

    int32_t  precision;          /* QD_PRECISION_F32: float32 FFT/quantizer (fast path);
                                    QD_PRECISION_F64: the same kernels instantiated in float64 -- the parity path
                                    for ill-conditioned configurations (band mask wide open, n_fft 8192) */
    int32_t  spectral_freeze;    /* dsp/pipeline.py:285-287, 303-304: every frame takes the magnitudes of frame 0 */
    double   formant_ratio;      /* 2^(formant_shift/12), dsp/spectral_fx.py:173; 0 = off (dsp/pipeline.py:306-310) */
    int32_t  formant_order;      /* cepstral lifter order, dsp/spectral_fx.py:120 (30) */
    int32_t  no_spectral;        /* 1: no STFT pass at all -- x_pre = band, distortion, limiter, mix.  What
                                    quantize_mode="autotune_v1" does when its pitch stage is gated off (pre_quant off or
                                    snap_strength <= 0, dsp/pipeline.py:537-601), the only form in which that mode
                                    survives inside a multiband render (:1326-1327, :1076) */
} qd_params;

#define QD_PRECISION_F32 0
#define QD_PRECISION_F64 1

/*
 * Integer/float tables built on the host in float64 (bit-exact with the reference):
 *   target_bins  dsp/quantizer.py:127-196 (or :199-250 for harmonic lock), int32[n_bins]
 *   active_mask  dsp/pipeline.py:164-177, uint8[n_bins]
 *   smear_w      dsp/quantizer.py:460-465 kernel, 5 taps, float64
 * The library derives its gather (CSR) form from these.
 */
typedef struct qd_tables {
    int32_t        n_bins;          /* n_fft/2 + 1 */
    const int32_t *target_bins;
    const uint8_t *active_mask;
    double         snap;            /* clip(snap_strength, 0, 1)  dsp/quantizer.py:405 */
    double         smear;           /* clip(smear, 0, 1)          dsp/quantizer.py:406 */
    int32_t        smear_radius;    /* 2 */
    const double  *smear_w;         /* [2*smear_radius+1] */
} qd_tables;

/* Optional extra outputs (dsp/pipeline.py:914-918, 1104-1109); NULL = not wanted. */
typedef struct qd_taps {
    float *pre_quant;   /* [batch, n_samples], or packed like x in a ragged render */
    float *post_dist;   /* [batch, n_samples], or packed like x in a ragged render */
} qd_taps;

typedef struct qd_plan qd_plan;

int         qd_abi_version(void);
const char *qd_last_error(void);
/* number of visible CUDA devices with compute capability 10.x; <= 0 means unusable */
int         qd_device_count(void);

int    qd_plan_create(const qd_params *params, const qd_tables *tables, qd_plan **out);
void   qd_plan_destroy(qd_plan *plan);
/* bytes of device scratch qd_render_device needs for `batch` clips */
size_t qd_plan_workspace_bytes(const qd_plan *plan, int64_t batch);
/* number of kernels one qd_render_device call launches (for launch accounting) */
int    qd_plan_launches_per_render(const qd_plan *plan);

/*
 * Optional device-side timing: when enabled, qd_render_device brackets the launches of each
 * kernel class with CUDA events on the launch stream.  qd_plan_read_timing waits for the
 * recorded events, returns the accumulated milliseconds and launch counts per class since
 * the last read, and resets them.
 */
#define QD_KERNEL_SPECTRAL  0   /* STFT -> FX -> quantizer -> iSTFT -> OLA (-> distortion) */
#define QD_KERNEL_LIMITER   1   /* lookahead limiter + dry/wet + trim + recombine + delta */
#define QD_KERNEL_CROSSOVER 2   /* LR4 split + low-band delay/saturation */
#define QD_KERNEL_OTHER     3
#define QD_KERNEL_CLASSES   4
int qd_plan_enable_timing(qd_plan *plan, int on);
int qd_plan_read_timing(qd_plan *plan, double ms[QD_KERNEL_CLASSES], int64_t launches[QD_KERNEL_CLASSES]);

/*
 * FX random tables replayed from np.random on the host (SURVEY.md appendix C.11):
 *   SCRAMBLE_PICK: int16 source index per bin   [tables][2 passes][frames][n_bins]
 *   SCRAMBLE_SWAP: int16 source index per bin   (same shape; the swap permutation)
 *   PHASE_DISPERSAL (randomized): float32 jitter in [-1,1)  (same shape)
 * `device_table` stays owned by the caller and must outlive the renders.
 */
int qd_plan_set_fx_table(qd_plan *plan, const void *device_table, int64_t n_tables);

/*
 * Replacement for one process_audio call per clip (dsp/pipeline.py:1113):
 *   x [batch, n_samples] float32 mono clips (device)  ->  y [batch, n_samples] float32.
 * Inputs are not modified.  Asynchronous on `stream`.
 */
int qd_render_device(qd_plan *plan, const float *x, float *y, int64_t batch,
                     const qd_taps *taps, void *workspace, size_t workspace_bytes,
                     void *stream);

/*
 * Same render with HOST buffers (pinned for full speed): clips are cut into chunks of
 * `chunk_clips`, and H2D copy, kernels and D2H copy of consecutive chunks overlap on
 * three streams.  Synchronous: returns when y_host is complete.
 */
int qd_render_host(qd_plan *plan, const float *x_host, float *y_host, int64_t batch,
                   int64_t chunk_clips);

/*
 * The same with 16-bit PCM on the PCIe link -- what a WAV-to-WAV batch render (dsp/harness.py:24-63 around
 * io/audio_io.py:10-26) actually moves.  The conversions run on the device with libsndfile's rules, the ones the
 * reference's file I/O applies on the CPU: sample / 32768 on the way in, lrint(y * 32767) clipped to int16 on the
 * way out.  Half the bytes of qd_render_host per clip.
 */
int qd_render_host_pcm16(qd_plan *plan, const int16_t *x_host, int16_t *y_host, int64_t batch,
                         int64_t chunk_clips);

/* General form: either side float32 or PCM16.  Host buffers may be pinned (cudaHostAlloc / cudaHostRegister /
 * qd_host_alloc: copied directly) or pageable (staged through an internal ring of pinned buffers by copy
 * threads, QD_HOST_COPY_THREADS per direction, default 8 on hosts with 16 or more cores).  On any error the call drains its streams before it
 * returns. */
#define QD_SAMPLE_F32   0
#define QD_SAMPLE_PCM16 1
int qd_render_host_ex(qd_plan *plan, const void *x_host, void *y_host, int64_t batch, int64_t chunk_clips,
                      int32_t in_format, int32_t out_format);

/*
 * Ragged batch: clips of different lengths in one render.  Clip c occupies x[starts[c] - starts[0] ... + lengths[c])
 * and the same span of y and of each tap.  starts: int64[batch], non-decreasing, spans do not overlap (gaps allowed:
 * the Python packer aligns every start to 16 bytes); lengths: int32[batch], each <= the plan's n_samples (the plan's
 * n_samples is the longest clip it accepts, and sizes its FX tables).  Offsets are relative to starts[0], so a
 * sub-range of clips is addressed by advancing x, y, starts and lengths together.  Samples in the gaps of y and of
 * the taps are unspecified.
 *   span_samples  packed extent, starts[batch-1] - starts[0] + lengths[batch-1]: sizes the workspace, whose
 *                 intermediates are packed like x
 *   max_samples   the longest clip of the batch (<= n_samples): sizes the grid
 * qd_render_device_varlen never reads `starts` / `lengths` on the host (device arrays; the caller validates them);
 * qd_render_host_varlen takes host arrays, validates them (QD_ERR_INVALID_ARG), uploads them once per call and cuts
 * the batch into clip ranges whose packed span fits `chunk_samples` (a longer clip gets a chunk of its own).  The
 * uniform entry points above are the special case starts[c] = c * n_samples, lengths[c] = n_samples.
 */
size_t qd_plan_workspace_bytes_varlen(const qd_plan *plan, int64_t batch, int64_t span_samples);
int qd_render_device_varlen(qd_plan *plan, const float *x, float *y, const int64_t *starts /* device */,
                            const int32_t *lengths /* device */, int64_t batch, int64_t span_samples,
                            int32_t max_samples, const qd_taps *taps, void *workspace, size_t workspace_bytes,
                            void *stream);
int qd_render_host_varlen(qd_plan *plan, const void *x_host, void *y_host, const int64_t *starts /* host */,
                          const int32_t *lengths /* host */, int64_t batch, int64_t chunk_samples,
                          int32_t in_format, int32_t out_format);

/* Stage-level entry points (parity ladder, SURVEY.md section 7.3b). All async on `stream`. */
/* dsp/limiter.py:14-80 on [batch, n] */
int qd_limiter_device(const float *x, float *y, int64_t batch, int64_t n, int32_t lookahead,
                      double ceiling_lin, double release_coeff, void *stream);
/* dsp/crossover.py:71-118 on [batch, n]: float32 low and high bands */
int qd_crossover_device(const float *x, float *low, float *high, int64_t batch, int64_t n,
                        const double sos_low[2][6], const double sos_high[2][6], void *stream);
/* dsp/distortion.py:93-114 elementwise on `count` samples */
int qd_distort_device(const float *x, float *y, int64_t count, int32_t mode, double fold_amount,
                      double bias, float tube_gain, float tube_norm, void *stream);

/*
 * Device half of the scale-alignment metric avg_cents_offset_from_scale (dsp/analyses.py:53-142):
 * the STFT of every clip (dsp/stft_utils.py:11-97, n_fft = frame_length, hop n_fft/4, centre padded) and, per
 * frame, the `topn` (<= 8) strongest bins in descending magnitude among bins 1..n_fft/2 whose magnitude is
 * >= min_mag = 10^(min_db/20); bins [batch][1 + n/hop][topn] int16, -1 where fewer qualify.  The caller maps
 * bins to cents with its float64 table (quantumdistortion_b200/analyses.py).  precision: QD_PRECISION_*.
 */
int qd_spectral_peaks_device(const float *x, int64_t batch, int32_t n_samples, int32_t n_fft, int32_t topn,
                             double min_mag, int32_t precision, int16_t *bins, void *stream);

/*
 * quantize_mode = "autotune_v1", the reference's default mode (dsp/autotune.py:426-447 behind dsp/pipeline.py:537-601):
 * zero-phase band split -> YIN pitch track -> note hold -> granular pitch shifter -> sub layer, then the same
 * distortion / limiter / mix tail as the STFT path.  Everything the reference derives on the CPU (Butterworth
 * sections and sosfilt_zi from scipy, sample counts, key / scale tables) arrives resolved in this struct
 * (quantumdistortion_b200/autotune.py builds it).
 */
typedef struct qd_autotune_params {
    uint32_t struct_size;
    int32_t  sample_rate;
    int32_t  n_samples;
    int32_t  apply;              /* pre_quant and snap_strength > 0 (dsp/pipeline.py:538); 0: x_pre = x */
    /* zero-phase 4th-order Butterworth filters, dsp/autotune.py:88-127: [0] sub low-pass, [1] air high-pass,
       [2] detector high-pass, [3] detector low-pass; filt_on = 0 when the cutoff is <= 0 */
    int32_t  filt_on[4];
    double   sos[4][2][6];
    double   zi[4][2][2];        /* scipy.signal.sosfilt_zi */
    /* detector, dsp/autotune.py:140-236 */
    int32_t  frame_size;         /* 4096 */
    int32_t  hop;                /* 512 */
    int32_t  min_tau, max_tau;   /* dsp/autotune.py:153-154 */
    double   min_freq, max_freq, yin_threshold;
    double   rms_thr, flat_thr, conf_thr;
    /* note hold, dsp/autotune.py:65-85, 238-277 */
    int32_t  root_pc, n_intervals, intervals[8];
    double   strength, change_cents;
    int32_t  confirm_frames, release_frames;
    /* granular shifter, dsp/autotune.py:301-360 */
    int32_t  max_delay;          /* max(256, grain_size) */
    int32_t  buffer_size;        /* power of two >= 2 * max_delay */
    /* sub layer and mix, dsp/autotune.py:363-437 */
    int32_t  sub_enabled;
    int32_t  layer_on;           /* sub_enabled and sub_level > 0 and sub frequency > 0 */
    float    env_attack, env_release;   /* float32(exp(-1 / max(1, ms * sr / 1000))) */
    float    sub_level, sub_preserve, air_mix;
    float    phase_k;            /* float32(2 pi f_sub) */
    /* shared tail, same meaning as in qd_params */
    int32_t  distortion_mode;
    float    tube_gain, tube_norm;
    int32_t  limiter_on, lookahead;
    double   fold_amount, bias;
    double   ceiling_lin, release_coeff;
    float    wet, dry, trim_gain;
    int32_t  apply_trim, delta_listen;
} qd_autotune_params;

/* optional device outputs of the intermediate stages (parity ladder); NULL members are skipped */
typedef struct qd_autotune_debug {
    float  *sub, *body, *air, *det;     /* [batch, n] bands and detector side chain */
    float  *ratio_track;                /* [batch, n] */
    float  *corrected;                  /* [batch, n] shifted body */
    float  *sub_layer;                  /* [batch, n] */
    double *features;                   /* [batch, ceil(n / hop), 4]: rms, flatness, pitch, confidence */
} qd_autotune_debug;

size_t qd_autotune_workspace_bytes(const qd_autotune_params *params, int64_t batch);
int    qd_autotune_render_device(const qd_autotune_params *params, const float *x, float *y, int64_t batch,
                                 const qd_taps *taps, const qd_autotune_debug *debug, void *workspace,
                                 size_t workspace_bytes, void *stream);

/*
 * Ragged batch of the autotune_v1 mode: clips of different lengths in one call, packed as in qd_render_device_varlen
 * (clip c at x[starts[c] - starts[0] ... + lengths[c]), y and the taps packed the same way, gap samples unspecified;
 * starts / lengths are device arrays that are not read on the host).  params->n_samples is the longest clip the call
 * accepts; max_samples is the longest clip of the batch.  Every clip renders exactly as it does alone.  With the
 * pitch stage on (params->apply), a clip of 1..15 samples is not rendered (the caller rejects it, as
 * qd_autotune_render_device rejects such a batch); a zero-length clip is skipped.  No debug outputs: those are for
 * uniform batches.  qd_autotune_render_device is the special case starts[c] = c * n_samples.
 */
size_t qd_autotune_workspace_bytes_varlen(const qd_autotune_params *p, int64_t batch, int64_t span_samples);
int    qd_autotune_render_device_varlen(const qd_autotune_params *p, const float *x, float *y,
                                        const int64_t *starts /* device */, const int32_t *lengths /* device */,
                                        int64_t batch, int64_t span_samples, int32_t max_samples,
                                        const qd_taps *taps, void *workspace, size_t workspace_bytes, void *stream);

/*
 * Measurement helper for the roofline report: FP32 throughput of the CUDA cores in TFLOP/s, measured with the packed
 * fma.rn.f32x2 (FFMA2) instruction the spectral pass is built from (best of a few launches on `stream`; synchronous).
 */
int qd_measure_fp32_peak(double *tflops, void *stream);

/* pinned host memory helpers for qd_render_host callers */
void *qd_host_alloc(size_t bytes);
void  qd_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* QD_B200_H */
