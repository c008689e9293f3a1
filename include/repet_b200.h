/*
 * repet_b200.h -- C ABI of the B200-native REPET separation path (librepet_b200.so).
 *
 * The reference (zafarrafii/REPET-Python, repet.py) has no FFI: its boundary is the Python
 * module surface `repet.original/extended/adaptive/sim/simonline(audio_signal, fs)` plus the
 * private helpers `_stft ... _simmask`.  Each entry point below names the reference
 * function (repet.py line) it replaces; `repet-python_b200/repet/_host.py` is the ctypes
 * binding a maintainer of the reference would add (see INTEGRATION.md).
 *
 * Conventions
 *  - Plain pointers and sizes only; no torch / numpy types.  Every function returns an int
 *    status: 0 = REPET_OK, negative = error; `repet_last_error(h)` gives the message.
 *  - "_dev" functions take DEVICE pointers and enqueue on the handle's stream without
 *    synchronising (unless a host output such as `periods_host` is requested).  The others
 *    take HOST pointers and include the host<->device copies.
 *  - Audio is fp32 planar [clip][channel][sample] unless the name says f64 (the reference's
 *    float64 (sample, channel) NumPy layout, repet.py:73-77).
 *  - The caller owns every buffer.  Calls on one handle are stream-ordered and not
 *    re-entrant; use one handle per GPU and per host thread.
 *  - All derived integers (period range in frames, cutoff bin, segment sizes ...) are computed
 *    by the host with the reference's own Python expressions and passed in `repet_params`.
 */
#ifndef REPET_B200_H
#define REPET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REPET_OK 0
#define REPET_E_INVALID_ARG (-1) /* maps to ValueError on the Python side (quirk Q17) */
#define REPET_E_TOO_SHORT (-2)   /* clip too short for the period search: ValueError in the reference */
#define REPET_E_CUDA (-3)
#define REPET_E_OOM (-4)
#define REPET_E_UNSUPPORTED (-5) /* e.g. a window length this build has no transform for */

typedef struct repet_handle repet_handle;

/* Derived parameters; host computes them exactly as the reference does. */
typedef struct repet_params {
    int32_t window_length;    /* N  = 2^ceil(log2(0.04 fs))              repet.py:130 */
    int32_t step_length;      /* H  = N/2                                repet.py:132 */
    int32_t period_lo;        /* round(period_range[0]*fs/H)             repet.py:165 */
    int32_t period_hi;        /* round(period_range[1]*fs/H)             repet.py:165 */
    int32_t cutoff_bins;      /* round(cutoff_frequency*N/fs)            repet.py:173 */
    int32_t segment_length;   /* extended: samples (repet.py:266); adaptive: frames (repet.py:519) */
    int32_t segment_step;     /* extended: samples (repet.py:267); adaptive: frames (repet.py:520) */
    int32_t filter_order;     /* adaptive median order                   repet.py:54   */
    int32_t similarity_distance; /* frames                               repet.py:670 */
    int32_t similarity_number;   /*                                      repet.py:60  */
    int32_t buffer_frames;    /* simonline ring length in frames         repet.py:787 */
    int32_t online_frame_base; /* simonline on a window of a longer stream: absolute index of the window's
                                * first frame (ring slot = absolute frame mod buffer_frames, quirk Q6); 0 otherwise */
    double similarity_threshold; /*                                      repet.py:58  */
    double cola_gain;         /* sum(window[0:N:H])                      repet.py:1103 */
} repet_params;

/* ---- lifetime --------------------------------------------------------------------------- */
int repet_create(int device, repet_handle** out);
int repet_destroy(repet_handle* h);
const char* repet_last_error(repet_handle* h);
/* Use an existing CUDA stream (cudaStream_t passed as void*); NULL restores the handle's own
 * stream; pass cudaStreamLegacy ((void*)0x1) for the legacy default stream. */
int repet_set_stream(repet_handle* h, void* cuda_stream);
/* Analysis window, HOST pointer, n = window length (built with SciPy's periodic Hamming by the
 * host, repet.py:131 -- SciPy's values differ from the closed form by up to 1 ulp). */
int repet_set_window(repet_handle* h, const double* window, int n);
/* Cap on the workspace (bytes) a batch call may use per chunk of clips; 0 = default (min(24 GiB, 40 % of the
 * device memory free when the handle first asks)).  A chunk never holds less than one clip, so one clip whose
 * workspace alone exceeds the cap still runs.  REPET-SIM honours the cap for long tracks too: when a track's
 * similarity matrix does not fit, it is formed and consumed in row panels as high as the cap leaves room for
 * (at least 128 rows), one track at a time.  repet_general_f64's REPET-SIM honours the cap as well: its float64
 * similarity matrix and selection scratch are formed in row panels (multiples of 64 rows, at least 64) when the whole
 * matrix does not fit; its buffers that grow linearly with the track are not counted.  Buffers an entry point stages
 * its own input and output in come on top. */
int repet_set_workspace_limit(repet_handle* h, uint64_t bytes);
/* Bytes of device workspace the handle holds now (it grows on demand and is kept for later calls). */
uint64_t repet_workspace_bytes(repet_handle* h);
int repet_synchronize(repet_handle* h);
/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
uint64_t repet_launch_count(repet_handle* h);
const char* repet_version(void);

/* Per-kernel device time for the roofline report: with profiling on, every launch is
 * bracketed by a CUDA event pair on the handle's stream.  repet_profile_read synchronises the
 * stream and returns accumulated milliseconds and launch counts per kernel id. */
#define REPET_NUM_KERNELS 12
#define REPET_K_STFT 0
#define REPET_K_BEAT 1
#define REPET_K_PERIODS 2
#define REPET_K_MODEL 3
#define REPET_K_MASK_ISTFT 4
#define REPET_K_CONVERT 5
#define REPET_K_XFADE 6
#define REPET_K_NORMALIZE 7
#define REPET_K_SIMGEMM 8
#define REPET_K_TOPK 9
/* Process-wide launch-shape knobs for experiments: "stft_minb", "mask_minb" (resident CTAs per SM
 * the FFT kernels are compiled for: 4, 5, 6), "frames_per_cta", "beat_parts" (0 = automatic), "simgemm_tc" (2 = tcgen05 3xTF32 split
 * similarity GEMM, 1 = single-pass TF32, 0 = fp32 CUDA-core cross-check kernel), "sim_frames64" (1 = similarity
 * operand from the float64 front end, 0 = from the fp32 magnitudes), "cert_rel_ppm" (period certification window). */
int repet_set_tuning(const char* name, int value);
int repet_set_profiling(repet_handle* h, int on);
int repet_profile_read(repet_handle* h, double* ms, uint64_t* counts, int reset);
const char* repet_kernel_name(int id);

/* ---- drivers ---------------------------------------------------------------------------- */
/* repet.original (repet.py:67-202) over a batch of equally long clips, device resident.
 * audio/background: [n_clips][n_channels][n_samples] fp32 on the device.
 * periods_dev: optional int32[n_clips] on the device; periods_host: optional host copy
 * (forces a stream synchronise). */
int repet_original_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                             const repet_params* p, float* background, int32_t* periods_dev, int32_t* periods_host);
/* Same with HOST buffers (pinned memory recommended); copies are chunked and overlapped. */
int repet_original_batch(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                         const repet_params* p, float* background, int32_t* periods_host);
/* Same with int16 PCM input in WAV order [n_clips][n_samples][n_channels] (what wavread reads before it
 * normalises by 2^15, repet.py:926-929): half the host-to-device bytes; output fp32 planar. */
int repet_original_batch_pcm16(repet_handle* h, const int16_t* audio, int n_clips, int n_channels, int64_t n_samples,
                               const repet_params* p, float* background, int32_t* periods_host);
/* Any driver (method 0 original, 1 extended, 2 adaptive, 3 sim, 4 simonline) over a batch of equally long clips in
 * HOST memory, with the sample format of either side chosen by the caller:
 *   REPET_FMT_F32_PLANAR  [n_clips][n_channels][n_samples] fp32
 *   REPET_FMT_PCM16       [n_clips][n_samples][n_channels] int16, WAV order: what scipy.io.wavfile.read hands
 *                         repet.wavread before it normalises by 2^15 (repet.py:926-929), and what an int16 WAVE
 *                         writer stores after the separation (repet.wavwrite, repet.py:934-946).  Input is
 *                         normalised on the device; output is round(y * 2^15) saturated to int16 (LOSSY: adds up to
 *                         2^-16 of absolute error on top of the fp32 path's).
 * PCM16 on both sides moves 2 + 2 bytes per sample over the host link instead of 4 + 4.
 * ints_host: optional, [n_clips][repet_ints_per_clip(method, p, n_samples)]. */
#define REPET_FMT_F32_PLANAR 0
#define REPET_FMT_PCM16 1
int repet_separate_batch(repet_handle* h, int method, const void* audio, int in_format, int n_clips, int n_channels,
                         int64_t n_samples, const repet_params* p, void* background, int out_format, int32_t* ints_host);
int64_t repet_ints_per_clip(int method, const repet_params* p, int64_t n_samples);
/* Page-locked host memory for the host-buffer entry points (portable across the GPUs of the process): allocate
 * it, or pin an existing allocation in place (e.g. a NumPy array) for the duration of the calls. */
int repet_host_alloc(void** out, uint64_t bytes);
int repet_host_free(void* ptr);
int repet_host_register(void* ptr, uint64_t bytes);
int repet_host_unregister(void* ptr);
int repet_device_count(void);
/* The reference's exact calling convention for one clip: float64 (n_samples, n_channels)
 * in and out, host pointers (repet.py:73-77). */
int repet_original_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels,
                       const repet_params* p, double* background, int32_t* period_host);

/* repet.extended (repet.py:205-419): `original` on 10 s segments every 5 s with a triangular
 * cross-fade.  p->segment_length / segment_step are in SAMPLES.  Integer output: the period of
 * every segment, [n_clips][repet_extended_segments(p, n_samples)]. */
int repet_extended_segments(const repet_params* p, int64_t n_samples);
int repet_extended_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                             const repet_params* p, float* background, int32_t* periods_dev, int32_t* periods_host);
int repet_extended_batch(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                         const repet_params* p, float* background, int32_t* periods_host);
int repet_extended_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                       double* background, int32_t* periods_host, int periods_capacity);

/* repet.adaptive (repet.py:422-568): sliding beat spectrogram, per-frame periods, per-frame
 * median over <= filter_order period-offset frames.  p->segment_length / segment_step are in
 * FRAMES.  Integer output: the period of every frame, [n_clips][n_frames]. */
int repet_adaptive_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                             const repet_params* p, float* background, int32_t* periods_dev, int32_t* periods_host);
int repet_adaptive_batch(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                         const repet_params* p, float* background, int32_t* periods_host);
int repet_adaptive_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                       double* background, int32_t* periods_host, int periods_capacity);

/* repet.sim (repet.py:571-709): cosine self-similarity of the channel-mean magnitude frames,
 * per-frame lists of the most similar frames (strict local maxima within +-similarity_distance
 * frames, >= similarity_threshold, best similarity_number by value), median over each list.
 * The fast similarity matrix only proposes candidates; every decision is certified with exact
 * float64 dot products.  Integer output per clip: [counts n_frames][indices n_frames x number]
 * (n_frames = the centred frame count; list i holds counts[i] valid frame indices, most similar
 * first). */
int repet_sim_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                        const repet_params* p, float* background, int32_t* lists_dev, int32_t* lists_host);
int repet_sim_batch(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                    const repet_params* p, float* background, int32_t* lists_host);
int repet_sim_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                  double* background, int32_t* lists_host, int lists_capacity);

/* repet.simonline (repet.py:712-911): every frame j >= buffer_frames-1 against the previous
 * buffer_frames-1 frames in ring-buffer slot order; frames are NOT centred and earlier frames are
 * never synthesised.  All frames are independent, so the whole signal is processed in parallel.
 * Integer output per clip as for repet_sim with n_frames = repet_simonline_frames(p, n_samples);
 * lists hold FRAME indices. */
int repet_simonline_frames(const repet_params* p, int64_t n_samples);
int repet_simonline_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                              const repet_params* p, float* background, int32_t* lists_dev, int32_t* lists_host);
int repet_simonline_batch(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                          const repet_params* p, float* background, int32_t* lists_host);
int repet_simonline_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                        double* background, int32_t* lists_host, int lists_capacity);

/* Stateful stream of the online REPET-SIM (repet.py:712-911 fed block by block; SURVEY.md section 8(b)).  The
 * stream keeps its sample history (the last buffer_length seconds) in device memory: a block costs one upload
 * of the new samples and one download of the samples that became final.  repet_simonline_block takes the next
 * n_samples x n_channels float64 samples (host) and writes the background samples that have become final (every
 * frame covering them is complete: a latency of one hop); repet_simonline_flush returns the rest, zero-padding
 * the last frame as the reference does.  The concatenated outputs equal repet_simonline_f64 on the whole signal
 * (same ring-slot order, quirk Q6; nothing before frame buffer_frames-1, quirk Q5).  `capacity` = samples per
 * channel the background buffer holds (a block can release at most n_samples + one hop of them); *n_out = samples
 * per channel written.  One stream per handle at a time (calls are stream-ordered on the handle). */
typedef struct repet_stream repet_stream;
int repet_simonline_open(repet_handle* h, const repet_params* p, int n_channels, repet_stream** out);
int repet_simonline_block(repet_stream* s, const double* block, int64_t n_samples, double* background, int64_t capacity,
                          int64_t* n_out);
int repet_simonline_flush(repet_stream* s, double* background, int64_t capacity, int64_t* n_out);
int repet_simonline_close(repet_stream* s);

/* ---- by-products of a separation (README.md:64-81 of the reference) ---------------------- */
/* One call for the reference's documented usage: background = method(audio) (method 0 original, 1 extended,
 * 2 adaptive, 3 sim, 4 simonline), foreground = audio - background (README.md:68), and the three display
 * spectrograms abs(_stft(mean(x, axis=1)))[0:F] of mixture, background and foreground (README.md:79-81),
 * all from buffers already resident on the device.  float64 (n_samples, n_channels) in and out, HOST
 * pointers; foreground (optional) like background; spectrograms (optional) fp32
 * [3][repet_spectrogram_frames][repet_spectrogram_pitch], bins 0..N/2 of every row valid; ints as the
 * method's own *_f64 entry point. */
int repet_separate_f64(repet_handle* h, int method, const double* audio, int64_t n_samples, int n_channels,
                       const repet_params* p, double* background, double* foreground, float* spectrograms,
                       int32_t* ints_host, int ints_capacity);
int repet_spectrogram_pitch(const repet_params* p);                     /* floats per spectrogram row: F rounded up to 8 */
int repet_spectrogram_frames(const repet_params* p, int64_t n_samples); /* repet.py:1018-1028 */
/* Display spectrogram of every clip of a device-resident batch: audio [n_clips][n_channels][n_samples] fp32 ->
 * spectrogram [n_clips][frames][pitch] fp32 (device). */
int repet_spectrogram_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                                const repet_params* p, float* spectrogram);
/* foreground = audio - background over n_elements fp32 values, device pointers (16-byte aligned). */
int repet_foreground_dev(repet_handle* h, const float* audio, const float* background, int64_t n_elements,
                         float* foreground);

/* ---- helpers (unit parity with the reference's private functions), HOST pointers -------- */
/* _stft (repet.py:1001-1060) of n_channels (1 or 2) real signals at once.
 * signal: [n_channels][n_samples] fp32; spectrum: [n_frames][n_channels][N/2] float2 with
 * bin 0 = (DC.re, Nyquist.re); power (optional): [n_frames][1025] fp32 = (mean_c |X|)^2. */
int repet_stft(repet_handle* h, const float* signal, int n_channels, int64_t n_samples, float* spectrum,
               float* power, int32_t* n_frames_out);
/* _istft (repet.py:1063-1105): spectrum as above -> signal [n_channels][(n_frames-1)*H]. */
int repet_istft(repet_handle* h, const float* spectrum, int n_channels, int n_frames, double cola_gain,
                float* signal);
/* _beatspectrum (repet.py:1142-1158): spectrogram [n_frames][n_rows] fp32 (time major),
 * n_rows <= 1025, 2*n_frames-1 <= 2048 -> beat[n_frames] float64. */
int repet_beatspectrum(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, double* beat);
/* _periods on the device beat spectrum of the same input (repet.py:1249-1291): returns the
 * period for lags [period_lo, min(period_hi, n_frames/3)). */
int repet_period(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, int period_lo, int period_hi,
                 int32_t* period);
/* _mask (repet.py:1386-1458): magnitude spectrogram [n_frames][1025] fp32 + period ->
 * mask [n_frames][1025] fp32. */
int repet_mask(repet_handle* h, const float* magnitude, int n_frames, int period, float* mask);

/* _adaptivemask (repet.py:1461-1508): magnitudes [n_frames][1025], per-frame periods, order ->
 * mask [n_frames][1025]. */
int repet_adaptivemask(repet_handle* h, const float* magnitude, int n_frames, const int32_t* periods, int filter_order,
                       float* mask);
/* _beatspectrogram (repet.py:1161-1206) before the column replication: the beat spectrum of
 * every segment i = 0, step, 2 step, ... -> beat[n_segments][segment_length] float64. */
int repet_beatspectrogram(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, int segment_length,
                          int segment_step, double* beat, int32_t* n_segments_out);
/* _selfsimilaritymatrix (repet.py:1209-1225), fast pass only: magnitudes [n_frames][n_rows<=1025]
 * -> fp32 cosine similarity [n_frames][n_frames] (TF32 tensor-core product; the drivers certify
 * every decision they take from it in float64). */
int repet_selfsimilarity(repet_handle* h, const float* magnitude, int n_frames, int n_rows, float* similarity);
/* _periods (repet.py:1249-1291) on a caller-provided beat spectrum (n_columns = 1) or beat
 * spectrogram, beat[n_lags][n_columns] row-major float64 -> periods[n_columns]. */
int repet_periods(repet_handle* h, const double* beat, int n_lags, int n_columns, int period_lo, int period_hi,
                  int32_t* periods);

/* _similaritymatrix / _selfsimilaritymatrix (repet.py:1209-1246) in exact float64: magnitudes
 * [n_frames1][n_rows], [n_frames2][n_rows] (n_rows <= 1025) -> cosine similarity [n_frames1][n_frames2]. */
int repet_similarity(repet_handle* h, const float* magnitude1, int n_frames1, const float* magnitude2, int n_frames2,
                     int n_rows, double* similarity);
/* _localmaxima (n_columns = 1) / _indices (repet.py:1294-1383) on caller-provided float64 data
 * [n][n_columns] row-major: per column the indices (and optionally values) of the strict local maxima,
 * best first; indices/values [n_columns][number_values], counts [n_columns]. */
int repet_localmaxima(repet_handle* h, const double* data, int n, int n_columns, double minimum_value,
                      int minimum_distance, int number_values, int32_t* indices, int32_t* counts, double* values);
/* _simmask (repet.py:1511-1545): magnitudes [n_frames][1025], lists indices[n_frames][number] with
 * counts[n_frames] -> mask [n_frames][1025]. */
int repet_simmask(repet_handle* h, const float* magnitude, int n_frames, const int32_t* indices, const int32_t* counts,
                  int number, float* mask);
/* _acorr (repet.py:1108-1139): data [n_rows][n_columns] fp32 row-major, 2*n_rows-1 <= 2048 ->
 * unbiased autocorrelation of every column, float64 [n_rows][n_columns]. */
int repet_acorr(repet_handle* h, const float* data, int n_rows, int n_columns, double* autocorrelation);

/* ---- general-size float64 helpers ----------------------------------------------------------
 * The reference's private helpers take ANY window, step and matrix size (its README calls _stft directly,
 * README.md:79-81); these entry points do too, in float64 throughout (power-of-two transforms by radix-2 passes,
 * any other length by Bluestein's algorithm).  HOST pointers. */
/* number of frames of _stft (repet.py:1018-1028) for any window length and step */
int repet_stft_frames(int64_t n_samples, int window_length, int step_length);
/* _stft (repet.py:1001-1060): signal[n_samples], window[window_length] -> spectrum, the reference's own layout:
 * (window_length, n_frames) C-order complex128, i.e. double[window_length][n_frames][2], all bins. */
int repet_stft_f64(repet_handle* h, const double* signal, int64_t n_samples, const double* window, int window_length,
                   int step_length, double* spectrum, int32_t* n_frames_out);
/* _istft (repet.py:1063-1105): spectrum as above -> signal[n_frames*step - (window_length - step)]
 * (real part of the inverse transforms, overlap-add, trim, divide by sum(window[0:N:step])). */
int repet_istft_f64(repet_handle* h, const double* spectrum, int window_length, int n_frames, const double* window,
                    int step_length, double* signal, int64_t* n_samples_out);
/* _acorr (repet.py:1108-1139), any n_rows: data[n_rows][n_columns] float64 row-major -> same shape. */
int repet_acorr_f64(repet_handle* h, const double* data, int n_rows, int n_columns, double* autocorrelation);
/* _beatspectrum (repet.py:1142-1158), any size: spectrogram[n_frequencies][n_times] float64 -> beat[n_times]. */
int repet_beatspectrum_f64(repet_handle* h, const double* spectrogram, int n_frequencies, int n_times, double* beat);

/* ---- general float64 drivers ---------------------------------------------------------------
 * repet.original / extended / adaptive / sim / simonline (repet.py:67-911; method 0..4) for the inputs the fast fp32
 * kernels are not compiled for: window lengths other than 512 / 1024 / 2048 (sampling rates above 51.2 kHz: 4096
 * points at 96 kHz, 8192 at 192 kHz, repet.py:130), any number of channels (repet.py:152-155), period ranges above
 * 1024 frames, segments longer than one beat transform.  float64 end to end on the device (integer decisions need no
 * certification), built for generality, not speed.  audio / background: (n_samples, n_channels) float64, HOST;
 * window: the analysis window (window_length doubles, HOST); ints_host as repet_ints_per_clip(method, p, n_samples).
 * REPET-SIM (method 3) forms the T x T float64 similarity matrix whole when it and the selection scratch fit the
 * handle's workspace limit (repet_set_workspace_limit), else in row panels of the largest multiple of 64 rows that
 * fits; the matrix is bitwise symmetric, so panels give the same lists and background bit for bit.  The buffers
 * linear in T (spectra, magnitudes, staging: about 36 GB for one hour of 96 kHz mono) are outside the limit, and a
 * clip needs T * window_length < 2e9 (about 2.9 h at 96 kHz) or the call returns REPET_E_UNSUPPORTED. */
int repet_general_f64(repet_handle* h, int method, const double* audio, int64_t n_samples, int n_channels,
                      const repet_params* p, const double* window, double* background, int32_t* ints_host,
                      int64_t ints_capacity);

#ifdef __cplusplus
}
#endif
#endif /* REPET_B200_H */
