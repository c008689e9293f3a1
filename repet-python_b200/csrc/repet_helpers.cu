// Helper-level entry points (repet.py:1001-1545) of one window-length instantiation, and its entry
// table.  The extern "C" functions in repet_abi.cu dispatch here.
#include "repet_internal.h"

#include <cmath>
#include <cstdio>
#include <cstring>

namespace repet {

int drv_batch_dev(repet_handle*, int, const float*, int, int, int64_t, const repet_params*, float*, int32_t*, int32_t*);
int drv_batch_host(repet_handle*, int, const void*, int, int, int, int64_t, const repet_params*, void*, int, int32_t*);
int drv_single_f64(repet_handle*, int, const double*, int64_t, int, const repet_params*, double*, int32_t*, int64_t);
int drv_separate_f64(repet_handle*, int, const double*, int64_t, int, const repet_params*, double*, double*, float*,
                     int32_t*, int64_t);
int drv_spectrogram_dev(repet_handle*, const float*, int, int, int64_t, const repet_params*, float*);
int drv_foreground_dev(repet_handle*, const float*, const float*, int64_t, float*);
int drv_single_f64_dev(repet_handle*, int, const double*, int64_t, int, const repet_params*, double*);

// ---------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------
int hlp_stft(repet_handle* h, const float* signal, int n_channels, int64_t n_samples, float* spectrum, float* power,
               int32_t* n_frames_out) {
    if (!h) return REPET_E_INVALID_ARG;
    if (n_channels < 1 || n_channels > 2) return fail(h, REPET_E_UNSUPPORTED, "1 or 2 channels supported");
    if (!h->win[WIN_SLOT].window_set) return fail(h, REPET_E_INVALID_ARG, "repet_set_window has not been called");
    if (!signal || !spectrum || n_samples < 0) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const int T = frames_of(n_samples);
    if (n_frames_out) *n_frames_out = T;
    const size_t n = (size_t)n_samples * n_channels;
    const size_t x_elems = (size_t)T * n_channels * XPITCH;
    float *in, *P; float2* X;
    int rc = carve_arena(h, [&](Bump& b) {
        in = b.take<float>(n);
        X = b.take<float2>(x_elems);
        P = b.take<float>((size_t)T * PPITCH);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(in, signal, n * sizeof(float), cudaMemcpyHostToDevice, st));
    Geom g{1, 1, 0, 0, n_samples, 0, (int)n_samples, T};
    launch_stft(st, in, g, n_channels, window_of(h), tables(h), X, power ? P : nullptr, P_POWER, 8);
    h->launches += 1;
    CU(cudaMemcpyAsync(spectrum, X, x_elems * sizeof(float2), cudaMemcpyDeviceToHost, st));
    if (power)
        CU(cudaMemcpy2DAsync(power, NBIN * sizeof(float), P, PPITCH * sizeof(float), NBIN * sizeof(float), T,
                             cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_istft(repet_handle* h, const float* spectrum, int n_channels, int n_frames, double cola_gain, float* signal) {
    if (!h) return REPET_E_INVALID_ARG;
    if (n_channels < 1 || n_channels > 2) return fail(h, REPET_E_UNSUPPORTED, "1 or 2 channels supported");
    if (!spectrum || !signal || n_frames < 2) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const long long S = (long long)(n_frames - 1) * HOP;
    const size_t x_elems = (size_t)n_frames * n_channels * XPITCH;
    float2* X; float* out;
    int rc = carve_arena(h, [&](Bump& b) {
        X = b.take<float2>(x_elems);
        out = b.take<float>((size_t)S * n_channels);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(X, spectrum, x_elems * sizeof(float2), cudaMemcpyHostToDevice, st));
    Geom g{1, 1, 0, 0, S, 0, (int)S, n_frames};
    launch_istft(st, X, g, n_channels, (float)(1.0 / ((double)WIN_N * cola_gain)), tables(h), out, 8);
    h->launches += 1;
    CU(cudaMemcpyAsync(signal, out, (size_t)S * n_channels * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_beat_common(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, int lag_lo, int lag_hi,
                       double* beat, int32_t* period) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!spectrogram || n_frames < 1 || n_rows < 1 || n_rows > NBIN)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size (n_rows <= window_length / 2 + 1)");
    const int max_lag = beat ? n_frames - 1 : lag_hi - 1;
    if (n_frames + max_lag > BEAT_L)
        return fail(h, REPET_E_UNSUPPORTED, "n_frames + max lag exceeds the 2048-point beat transform");
    CU(cudaSetDevice(h->device));
    const int n_parts = 17, f_per_part = 64;
    float *P, *psd; double* b; int32_t* per;
    int rc = carve_arena(h, [&](Bump& w) {
        P = w.take<float>((size_t)n_frames * PPITCH);
        psd = w.take<float>((size_t)n_parts * BEAT_L);
        b = w.take<double>(BEAT_L);
        per = w.take<int32_t>(1);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemsetAsync(P, 0, (size_t)n_frames * PPITCH * sizeof(float), st));
    CU(cudaMemcpy2DAsync(P, PPITCH * sizeof(float), spectrogram, n_rows * sizeof(float), n_rows * sizeof(float),
                         n_frames, cudaMemcpyHostToDevice, st));
    launch_beat(st, P, 1, n_frames, 0, n_frames, 0, 1, tables(h), psd, n_parts, f_per_part);
    launch_periods(st, psd, nullptr, 1, n_parts, n_frames, (double)n_rows, lag_lo, lag_hi, 0, beat ? n_frames : 0,
                   beat ? b : nullptr, BEAT_L, period ? per : nullptr, nullptr, nullptr);
    h->launches += 2;
    if (beat) CU(cudaMemcpyAsync(beat, b, (size_t)n_frames * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (period) CU(cudaMemcpyAsync(period, per, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

// magnitudes [n_frames][NBIN] as purely real spectra; bin 0 packs (DC, Nyquist)
static void pack_magnitudes(const float* magnitude, int T, std::vector<float2>& host) {
    host.resize((size_t)T * XPITCH);
    for (int j = 0; j < T; ++j) {
        const float* row = magnitude + (size_t)j * NBIN;
        host[(size_t)j * XPITCH] = make_float2(row[0], row[XPITCH]);
        for (int k = 1; k < XPITCH; ++k) host[(size_t)j * XPITCH + k] = make_float2(row[k], 0.f);
    }
}

int hlp_mask(repet_handle* h, const float* magnitude, int n_frames, int period, float* mask) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!magnitude || !mask || n_frames < 1 || period < 1) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const int T = n_frames;
    const size_t x_elems = (size_t)T * XPITCH;
    float2* X; float *model, *M; int32_t* per;
    int rc = carve_arena(h, [&](Bump& b) {
        X = b.take<float2>(x_elems);
        model = b.take<float>((size_t)period * PPITCH);
        M = b.take<float>((size_t)T * PPITCH);
        per = b.take<int32_t>(1);
    });
    if (rc) return rc;
    std::vector<float2> host;
    pack_magnitudes(magnitude, T, host);
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(X, host.data(), x_elems * sizeof(float2), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(per, &period, sizeof(int32_t), cudaMemcpyHostToDevice, st));
    launch_model(st, X, 1, T, 1, per, period, model);
    launch_mask_only(st, X, 1, T, 1, per, period, model, M);
    h->launches += 2;
    CU(cudaMemcpy2DAsync(mask, NBIN * sizeof(float), M, PPITCH * sizeof(float), NBIN * sizeof(float), T,
                         cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_adaptivemask(repet_handle* h, const float* magnitude, int n_frames, const int32_t* periods, int filter_order,
                       float* mask) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!magnitude || !mask || !periods || n_frames < 1 || filter_order < 1)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const int T = n_frames;
    const size_t x_elems = (size_t)T * XPITCH;
    float2* X; float *model, *M; int32_t* per;
    int rc = carve_arena(h, [&](Bump& b) {
        X = b.take<float2>(x_elems);
        model = b.take<float>((size_t)T * PPITCH);
        M = b.take<float>((size_t)T * PPITCH);
        per = b.take<int32_t>(T);
    });
    if (rc) return rc;
    std::vector<float2> host;
    pack_magnitudes(magnitude, T, host);
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(X, host.data(), x_elems * sizeof(float2), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(per, periods, (size_t)T * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    launch_adaptive_model(st, X, 1, T, 1, per, filter_order, model);
    launch_mask_only(st, X, 1, T, 1, nullptr, T, model, M);
    h->launches += 2;
    CU(cudaMemcpy2DAsync(mask, NBIN * sizeof(float), M, PPITCH * sizeof(float), NBIN * sizeof(float), T,
                         cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_beatspectrogram(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, int segment_length,
                          int segment_step, double* beat, int32_t* n_segments_out) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!spectrogram || !beat || n_frames < 1 || n_rows < 1 || n_rows > NBIN || segment_length < 1 || segment_step < 1)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size (n_rows <= window_length / 2 + 1)");
    if (2 * segment_length - 1 > BEAT_L)
        return fail(h, REPET_E_UNSUPPORTED, "segment_length exceeds the 2048-point beat transform");
    CU(cudaSetDevice(h->device));
    const int n_seg = (n_frames + segment_step - 1) / segment_step;
    if (n_segments_out) *n_segments_out = n_seg;
    const int n_parts = 9, f_per_part = 120;
    float *P, *psd; double* b;
    int rc = carve_arena(h, [&](Bump& w) {
        P = w.take<float>((size_t)n_frames * PPITCH);
        psd = w.take<float>((size_t)n_seg * n_parts * BEAT_L);
        b = w.take<double>((size_t)n_seg * segment_length);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemsetAsync(P, 0, (size_t)n_frames * PPITCH * sizeof(float), st));
    CU(cudaMemcpy2DAsync(P, PPITCH * sizeof(float), spectrogram, n_rows * sizeof(float), n_rows * sizeof(float), n_frames,
                         cudaMemcpyHostToDevice, st));
    const int left = segment_length / 2;  // ceil((L-1)/2), repet.py:1182
    launch_beat(st, P, 1, n_frames, -left, segment_length, segment_step, n_seg, tables(h), psd, n_parts, f_per_part);
    launch_periods(st, psd, nullptr, n_seg, n_parts, segment_length, (double)n_rows, 0, 0, 0, segment_length, b, segment_length,
                   nullptr, nullptr, nullptr);
    h->launches += 2;
    CU(cudaMemcpyAsync(beat, b, (size_t)n_seg * segment_length * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_selfsimilarity(repet_handle* h, const float* magnitude, int n_frames, int n_rows, float* similarity) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!magnitude || !similarity || n_frames < 1 || n_rows < 1 || n_rows > NBIN)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size (n_rows <= window_length / 2 + 1)");
    CU(cudaSetDevice(h->device));
    const int T = n_frames;
    float *V, *An32, *An32lo, *S;
    int rc = carve_arena(h, [&](Bump& b) {
        V = b.take<float>((size_t)T * PPITCH);
        An32 = b.take<float>((size_t)T * KPAD);
        An32lo = b.take<float>((size_t)T * KPAD);
        S = b.take<float>((size_t)T * T);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemsetAsync(V, 0, (size_t)T * PPITCH * sizeof(float), st));
    CU(cudaMemcpy2DAsync(V, PPITCH * sizeof(float), magnitude, n_rows * sizeof(float), n_rows * sizeof(float), T,
                         cudaMemcpyHostToDevice, st));
    const bool split = g_tuning.simgemm_tc >= 2;
    launch_normalize(st, V, T, nullptr, An32, split ? An32lo : nullptr, g_tuning.simgemm_tc ? 1 : 0);
    if (g_tuning.simgemm_tc) {
        if (launch_selfsim_tc(st, An32, split ? An32lo : nullptr, 1, T, S, h->sm_count))
            return fail(h, REPET_E_CUDA, "tensor-map encode failed");
    } else {
        launch_selfsim_simt(st, An32, 1, T, S);
    }
    h->launches += 2;
    CU(cudaMemcpyAsync(similarity, S, (size_t)T * T * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_periods(repet_handle* h, const double* beat, int n_lags, int n_columns, int period_lo, int period_hi,
                  int32_t* periods) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!beat || !periods || n_lags < 1 || n_columns < 1) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    const int lag_hi = std::min(period_hi, n_lags / 3);  // repet.py:1265-1267
    if (period_lo < 0 || lag_hi <= period_lo)
        return fail(h, REPET_E_TOO_SHORT, "attempt to get argmax of an empty sequence");
    CU(cudaSetDevice(h->device));
    const size_t n = (size_t)n_lags * n_columns;
    double* b; int32_t* per;
    int rc = carve_arena(h, [&](Bump& w) {
        b = w.take<double>(n);
        per = w.take<int32_t>(n_columns);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(b, beat, n * sizeof(double), cudaMemcpyHostToDevice, st));
    launch_argmax_columns(st, b, n_lags, n_columns, period_lo, lag_hi, per);
    h->launches += 1;
    CU(cudaMemcpyAsync(periods, per, (size_t)n_columns * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

// upload a [n][n_rows] fp32 matrix into rows of PPITCH floats (zero padded)
static int upload_rows(repet_handle* h, const float* host, int n, int n_rows, float* dev) {
    CU(cudaMemsetAsync(dev, 0, (size_t)n * PPITCH * sizeof(float), h->stream));
    CU(cudaMemcpy2DAsync(dev, PPITCH * sizeof(float), host, n_rows * sizeof(float), n_rows * sizeof(float), n,
                         cudaMemcpyHostToDevice, h->stream));
    return REPET_OK;
}

int hlp_similarity(repet_handle* h, const float* magnitude1, int n_frames1, const float* magnitude2, int n_frames2,
                     int n_rows, double* similarity) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!magnitude1 || !magnitude2 || !similarity || n_frames1 < 1 || n_frames2 < 1 || n_rows < 1 || n_rows > NBIN)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size (n_rows <= window_length / 2 + 1)");
    CU(cudaSetDevice(h->device));
    const size_t n1 = n_frames1, n2 = n_frames2;
    float* V; double *An, *out;
    int rc = carve_arena(h, [&](Bump& b) {
        V = b.take<float>((n1 + n2) * PPITCH);
        An = b.take<double>((n1 + n2) * APITCH64);
        out = b.take<double>(n1 * n2);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    if ((rc = upload_rows(h, magnitude1, n_frames1, n_rows, V))) return rc;
    if ((rc = upload_rows(h, magnitude2, n_frames2, n_rows, V + n1 * PPITCH))) return rc;
    launch_normalize(st, V, n_frames1 + n_frames2, An, nullptr, nullptr, 0);
    launch_cosine64(st, An, n_frames1, An + n1 * APITCH64, n_frames2, out);
    h->launches += 2;
    CU(cudaMemcpyAsync(similarity, out, n1 * n2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_localmaxima(repet_handle* h, const double* data, int n, int n_columns, double minimum_value,
                      int minimum_distance, int number_values, int32_t* indices, int32_t* counts, double* values) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!data || !indices || !counts || n < 1 || n_columns < 1 || number_values < 1 || minimum_distance < 0)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const size_t total = (size_t)n * n_columns, lists = (size_t)n_columns * number_values;
    double *d, *val; int32_t *idx, *cnt;
    int rc = carve_arena(h, [&](Bump& b) {
        d = b.take<double>(total);
        idx = b.take<int32_t>(lists);
        cnt = b.take<int32_t>(n_columns);
        val = b.take<double>(lists);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(d, data, total * sizeof(double), cudaMemcpyHostToDevice, st));
    if (launch_localmaxima64(st, d, n, n_columns, minimum_value, minimum_distance, number_values, idx, cnt, val))
        return fail(h, REPET_E_UNSUPPORTED, "vector too long for the shared-memory local-maximum scan");
    h->launches += 1;
    CU(cudaMemcpyAsync(indices, idx, lists * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(counts, cnt, (size_t)n_columns * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (values) CU(cudaMemcpyAsync(values, val, lists * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_simmask(repet_handle* h, const float* magnitude, int n_frames, const int32_t* indices, const int32_t* counts,
                  int number, float* mask) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!magnitude || !indices || !counts || !mask || n_frames < 1 || number < 1)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const int T = n_frames;
    const size_t x_elems = (size_t)T * XPITCH;
    float2* X; float *model, *M, *Vsq; int32_t *idx, *cnt;
    int rc = carve_arena(h, [&](Bump& b) {
        X = b.take<float2>(x_elems);
        model = b.take<float>((size_t)T * PPITCH);
        M = b.take<float>((size_t)T * PPITCH);
        Vsq = b.take<float>((size_t)T * PPITCH);
        idx = b.take<int32_t>((size_t)T * number);
        cnt = b.take<int32_t>(T);
    });
    if (rc) return rc;
    std::vector<float2> host;
    pack_magnitudes(magnitude, T, host);
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(X, host.data(), x_elems * sizeof(float2), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(idx, indices, (size_t)T * number * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(cnt, counts, (size_t)T * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    launch_sqmag(st, X, T, Vsq);
    if (launch_simmodel(st, X, Vsq, 1, T, 1, idx, cnt, number, 0, model))
        return fail(h, REPET_E_UNSUPPORTED, "lists too long for the shared-memory median");
    launch_mask_only(st, X, 1, T, 1, nullptr, T, model, M);
    h->launches += 2;
    CU(cudaMemcpy2DAsync(mask, NBIN * sizeof(float), M, PPITCH * sizeof(float), NBIN * sizeof(float), T,
                         cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int hlp_acorr(repet_handle* h, const float* data, int n_rows, int n_columns, double* autocorrelation) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!data || !autocorrelation || n_rows < 1 || n_columns < 1) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    if (2 * n_rows - 1 > BEAT_L) return fail(h, REPET_E_UNSUPPORTED, "more rows than the 2048-point transform holds");
    CU(cudaSetDevice(h->device));
    // every column becomes one beat item whose only non-zero frequency row is that column
    const int chunk = std::max(1, std::min(n_columns, (int)(((size_t)512 << 20) / ((size_t)n_rows * PPITCH * sizeof(float)))));
    float *P, *psd; double* b;
    int rc = carve_arena(h, [&](Bump& w) {
        P = w.take<float>((size_t)chunk * n_rows * PPITCH);
        psd = w.take<float>((size_t)chunk * BEAT_L);
        b = w.take<double>((size_t)chunk * n_rows);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    std::vector<double> host((size_t)chunk * n_rows);
    for (int c0 = 0; c0 < n_columns; c0 += chunk) {
        const int g = std::min(chunk, n_columns - c0);
        CU(cudaMemsetAsync(P, 0, (size_t)g * n_rows * PPITCH * sizeof(float), st));
        for (int c = 0; c < g; ++c)  // column c0+c -> item c, frequency row 0
            CU(cudaMemcpy2DAsync(P + (size_t)c * n_rows * PPITCH, PPITCH * sizeof(float), data + c0 + c,
                                 n_columns * sizeof(float), sizeof(float), n_rows, cudaMemcpyHostToDevice, st));
        launch_beat(st, P, g, n_rows, 0, n_rows, 0, 1, tables(h), psd, 1, 8);
        launch_periods(st, psd, nullptr, g, 1, n_rows, 1.0, 0, 0, 0, n_rows, b, n_rows, nullptr, nullptr, nullptr);
        h->launches += 2;
        CU(cudaMemcpyAsync(host.data(), b, (size_t)g * n_rows * sizeof(double), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (int c = 0; c < g; ++c)
            for (int l = 0; l < n_rows; ++l) autocorrelation[(size_t)l * n_columns + c0 + c] = host[(size_t)c * n_rows + l];
    }
    CU(cudaGetLastError());
    return REPET_OK;
}


const repet_entry* entry_table() {
    static const repet_entry table = {WIN_N,         drv_batch_dev,  drv_batch_host,      drv_single_f64,     hlp_stft,
                                      hlp_istft,     hlp_beat_common, hlp_mask,           hlp_adaptivemask,   hlp_beatspectrogram,
                                      hlp_selfsimilarity, hlp_periods, hlp_similarity,    hlp_localmaxima,    hlp_simmask,
                                      hlp_acorr,     drv_separate_f64, drv_spectrogram_dev, drv_foreground_dev, drv_single_f64_dev};
    return &table;
}

}  // namespace repet
