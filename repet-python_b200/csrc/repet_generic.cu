// General-size float64 paths of the transform helpers: _stft / _istft for ANY window length and step
// (repet.py:1001-1105), _acorr / _beatspectrum for ANY number of rows (repet.py:1108-1158).
//
// The drivers and the fast helper entry points run register-blocked fp32 transforms of 512 / 1024 / 2048 points
// with a hop of half a window; the reference's private helpers take any window, any step and any matrix size, and
// its examples call them directly (README.md:79-81).  This file is the catch-all behind those helpers: batched
// complex float64 FFTs of any length -- Stockham radix-2 passes through global memory for powers of two,
// Bluestein's chirp-z on top of them for everything else -- compiled once, independent of REPET_WIN_N.
// Throughput is not the point here (a 30 s clip takes ~1 ms); float64 accuracy and generality are.
#include "repet_internal.h"

#include <cmath>

namespace {

using repet::fail;
using repet::Bump;
using repet::carve_arena;
using repet::default_ws_limit;

__device__ __forceinline__ double2 zmul(double2 a, double2 b) {
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}

// One radix-2 Stockham pass (autosort: natural order in, natural order out after log2(L) passes):
// butterfly j of row `row` combines src[j] and src[j + L/2] with the twiddle of its position inside the current
// sub-transform of length 2 * ns and writes to dst[(j / ns) * 2 ns + j % ns (+ ns)].
__global__ void __launch_bounds__(256)
k_stockham_pass(const double2* __restrict__ src, double2* __restrict__ dst, int L, long long n_rows, int ns, int inverse) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int half = L >> 1;
    const long long row = gid / half;
    if (row >= n_rows) return;
    const int j = (int)(gid - row * half);
    const int k = j & (ns - 1);
    double sn, cs;
    sincospi((inverse ? 1.0 : -1.0) * (double)k / (double)ns, &sn, &cs);
    const double2* __restrict__ s = src + row * L;
    double2* __restrict__ d = dst + row * L;
    const double2 a = s[j];
    const double2 b = zmul(s[j + half], make_double2(cs, sn));
    const int o = ((j - k) << 1) + k;
    d[o] = make_double2(a.x + b.x, a.y + b.y);
    d[o + ns] = make_double2(a.x - b.x, a.y - b.y);
}

// in-place-looking batched FFT of power-of-two length L: data and tmp are [n_rows][L]; the result ends in `data`
// (unnormalised in both directions)
void fft_pow2(cudaStream_t st, double2* data, double2* tmp, int L, long long n_rows, bool inverse) {
    if (L < 2) return;
    int passes = 0;
    for (int v = L; v > 1; v >>= 1) ++passes;
    double2* src = data;
    double2* dst = tmp;
    if (passes & 1) {  // odd number of passes: start from tmp so that the last pass writes `data`
        cudaMemcpyAsync(tmp, data, (size_t)n_rows * L * sizeof(double2), cudaMemcpyDeviceToDevice, st);
        src = tmp;
        dst = data;
    }
    const long long threads = n_rows * (L >> 1);
    const unsigned blocks = (unsigned)((threads + 255) / 256);
    for (int ns = 1; ns < L; ns <<= 1) {
        k_stockham_pass<<<blocks, 256, 0, st>>>(src, dst, L, n_rows, ns, inverse ? 1 : 0);
        double2* t = src;
        src = dst;
        dst = t;
    }
}

int next_pow2(long long v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

// ---- Bluestein: DFT of any length N as a circular convolution of length M = pow2 >= 2N - 1 ----------------
// X[k] = conj(c[k]) * sum_n (x[n] conj(c[n])) c[k - n],  c[n] = exp(i pi n^2 / N)   (forward; the inverse
// conjugates c).  n^2 is reduced mod 2N in integers so that the chirp stays exact for long transforms.
__device__ __forceinline__ double2 chirp(long long n, int N, int inverse) {
    const long long r = (n * n) % (2LL * N);
    double sn, cs;
    sincospi((double)r / (double)N, &sn, &cs);
    return make_double2(cs, inverse ? -sn : sn);
}
__global__ void k_bluestein_filter(double2* __restrict__ filt, int N, int M, int inverse) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    double2 v = make_double2(0.0, 0.0);
    if (m < N) v = chirp(m, N, inverse);
    else if (M - m < N) v = chirp(M - m, N, inverse);
    filt[m] = v;
}
__global__ void k_bluestein_pre(const double2* __restrict__ x, double2* __restrict__ a, int N, int M, long long n_rows,
                                int inverse) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = gid / M;
    if (row >= n_rows) return;
    const int m = (int)(gid - row * M);
    double2 v = make_double2(0.0, 0.0);
    if (m < N) {
        const double2 c = chirp(m, N, inverse);
        v = zmul(x[row * N + m], make_double2(c.x, -c.y));
    }
    a[gid] = v;
}
__global__ void k_pointwise_mul(double2* __restrict__ a, const double2* __restrict__ f, int M, long long n_rows) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_rows * M) return;
    a[gid] = zmul(a[gid], f[gid % M]);
}
__global__ void k_bluestein_post(const double2* __restrict__ a, double2* __restrict__ x, int N, int M, long long n_rows,
                                 int inverse) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long row = gid / N;
    if (row >= n_rows) return;
    const int k = (int)(gid - row * N);
    const double2 c = chirp(k, N, inverse);
    const double2 v = a[row * M + k];
    const double s = 1.0 / (double)M;  // the inverse transform of the convolution
    x[gid] = zmul(make_double2(v.x * s, v.y * s), make_double2(c.x, -c.y));
}

// workspace (in double2 elements) fft_any needs besides `data` [n_rows][N]
size_t fft_any_workspace(int N, long long n_rows) {
    if ((N & (N - 1)) == 0) return (size_t)n_rows * N;
    const int M = next_pow2(2LL * N - 1);
    return 2 * (size_t)n_rows * M + (size_t)2 * M;
}

// batched DFT of any length N, unnormalised, result in `data`
void fft_any(cudaStream_t st, double2* data, double2* ws, int N, long long n_rows, bool inverse) {
    if ((N & (N - 1)) == 0) {
        fft_pow2(st, data, ws, N, n_rows, inverse);
        return;
    }
    const int M = next_pow2(2LL * N - 1);
    double2* a = ws;
    double2* tmp = a + (size_t)n_rows * M;
    double2* filt = tmp + (size_t)n_rows * M;
    double2* filt_tmp = filt + M;
    const int inv = inverse ? 1 : 0;
    k_bluestein_filter<<<(M + 255) / 256, 256, 0, st>>>(filt, N, M, inv);
    fft_pow2(st, filt, filt_tmp, M, 1, false);
    const long long total = n_rows * M;
    k_bluestein_pre<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(data, a, N, M, n_rows, inv);
    fft_pow2(st, a, tmp, M, n_rows, false);
    k_pointwise_mul<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(a, filt, M, n_rows);
    fft_pow2(st, a, tmp, M, n_rows, true);
    const long long outs = n_rows * N;
    k_bluestein_post<<<(unsigned)((outs + 255) / 256), 256, 0, st>>>(a, data, N, M, n_rows, inv);
}

// ---- _stft ---------------------------------------------------------------------------------------------------
// frames[j][n] = w[n] * padded[j*step + n], padded = floor(N/2) zeros + signal + zeros     repet.py:1018-1055
__global__ void k_frames(const double* __restrict__ signal, long long S, const double* __restrict__ window, int N,
                         int step, int pad, long long T, double2* __restrict__ frames) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= T * N) return;
    const long long j = gid / N;
    const int n = (int)(gid - j * N);
    const long long m = j * step + n - pad;
    frames[gid] = make_double2((m >= 0 && m < S) ? window[n] * signal[m] : 0.0, 0.0);
}
// [T][N] -> the reference's (N, T) C-order layout, through a 32 x 32 shared-memory tile
__global__ void k_transpose(const double2* __restrict__ in, long long rows, int cols, double2* __restrict__ out) {
    __shared__ double2 tile[32][33];
    const long long r0 = (long long)blockIdx.y * 32;
    const int c0 = blockIdx.x * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const long long r = r0 + i;
        const int c = c0 + threadIdx.x;
        if (r < rows && c < cols) tile[i][threadIdx.x] = in[r * cols + c];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = c0 + i;
        const long long r = r0 + threadIdx.x;
        if (r < rows && c < cols) out[(long long)c * rows + r] = tile[threadIdx.x][i];
    }
}
void transpose(cudaStream_t st, const double2* in, long long rows, int cols, double2* out) {
    dim3 grid((cols + 31) / 32, (unsigned)((rows + 31) / 32));
    k_transpose<<<grid, dim3(32, 8), 0, st>>>(in, rows, cols, out);
}

// ---- _istft --------------------------------------------------------------------------------------------------
// y[m] = (1/g) sum_j real(ifft(Y[:, j]))[m + (N - step) - j*step] over the frames covering it  repet.py:1085-1103
__global__ void k_overlap_add(const double2* __restrict__ frames, int N, int step, long long T, long long n_out,
                              double inv_norm, double* __restrict__ out) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_out) return;
    const long long pos = m + (N - step);  // index into the untrimmed overlap-add buffer
    long long j_hi = pos / step;
    if (j_hi > T - 1) j_hi = T - 1;
    // smallest j with pos - j*step < N: ceil((pos - N + 1) / step), clipped at 0
    const long long j_lo = pos - N + 1 <= 0 ? 0 : (pos - N + step) / step;
    double acc = 0.0;
    for (long long j = j_lo; j <= j_hi; ++j) acc += frames[j * N + (pos - j * step)].x;  // frame order, as the reference adds
    out[m] = acc * inv_norm;
}

// ---- _acorr / _beatspectrum -------------------------------------------------------------------------------------
// data [n_rows][n_cols] (row-major, float64) -> columns as zero-padded complex rows [n_cols][L]
__global__ void k_load_columns(const double* __restrict__ data, int n_rows, int n_cols, int L, double2* __restrict__ z) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_cols * L) return;
    const int c = (int)(gid / L), l = (int)(gid - (long long)c * L);
    z[gid] = make_double2(l < n_rows ? data[(size_t)l * n_cols + c] : 0.0, 0.0);
}
__global__ void k_power(double2* __restrict__ z, long long n) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n) return;
    const double2 v = z[gid];
    z[gid] = make_double2(fma(v.x, v.x, v.y * v.y), 0.0);
}
// autocorrelation[l][c] = real(ifft)[l] / L / (n_rows - l)          repet.py:1129-1137
__global__ void k_store_acorr(const double2* __restrict__ z, int n_rows, int n_cols, int L, double* __restrict__ out) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_rows * n_cols) return;
    const int l = (int)(gid / n_cols), c = (int)(gid - (long long)l * n_cols);
    out[gid] = z[(size_t)c * L + l].x / (double)L / (double)(n_rows - l);
}
// contiguous sequences [n_seq][n] -> zero-padded complex rows [n_seq][L]
__global__ void k_load_rows(const double* __restrict__ data, int n, int n_seq, int L, double2* __restrict__ z) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_seq * L) return;
    const int c = (int)(gid / L), l = (int)(gid - (long long)c * L);
    z[gid] = make_double2(l < n ? data[(size_t)c * n + l] : 0.0, 0.0);
}
// beat[l] += sum over this chunk's rows of their unbiased autocorrelation at lag l (repet.py:1135-1137, 1156):
// fixed-order sum, one thread per lag
__global__ void k_accumulate_beat(const double2* __restrict__ z, int n, int n_seq, int L, double* __restrict__ beat) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n) return;
    double acc = beat[l];
    const double scale = 1.0 / (double)L / (double)(n - l);
    for (int c = 0; c < n_seq; ++c) acc += z[(size_t)c * L + l].x * scale;
    beat[l] = acc;
}
__global__ void k_scale_beat(double* __restrict__ beat, int n, int n_seq) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < n) beat[l] /= (double)n_seq;
}

// z, tmp: [n_cols][L] each, L = next_pow2(2 n_rows)
int acorr_device(repet_handle* h, const double* d_data, int n_rows, int n_cols, double* d_out, double2* z, double2* tmp) {
    // any L >= 2 n_rows - 1 gives the same linear autocorrelation as the reference's length 2 n_rows (quirk Q13)
    const int L = next_pow2(2LL * n_rows);
    cudaStream_t st = h->stream;
    const long long total = (long long)n_cols * L;
    k_load_columns<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_data, n_rows, n_cols, L, z);
    fft_pow2(st, z, tmp, L, n_cols, false);
    k_power<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(z, total);
    fft_pow2(st, z, tmp, L, n_cols, true);
    const long long outs = (long long)n_rows * n_cols;
    k_store_acorr<<<(unsigned)((outs + 255) / 256), 256, 0, st>>>(z, n_rows, n_cols, L, d_out);
    h->launches += 3 + 2 * 20;
    return REPET_OK;
}

}  // namespace

extern "C" {

int repet_stft_frames(int64_t n_samples, int window_length, int step_length) {
    if (window_length < 1 || step_length < 1 || n_samples < 0) return 0;
    const int64_t pad = window_length / 2;
    const int64_t span = n_samples + 2 * pad - window_length;
    // ceil(span / step) + 1 with Python's rounding for negative spans (repet.py:1021-1028)
    const int64_t q = span >= 0 ? (span + step_length - 1) / step_length : -((-span) / step_length);
    return (int)(q + 1);
}

int repet_stft_f64(repet_handle* h, const double* signal, int64_t n_samples, const double* window, int window_length,
                   int step_length, double* spectrum, int32_t* n_frames_out) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!signal || !window || !spectrum || n_samples < 0 || window_length < 1 || step_length < 1)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    const int N = window_length;
    const long long T = repet_stft_frames(n_samples, window_length, step_length);
    if (n_frames_out) *n_frames_out = (int32_t)T;
    if (T < 1) return fail(h, REPET_E_INVALID_ARG, "signal too short for one frame");
    CU(cudaSetDevice(h->device));
    const size_t elems = (size_t)T * N;
    double *d_sig, *d_win; double2 *frames, *out, *ws;
    int rc = carve_arena(h, [&](Bump& b) {
        d_sig = b.take<double>((size_t)std::max<int64_t>(n_samples, 1));
        d_win = b.take<double>(N);
        frames = b.take<double2>(elems);
        out = b.take<double2>(elems);
        ws = b.take<double2>(fft_any_workspace(N, T));
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    if (n_samples > 0) CU(cudaMemcpyAsync(d_sig, signal, (size_t)n_samples * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_win, window, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st));
    k_frames<<<(unsigned)((elems + 255) / 256), 256, 0, st>>>(d_sig, n_samples, d_win, N, step_length, N / 2, T, frames);
    fft_any(st, frames, ws, N, T, false);
    transpose(st, frames, T, N, out);
    h->launches += 2 + 12;
    CU(cudaMemcpyAsync(spectrum, out, elems * sizeof(double2), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int repet_istft_f64(repet_handle* h, const double* spectrum, int window_length, int n_frames, const double* window,
                    int step_length, double* signal, int64_t* n_samples_out) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!spectrum || !window || !signal || window_length < 1 || step_length < 1 || n_frames < 1)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    const int N = window_length;
    const long long T = n_frames;
    // untrimmed length T*step + (N - step), minus N - step at both ends (repet.py:1079, 1098-1100)
    const long long n_out = T * step_length - (long long)(N - step_length);
    if (n_samples_out) *n_samples_out = std::max<long long>(n_out, 0);
    if (n_out <= 0) return REPET_OK;
    double gain = 0.0;
    for (int i = 0; i < N; i += step_length) gain += window[i];  // sum(window[0:N:step]), repet.py:1103
    CU(cudaSetDevice(h->device));
    const size_t elems = (size_t)T * N;
    double2 *in, *frames, *ws; double* out;
    int rc = carve_arena(h, [&](Bump& b) {
        in = b.take<double2>(elems);
        frames = b.take<double2>(elems);
        ws = b.take<double2>(fft_any_workspace(N, T));
        out = b.take<double>((size_t)n_out);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(in, spectrum, elems * sizeof(double2), cudaMemcpyHostToDevice, st));
    transpose(st, in, N, (int)T, frames);  // (N, T) -> [T][N]
    fft_any(st, frames, ws, N, T, true);
    k_overlap_add<<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>(frames, N, step_length, T, n_out, 1.0 / ((double)N * gain), out);
    h->launches += 2 + 12;
    CU(cudaMemcpyAsync(signal, out, (size_t)n_out * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int repet_acorr_f64(repet_handle* h, const double* data, int n_rows, int n_columns, double* autocorrelation) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!data || !autocorrelation || n_rows < 1 || n_columns < 1) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    const int L = next_pow2(2LL * n_rows);
    const size_t n = (size_t)n_rows * n_columns;
    // columns in chunks so that the two transform buffers stay below ~4 GB
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_columns, ((size_t)2 << 30) / ((size_t)L * sizeof(double2))));
    double *d_in, *d_out, *c_in, *c_out; double2 *z, *tmp;
    int rc = carve_arena(h, [&](Bump& b) {
        d_in = b.take<double>(n);
        d_out = b.take<double>(n);
        c_in = b.take<double>((size_t)n_rows * chunk);
        c_out = b.take<double>((size_t)n_rows * chunk);
        z = b.take<double2>((size_t)chunk * L);
        tmp = b.take<double2>((size_t)chunk * L);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(d_in, data, n * sizeof(double), cudaMemcpyHostToDevice, st));
    for (int c0 = 0; c0 < n_columns; c0 += chunk) {
        const int g = std::min(chunk, n_columns - c0);
        if (g == n_columns) {
            if ((rc = acorr_device(h, d_in, n_rows, n_columns, d_out, z, tmp))) return rc;
        } else {  // a block of columns: gather it into a dense [n_rows][g] matrix, scatter the result back
            CU(cudaMemcpy2DAsync(c_in, (size_t)g * sizeof(double), d_in + c0, (size_t)n_columns * sizeof(double),
                                 (size_t)g * sizeof(double), n_rows, cudaMemcpyDeviceToDevice, st));
            if ((rc = acorr_device(h, c_in, n_rows, g, c_out, z, tmp))) return rc;
            CU(cudaMemcpy2DAsync(d_out + c0, (size_t)n_columns * sizeof(double), c_out, (size_t)g * sizeof(double),
                                 (size_t)g * sizeof(double), n_rows, cudaMemcpyDeviceToDevice, st));
        }
    }
    CU(cudaMemcpyAsync(autocorrelation, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

int repet_beatspectrum_f64(repet_handle* h, const double* spectrogram, int n_frequencies, int n_times, double* beat) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!spectrogram || !beat || n_frequencies < 1 || n_times < 1) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    // _beatspectrum(V) = mean(_acorr(V.T), axis=1) (repet.py:1153-1156): every frequency row of V is one contiguous
    // sequence of n_times samples; rows go through the transforms in chunks, the mean is accumulated row by row in a
    // fixed order
    const int L = next_pow2(2LL * n_times);
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_frequencies, ((size_t)2 << 30) / ((size_t)L * sizeof(double2))));
    const size_t n = (size_t)n_frequencies * n_times;
    double *d_v, *d_beat; double2 *z, *tmp;
    int rc = carve_arena(h, [&](Bump& b) {
        d_v = b.take<double>(n);
        z = b.take<double2>((size_t)chunk * L);
        tmp = b.take<double2>((size_t)chunk * L);
        d_beat = b.take<double>(n_times);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(d_v, spectrogram, n * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d_beat, 0, (size_t)n_times * sizeof(double), st));
    for (int f0 = 0; f0 < n_frequencies; f0 += chunk) {
        const int g = std::min(chunk, n_frequencies - f0);
        const long long total = (long long)g * L;
        k_load_rows<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_v + (size_t)f0 * n_times, n_times, g, L, z);
        fft_pow2(st, z, tmp, L, g, false);
        k_power<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(z, total);
        fft_pow2(st, z, tmp, L, g, true);
        k_accumulate_beat<<<(n_times + 127) / 128, 128, 0, st>>>(z, n_times, g, L, d_beat);
        h->launches += 3 + 2 * 20;
    }
    k_scale_beat<<<(n_times + 127) / 128, 128, 0, st>>>(d_beat, n_times, n_frequencies);
    CU(cudaMemcpyAsync(beat, d_beat, (size_t)n_times * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

}  // extern "C"

// =====================================================================================================================
// General float64 DRIVERS: repet.original / extended / adaptive / sim / simonline (repet.py:67-911) for the inputs the
// register-blocked fp32 kernels are not compiled for -- window lengths other than 512 / 1024 / 2048 (sampling rates
// above 51.2 kHz: 4096 points at 96 kHz, 8192 at 192 kHz, repet.py:130), more than two channels (the reference
// loops over any number, repet.py:152-155), period ranges above 1024 frames, segments longer than one beat transform,
// very long similar-frame lists.  Same pipeline, written for generality instead of speed: float64 end to end (so the
// integer decisions need no certification), simple kernels, transforms by the Stockham passes above.
// =====================================================================================================================
namespace {

enum { GEN_ORIGINAL = 0, GEN_EXTENDED = 1, GEN_ADAPTIVE = 2, GEN_SIM = 3, GEN_SIMONLINE = 4 };

// Device allocations of one call, released together.  Stream-ordered (cudaMallocAsync): the driver's memory pool
// keeps up to 8 GB of freed blocks, so the per-segment calls of `extended` and repeated calls reuse them instead of
// paying cudaMalloc / cudaFree (which synchronise the device) every time.
struct Pool {
    cudaStream_t st;
    std::vector<void*> ptrs;
    bool ok = true;
    explicit Pool(cudaStream_t stream) : st(stream) {
        static bool configured[64] = {false};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!configured[dev & 63]) {
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                uint64_t keep = (uint64_t)8 << 30;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
            (void)cudaGetLastError();
            configured[dev & 63] = true;
        }
    }
    template <typename T>
    T* get(size_t n) {
        void* p = nullptr;
        if (cudaMallocAsync(&p, std::max<size_t>(n, 1) * sizeof(T), st) != cudaSuccess) {
            (void)cudaGetLastError();
            ok = false;
            return nullptr;
        }
        ptrs.push_back(p);
        return static_cast<T*>(p);
    }
    void release(void* p) {
        for (size_t i = 0; i < ptrs.size(); ++i)
            if (ptrs[i] == p) {
                cudaFreeAsync(p, st);
                ptrs.erase(ptrs.begin() + i);
                return;
            }
    }
    ~Pool() {
        for (void* p : ptrs) cudaFreeAsync(p, st);
    }
};

inline unsigned blocks_for(long long n, int per = 256) { return (unsigned)((n + per - 1) / per); }

// frames[c][j][n] = w[n] * x[j*H + n - pad][c]  (zero outside the signal); audio (S, C) interleaved, row pitch `ld`
__global__ void k_gen_frames(const double* __restrict__ audio, long long S, int C, int ld, const double* __restrict__ window,
                             int N, int H, int pad, long long T, double2* __restrict__ frames) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)C * T * N) return;
    const int n = (int)(gid % N);
    const long long j = (gid / N) % T;
    const int c = (int)(gid / ((long long)N * T));
    const long long m = j * H + n - pad;
    frames[gid] = make_double2((m >= 0 && m < S) ? window[n] * audio[m * ld + c] : 0.0, 0.0);
}
// V[c][t][f] = |X[c][t][f]|, f <= N/2 (repet.py:158); Vm[t][f] = mean over channels (repet.py:162, 667)
__global__ void k_gen_magnitude(const double2* __restrict__ X, int C, long long T, int N, int F, double* __restrict__ V,
                                double* __restrict__ Vm) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= T * F) return;
    const long long t = gid / F;
    const int f = (int)(gid - t * F);
    double sum = 0.0;
    for (int c = 0; c < C; ++c) {
        const double2 x = X[((long long)c * T + t) * N + f];
        const double v = hypot(x.x, x.y);
        V[((long long)c * T + t) * F + f] = v;
        sum += v;
    }
    Vm[gid] = sum / (double)C;
}
// time sequences of the squared channel-mean magnitudes, one per (segment, frequency): z[(s*F + f)][l] =
// Vm[ts_s + l][f]^2 for l < len and 0 <= ts_s + l < T, else 0          (repet.py:162, 1123, 1177-1198)
__global__ void k_gen_load_seq(const double* __restrict__ Vm, long long T, int F, int f0, int nf, long long ts0, int seg_step,
                               int n_seg, int len, int L, double2* __restrict__ z) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)n_seg * nf * L) return;
    const int l = (int)(gid % L);
    const int f = (int)((gid / L) % nf);
    const int s = (int)(gid / ((long long)L * nf));
    const long long t = ts0 + (long long)s * seg_step + l;
    double v = 0.0;
    if (l < len && t >= 0 && t < T) {
        v = Vm[t * F + f0 + f];
        v *= v;
    }
    z[gid] = make_double2(v, 0.0);
}
// beat[s][l] += sum over this chunk's frequency rows of acorr / (len - l)     (repet.py:1135-1137)
__global__ void k_gen_accumulate_beat(const double2* __restrict__ z, int nf, int n_seg, int len, int L, int n_lags,
                                      double* __restrict__ beat) {
    const int gid = blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_seg * n_lags) return;
    const int s = gid / n_lags, l = gid - s * n_lags;
    double acc = beat[gid];
    const double scale = 1.0 / (double)L / (double)(len - l);
    for (int f = 0; f < nf; ++f) acc += z[((long long)s * nf + f) * L + l].x * scale;
    beat[gid] = acc;
}
// period = first argmax over lags [lo, hi) + 1 (repet.py:1262-1289, quirks Q1, Q2); the common 1/F factor is omitted
__global__ void k_gen_argmax(const double* __restrict__ beat, int n_seg, int n_lags, int lo, int hi, int* __restrict__ period) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const double* __restrict__ b = beat + (long long)s * n_lags;
    int arg = lo;
    double best = b[lo];
    for (int l = lo + 1; l < hi; ++l)
        if (b[l] > best) {
            best = b[l];
            arg = l;
        }
    period[s] = arg + 1;
}
// per-frame periods of the adaptive REPET with the all-zero column of quirk Q3 (repet.py:1194-1204)
__global__ void k_gen_expand(const int* __restrict__ seg_period, long long T, int step, int lo, int* __restrict__ frame_period) {
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= T) return;
    const long long s = j / step;
    const bool zero_column = step > 1 && (j - s * step) == step - 1;
    frame_period[j] = zero_column ? lo + 1 : seg_period[s];
}
// An[t][f] = Vm[t][f] / ||Vm[t]||  (repet.py:1220, 1240); an all-zero frame gives 0/0 = NaN as in the reference (Q18)
__global__ void k_gen_normalize(const double* __restrict__ Vm, long long T, int F, double* __restrict__ An) {
    const long long t = blockIdx.x;
    __shared__ double s_red[256];
    double acc = 0.0;
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        const double v = Vm[t * F + f];
        acc += v * v;
    }
    s_red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o];
        __syncthreads();
    }
    const double norm = sqrt(s_red[0]);
    for (int f = threadIdx.x; f < F; f += blockDim.x) An[t * F + f] = Vm[t * F + f] / norm;
}
// Rows [r0, r0 + rows) of S = An An^T, float64, 64 x 64 tiles, into S row-major with pitch T (the whole matrix: r0 = 0,
// rows = T).  Every element is one fma chain over ascending k from 0.0, whichever tile forms it, and fma(a, b, c) =
// fma(b, a, c): S is bitwise symmetric, and a panel holds bit for bit the rows of the whole matrix.
__global__ void __launch_bounds__(256)
k_gen_gram(const double* __restrict__ An, long long T, int F, long long r0, long long rows, double* __restrict__ S) {
    __shared__ double sa[16][65];
    __shared__ double sb[16][65];
    const int ti = threadIdx.x & 15, tj = threadIdx.x >> 4;
    const long long i0 = (long long)blockIdx.x * 64, j0 = r0 + (long long)blockIdx.y * 64, j_end = r0 + rows;
    double acc[4][4] = {};
    for (int k0 = 0; k0 < F; k0 += 16) {
        for (int e = 0; e < 4; ++e) {
            const int idx = threadIdx.x + 256 * e;
            const int row = idx >> 4, kk = idx & 15;
            const long long ri = i0 + row, rj = j0 + row;
            sa[kk][row] = (ri < T && k0 + kk < F) ? An[ri * F + k0 + kk] : 0.0;
            sb[kk][row] = (rj < j_end && k0 + kk < F) ? An[rj * F + k0 + kk] : 0.0;
        }
        __syncthreads();
        for (int kk = 0; kk < 16; ++kk) {
            double av[4], bv[4];
            for (int a = 0; a < 4; ++a) av[a] = sa[kk][ti + 16 * a];
            for (int b = 0; b < 4; ++b) bv[b] = sb[kk][tj + 16 * b];
            for (int a = 0; a < 4; ++a)
                for (int b = 0; b < 4; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
        }
        __syncthreads();
    }
    for (int a = 0; a < 4; ++a)
        for (int b = 0; b < 4; ++b) {
            const long long i = i0 + ti + 16 * a, j = j0 + tj + 16 * b;
            if (i < T && j < j_end) S[(j - r0) * T + i] = acc[a][b];
        }
}
// _localmaxima of one vector held in shared memory (repet.py:1309-1343): v >= thr and strictly above every neighbour
// within +-d (windows clipped, NaN never wins), ranked by value descending (ties: descending index), first `number`.
// `kept` is scratch for n ints.  slot_frame (optional) maps a position to the frame index written out (simonline).
__device__ void gen_localmaxima(const double* __restrict__ v, int n, double thr, int d, int number, int* __restrict__ kept,
                                int* __restrict__ s_count, int* __restrict__ idx_out, int* __restrict__ cnt_out, int j_online,
                                int B_online, int base_online = 0) {
    if (threadIdx.x == 0) *s_count = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double x = v[i];
        bool keep = x >= thr;
        const int lo = max(i - d, 0), hi = min(i + d, n - 1);
        for (int u = lo; u <= hi && keep; ++u)
            if (u != i && !(x > v[u])) keep = false;
        if (keep) kept[atomicAdd(s_count, 1)] = i;
    }
    __syncthreads();
    const int K = *s_count;
    for (int q = threadIdx.x; q < K; q += blockDim.x) {
        const int i = kept[q];
        const double x = v[i];
        int rank = 0;
        for (int r = 0; r < K && rank < number; ++r) {  // a candidate ranked `number` or below is out either way
            const int io = kept[r];
            rank += (v[io] > x) || (v[io] == x && io > i);
        }
        if (rank < number) {
            int out = i;
            if (B_online > 0) {  // ring slot -> frame index (repet.py:837, 852; quirk Q6); j_online carries the base
                const int j0 = j_online % B_online;
                out = (i <= j0 ? j_online - (j0 - i) : j_online - (j0 - i) - B_online) - base_online;
            }
            idx_out[rank] = out;
        }
    }
    if (threadIdx.x == 0) *cnt_out = min(K, number);
    __syncthreads();
}
// REPET-SIM: the similar-frame lists of columns r0 .. r0 + rows - 1 of S (repet.py:1370-1381), from the panel S that
// holds rows [r0, r0 + rows) of the symmetric S with pitch T.  Persistent CTAs walk the columns; a column (= row of
// S) is examined in chunks of GEN_IDX_CHUNK elements staged in shared memory with a halo of d on both sides, so a
// track of any length fits; the survivors' indices go to a per-CTA global scratch list and are ranked by value (ties:
// descending index) as _localmaxima does.  idx / cnt are indexed by absolute frame.
constexpr int GEN_IDX_CHUNK = 4096;
__global__ void __launch_bounds__(512)
k_gen_indices(const double* __restrict__ S, int T, int r0, int rows, double thr, int d, int number, int* __restrict__ idx,
              int* __restrict__ cnt, int* __restrict__ kept_scratch) {
    extern __shared__ __align__(16) unsigned char gsm[];
    double* v = reinterpret_cast<double*>(gsm);  // [GEN_IDX_CHUNK + 2 d]
    __shared__ int s_count;
    int* __restrict__ kept = kept_scratch + (size_t)blockIdx.x * T;
    for (int c = r0 + blockIdx.x; c < r0 + rows; c += gridDim.x) {
        const double* __restrict__ row = S + (long long)(c - r0) * T;
        __syncthreads();
        if (threadIdx.x == 0) s_count = 0;
        for (int g0 = 0; g0 < T; g0 += GEN_IDX_CHUNK) {
            __syncthreads();
            const int n_stage = min(GEN_IDX_CHUNK, T - g0) + 2 * d;
            for (int x = threadIdx.x; x < n_stage; x += blockDim.x) {
                const int g = g0 - d + x;
                v[x] = (g >= 0 && g < T) ? row[g] : -INFINITY;  // beyond the ends: clipped windows (never above a value)
            }
            __syncthreads();
            for (int x = threadIdx.x; x < min(GEN_IDX_CHUNK, T - g0); x += blockDim.x) {
                const double a = v[x + d];
                bool keep = a >= thr;
                for (int u = x; u <= x + 2 * d && keep; ++u)
                    if (u != x + d && !(a > v[u])) {
                        // -inf padding stands for "no neighbour": it must not veto a maximum of value -inf itself
                        const int g = g0 - d + u;
                        if (g >= 0 && g < T) keep = false;
                    }
                if (keep) kept[atomicAdd(&s_count, 1)] = g0 + x;
            }
        }
        __syncthreads();
        const int K = s_count;
        for (int q = threadIdx.x; q < K; q += blockDim.x) {
            const int i = kept[q];
            const double a = row[i];
            int rank = 0;
            for (int r = 0; r < K && rank < number; ++r) {  // a candidate ranked `number` or below is out either way
                const int io = kept[r];
                const double b = row[io];
                rank += (b > a) || (b == a && io > i);
            }
            if (rank < number) idx[(long long)c * number + rank] = i;
        }
        if (threadIdx.x == 0) cnt[c] = min(K, number);
    }
}
// online REPET-SIM: frame j >= B-1 against the B frames of its ring buffer in SLOT order (repet.py:834-866, quirk Q6)
// Rows are frames base .. base + T - 1 of a longer stream (base = repet_params.online_frame_base; 0 for a whole
// signal): the ring slot of a frame is its ABSOLUTE index mod B, and slots whose frame lies before the window hold
// no data (-inf: never a maximum), exactly as in the fast path's k_online_select.
__global__ void __launch_bounds__(256)
k_gen_online(const double* __restrict__ An, int T, int F, int B, int base, int row_first, double thr, int d, int number,
             int* __restrict__ idx, int* __restrict__ cnt) {
    extern __shared__ __align__(16) unsigned char gsm[];
    double* v = reinterpret_cast<double*>(gsm);       // [B] similarity by slot
    int* kept = reinterpret_cast<int*>(v + B);        // [B]
    __shared__ int s_count;
    const int j = blockIdx.x + row_first;             // row inside the window
    if (j >= T) return;
    const int ja = j + base;                          // absolute frame index
    const int j0 = ja % B;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const double* __restrict__ a = An + (long long)j * F;
    for (int b = warp; b < B; b += nwarp) {
        const int u = (b <= j0 ? ja - (j0 - b) : ja - (j0 - b) - B) - base;  // row of the frame in slot b
        double acc = -INFINITY;
        if (u >= 0) {
            const double* __restrict__ x = An + (long long)u * F;
            acc = 0.0;
            for (int f = lane; f < F; f += 32) acc = fma(a[f], x[f], acc);
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        }
        if (lane == 0) v[b] = acc;
    }
    __syncthreads();
    gen_localmaxima(v, B, thr, d, number, kept, &s_count, idx + (long long)j * number, cnt + j, ja, B, base);
}

// median of n values fetched by `fetch(s)`: insertion sort in local memory up to GEN_SORT_MAX, exact rank selection
// beyond; np.median's even-count rule (mean of the two middle values); n = 0 gives NaN (np.median of an empty slice)
constexpr int GEN_SORT_MAX = 128;
template <typename Fetch>
__device__ double gen_median(int n, Fetch fetch) {
    if (n <= 0) return nan("");
    if (n <= GEN_SORT_MAX) {
        double v[GEN_SORT_MAX];
        for (int s = 0; s < n; ++s) {
            const double x = fetch(s);
            int q = s;
            while (q > 0 && v[q - 1] > x) {
                v[q] = v[q - 1];
                --q;
            }
            v[q] = x;
        }
        return (n & 1) ? v[n >> 1] : 0.5 * (v[(n >> 1) - 1] + v[n >> 1]);
    }
    const int k_lo = (n - 1) >> 1, k_hi = n >> 1;
    double v_lo = 0.0, v_hi = 0.0;
    bool got_lo = false, got_hi = false;
    for (int i = 0; i < n && !(got_lo && got_hi); ++i) {
        const double vi = fetch(i);
        int less = 0, equal = 0;
        for (int s = 0; s < n; ++s) {
            const double vs = fetch(s);
            less += vs < vi;
            equal += vs == vi;
        }
        if (!got_lo && less <= k_lo && k_lo < less + equal) {
            v_lo = vi;
            got_lo = true;
        }
        if (!got_hi && less <= k_hi && k_hi < less + equal) {
            v_hi = vi;
            got_hi = true;
        }
    }
    return 0.5 * (v_lo + v_hi);
}

// the repeating segment of _mask (repet.py:1398-1438): model[c][q][f] = median over s of V[c][q + s p][f], with r or
// r - 1 values per phase (quirk Q9) -- one median per (channel, phase, bin), shared by every frame of that phase
__global__ void k_gen_period_model(const double* __restrict__ V, int C, long long T, int F, int period,
                                   double* __restrict__ model) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)C * period * F) return;
    const int f = (int)(gid % F);
    const long long q = (gid / F) % period;
    const int c = (int)(gid / ((long long)F * period));
    const double* __restrict__ Vc = V + (long long)c * T * F;
    const long long r = (T + period - 1) / period;
    const int n = q >= T ? 0 : (int)(q < T - (r - 1) * period ? r : r - 1);
    model[gid] = gen_median(n, [&](int s) { return Vc[(q + (long long)s * period) * F + f]; });
}

// repeating model + soft mask + high-pass + mirror + apply, in place on X (repet.py:1398-1456, 1474-1506, 1529-1543,
// 185-197).  mode 0: period-strided frames of a phase (quirk Q9); 1: the in-range frames t + c p_t; 2: listed frames.
__global__ void k_gen_mask_apply(double2* __restrict__ X, const double* __restrict__ V, int C, long long T, int N, int F,
                                 int mode, int period, const double* __restrict__ period_model,
                                 const int* __restrict__ frame_period, int order, const int* __restrict__ idx,
                                 const int* __restrict__ cnt, int number, int first_frame, int cutoff) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= (long long)C * T * F) return;
    const int f = (int)(gid % F);
    const long long t = (gid / F) % T;
    const int c = (int)(gid / ((long long)F * T));
    if (t < first_frame) return;  // online frames before the buffer is full are never synthesised (quirk Q5)
    const double* __restrict__ Vc = V + (long long)c * T * F;
    double model;
    if (mode == 0) {
        model = period_model[((long long)c * period + t % period) * F + f];
    } else if (mode == 1) {
        const int p = frame_period[t];
        const int half = (order + 1) / 2;
        long long c_lo = 1 - half, c_hi = order - half;
        if (p > 0) {
            c_lo = max(c_lo, -(t / p));
            c_hi = min(c_hi, (T - 1 - t) / p);
        } else {
            c_lo = c_hi = 0;
        }
        const int n = (int)(c_hi - c_lo + 1);
        model = gen_median(n, [&](int s) { return Vc[(t + (c_lo + s) * p) * F + f]; });
    } else {
        const int n = cnt[t];
        const int* __restrict__ list = idx + t * number;
        model = gen_median(n, [&](int s) { return Vc[(long long)list[s] * F + f]; });
    }
    const double v = Vc[t * F + f];
    const double eps = 2.220446049250313e-16;
    double rep = (model != model) ? model : fmin(v, model);  // np.minimum keeps NaN
    double m = (rep + eps) / (v + eps);
    if (f >= 1 && f <= cutoff) m = 1.0;  // high-pass rows 1..cutoff, DC kept (quirk Q11)
    double2* __restrict__ row = X + ((long long)c * T + t) * N;
    double2 x = row[f];
    row[f] = make_double2(m * x.x, m * x.y);
    if (f >= 1 && f < N - f) {  // mirrored bin N - f (repet.py:188-190); f = N/2 is its own mirror
        x = row[N - f];
        row[N - f] = make_double2(m * x.x, m * x.y);
    }
}
// overlap-add of real(ifft) frames of every channel, interleaved output (repet.py:1089-1103, 898-909).
// trim = samples dropped at the start (N - H for centred frames, 0 online); frames below first_frame are skipped.
__global__ void k_gen_overlap_add(const double2* __restrict__ frames, int C, long long T, int N, int H, long long trim,
                                  int first_frame, long long S, double inv_norm, double* __restrict__ out, int ld) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= S * C) return;
    const long long m = gid / C;
    const int c = (int)(gid - m * C);
    const long long pos = m + trim;
    long long j_hi = pos / H;
    if (j_hi > T - 1) j_hi = T - 1;
    long long j_lo = pos - N + 1 <= 0 ? 0 : (pos - N + H) / H;
    if (j_lo < first_frame) j_lo = first_frame;
    double acc = 0.0;
    for (long long j = j_lo; j <= j_hi; ++j) acc += frames[((long long)c * T + j) * N + (pos - j * H)].x;
    out[m * ld + c] = acc * inv_norm;
}
// one step of the reference's in-place cross-fade (repet.py:388-414)
__global__ void k_gen_xfade(double* __restrict__ bg, const double* __restrict__ seg, long long k, long long len, long long ov,
                            int C, int first) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= len * C) return;
    const long long i = gid / C;
    double* __restrict__ dst = bg + k * C + gid;
    if (!first && i < ov) {
        const double up = (double)(2 * i + 1) / (double)(2 * ov);                 // triang(2 ov)[i]
        const double down = (double)(2 * (ov - 1 - i) + 1) / (double)(2 * ov);    // triang(2 ov)[ov + i]
        *dst = *dst * down + seg[gid] * up;
    } else {
        *dst += seg[gid];
    }
}

struct GenShape {
    int N, H, F, C;
    const double* d_window;
    double gain;
};

// the beat spectra of n_seg segments (rows [ts0 + s*seg_step, ... + len) of Vm^2, zero outside the clip), lags < n_lags
int gen_beat(repet_handle* h, Pool& pool, const GenShape& g, const double* Vm, long long T, long long ts0, int seg_step,
             int n_seg, int len, int n_lags, double* beat) {
    cudaStream_t st = h->stream;
    const int L = next_pow2((long long)len + n_lags);
    CU(cudaMemsetAsync(beat, 0, (size_t)n_seg * n_lags * sizeof(double), st));
    // (segments x frequency rows) in chunks of at most ~1 GB per transform buffer
    const size_t row_bytes = (size_t)L * sizeof(double2);
    const int seg_chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_seg, ((size_t)1 << 30) / (row_bytes * g.F)));
    const int f_chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)g.F, ((size_t)1 << 30) / (row_bytes * seg_chunk)));
    double2* z = pool.get<double2>((size_t)seg_chunk * f_chunk * L);
    double2* tmp = pool.get<double2>((size_t)seg_chunk * f_chunk * L);
    if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general beat spectrum");
    for (int s0 = 0; s0 < n_seg; s0 += seg_chunk) {
        const int ns = std::min(seg_chunk, n_seg - s0);
        for (int f0 = 0; f0 < g.F; f0 += f_chunk) {
            const int nf = std::min(f_chunk, g.F - f0);
            const long long total = (long long)ns * nf * L;
            k_gen_load_seq<<<blocks_for(total), 256, 0, st>>>(Vm, T, g.F, f0, nf, ts0 + (long long)s0 * seg_step, seg_step, ns,
                                                              len, L, z);
            fft_pow2(st, z, tmp, L, (long long)ns * nf, false);
            k_power<<<blocks_for(total), 256, 0, st>>>(z, total);
            fft_pow2(st, z, tmp, L, (long long)ns * nf, true);
            k_gen_accumulate_beat<<<blocks_for((long long)ns * n_lags, 128), 128, 0, st>>>(z, nf, ns, len, L, n_lags,
                                                                                          beat + (size_t)s0 * n_lags);
            h->launches += 3 + 2 * 16;
        }
    }
    pool.release(z);
    pool.release(tmp);
    return REPET_OK;
}

// One clip (or one segment of `extended`) through the pipeline.  d_audio: (S, C) float64 with row pitch ld on the
// device; d_out: same layout; d_ints: integer outputs of `method` on the device.
int gen_run(repet_handle* h, int method, const double* d_audio, long long S, int ld, const GenShape& g,
            const repet_params* p, double* d_out, int* d_ints) {
    cudaStream_t st = h->stream;
    Pool pool(st);
    const int N = g.N, H = g.H, F = g.F, C = g.C;
    const bool online = method == GEN_SIMONLINE;
    long long T;
    int pad, first_frame = 0;
    if (online) {
        const int B = p->buffer_frames;
        if (B < 1) return fail(h, REPET_E_INVALID_ARG, "buffer_length must cover at least one frame");
        if (p->online_frame_base < 0) return fail(h, REPET_E_INVALID_ARG, "online_frame_base must not be negative");
        // the reference's warm-up loop fails to broadcast (repet.py:801-804); a window of a longer stream
        // (online_frame_base > 0) has had its warm-up earlier
        if (S < N || (p->online_frame_base == 0 && (long long)(B - 2) * H + N > S))
            return fail(h, REPET_E_INVALID_ARG, "operands could not be broadcast together (signal shorter than the buffer)");
        T = (S - N + H - 1) / H + 1;  // repet.py:781
        pad = 0;
        first_frame = std::max(0, B - 1 - p->online_frame_base);
    } else {
        T = (S + H - 1) / H + 1;  // repet.py:1018-1028 with N = 2H
        pad = N / 2;
    }
    if (T > 2000000000LL / std::max(N, 1)) return fail(h, REPET_E_UNSUPPORTED, "clip too long for the general path");
    double2* X = pool.get<double2>((size_t)C * T * N);
    double2* tmp = pool.get<double2>((size_t)C * T * N);
    double* V = pool.get<double>((size_t)C * T * F);
    double* Vm = pool.get<double>((size_t)T * F);
    if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
    k_gen_frames<<<blocks_for((long long)C * T * N), 256, 0, st>>>(d_audio, S, C, ld, g.d_window, N, H, pad, T, X);
    fft_pow2(st, X, tmp, N, (long long)C * T, false);
    k_gen_magnitude<<<blocks_for(T * F), 256, 0, st>>>(X, C, T, N, F, V, Vm);
    h->launches += 2 + 13;

    int mode = 0, period_host = 0, *frame_period = nullptr, *idx = nullptr, *cnt = nullptr;
    if (method == GEN_ORIGINAL) {
        const int lag_hi = (int)std::min<long long>(p->period_hi, T / 3);  // quirk Q2
        if (p->period_lo < 0 || lag_hi <= p->period_lo)
            return fail(h, REPET_E_TOO_SHORT, "attempt to get argmax of an empty sequence (signal too short for the period range)");
        double* beat = pool.get<double>(lag_hi);
        if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
        int rc = gen_beat(h, pool, g, Vm, T, 0, 0, 1, (int)T, lag_hi, beat);
        if (rc) return rc;
        k_gen_argmax<<<1, 32, 0, st>>>(beat, 1, lag_hi, p->period_lo, lag_hi, d_ints);
        CU(cudaMemcpyAsync(&period_host, d_ints, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        mode = 0;
    } else if (method == GEN_ADAPTIVE) {
        const int L = p->segment_length, step = p->segment_step;
        if (L <= 0 || step <= 0) return fail(h, REPET_E_INVALID_ARG, "segment length and step must be positive");
        if (p->filter_order < 1) return fail(h, REPET_E_INVALID_ARG, "filter_order must be at least 1");
        const int lag_hi = std::min(p->period_hi, L / 3);
        if (p->period_lo < 0 || lag_hi <= p->period_lo)
            return fail(h, REPET_E_TOO_SHORT, "attempt to get argmax of an empty sequence (segment too short for the period range)");
        const int n_seg = (int)((T + step - 1) / step);
        const int left = L / 2;  // ceil((L - 1) / 2), repet.py:1182
        double* beat = pool.get<double>((size_t)n_seg * lag_hi);
        int* seg_period = pool.get<int>(n_seg);
        if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
        int rc = gen_beat(h, pool, g, Vm, T, -left, step, n_seg, L, lag_hi, beat);
        if (rc) return rc;
        k_gen_argmax<<<blocks_for(n_seg, 128), 128, 0, st>>>(beat, n_seg, lag_hi, p->period_lo, lag_hi, seg_period);
        k_gen_expand<<<blocks_for(T), 256, 0, st>>>(seg_period, T, step, p->period_lo, d_ints);
        frame_period = d_ints;
        mode = 1;
    } else if (method == GEN_SIM || online) {
        if (p->similarity_number < 1) return fail(h, REPET_E_INVALID_ARG, "similarity_number must be at least 1");
        if (p->similarity_distance < 0) return fail(h, REPET_E_INVALID_ARG, "similarity_distance must not be negative");
        const int number = p->similarity_number;
        double* An = pool.get<double>((size_t)T * F);
        if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
        k_gen_normalize<<<(unsigned)T, 256, 0, st>>>(Vm, T, F, An);
        cnt = d_ints;
        idx = d_ints + T;
        CU(cudaMemsetAsync(cnt, 0, (size_t)T * sizeof(int), st));
        if (online) {
            const int B = p->buffer_frames;
            const size_t smem = (size_t)B * 12 + 16;
            if (smem > 200 * 1024) return fail(h, REPET_E_UNSUPPORTED, "buffer_length too long for the general online selection");
            if (smem > 48 * 1024) CU(cudaFuncSetAttribute(k_gen_online, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            if (T > first_frame)
                k_gen_online<<<(unsigned)(T - first_frame), 256, smem, st>>>(An, (int)T, F, B, p->online_frame_base, first_frame,
                                                                            p->similarity_threshold, p->similarity_distance,
                                                                            number, idx, cnt);
        } else {
            const size_t smem = (size_t)(GEN_IDX_CHUNK + 2 * (size_t)p->similarity_distance) * sizeof(double);
            if (smem > 200 * 1024) return fail(h, REPET_E_UNSUPPORTED, "similarity_distance too long for the general similar-frame selection");
            if (smem > 48 * 1024) CU(cudaFuncSetAttribute(k_gen_indices, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            // S and k_gen_indices' per-CTA kept lists are the quadratic part of the call, and the workspace limit
            // governs them: need(P) = P rows of S + one list of T ints per selection CTA.  The whole matrix when
            // need(T) fits; otherwise panels of P rows, the largest multiple of the Gram tile (64) that fits, 64 at
            // least.  S is bitwise symmetric, so a panel's rows are the columns whose lists it settles: panels give
            // the whole matrix's lists exactly.  The linear buffers (X, tmp, V, Vm, An and the entry point's staging)
            // are not counted against the limit.
            const long long max_ctas = 2LL * h->sm_count;
            auto need = [&](long long P) { return (size_t)P * T * sizeof(double) + (size_t)std::min(P, max_ctas) * T * sizeof(int); };
            const size_t limit = default_ws_limit(h);
            long long P = T;
            if (need(T) > limit) {
                P = std::min<long long>(T, (long long)(limit / ((size_t)T * sizeof(double)))) / 64 * 64;
                while (P > 64 && need(P) > limit) P -= 64;
                P = std::min(T, std::max(P, 64LL));
            }
            double* Sm = pool.get<double>((size_t)P * T);
            int* kept_scratch = pool.get<int>((size_t)std::min(P, max_ctas) * T);
            if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory for the similarity matrix");
            for (long long r0 = 0; r0 < T; r0 += P) {
                const long long rows = std::min(P, T - r0);
                dim3 grid((unsigned)((T + 63) / 64), (unsigned)((rows + 63) / 64));
                k_gen_gram<<<grid, 256, 0, st>>>(An, T, F, r0, rows, Sm);
                k_gen_indices<<<(unsigned)std::min(rows, max_ctas), 512, smem, st>>>(Sm, (int)T, (int)r0, (int)rows,
                                                                                    p->similarity_threshold,
                                                                                    p->similarity_distance, number, idx,
                                                                                    cnt, kept_scratch);
                h->launches += 2;
            }
            pool.release(kept_scratch);
            pool.release(Sm);
        }
        mode = 2;
    } else {
        return fail(h, REPET_E_INVALID_ARG, "unknown method");
    }
    double* period_model = nullptr;
    if (mode == 0) {
        period_model = pool.get<double>((size_t)C * period_host * F);
        if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
        k_gen_period_model<<<blocks_for((long long)C * period_host * F), 256, 0, st>>>(V, C, T, F, period_host, period_model);
    }
    k_gen_mask_apply<<<blocks_for((long long)C * T * F), 256, 0, st>>>(X, V, C, T, N, F, mode, period_host, period_model,
                                                                      frame_period, p->filter_order, idx, cnt,
                                                                      p->similarity_number, first_frame, p->cutoff_bins);
    fft_pow2(st, X, tmp, N, (long long)C * T, true);
    k_gen_overlap_add<<<blocks_for(S * C), 256, 0, st>>>(X, C, T, N, H, online ? 0 : N - H, first_frame, S,
                                                        1.0 / ((double)N * g.gain), d_out, ld);
    h->launches += 4 + 13;
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

}  // namespace

extern "C" {

int repet_general_f64(repet_handle* h, int method, const double* audio, int64_t n_samples, int n_channels,
                      const repet_params* p, const double* window, double* background, int32_t* ints_host,
                      int64_t ints_capacity) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!audio || !p || !window || !background || n_samples < 1 || n_channels < 1)
        return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    const int N = p->window_length, H = p->step_length;
    if (N < 4 || (N & (N - 1)) || 2 * H != N)
        return fail(h, REPET_E_INVALID_ARG, "window_length must be a power of two and step_length half of it (repet.py:130-132)");
    if (method < GEN_ORIGINAL || method > GEN_SIMONLINE) return fail(h, REPET_E_INVALID_ARG, "unknown method");
    CU(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    Pool pool(st);
    const long long S = n_samples;
    const int C = n_channels;
    const long long need = repet_ints_per_clip(method, p, n_samples);
    if (ints_host && ints_capacity < need) return fail(h, REPET_E_INVALID_ARG, "integer output buffer too small");
    double* d_audio = pool.get<double>((size_t)S * C);
    double* d_out = pool.get<double>((size_t)S * C);
    double* d_window = pool.get<double>(N);
    int* d_ints = pool.get<int>((size_t)std::max<long long>(need, 1));
    if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
    CU(cudaMemcpyAsync(d_audio, audio, (size_t)S * C * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_window, window, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st));
    GenShape g{N, H, N / 2 + 1, C, d_window, p->cola_gain};
    int rc = REPET_OK;
    if (method == GEN_EXTENDED && S >= (long long)p->segment_length + p->segment_step) {
        // repet.py:263-419: `original` per segment, the last one takes the remainder, cross-faded in order
        const long long seg_len = p->segment_length, step = p->segment_step, ov = seg_len - step;
        if (seg_len <= 0 || step <= 0 || ov <= 0) return fail(h, REPET_E_INVALID_ARG, "segment_length must exceed segment_step (both positive)");
        const int n_seg = 1 + (int)((S - seg_len) / step);
        const long long last_len = S - (long long)(n_seg - 1) * step;
        double* d_seg = pool.get<double>((size_t)std::max(seg_len, last_len) * C);
        if (!pool.ok) return fail(h, REPET_E_OOM, "out of device memory in the general path");
        CU(cudaMemsetAsync(d_out, 0, (size_t)S * C * sizeof(double), st));
        long long k = 0;
        for (int j = 0; j < n_seg && !rc; ++j, k += step) {
            const long long len = j < n_seg - 1 ? seg_len : last_len;
            rc = gen_run(h, GEN_ORIGINAL, d_audio + k * C, len, C, g, p, d_seg, d_ints + j);
            if (!rc) k_gen_xfade<<<blocks_for(len * C), 256, 0, st>>>(d_out, d_seg, k, len, ov, C, j == 0 ? 1 : 0);
        }
    } else {
        rc = gen_run(h, method == GEN_EXTENDED ? GEN_ORIGINAL : method, d_audio, S, C, g, p, d_out, d_ints);
    }
    if (rc) return rc;
    CU(cudaMemcpyAsync(background, d_out, (size_t)S * C * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (ints_host && need > 0) CU(cudaMemcpyAsync(ints_host, d_ints, (size_t)need * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    return REPET_OK;
}

}  // extern "C"
