// Hand-written sm_100a kernels of the REPET separation path (fp32 arithmetic, fp64 for the
// one-per-clip period search).  Reference semantics: /root/reference/repet.py, cited per kernel.
//
// Data layout in HBM (per batch item = clip or 10 s segment):
//   audio  [clip][channel][sample]  fp32 planar
//   X      [item][frame][channel][1024] float2  half spectrum; bin 0 = (DC.re, Nyquist.re)
//   P      [item][frame][1032] fp32   (mean_c |X|)^2 (beat spectrum) or mean_c |X| (similarity)
//   model  [item][channel][phase][1032] fp32   median over the period-strided frames
// Frames are the slow axis, bins the fast one: every gather along time (period-strided
// medians, similar-frame medians) is a coalesced row read.
#include "repet_kernels.cuh"
#include "fft_core.cuh"
#include "median_networks.cuh"

namespace repet {

using FF = Fft<WIN_N>;  // frame transforms (STFT / ISTFT)
using TF = Fft<2048>;   // time-axis transforms of the beat spectrum


// ------------------------------------------------------------------------------------------
// k_stft  --  _stft + abs + channel mean (+ square)      repet.py:1001-1060, 158, 162, 667
// One CTA of 128 threads walks K consecutive frames of one item.  Both channels ride in one
// complex transform (z = w*(xL + i xR)) and are separated by Hermitian symmetry afterwards.
// The second half of frame j is the first half of frame j+1 and lands in the SAME thread
// (n = n1*128 + t), so the overlap is carried in registers: 16 new samples per thread-frame.
// Algorithmic bytes per frame: 2*4 KB audio in, 16 KB X out, 4.1 KB P out.
// ------------------------------------------------------------------------------------------
// one output bin of the Hermitian split: a = Z[k]/2, b = Z[2048-k]/2 (the window is pre-halved)
//   XL[k] = a + conj(b)            XR[k] = -i (a - conj(b))
// VSQ: also write the squared magnitudes |X_c|^2 of every channel to vrow[c * PPITCH + k] (the adaptive median
// gathers 5 rows per frame: 4-byte magnitudes halve its L2 traffic against the 8-byte spectra)
template <int NCH, bool VSQ = false>
__device__ __forceinline__ void stft_emit(float2 a, float2 b, int k, float2* __restrict__ xrow, float* __restrict__ prow,
                                          int pmode, float* __restrict__ vrow = nullptr) {
    const float2 xl = __ffma2_rn(b, make_float2(1.f, -1.f), a);
    xrow[k] = xl;
    const float l2 = cmag2(xl);
    float mean = fast_sqrt(l2);
    if (VSQ) vrow[k] = l2;
    if (NCH == 2) {
        const float2 d = __ffma2_rn(b, make_float2(-1.f, 1.f), a);  // a - conj(b); XR = (d.y, -d.x)
        xrow[XPITCH + k] = make_float2(d.y, -d.x);
        const float r2 = cmag2(d);
        mean = 0.5f * (mean + fast_sqrt(r2));
        if (VSQ) vrow[PPITCH + k] = r2;
    }
    if (prow) prow[k] = pmode == P_POWER ? mean * mean : mean;
}

// display spectrogram |STFT(mean_c x)| (README.md:79-81): the transform is linear, so the STFT of the channel
// mean is the mean of the channel spectra; only the magnitude row is written
template <int NCH>
__device__ __forceinline__ void stft_emit_mixdown(float2 a, float2 b, int k, float* __restrict__ prow) {
    const float2 xl = __ffma2_rn(b, make_float2(1.f, -1.f), a);
    if (NCH == 2) {
        const float2 d = __ffma2_rn(b, make_float2(-1.f, 1.f), a);  // XR = (d.y, -d.x)
        prow[k] = 0.5f * cmag(make_float2(xl.x + d.y, xl.y - d.x));
    } else {
        prow[k] = cmag(xl);
    }
}

template <int NCH, int MINB, bool MIXDOWN = false, bool VSQ = false>
__global__ void __launch_bounds__(FF::THREADS, MINB)
k_stft(const float* __restrict__ audio, Geom g, const float* __restrict__ window, FftTables tb,
       float2* __restrict__ X, float* __restrict__ P, int pmode, int K, float* __restrict__ Vsq = nullptr) {
    __shared__ float2 s_bufA[FF::BUF];
    __shared__ float2 s_bufB[FF::BUF];
    __shared__ float2 s_tw2[FF::TW2];
    __shared__ float s_win[WIN_N];  // half the window: the 1/2 of the channel split is folded in here
    const int t = threadIdx.x;
    const int item = blockIdx.y;
    const int j0 = blockIdx.x * K;
    const int j1 = min(j0 + K, g.T);
    s_tw2[t] = tb.tw2[t];
    FF::Twiddle1 tw;
    tw.load(tb.tw1, t);
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) s_win[n1 * FF::THREADS + t] = 0.5f * __ldg(&window[n1 * FF::THREADS + t]);
    const int gitem = g.item0 + item;
    const int clip = gitem / g.seg_per_clip, sg = gitem - clip * g.seg_per_clip;
    const float* __restrict__ a0 = audio + g.first_offset + (long long)clip * g.clip_stride + (long long)sg * g.seg_stride;
    const float* __restrict__ a1 = a0 + g.chan_stride;
    // The window lives in shared memory so that the registers can hold TWO half frames: the first half of the
    // current frame (= the previous frame's second half) and the second half, which is fetched one frame ahead --
    // its global-load latency hides behind the previous frame's transform instead of stalling the window multiply.
    float cl[8], cr[8], nl[8], nr[8];
    auto fetch_half = [&](int j, float (&dl)[8], float (&dr)[8]) {  // second half of frame j
        const long long base = (long long)(j + g.frame_shift) * HOP + t;
        if (base - t >= 0 && base - t + HOP <= g.S) {  // whole half frame inside the signal: no bounds checks
#pragma unroll
            for (int n1 = 0; n1 < 8; ++n1) {
                dl[n1] = __ldg(a0 + base + n1 * FF::THREADS);
                dr[n1] = NCH == 2 ? __ldg(a1 + base + n1 * FF::THREADS) : 0.f;
            }
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 8; ++n1) {
                const long long idx = base + n1 * FF::THREADS;
                const bool ok = idx >= 0 && idx < g.S;
                dl[n1] = ok ? __ldg(a0 + idx) : 0.f;
                dr[n1] = (NCH == 2 && ok) ? __ldg(a1 + idx) : 0.f;
            }
        }
    };
    fetch_half(j0 - 1, cl, cr);  // first half of the first frame
    fetch_half(j0, nl, nr);
    __syncthreads();
    for (int j = j0; j < j1; ++j) {
        float2 r[16];
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) {
            const float w_lo = s_win[n1 * FF::THREADS + t], w_hi = s_win[(8 + n1) * FF::THREADS + t];
            r[n1] = make_float2(w_lo * cl[n1], w_lo * cr[n1]);
            r[8 + n1] = make_float2(w_hi * nl[n1], w_hi * nr[n1]);
            cl[n1] = nl[n1];
            cr[n1] = nr[n1];
        }
        if (j + 1 < j1) fetch_half(j + 1, nl, nr);  // consumed one transform from now
        FF::stage1(r, tw, s_bufA, t);
        __syncthreads();
        FF::stage2(r, s_bufA, s_bufB, s_tw2, t);
        __syncthreads();
        FF::stage3(r, s_bufB, t);
        // the thread now holds Z[k]/2 and Z[N-k]/2 for its 8 bins k < N/2: split in registers
        const size_t frame = (size_t)item * g.T + j;
        float2* __restrict__ xrow = X + frame * (size_t)(NCH * XPITCH);
        float* __restrict__ prow = P ? P + frame * (size_t)PPITCH : nullptr;
        float* __restrict__ vrow = VSQ ? Vsq + frame * (size_t)(NCH * PPITCH) : nullptr;
        if (prow && t >= 1 && t < PPITCH - XPITCH) prow[XPITCH + t] = 0.f;  // rows 1025..1031: zero padding
        if (MIXDOWN) {
            if (t != 0) {
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int k3 = 0; k3 < 4; ++k3)
                        stft_emit_mixdown<NCH>(r[h * 8 + k3], r[(1 - h) * 8 + 7 - k3], (h == 0 ? t : FF::CCOLS - t) + FF::CCOLS * k3, prow);
            } else {
                const float2 dc = r[0], ny = r[4];
                prow[0] = NCH == 2 ? fabsf(dc.x + dc.y) : 2.f * fabsf(dc.x);
                prow[XPITCH] = NCH == 2 ? fabsf(ny.x + ny.y) : 2.f * fabsf(ny.x);
#pragma unroll
                for (int k3 = 1; k3 < 4; ++k3) stft_emit_mixdown<NCH>(r[k3], r[8 - k3], FF::CCOLS * k3, prow);
#pragma unroll
                for (int k3 = 0; k3 < 4; ++k3) stft_emit_mixdown<NCH>(r[8 + k3], r[8 + 7 - k3], FF::THREADS + FF::CCOLS * k3, prow);
            }
            continue;
        }
        if (t != 0) {
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int k3 = 0; k3 < 4; ++k3)
                    stft_emit<NCH, VSQ>(r[h * 8 + k3], r[(1 - h) * 8 + 7 - k3], (h == 0 ? t : FF::CCOLS - t) + FF::CCOLS * k3, xrow, prow, pmode, vrow);
        } else {
            // thread 0 owns the self-mirrored columns 0 and 128; bin 0 packs (DC, Nyquist), both real
            const float2 dc = r[0], ny = r[4];
            xrow[0] = make_float2(2.f * dc.x, 2.f * ny.x);
            if (NCH == 2) xrow[XPITCH] = make_float2(2.f * dc.y, 2.f * ny.y);
            if (VSQ) {
                vrow[0] = __fmul_rn(2.f * dc.x, 2.f * dc.x);
                vrow[XPITCH] = __fmul_rn(2.f * ny.x, 2.f * ny.x);
                if (NCH == 2) {
                    vrow[PPITCH] = __fmul_rn(2.f * dc.y, 2.f * dc.y);
                    vrow[PPITCH + XPITCH] = __fmul_rn(2.f * ny.y, 2.f * ny.y);
                }
            }
            if (prow) {
                const float m0 = NCH == 2 ? fabsf(dc.x) + fabsf(dc.y) : 2.f * fabsf(dc.x);
                const float mn = NCH == 2 ? fabsf(ny.x) + fabsf(ny.y) : 2.f * fabsf(ny.x);
                prow[0] = pmode == P_POWER ? m0 * m0 : m0;
                prow[XPITCH] = pmode == P_POWER ? mn * mn : mn;
            }
#pragma unroll
            for (int k3 = 1; k3 < 4; ++k3) stft_emit<NCH, VSQ>(r[k3], r[8 - k3], FF::CCOLS * k3, xrow, prow, pmode, vrow);
#pragma unroll
            for (int k3 = 0; k3 < 4; ++k3) stft_emit<NCH, VSQ>(r[8 + k3], r[8 + 7 - k3], FF::THREADS + FF::CCOLS * k3, xrow, prow, pmode, vrow);
        }
    }
}


void launch_stft(cudaStream_t st, const float* audio, Geom g, int nch, const float* window, FftTables tb, float2* X,
                 float* P, int pmode, int frames_per_cta, float* Vsq) {
    dim3 grid((g.T + frames_per_cta - 1) / frames_per_cta, g.n_items);
    if (Vsq) {  // X, P and the squared magnitudes of every channel (adaptive)
        if (nch == 2) k_stft<2, 4, false, true><<<grid, FF::THREADS, 0, st>>>(audio, g, window, tb, X, P, pmode, frames_per_cta, Vsq);
        else k_stft<1, 4, false, true><<<grid, FF::THREADS, 0, st>>>(audio, g, window, tb, X, P, pmode, frames_per_cta, Vsq);
        return;
    }
#define REPET_GO(NCH, MINB) k_stft<NCH, MINB><<<grid, FF::THREADS, 0, st>>>(audio, g, window, tb, X, P, pmode, frames_per_cta)
    if (pmode == P_MIXDOWN) {  // spectrogram only: X is not written
        if (nch == 2) k_stft<2, 4, true><<<grid, FF::THREADS, 0, st>>>(audio, g, window, tb, nullptr, P, pmode, frames_per_cta);
        else k_stft<1, 4, true><<<grid, FF::THREADS, 0, st>>>(audio, g, window, tb, nullptr, P, pmode, frames_per_cta);
        return;
    }
    if (nch == 2) {
        if (g_tuning.stft_minb >= 6) REPET_GO(2, 6);
        else if (g_tuning.stft_minb == 5) REPET_GO(2, 5);
        else REPET_GO(2, 4);
    } else {
        REPET_GO(1, 4);
    }
#undef REPET_GO
}

// ------------------------------------------------------------------------------------------
// k_beat  --  _acorr / _beatspectrum in the FFT domain        repet.py:1108-1158, 1161-1206
// b[l] = mean_f (1/(R-l)) sum_t P[f,t] P[f,t+l].  Per frequency row the autocorrelation is
// the inverse transform of |FFT_L(P_f)|^2 (L = 2048 >= R + max lag, so no circular alias for
// the lags consumed); by linearity the PSDs are SUMMED over f first and inverted once per clip
// (k_periods).  Two rows f, f+1 ride in one complex transform: |Fa|^2 + |Fb|^2 =
// (|Z[k]|^2 + |Z[-k]|^2)/2, so the kernel only accumulates |Z[k]|^2 per thread-owned bin, in
// registers, over all the rows the CTA owns -- no exchange, no atomics, deterministic.
// The CTA stages an 8-row x R tile of P (32 B per frame row: full sectors) transposed in
// shared memory.  Algorithmic bytes: P read once (4.1 KB per frame).
// ------------------------------------------------------------------------------------------
// 16-byte asynchronous global -> shared copy; src_bytes = 0 writes zeros (frames outside the clip)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src), "r"(src_bytes)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// BL = transform length: 2048, or 1024 when rows + max lag fit (10 s segments of `extended` / `adaptive`: less
// than half the butterflies).  Partials are written with a pitch of BEAT_L floats either way.
template <int BL>
__global__ void __launch_bounds__(BL / 16)
k_beat(const float* __restrict__ P, int T, int t_first, int t_len, int seg_step, int n_seg, FftTables tb,
       float* __restrict__ psd_part, int n_parts, int f_per_part, int TP) {
    using TF = Fft<BL>;
    extern __shared__ __align__(16) unsigned char s_raw[];
    float2* s_bufA = reinterpret_cast<float2*>(s_raw);
    float2* s_bufB = s_bufA + TF::BUF;
    float2* s_tw2 = s_bufB + TF::BUF;
    float4* s_tile = reinterpret_cast<float4*>(s_tw2 + TF::TW2);  // 2 x [TP] frames x 4 rows (16 B per frame)
    const int t = threadIdx.x;
    const int bi = blockIdx.y;
    const int item = bi / n_seg, sg = bi - item * n_seg;
    const int ts = t_first + sg * seg_step;
    const int f_begin = blockIdx.x * f_per_part;
    const int f_end = min(NBIN, f_begin + f_per_part);
    s_tw2[t] = (BL == 2048 ? tb.tw2_t : tb.tw2_t1k)[t];
    typename TF::Twiddle1 tw;
    tw.load(BL == 2048 ? tb.tw1_t : tb.tw1_t1k, t);
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    const float* __restrict__ Pitem = P + (size_t)item * T * PPITCH;
    // tiles of 4 rows x t_len frames, double buffered with cp.async: tile i+1 streams in while the
    // two transforms of tile i run.  Rows >= 1025 are the zero padding of P.
    auto fetch = [&](int f0, int buf) {
        float4* dst = s_tile + buf * TP;
        for (int row = t; row < t_len; row += TF::THREADS) {
            const int frame = ts + row;
            const bool ok = frame >= 0 && frame < T;
            cp_async16(dst + row, Pitem + (size_t)(ok ? frame : 0) * PPITCH + f0, ok ? 16 : 0);
        }
        cp_async_commit();
    };
    const int n_tiles = (f_end - f_begin + 3) >> 2;
    if (n_tiles > 0) fetch(f_begin, 0);
    for (int tile = 0; tile < n_tiles; ++tile) {
        const int f0 = f_begin + 4 * tile;
        if (tile + 1 < n_tiles) {
            fetch(f0 + 4, (tile + 1) & 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float* __restrict__ cur = reinterpret_cast<const float*>(s_tile + (tile & 1) * TP);
        const int npairs = (min(4, f_end - f0) + 1) >> 1;
        for (int pr = 0; pr < npairs; ++pr) {
            float2 r[16];
#pragma unroll
            for (int n1 = 0; n1 < 16; ++n1) {
                const int n = n1 * TF::THREADS + t;
                r[n1] = n < t_len ? *reinterpret_cast<const float2*>(cur + 4 * n + 2 * pr) : make_float2(0.f, 0.f);
            }
            TF::stage1(r, tw, s_bufA, t);
            __syncthreads();
            TF::stage2(r, s_bufA, s_bufB, s_tw2, t);
            __syncthreads();
            TF::stage3(r, s_bufB, t);
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = fmaf(r[i].x, r[i].x, fmaf(r[i].y, r[i].y, acc[i]));
        }
        // the buffer just consumed is refilled two iterations from now, after the barriers above
    }
    float* __restrict__ out = psd_part + ((size_t)bi * n_parts + blockIdx.x) * BEAT_L;
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int k3 = 0; k3 < 8; ++k3) out[TF::out_column(t, h) + TF::CCOLS * k3] = acc[h * 8 + k3];
}

template <int BL>
static size_t beat_smem_bytes(int t_len, int* TP_out) {
    int TP = ((t_len + 7) / 8) * 8 + 8;
    *TP_out = TP;
    return (size_t)(2 * Fft<BL>::BUF + Fft<BL>::TW2) * sizeof(float2) + (size_t)2 * TP * sizeof(float4);
}

template <int BL>
static void go_beat(cudaStream_t st, const float* P, int n_items, int T, int t_first, int t_len, int seg_step, int n_seg,
                    FftTables tb, float* psd_part, int n_parts, int f_per_part) {
    int TP;
    size_t smem = beat_smem_bytes<BL>(t_len, &TP);
    static SmemOptIn opt_in;
    smem_opt_in(k_beat<BL>, smem, opt_in);
    dim3 grid(n_parts, n_items * n_seg);
    k_beat<BL><<<grid, BL / 16, smem, st>>>(P, T, t_first, t_len, seg_step, n_seg, tb, psd_part, n_parts, f_per_part, TP);
}

void launch_beat(cudaStream_t st, const float* P, int n_items, int T, int t_first, int t_len, int seg_step, int n_seg,
                 FftTables tb, float* psd_part, int n_parts, int f_per_part, int L) {
    if (L == 1024) go_beat<1024>(st, P, n_items, T, t_first, t_len, seg_step, n_seg, tb, psd_part, n_parts, f_per_part);
    else go_beat<2048>(st, P, n_items, T, t_first, t_len, seg_step, n_seg, tb, psd_part, n_parts, f_per_part);
}

// ------------------------------------------------------------------------------------------
// k_periods  --  inverse transform of the summed PSD, unbiased normalisation, argmax
//                                                             repet.py:1129-1137, 1156, 1249-1291
// One CTA per clip (or per adaptive segment), fp64: the summed PSD is dominated by its DC
// bin, and doing this single small transform in double keeps the fp32 front end's error out
// of the argmax.  period = first argmax over lags [lo, hi) + 1 (quirks Q1, Q2).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_periods(const float* __restrict__ psd_part, const float* __restrict__ psd_part_im, int n_parts, int t_len,
          double norm_rows, int lag_lo, int lag_hi, int out_lo, int out_hi, double* __restrict__ beat_out,
          int beat_pitch, int* __restrict__ period, double* __restrict__ stats, int* __restrict__ cert, double cert_rel, int L) {
    // L = length of the time-axis transforms that produced the partials (1024 for short segments, else 2048);
    // the partials keep a pitch of L floats either way
    extern __shared__ __align__(16) unsigned char s_raw_periods[];
    double* s_cos = reinterpret_cast<double*>(s_raw_periods);  // [L]      cos(2 pi k / L)
    double* s_b = s_cos + L;                              // [L]      partial sums, then b[l]
    double* s_psd = s_b + L;                              // [L/2+1]  symmetric part of Re G
    double* s_im = s_psd + L / 2 + 1;                     // [L/2+1]  antisymmetric part of Im G
    const int t = threadIdx.x;
    const int bi = blockIdx.x;
    for (int k = t; k < L; k += 256) {
        double a = 0.0;
        const float* __restrict__ src = psd_part + (size_t)bi * n_parts * BEAT_L + k;
        for (int part = 0; part < n_parts; ++part) a += (double)src[(size_t)part * BEAT_L];
        s_b[k] = a;
        s_cos[k] = cospi((double)k / (double)(L / 2));
    }
    __syncthreads();
    for (int k = t; k <= L / 2; k += 256) s_psd[k] = 0.5 * (s_b[k] + s_b[(L - k) & (L - 1)]);
    __syncthreads();
    if (psd_part_im) {
        // blocked cross-spectrum G = sum conj(A) C: r[l] = (1/L) sum_k Re G cos - Im G sin, G Hermitian
        for (int k = t; k < L; k += 256) {
            double a = 0.0;
            const float* __restrict__ src = psd_part_im + (size_t)bi * n_parts * BEAT_L + k;
            for (int part = 0; part < n_parts; ++part) a += (double)src[(size_t)part * BEAT_L];
            s_b[k] = a;
        }
        __syncthreads();
        for (int k = t; k <= L / 2; k += 256) s_im[k] = 0.5 * (s_b[k] - s_b[(L - k) & (L - 1)]);
        __syncthreads();
    }
    int l0 = out_lo, l1 = out_hi;
    if (period) {
        l0 = (out_hi > out_lo) ? min(out_lo, lag_lo) : lag_lo;
        l1 = (out_hi > out_lo) ? max(out_hi, lag_hi) : lag_hi;
    }
    for (int l = l0 + t; l < l1; l += 256) {
        double s = 0.0;
        if (!beat_out) {
            // period search only: Clenshaw's recurrence for sum_k a_k cos(k theta) (and b_1 sin(theta) for the
            // sine series) -- one broadcast load and one dependent DFMA per term instead of a table lookup with
            // lane-dependent stride.  Its rounding (~1e-12 relative for the lags in range) is far inside the
            // 100 ppm window below which k_period_certify re-decides the argmax from exact sums.
            double sn, c;
            sincospi((double)l / (double)(L / 2), &sn, &c);
            const double c2 = 2.0 * c;
            double b1 = 0.0, b2 = 0.0, d1 = 0.0, d2 = 0.0;
            if (psd_part_im) {
                for (int k = L / 2 - 1; k >= 1; --k) {
                    const double b0 = fma(c2, b1, s_psd[k] - b2);
                    const double d0 = fma(c2, d1, s_im[k] - d2);
                    b2 = b1;
                    b1 = b0;
                    d2 = d1;
                    d1 = d0;
                }
            } else {
                for (int k = L / 2 - 1; k >= 1; --k) {
                    const double b0 = fma(c2, b1, s_psd[k] - b2);
                    b2 = b1;
                    b1 = b0;
                }
            }
            s = fma(b1, c, -b2) - d1 * sn;
        } else if (psd_part_im) {
            for (int k = 1; k < L / 2; ++k) {
                const int ph = (k * l) & (L - 1);
                s = fma(s_psd[k], s_cos[ph], s);
                s = fma(-s_im[k], s_cos[(ph - L / 4) & (L - 1)], s);  // sin(x) = cos(x - pi/2)
            }
        } else {
            for (int k = 1; k < L / 2; ++k) s = fma(s_psd[k], s_cos[(k * l) & (L - 1)], s);
        }
        s = 2.0 * s + s_psd[0] + ((l & 1) ? -s_psd[L / 2] : s_psd[L / 2]);
        s_b[l] = s / (double)L / ((double)(t_len - l) * norm_rows);
    }
    __syncthreads();
    if (beat_out)
        for (int l = out_lo + t; l < out_hi; l += 256) beat_out[(size_t)bi * beat_pitch + (l - out_lo)] = s_b[l];
    if (period && t == 0) {
        double best = s_b[lag_lo], second = -1.0e300;
        int arg = lag_lo, arg2 = -1;
        for (int l = lag_lo + 1; l < lag_hi; ++l) {
            const double v = s_b[l];
            if (v > best) {
                second = best;
                arg2 = arg;
                best = v;
                arg = l;
            } else if (v > second) {
                second = v;
                arg2 = l;
            }
        }
        period[bi] = arg + 1;
        if (cert) {
            // lags whose value is within CERT_REL of the best: k_period_certify re-evaluates them exactly.
            // If more than CERT_MAX qualify the CERT_MAX largest are kept (the maximum is always among
            // them); they are stored in ascending lag order, which the first-maximum rule relies on.
            int n = 0;
            int lags[CERT_MAX];
            const double floor_v = best - fabs(best) * cert_rel;
            for (int l = lag_lo; l < lag_hi; ++l) {
                if (!(s_b[l] >= floor_v)) continue;
                if (n < CERT_MAX) {
                    lags[n++] = l;
                } else {
                    int weakest = 0;
                    for (int q = 1; q < CERT_MAX; ++q)
                        if (s_b[lags[q]] < s_b[lags[weakest]]) weakest = q;
                    if (s_b[l] > s_b[lags[weakest]]) {  // drop the weakest, keep ascending order
                        for (int q = weakest; q + 1 < CERT_MAX; ++q) lags[q] = lags[q + 1];
                        lags[CERT_MAX - 1] = l;
                    }
                }
            }
            for (int q = 0; q < n; ++q) cert[bi * (CERT_MAX + 1) + 1 + q] = lags[q];
            cert[bi * (CERT_MAX + 1)] = n >= 2 ? n : 0;
        }
        if (stats) {
            stats[4 * bi + 0] = best;
            stats[4 * bi + 1] = second;
            stats[4 * bi + 2] = (double)arg;
            stats[4 * bi + 3] = (double)arg2;
        }
    }
}

void launch_periods(cudaStream_t st, const float* psd_part, const float* psd_part_im, int n_beat_items, int n_parts,
                    int t_len, double norm_rows, int lag_lo, int lag_hi, int out_lo, int out_hi, double* beat_out,
                    int beat_pitch, int* period, double* stats, int* cert, int L) {
    const size_t smem = (size_t)(2 * BEAT_L + 2 * (BEAT_L / 2 + 1)) * sizeof(double);
    static SmemOptIn opt_in;
    smem_opt_in(k_periods, smem, opt_in);
    k_periods<<<n_beat_items, 256, smem, st>>>(psd_part, psd_part_im, n_parts, t_len, norm_rows, lag_lo, lag_hi, out_lo,
                                              out_hi, beat_out, beat_pitch, period, stats, cert,
                                              g_tuning.cert_rel_ppm > 0 ? 1e-6 * g_tuning.cert_rel_ppm : CERT_REL, L);
}

// ------------------------------------------------------------------------------------------
// k_period_certify / k_period_finalize  --  near-tied period candidates decided in float64
// When several lags sit within CERT_REL of the maximum of the beat spectrum, the fp32 time-axis
// transforms of k_beat could flip their order.  Each candidate lag is re-evaluated exactly,
// b[l] = (1/(R-l)) sum_f sum_t P[f,t] P[f,t+l] (R rows of the clip or of the adaptive segment, zero outside the
// clip) accumulated in float64 straight from P (the 1/F factor
// is common), and the first maximum wins, as np.argmax does.  Unflagged clips cost one flag read.
// ------------------------------------------------------------------------------------------
constexpr int CERT_GROUP = 32;   // beat items whose flags one CTA scans (one per lane of warp 0)

__global__ void __launch_bounds__(256)
k_period_certify(const float* __restrict__ P, int T, int n_items, int t_first, int t_len, int seg_step, int n_seg,
                 const int* __restrict__ cert, double* __restrict__ cert_part) {
    // grid = (candidate slot, time chunk, group of 32 beat items): flagged items are rare, so the CTA reads
    // the 32 flags of its group at once and only walks the items that need this slot
    const int slot = blockIdx.x, chunk = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __shared__ unsigned s_flags;
    __shared__ double s_red[8];
    if (warp == 0) {
        const int mine = blockIdx.z * CERT_GROUP + lane;
        const unsigned flags = __ballot_sync(0xffffffffu, mine < n_items && cert[mine * (CERT_MAX + 1)] > slot);
        if (lane == 0) s_flags = flags;
    }
    __syncthreads();
    unsigned flags = s_flags;
    while (flags) {
        const int item = blockIdx.z * CERT_GROUP + __ffs(flags) - 1;
        flags &= flags - 1;
        const int lag = cert[item * (CERT_MAX + 1) + 1 + slot];
        // beat item = (clip, segment): rows [ts, ts + t_len) of the clip's P, zero outside [0, T)
        const int clip = item / n_seg, ts = t_first + (item - clip * n_seg) * seg_step;
        const float* __restrict__ Pi = P + (size_t)clip * T * PPITCH;
        const int rows = t_len - lag;
        const int per = (rows + CERT_TSPLIT - 1) / CERT_TSPLIT;
        const int t_begin = max(ts + chunk * per, 0), t_end = min(ts + min(rows, (chunk + 1) * per), T - lag);
        double acc = 0.0;
        for (int t = t_begin + warp; t < t_end; t += 8) {
            const float* __restrict__ a = Pi + (size_t)t * PPITCH;
            const float* __restrict__ b = Pi + (size_t)(t + lag) * PPITCH;
            constexpr int DOTN = (NBIN + 31) / 32;
            float av[DOTN], bv[DOTN];
#pragma unroll
            for (int i = 0; i < DOTN; ++i) {
                const int f = lane + 32 * i;
                av[i] = f < NBIN ? __ldg(a + f) : 0.f;
                bv[i] = f < NBIN ? __ldg(b + f) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < DOTN; ++i) acc = fma((double)av[i], (double)bv[i], acc);
        }
        // fixed-order reduction: lanes by butterfly, then the 8 warps in order
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) s_red[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double total = 0.0;
            for (int w = 0; w < 8; ++w) total += s_red[w];
            cert_part[((size_t)item * CERT_MAX + slot) * CERT_TSPLIT + chunk] = total;
        }
        __syncthreads();
    }
}

__global__ void k_period_finalize(const int* __restrict__ cert, const double* __restrict__ cert_part, int n_items,
                                  int t_len, int* __restrict__ period) {
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= n_items) return;
    const int n = cert[item * (CERT_MAX + 1)];
    if (n < 2) return;
    int arg = -1;
    double best = 0.0;
    for (int s = 0; s < n; ++s) {
        const int lag = cert[item * (CERT_MAX + 1) + 1 + s];
        double v = 0.0;
        for (int c = 0; c < CERT_TSPLIT; ++c) v += cert_part[((size_t)item * CERT_MAX + s) * CERT_TSPLIT + c];
        v /= (double)(t_len - lag);
        if (arg < 0 || v > best) {  // candidates are in ascending lag order: strict > keeps the first maximum
            best = v;
            arg = lag;
        }
    }
    period[item] = arg + 1;
}

void launch_period_certify(cudaStream_t st, const float* P, int n_items, int T, int t_first, int t_len, int seg_step,
                           int n_seg, const int* cert, double* cert_val, int* period) {
    dim3 grid(CERT_MAX, CERT_TSPLIT, (n_items + CERT_GROUP - 1) / CERT_GROUP);
    k_period_certify<<<grid, 256, 0, st>>>(P, T, n_items, t_first, t_len, seg_step, n_seg, cert, cert_val);
    k_period_finalize<<<(n_items + 127) / 128, 128, 0, st>>>(cert, cert_val, n_items, t_len, period);
}

// ------------------------------------------------------------------------------------------
// k_beat_blocked  --  the beat spectrum of clips longer than one transform
// For T + max lag > 2048 the time axis is cut into blocks of Bk = 2048 - max lag + 1 frames.
// Block b correlates a = P[b Bk .. b Bk + Bk) with c = P[b Bk .. b Bk + Bk + max lag - 1) (zero past
// T): sum_t a[t] c[t + l] has no circular alias for l < max lag.  One complex transform of
// z = a + i c gives A = (Z[k] + conj Z[-k])/2 and C = (Z[k] - conj Z[-k])/(2i); the kernel
// accumulates the cross-spectrum G[k] = conj(A) C over its rows in registers (thread-owned bins
// k and -k are paired through shared memory) and k_periods inverts sum G once per clip.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TF::THREADS)
k_beat_blocked(const float* __restrict__ P, int T, int Bk, int max_lag, FftTables tb, float* __restrict__ g_re,
               float* __restrict__ g_im, int n_fparts, int f_per_part, int TP) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    float2* s_bufA = reinterpret_cast<float2*>(s_raw);
    float2* s_bufB = s_bufA + TF::BUF;
    float2* s_tw2 = s_bufB + TF::BUF;
    float* s_tile = reinterpret_cast<float*>(s_tw2 + TF::TW2);  // [8][TP] rows of P, time contiguous
    const int t = threadIdx.x;
    const int item = blockIdx.z;
    const int blk = blockIdx.y;
    const int fpart = blockIdx.x;
    const int n_blocks = gridDim.y;
    const int t0 = blk * Bk;
    const int span = min(Bk + max_lag - 1, T - t0);  // valid frames of c
    const int a_len = min(Bk, T - t0);               // valid frames of a
    const int f_begin = fpart * f_per_part;
    const int f_end = min(NBIN, f_begin + f_per_part);
    s_tw2[t] = tb.tw2_t[t];
    TF::Twiddle1 tw;
    tw.load(tb.tw1_t, t);
    float acc_re[16], acc_im[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc_re[i] = acc_im[i] = 0.f;
    const float* __restrict__ Pitem = P + (size_t)item * T * PPITCH;
    for (int f0 = f_begin; f0 < f_end; f0 += 8) {
        __syncthreads();
        for (int idx = t; idx < 2 * span; idx += TF::THREADS) {
            const int row = idx >> 1, half = idx & 1;
            float4 v = __ldg(reinterpret_cast<const float4*>(Pitem + (size_t)(t0 + row) * PPITCH + f0 + 4 * half));
            const int f = f0 + 4 * half;
            if (f + 0 >= f_end) v.x = 0.f;
            if (f + 1 >= f_end) v.y = 0.f;
            if (f + 2 >= f_end) v.z = 0.f;
            if (f + 3 >= f_end) v.w = 0.f;
            s_tile[(4 * half + 0) * TP + row] = v.x;
            s_tile[(4 * half + 1) * TP + row] = v.y;
            s_tile[(4 * half + 2) * TP + row] = v.z;
            s_tile[(4 * half + 3) * TP + row] = v.w;
        }
        __syncthreads();
        const int nrows = min(8, f_end - f0);
        for (int fr = 0; fr < nrows; ++fr) {
            float2 r[16];
            const float* __restrict__ col = s_tile + fr * TP;
#pragma unroll
            for (int n1 = 0; n1 < 16; ++n1) {
                const int n = n1 * TF::THREADS + t;
                const float c = n < span ? col[n] : 0.f;
                r[n1] = make_float2(n < a_len ? c : 0.f, c);
            }
            TF::stage1(r, tw, s_bufA, t);
            __syncthreads();
            TF::stage2(r, s_bufA, s_bufB, s_tw2, t);
            __syncthreads();
            TF::stage3(r, s_bufB, t);
            // Z[k] and Z[-k] are both in this thread's registers (fft_out_column): pair them here
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int k3 = 0; k3 < 8; ++k3) {
                    const float2 p = r[h * 8 + k3];
                    // mirror of column c, slot k3: column 256-c, slot 7-k3; the self-mirrored columns of
                    // thread 0 pair (0: k3 <-> (8-k3)%8, 128: k3 <-> 7-k3) inside the same column
                    float2 zq;
                    if (t != 0) zq = r[(1 - h) * 8 + 7 - k3];
                    else zq = (h == 0) ? r[(8 - k3) & 7] : r[8 + 7 - k3];
                    const float2 q = make_float2(zq.x, -zq.y);  // conj Z[-k]
                    // conj(A) C = conj(p + q) * (-i) (p - q) / 4
                    const float sx = p.x + q.x, sy = -(p.y + q.y);  // conj(p + q)
                    const float dx = p.y - q.y, dy = -(p.x - q.x);  // -i (p - q)
                    acc_re[h * 8 + k3] = fmaf(0.25f, sx * dx - sy * dy, acc_re[h * 8 + k3]);
                    acc_im[h * 8 + k3] = fmaf(0.25f, sx * dy + sy * dx, acc_im[h * 8 + k3]);
                }
        }
    }
    const size_t part = ((size_t)item * n_blocks + blk) * n_fparts + fpart;
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int k3 = 0; k3 < 8; ++k3) {
            const int k = TF::out_column(t, h) + TF::CCOLS * k3;
            g_re[part * BEAT_L + k] = acc_re[h * 8 + k3];
            g_im[part * BEAT_L + k] = acc_im[h * 8 + k3];
        }
}

void launch_beat_blocked(cudaStream_t st, const float* P, int n_items, int T, int Bk, int max_lag, FftTables tb,
                         float* g_re, float* g_im, int n_blocks, int n_fparts, int f_per_part) {
    const int rows = Bk + max_lag - 1;
    const int TP = ((rows + 7) / 8) * 8 + 4;
    const size_t smem = (size_t)(2 * TF::BUF + TF::TW2) * sizeof(float2) + (size_t)8 * TP * sizeof(float);
    static SmemOptIn opt_in;
    smem_opt_in(k_beat_blocked, smem, opt_in);
    dim3 grid(n_fparts, n_blocks, n_items);
    k_beat_blocked<<<grid, TF::THREADS, smem, st>>>(P, T, Bk, max_lag, tb, g_re, g_im, n_fparts, f_per_part, TP);
}

// ------------------------------------------------------------------------------------------
// Medians.  Magnitudes are compared through their SQUARES (monotonic), so a median costs one
// or two square roots instead of n.  For n <= 32 the values sit in registers and go through a
// generated selection network (median_networks.cuh: pruned odd-even merge sort, only the
// half-comparators that reach the middle outputs).  np.median's even-count rule (mean of the two
// middle values) applies to the magnitudes, i.e. after the square roots.
// ------------------------------------------------------------------------------------------
// squared magnitude of bin k (0..1024) of one (frame, channel) row of X; bin 0 packs (DC, Nyquist)
__device__ __forceinline__ float row_mag2(const float2* __restrict__ row, int k) {
    if (k == 0) {
        const float x = __ldg(&row[0]).x;
        return __fmul_rn(x, x);
    }
    if (k == XPITCH) {
        const float y = __ldg(&row[0]).y;
        return __fmul_rn(y, y);
    }
    return cmag2(__ldg(&row[k]));
}

// median of the magnitudes of two adjacent bins (k, k+1) over N frames `stride` apart, one
// 16-byte load per frame.  first_is_dc: bin k = 0 holds (DC.re, Nyquist.re); only DC is used here.
template <int N>
__device__ __forceinline__ float2 strided_median_pair(const float2* __restrict__ base, size_t stride, bool first_is_dc) {
    float v0[N], v1[N];
#pragma unroll
    for (int s = 0; s < N; ++s) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(base + (size_t)s * stride));
        v0[s] = first_is_dc ? __fmul_rn(x.x, x.x) : __fmaf_rn(x.x, x.x, __fmul_rn(x.y, x.y));
        v1[s] = __fmaf_rn(x.z, x.z, __fmul_rn(x.w, x.w));
    }
    median_select<N>(v0);
    median_select<N>(v1);
    if (N & 1) return make_float2(fast_sqrt(v0[(N - 1) / 2]), fast_sqrt(v1[(N - 1) / 2]));
    return make_float2(0.5f * (fast_sqrt(v0[(N - 1) / 2]) + fast_sqrt(v0[N / 2])),
                       0.5f * (fast_sqrt(v1[(N - 1) / 2]) + fast_sqrt(v1[N / 2])));
}

template <int N>
__device__ __forceinline__ float strided_median(const float2* __restrict__ base, size_t stride, int k) {
    float v[N];
#pragma unroll
    for (int s = 0; s < N; ++s) v[s] = row_mag2(base + (size_t)s * stride, k);
    median_select<N>(v);
    return (N & 1) ? fast_sqrt(v[(N - 1) / 2]) : 0.5f * (fast_sqrt(v[(N - 1) / 2]) + fast_sqrt(v[N / 2]));
}

// Fallback for n > 32: rank selection straight from memory (O(n^2), exact).  `fetch(s)` returns
// squared magnitude s.
template <typename Fetch>
__device__ float median_by_rank(int n, Fetch fetch) {
    const int k_lo = (n - 1) >> 1, k_hi = n >> 1;
    float v_lo = 0.f, v_hi = 0.f;
    bool got_lo = false, got_hi = false;
    for (int i = 0; i < n && !(got_lo && got_hi); ++i) {
        const float vi = fetch(i);
        int less = 0, equal = 0;
        for (int j = 0; j < n; ++j) {
            const float vj = fetch(j);
            less += vj < vi;
            equal += vj == vi;
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
    return 0.5f * (fast_sqrt(v_lo) + fast_sqrt(v_hi));
}

// ------------------------------------------------------------------------------------------
// k_model  --  the repeating segment of _mask                      repet.py:1398-1438
// model[f, q] = median over s of V[f, s*p + q]; r = ceil(T/p) values for phases
// q < T-(r-1)p, r-1 otherwise (the reference's zero padding is excluded, quirk Q9).
// Grid (phase groups + 1, items*channels).  A CTA of 128 threads owns MODEL_QB consecutive
// phases of one (item, channel); each thread takes bin PAIRS (16-byte loads) in 4 passes of 256
// bins, so every gather is a coalesced 2 KB row segment and a thread keeps 2n loads in flight.
// The extra CTA column does the Nyquist bin (packed in bin 0's imaginary slot), one phase per
// thread.  Algorithmic bytes: X read once.
// ------------------------------------------------------------------------------------------
constexpr int MODEL_QB = 8;

template <int N>
__device__ __forceinline__ void model_phase(const float2* __restrict__ base, size_t stride, float* __restrict__ out, int t) {
#pragma unroll 1
    for (int k = 2 * t; k < XPITCH; k += 256) {
        const float2 m = strided_median_pair<N>(base + k, stride, k == 0);
        *reinterpret_cast<float2*>(out + k) = m;
    }
}

__global__ void __launch_bounds__(128)
k_model(const float2* __restrict__ X, int T, int nch, const int* __restrict__ period, int pmax,
        float* __restrict__ model, int n_groups) {
    const int item = blockIdx.y / nch, c = blockIdx.y - item * nch;
    const int p = period[item];
    if (p <= 0) return;
    const int t = threadIdx.x;
    const int r = (T + p - 1) / p;
    const int k0 = T - (r - 1) * p;
    const size_t stride = (size_t)p * nch * XPITCH;
    const float2* __restrict__ chan = X + (size_t)item * T * (size_t)(nch * XPITCH) + (size_t)c * XPITCH;
    float* __restrict__ mrow = model + ((size_t)item * nch + c) * (size_t)pmax * PPITCH;
    if ((int)blockIdx.x == n_groups) {
        // Nyquist bins of every phase
        for (int q = t; q < p; q += 128) {
            const int n = q < k0 ? r : r - 1;
            const float2* __restrict__ base = chan + (size_t)q * (nch * XPITCH);
            float med;
            switch (n) {
#define REPET_CASE(N) case N: med = strided_median<N>(base, stride, XPITCH); break;
                REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
                REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
                REPET_CASE(15) REPET_CASE(16) REPET_CASE(17) REPET_CASE(18) REPET_CASE(19) REPET_CASE(20) REPET_CASE(21)
                REPET_CASE(22) REPET_CASE(23) REPET_CASE(24) REPET_CASE(25) REPET_CASE(26) REPET_CASE(27) REPET_CASE(28)
                REPET_CASE(29) REPET_CASE(30) REPET_CASE(31) REPET_CASE(32)
#undef REPET_CASE
                default:
                    med = n <= 0 ? nanf("")
                                 : median_by_rank(n, [&](int s) { return row_mag2(base + (size_t)s * stride, XPITCH); });
            }
            mrow[(size_t)q * PPITCH + XPITCH] = med;
        }
        return;
    }
    const int q_end = min(p, ((int)blockIdx.x + 1) * MODEL_QB);
    for (int q = blockIdx.x * MODEL_QB; q < q_end; ++q) {
        const int n = q < k0 ? r : r - 1;
        const float2* __restrict__ base = chan + (size_t)q * (nch * XPITCH);
        float* __restrict__ out = mrow + (size_t)q * PPITCH;
        switch (n) {
#define REPET_CASE(N) case N: model_phase<N>(base, stride, out, t); break;
            REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
            REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
            REPET_CASE(15) REPET_CASE(16) REPET_CASE(17) REPET_CASE(18) REPET_CASE(19) REPET_CASE(20) REPET_CASE(21)
            REPET_CASE(22) REPET_CASE(23) REPET_CASE(24) REPET_CASE(25) REPET_CASE(26) REPET_CASE(27) REPET_CASE(28)
            REPET_CASE(29) REPET_CASE(30) REPET_CASE(31) REPET_CASE(32)
#undef REPET_CASE
            default:
                for (int k = t; k < XPITCH; k += 128)
                    out[k] = n <= 0 ? nanf("")
                                    : median_by_rank(n, [&](int s) { return row_mag2(base + (size_t)s * stride, k); });
        }
    }
}

void launch_model(cudaStream_t st, const float2* X, int n_items, int T, int nch, const int* period, int pmax,
                  float* model) {
    const int n_groups = (pmax + MODEL_QB - 1) / MODEL_QB;
    dim3 grid(n_groups + 1, n_items * nch);
    k_model<<<grid, 128, 0, st>>>(X, T, nch, period, pmax, model, n_groups);
}

// Soft mask of one bin: (min(model, V) + eps) / (V + eps)          repet.py:1441-1448 (quirk Q10)
// computed from the squared magnitude as min(model * rsqrt(V^2), 1): no square root, no division.
// V = 0 gives model * inf = inf (or NaN for model = 0), and fminf(., 1) returns 1 -- the
// reference's eps/eps.  For model = 0 < V the reference's eps/(V+eps) ~ 1e-16/V becomes 0.
// ---- mbarrier / bulk-copy (TMA) primitives for the spectra ring of k_mask_istft ----
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_addr(bar)), "r"(parity)
        : "memory");
}
// one thread: global -> shared bulk copy of `bytes` (multiple of 16), completion on `bar`
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // earlier generic accesses to the buffer first
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

// mask = min(model, |X|) / |X| (repet.py:1441-1452 with eps = machine epsilon): model * rsqrt(|X|^2) capped at 1.
// |X| = 0 gives 0 * inf = NaN, which fminf drops in favour of 1 -- the reference's (0 + eps) / (0 + eps) (quirk Q10).
__device__ __forceinline__ float soft_mask(float model, float v2) { return fminf(model * fast_rsqrt(v2), 1.0f); }
// The same, but a NaN MODEL stays NaN, as np.minimum keeps it (a REPET-SIM frame whose similar-frame list is
// empty has np.median([]) = NaN as its model, and the reference's output is NaN over that frame).  Used for the
// DC bin only: one NaN bin makes the whole inverse transform of the frame NaN, so the other bins can keep the
// cheaper form.  |X|^2 + FLT_MIN keeps the silent-frame case finite (the masked value is mask * 0 = 0 anyway).
__device__ __forceinline__ float soft_mask_keep_nan(float model, float v2) {
    float r;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(model * fast_rsqrt(v2 + 1.17549435e-38f)), "f"(1.0f));
    return r;
}
// helper-level mask (returns the mask itself): exact in both special cases
__device__ __forceinline__ float soft_mask_exact(float model, float v2) {
    return model != model ? model : soft_mask(model, v2);
}

// ------------------------------------------------------------------------------------------
// k_mask_istft  --  rest of _mask + high-pass + mirror + apply + _istft
//                                                       repet.py:1441-1456, 185-200, 1063-1105
// One CTA of 128 threads produces `nblk` consecutive output blocks of H samples of one item;
// block b = second half of frame b + first half of frame b+1, so the CTA walks nblk+1 frames.
// Per frame: each bin's mask is computed once (both channels), the masked spectra are packed
// Z = YL + i YR with their Hermitian mirror, and ONE inverse complex transform (forward FFT of
// the re/im-swapped input) returns both channels' frames.  The output index n = pi + 256*k3
// keeps both halves of the overlap in the same thread: overlap-add happens in registers.
// MASKED = false is the plain _istft helper.
// Algorithmic bytes per frame: 16 KB X in, 8 KB audio out (+ model rows, L2 resident).
// ------------------------------------------------------------------------------------------
constexpr size_t MASK_ISTFT_SMEM = (size_t)(2 * WIN_N + FF::BUF + FF::TW2) * sizeof(float2) + 2 * sizeof(uint64_t);

template <int NCH, bool MASKED, int MINB>
__global__ void __launch_bounds__(FF::THREADS, MINB)
k_mask_istft(const float2* __restrict__ X, Geom g, const int* __restrict__ period, int pmax,
             const float* __restrict__ model, int cutoff, float scale, FftTables tb, float* __restrict__ out,
             int nblk) {
    // spectra ring: frame f's X rows (NCH x N/2 float2, one bulk copy) land in s_ring[f & 1] while
    // earlier frames are transformed; once read, the slot doubles as the transform's first exchange
    // buffer, and it is refilled (two frames ahead) when the second stage has drained it
    extern __shared__ __align__(128) unsigned char s_dyn[];  // MASK_ISTFT_SMEM bytes (above the static limit at N = 2048)
    float2(*s_ring)[WIN_N] = reinterpret_cast<float2(*)[WIN_N]>(s_dyn);  // y2 layout and a stereo frame: N float2 each
    float2* s_y1 = reinterpret_cast<float2*>(s_dyn) + 2 * WIN_N;
    float2* s_tw2 = s_y1 + FF::BUF;
    uint64_t* s_full = reinterpret_cast<uint64_t*>(s_tw2 + FF::TW2);
    constexpr uint32_t ROW_BYTES = NCH * XPITCH * sizeof(float2);
    const int t = threadIdx.x;
    const int item = blockIdx.y;
    const int b0 = blockIdx.x * nblk;               // first output block
    // output blocks: T-1 for centred frames; T+1 for online frames (frame j fills blocks j and j+1,
    // so the last block holds the second half of the last frame alone)
    const int n_blocks = g.T + 2 * g.frame_shift - 1;
    const int b1 = min(b0 + nblk, n_blocks);        // one past the last output block
    const float2* __restrict__ Xitem = X + (size_t)item * g.T * (size_t)(NCH * XPITCH);
    // frame jc (centred index) reads row jc - frame_shift; rows outside [first_frame, T) do not exist
    auto row_of = [&](int jc) { return jc - g.frame_shift; };
    auto exists = [&](int jc) { return jc <= b1 && row_of(jc) >= g.first_frame && row_of(jc) < g.T; };
    if (t == 0) {
        mbar_init(&s_full[0], 1);
        mbar_init(&s_full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    s_tw2[t] = tb.tw2[t];
    typename FF::TwiddleT tw;
    tw.load(tb.tw1, t);
    // 1 / (N * COLA gain) rides on the second-stage twiddles: every output passes through exactly one of them
#pragma unroll
    for (int i = 0; i < 16; ++i) tw.w[i] = make_float2(tw.w[i].x * scale, tw.w[i].y * scale);
    const int gitem = g.item0 + item;
    const int clip = gitem / g.seg_per_clip, sg = gitem - clip * g.seg_per_clip;
    float* __restrict__ o0 = out + g.first_offset + (long long)clip * g.clip_stride + (long long)sg * g.seg_stride;
    float* __restrict__ o1 = o0 + g.chan_stride;
    int p = 1;
    if (MASKED) p = period ? period[item] : pmax;  // no period array: one model row per frame (adaptive, sim)
    const bool t0 = t == 0;
    float carry_l[8], carry_r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) carry_l[i] = carry_r[i] = 0.f;
    __syncthreads();
    if (t == 0) {
#pragma unroll
        for (int d = 0; d < 2; ++d)
            if (exists(b0 + d))
                bulk_load(s_ring[d], Xitem + (size_t)row_of(b0 + d) * (NCH * XPITCH), ROW_BYTES, &s_full[d]);
    }
    // model rows (L2 resident) of frame jc, 8 bins per channel: issued one frame ahead, right after the previous
    // frame's masks have consumed these registers, so their latency hides behind that frame's transform
    float ml[2][4], mr[2][4];
    int q_cur = 0, q_next = 0;  // model row (phase) of the frame being processed / of the one prefetched
    auto load_model = [&](int jc) {
        if (!MASKED || !exists(jc)) return;
        const int q = row_of(jc) % p;
        q_next = q;
        const float* __restrict__ lrow = model + (((size_t)item * NCH + 0) * pmax + q) * PPITCH;
        const float* __restrict__ rrow = model + (((size_t)item * NCH + (NCH - 1)) * pmax + q) * PPITCH;
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int k3 = 0; k3 < 4; ++k3) {
                const int k = FF::out_column(t, h) + FF::CCOLS * k3;
                ml[h][k3] = __ldg(&lrow[k]);
                if (NCH == 2) mr[h][k3] = __ldg(&rrow[k]);
            }
    };
    load_model(b0);
    uint32_t phase = 0;  // bit s = parity of the next completion of slot s
    for (int jc = b0; jc <= b1; ++jc) {
        q_cur = q_next;
        const int j = row_of(jc);
        const int slot = (jc - b0) & 1;
        float2 r[16];
        if (!exists(jc)) {
            // a frame that does not exist (online: before the buffer is full): contributes zeros
#pragma unroll
            for (int i = 0; i < 16; ++i) r[i] = make_float2(0.f, 0.f);
            if (t == 0 && exists(jc + 2))
                bulk_load(s_ring[slot], Xitem + (size_t)row_of(jc + 2) * (NCH * XPITCH), ROW_BYTES, &s_full[slot]);
            load_model(jc + 1);
        } else {
        // the model rows of this frame were fetched while the previous frame was transformed (load_model)
        const float* __restrict__ ml_row = nullptr;
        const float* __restrict__ mr_row = nullptr;
        if (MASKED) {  // (only thread 0 dereferences these, for the Nyquist bin)
            ml_row = model + (((size_t)item * NCH + 0) * pmax + q_cur) * PPITCH;
            mr_row = model + (((size_t)item * NCH + (NCH - 1)) * pmax + q_cur) * PPITCH;
        }
        float2* __restrict__ ring = s_ring[slot];
        mbar_wait(&s_full[slot], (phase >> slot) & 1u);
        phase ^= 1u << slot;
        // The thread masks the 8 bins k < N/2 of its two columns (fft_core.cuh, transposed plan) and
        // forms Z[k] = YL + i YR and Z[N-k] = conj(YL) + i conj(YR) of the two packed channels, stored
        // re/im swapped (inverse transform by the forward stages); Z[N-k] lands in its other column.
        float2 zk[2][4], zm[2][4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int col = FF::out_column(t, h);
#pragma unroll
            for (int k3 = 0; k3 < 4; ++k3) {
                const int k = col + FF::CCOLS * k3;
                const float2 xl = ring[k];
                float2 xr = make_float2(0.f, 0.f);
                if (NCH == 2) xr = ring[XPITCH + k];
                if (h == 0 && k3 == 0 && t0) {
                    // bin 0 packs DC (mask kept, quirk Q11) and Nyquist, both purely real
                    float m_dc_l = 1.f, m_ny_l = 1.f, m_dc_r = 1.f, m_ny_r = 1.f;
                    if (MASKED) {
                        m_dc_l = soft_mask_keep_nan(ml[0][0], xl.x * xl.x);
                        m_ny_l = (XPITCH <= cutoff) ? 1.f : soft_mask(__ldg(&ml_row[XPITCH]), xl.y * xl.y);
                        if (NCH == 2) {
                            m_dc_r = soft_mask_keep_nan(mr[0][0], xr.x * xr.x);
                            m_ny_r = (XPITCH <= cutoff) ? 1.f : soft_mask(__ldg(&mr_row[XPITCH]), xr.y * xr.y);
                        }
                    }
                    zk[h][k3] = make_float2(m_dc_r * xr.x, m_dc_l * xl.x);  // Z[0]
                    zm[h][k3] = make_float2(m_ny_r * xr.y, m_ny_l * xl.y);  // Z[N/2]
                } else {
                    float m_l = 1.f, m_r = 1.f;
                    if (MASKED) {
                        if (k > cutoff) {
                            m_l = soft_mask(ml[h][k3], cmag2(xl));
                            if (NCH == 2) m_r = soft_mask(mr[h][k3], cmag2(xr));
                        }
                    }
                    const float2 yl = make_float2(m_l * xl.x, m_l * xl.y);
                    const float2 yr = make_float2(m_r * xr.x, m_r * xr.y);
                    zk[h][k3] = make_float2(yl.y + yr.x, yl.x - yr.y);
                    zm[h][k3] = make_float2(yr.x - yl.y, yl.x + yr.y);
                }
            }
        }
        // column t holds bins t + 2T k3, its mirrors sit in column 2T - t at 7 - k3; thread 0 owns the two
        // self-mirrored columns 0 (mirror 8 - k3, Nyquist at k3 = 4) and T (mirror 7 - k3)
#pragma unroll
        for (int k3 = 0; k3 < 4; ++k3) {
            r[k3] = zk[0][k3];
            r[8 + k3] = zk[1][k3];
        }
        r[4] = t0 ? zm[0][0] : zm[1][3];
        r[5] = t0 ? zm[0][3] : zm[1][2];
        r[6] = t0 ? zm[0][2] : zm[1][1];
        r[7] = t0 ? zm[0][1] : zm[1][0];
        r[12] = t0 ? zm[1][3] : zm[0][3];
        r[13] = t0 ? zm[1][2] : zm[0][2];
        r[14] = t0 ? zm[1][1] : zm[0][1];
        r[15] = t0 ? zm[1][0] : zm[0][0];
        load_model(jc + 1);
        __syncthreads();  // every thread has read its spectra: the slot becomes the y2 exchange buffer
        FF::tstage3(r, ring, s_tw2, t);
        __syncthreads();
        FF::tstage2(r, ring, s_y1, tw, t);
        __syncthreads();  // y2 drained: refill the slot with the frame two ahead
        if (t == 0 && exists(jc + 2))
            bulk_load(ring, Xitem + (size_t)row_of(jc + 2) * (NCH * XPITCH), ROW_BYTES, &s_full[slot]);
        FF::tstage1(r, s_y1, t);
        }
        // r[n1] = (yR, yL) / COLA gain at frame sample n = n1*T + t: n1 < 8 completes block jc - 1, the rest is carried
        if (jc > b0) {
            const long long blk = (long long)(jc - 1) * HOP;
#pragma unroll
            for (int n1 = 0; n1 < 8; ++n1) {
                const long long m = blk + n1 * FF::THREADS + t;
                if (m < g.S) {
                    o0[m] = carry_l[n1] + r[n1].y;
                    if (NCH == 2) o1[m] = carry_r[n1] + r[n1].x;
                }
            }
        }
#pragma unroll
        for (int n1 = 0; n1 < 8; ++n1) {
            carry_l[n1] = r[8 + n1].y;
            carry_r[n1] = r[8 + n1].x;
        }
    }
}

template <int NCH, bool MASKED, int MINB>
static void go_mask_istft(cudaStream_t st, dim3 grid, const float2* X, Geom g, const int* period, int pmax,
                          const float* model, int cutoff, float scale, FftTables tb, float* out, int blocks_per_cta) {
    static SmemOptIn opt_in;
    smem_opt_in(k_mask_istft<NCH, MASKED, MINB>, MASK_ISTFT_SMEM, opt_in);
    k_mask_istft<NCH, MASKED, MINB><<<grid, FF::THREADS, MASK_ISTFT_SMEM, st>>>(X, g, period, pmax, model, cutoff, scale,
                                                                                  tb, out, blocks_per_cta);
}

void launch_mask_istft(cudaStream_t st, const float2* X, Geom g, int nch, const int* period, int pmax,
                       const float* model, int cutoff, float scale, FftTables tb, float* out, int blocks_per_cta) {
    const int nblocks = g.T + 2 * g.frame_shift - 1;
    dim3 grid((nblocks + blocks_per_cta - 1) / blocks_per_cta, g.n_items);
#define REPET_GO(NCH, MINB) \
    go_mask_istft<NCH, true, MINB>(st, grid, X, g, period, pmax, model, cutoff, scale, tb, out, blocks_per_cta)
    if (nch == 2) {
        if (g_tuning.mask_minb >= 5) REPET_GO(2, 5);
        else if (g_tuning.mask_minb == 3) REPET_GO(2, 3);
        else REPET_GO(2, 4);
    } else {
        REPET_GO(1, 4);
    }
#undef REPET_GO
}
void launch_istft(cudaStream_t st, const float2* X, Geom g, int nch, float scale, FftTables tb, float* out,
                  int blocks_per_cta) {
    const int nblocks = g.T + 2 * g.frame_shift - 1;
    dim3 grid((nblocks + blocks_per_cta - 1) / blocks_per_cta, g.n_items);
    if (nch == 2) go_mask_istft<2, false, 4>(st, grid, X, g, nullptr, 0, nullptr, 0, scale, tb, out, blocks_per_cta);
    else go_mask_istft<1, false, 4>(st, grid, X, g, nullptr, 0, nullptr, 0, scale, tb, out, blocks_per_cta);
}

// ------------------------------------------------------------------------------------------
// k_mask_only  --  _mask as a helper: M[item][c][frame][bin]          repet.py:1441-1456
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_mask_only(const float2* __restrict__ X, int T, int nch, const int* __restrict__ period, int pmax,
            const float* __restrict__ model, float* __restrict__ mask_out) {
    const int item = blockIdx.z / nch, c = blockIdx.z - item * nch;
    const int j = blockIdx.x;  // frames on grid.x: there can be more than 65535 of them
    const int k = blockIdx.y * 128 + threadIdx.x;
    if (k > XPITCH) return;
    const int p = period ? period[item] : pmax;
    const float2* __restrict__ row = X + ((size_t)item * T + j) * (size_t)(nch * XPITCH) + (size_t)c * XPITCH;
    const float m = model[(((size_t)item * nch + c) * pmax + (j % p)) * PPITCH + k];
    mask_out[(((size_t)item * nch + c) * T + j) * PPITCH + k] = soft_mask_exact(m, row_mag2(row, k));
}

void launch_mask_only(cudaStream_t st, const float2* X, int n_items, int T, int nch, const int* period, int pmax,
                      const float* model, float* mask_out) {
    dim3 grid(T, (XPITCH + 128) / 128, n_items * nch);
    k_mask_only<<<grid, 128, 0, st>>>(X, T, nch, period, pmax, model, mask_out);
}

// ------------------------------------------------------------------------------------------
// k_expand_periods  --  per-frame periods of the adaptive REPET        repet.py:1194-1204, 1274-1289
// Segment i = 0, step, 2 step, ... of the beat spectrogram is replicated over columns
// i .. i+step-2; column i+step-1 stays all-zero in the reference, so its argmax is 0 and its
// period is lo + 1 (quirk Q3).
// ------------------------------------------------------------------------------------------
__global__ void k_expand_periods(const int* __restrict__ seg_period, int n_seg, int T, int step, int lag_lo,
                                 int* __restrict__ frame_period) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int item = blockIdx.y;
    if (j >= T) return;
    const int sI = j / step;
    const bool zero_column = step > 1 && (j - sI * step) == step - 1;
    frame_period[(size_t)item * T + j] = zero_column ? lag_lo + 1 : seg_period[(size_t)item * n_seg + sI];
}

void launch_expand_periods(cudaStream_t st, const int* seg_period, int n_items, int n_seg, int T, int step, int lag_lo,
                           int* frame_period) {
    dim3 grid((T + 255) / 256, n_items);
    k_expand_periods<<<grid, 256, 0, st>>>(seg_period, n_seg, T, step, lag_lo, frame_period);
}

// ------------------------------------------------------------------------------------------
// k_adaptive_model  --  the per-frame median of _adaptivemask            repet.py:1474-1498
// model[f, i] = median{ V[f, i + c p_i] : c in {1..order} - ceil(order/2), 0 <= i + c p_i < T }.
// The in-range offsets are contiguous in c, so every frame is a strided gather (start frame,
// stride p_i, count n) and reuses the pair-load median of k_model.  One model row per frame.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_adaptive_model(const float2* __restrict__ X, int T, int nch, const int* __restrict__ frame_period, int order,
                 float* __restrict__ model, int n_groups) {
    const int item = blockIdx.y / nch, c = blockIdx.y - item * nch;
    const int t = threadIdx.x;
    const int half = (order + 1) / 2;  // ceil(order / 2)
    const size_t row = (size_t)nch * XPITCH;
    const float2* __restrict__ chan = X + (size_t)item * T * row + (size_t)c * XPITCH;
    float* __restrict__ mrow = model + ((size_t)item * nch + c) * (size_t)T * PPITCH;
    const int* __restrict__ fp = frame_period + (size_t)item * T;
    const bool nyquist_cta = (int)blockIdx.x == n_groups;
    const int j_begin = nyquist_cta ? t : blockIdx.x * MODEL_QB;
    const int j_end = nyquist_cta ? T : min(T, j_begin + MODEL_QB);
    const int j_step = nyquist_cta ? 128 : 1;
    for (int j = j_begin; j < j_end; j += j_step) {
        const int p = fp[j];
        int c_lo = 1 - half, c_hi = order - half;
        if (p > 0) {
            c_lo = max(c_lo, -(j / p));
            c_hi = min(c_hi, (T - 1 - j) / p);
        } else {
            c_lo = c_hi = 0;
        }
        const int n = c_hi - c_lo + 1;
        const float2* __restrict__ base = chan + (size_t)(j + c_lo * p) * row;
        const size_t stride = (size_t)max(p, 0) * row;
        float* __restrict__ out = mrow + (size_t)j * PPITCH;
        if (nyquist_cta) {
            float med;
            switch (n) {
#define REPET_CASE(N) case N: med = strided_median<N>(base, stride, XPITCH); break;
                REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
                REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
                REPET_CASE(15) REPET_CASE(16)
#undef REPET_CASE
                default:
                    med = median_by_rank(n, [&](int s) { return row_mag2(base + (size_t)s * stride, XPITCH); });
            }
            out[XPITCH] = med;
            continue;
        }
        switch (n) {
#define REPET_CASE(N) case N: model_phase<N>(base, stride, out, t); break;
            REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
            REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
            REPET_CASE(15) REPET_CASE(16)
#undef REPET_CASE
            default:
                for (int k = t; k < XPITCH; k += 128)
                    out[k] = median_by_rank(n, [&](int s) { return row_mag2(base + (size_t)s * stride, k); });
        }
    }
}

// The same from the squared-magnitude plane Vsq [item][frame][channel][PPITCH] written by k_stft: a thread takes four
// adjacent bins (one 16-byte load per tap), so a tap costs 4 bytes per bin of L2 traffic instead of 8 -- the kernel
// runs at the L2 throughput cap (5 taps per frame: ~11 TB/s with the spectra as the source, profiles/r2a).
template <int N>
__device__ __forceinline__ void vsq_median_quad(const float* __restrict__ base, size_t stride, float* __restrict__ out) {
    float v0[N], v1[N], v2[N], v3[N];
#pragma unroll
    for (int s = 0; s < N; ++s) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(base + (size_t)s * stride));
        v0[s] = x.x;
        v1[s] = x.y;
        v2[s] = x.z;
        v3[s] = x.w;
    }
    median_select<N>(v0);
    median_select<N>(v1);
    median_select<N>(v2);
    median_select<N>(v3);
    float4 m;
    if (N & 1) {
        m = make_float4(fast_sqrt(v0[(N - 1) / 2]), fast_sqrt(v1[(N - 1) / 2]), fast_sqrt(v2[(N - 1) / 2]), fast_sqrt(v3[(N - 1) / 2]));
    } else {
        m = make_float4(0.5f * (fast_sqrt(v0[(N - 1) / 2]) + fast_sqrt(v0[N / 2])), 0.5f * (fast_sqrt(v1[(N - 1) / 2]) + fast_sqrt(v1[N / 2])),
                        0.5f * (fast_sqrt(v2[(N - 1) / 2]) + fast_sqrt(v2[N / 2])), 0.5f * (fast_sqrt(v3[(N - 1) / 2]) + fast_sqrt(v3[N / 2])));
    }
    *reinterpret_cast<float4*>(out) = m;
}
template <int N>
__device__ __forceinline__ float vsq_median_one(const float* __restrict__ base, size_t stride) {
    float v[N];
#pragma unroll
    for (int s = 0; s < N; ++s) v[s] = __ldg(base + (size_t)s * stride);
    median_select<N>(v);
    return (N & 1) ? fast_sqrt(v[(N - 1) / 2]) : 0.5f * (fast_sqrt(v[(N - 1) / 2]) + fast_sqrt(v[N / 2]));
}

constexpr int ADAPTIVE_V_MAX = 16;  // filter orders up to 16 take the Vsq kernel

__global__ void __launch_bounds__(128)
k_adaptive_model_v(const float* __restrict__ Vsq, int T, int nch, const int* __restrict__ frame_period, int order,
                   float* __restrict__ model) {
    const int item = blockIdx.y / nch, c = blockIdx.y - item * nch;
    const int t = threadIdx.x;
    const int half = (order + 1) / 2;  // ceil(order / 2)
    const size_t row = (size_t)nch * PPITCH;
    const float* __restrict__ chan = Vsq + (size_t)item * T * row + (size_t)c * PPITCH;
    float* __restrict__ mrow = model + ((size_t)item * nch + c) * (size_t)T * PPITCH;
    const int* __restrict__ fp = frame_period + (size_t)item * T;
    const int j_begin = blockIdx.x * MODEL_QB, j_end = min(T, j_begin + MODEL_QB);
    for (int j = j_begin; j < j_end; ++j) {
        const int p = fp[j];
        int c_lo = 1 - half, c_hi = order - half;
        if (p > 0) {
            c_lo = max(c_lo, -(j / p));
            c_hi = min(c_hi, (T - 1 - j) / p);
        } else {
            c_lo = c_hi = 0;
        }
        const int n = c_hi - c_lo + 1;
        const float* __restrict__ base = chan + (size_t)(j + c_lo * p) * row;
        const size_t stride = (size_t)max(p, 0) * row;
        float* __restrict__ out = mrow + (size_t)j * PPITCH;
        switch (n) {
#define REPET_CASE(N)                                                                           \
    case N:                                                                                     \
        for (int k = 4 * t; k < XPITCH; k += 512) vsq_median_quad<N>(base + k, stride, out + k); \
        if (t == 0) out[XPITCH] = vsq_median_one<N>(base + XPITCH, stride);                     \
        break;
            REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
            REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
            REPET_CASE(15) REPET_CASE(16)
#undef REPET_CASE
        }
    }
}

void launch_adaptive_model(cudaStream_t st, const float2* X, int n_items, int T, int nch, const int* frame_period,
                           int order, float* model, const float* Vsq) {
    const int n_groups = (T + MODEL_QB - 1) / MODEL_QB;
    if (Vsq && order <= ADAPTIVE_V_MAX) {
        dim3 grid(n_groups, n_items * nch);
        k_adaptive_model_v<<<grid, 128, 0, st>>>(Vsq, T, nch, frame_period, order, model);
        return;
    }
    dim3 grid(n_groups + 1, n_items * nch);
    k_adaptive_model<<<grid, 128, 0, st>>>(X, T, nch, frame_period, order, model, n_groups);
}

// ------------------------------------------------------------------------------------------
// k_xfade  --  the segment cross-fade of REPET extended                       repet.py:388-414
// Per output sample, the covering segments are visited in order exactly as the reference's
// in-place loop does: the first contributes as is; a later one scales what is already there by
// the falling half of triang(2*overlap) and adds itself scaled by the rising half over its
// first `overlap` samples, and simply adds beyond.
// ------------------------------------------------------------------------------------------
template <bool VEC4>
__global__ void k_xfade(const float* __restrict__ seg_main, const float* __restrict__ seg_last, int n_seg, int seg_len,
                        int last_len, int step, int nch, int S, float* __restrict__ out) {
    // 32-bit index arithmetic (a clip has fewer than 2^31 samples); 4 consecutive samples per thread
    const int u0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (u0 >= S) return;
    const int clip = blockIdx.y / nch, c = blockIdx.y - clip * nch;
    const int ov = seg_len - step;
    const float inv = 1.0f / (float)(2 * ov);
    const float* __restrict__ main_base = seg_main + ((size_t)clip * (n_seg - 1) * nch + c) * (size_t)seg_len;
    const float* __restrict__ last_base = seg_last + ((size_t)clip * nch + c) * (size_t)last_len;
    float* __restrict__ dst = out + ((size_t)clip * nch + c) * (size_t)S;
    const int q_hi = u0 / step;
    const int q_lo = u0 < seg_len ? -1 : (u0 - seg_len) / step;
    if (VEC4 && u0 + 3 < S) {
        // step, segment length and every buffer length are multiples of 4 samples: the 4 samples of the thread sit
        // in the same segments, on the same side of every overlap boundary, and every access is a 16-byte one
        const int sg_hi = min(q_hi, n_seg - 1);
        const int sg_lo = min(u0 < seg_len ? 0 : q_lo + 1, n_seg - 1);
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int sg = sg_lo; sg <= sg_hi; ++sg) {
            const int i = u0 - sg * step;
            const float4 x = __ldg(reinterpret_cast<const float4*>(
                sg < n_seg - 1 ? main_base + (size_t)sg * nch * seg_len + i : last_base + i));
            if (sg > 0 && i < ov) {
                const float xs[4] = {x.x, x.y, x.z, x.w};
                float v[4] = {val.x, val.y, val.z, val.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float up = (float)(2 * (i + e) + 1) * inv;               // triang(2 ov)[i]
                    const float down = (float)(2 * (ov - 1 - (i + e)) + 1) * inv;  // triang(2 ov)[ov + i]
                    v[e] = v[e] * down + xs[e] * up;
                }
                val = make_float4(v[0], v[1], v[2], v[3]);
            } else {
                val = make_float4(val.x + x.x, val.y + x.y, val.z + x.z, val.w + x.w);
            }
        }
        *reinterpret_cast<float4*>(dst + u0) = val;
        return;
    }
    // the covering segments of the 4 samples differ at most at segment boundaries: compute per sample,
    // but share the divisions
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int u = u0 + e;
        if (u >= S) break;
        int sg_hi = q_hi + ((u - q_hi * step) >= step ? 1 : 0);
        int sg_lo = u < seg_len ? 0 : q_lo + 1 + ((u - seg_len - q_lo * step) >= step ? 1 : 0);
        sg_hi = min(sg_hi, n_seg - 1);
        sg_lo = min(sg_lo, n_seg - 1);
        float val = 0.f;
        for (int sg = sg_lo; sg <= sg_hi; ++sg) {
            const int i = u - sg * step;
            const float x = sg < n_seg - 1 ? main_base[(size_t)sg * nch * seg_len + i] : last_base[i];
            if (sg > 0 && i < ov) {
                const float up = (float)(2 * i + 1) * inv;               // triang(2 ov)[i]
                const float down = (float)(2 * (ov - 1 - i) + 1) * inv;  // triang(2 ov)[ov + i]
                val = val * down + x * up;
            } else {
                val += x;
            }
        }
        dst[u] = val;
    }
}

void launch_xfade(cudaStream_t st, const float* seg_main, const float* seg_last, int n_clips, int n_seg, int seg_len,
                  int last_len, int step, int nch, long long S, float* out) {
    dim3 grid((unsigned)((S + 1023) / 1024), n_clips * nch);
    // 16-byte path: every offset a thread forms is a multiple of 4 samples (the workspace slices are 256-byte aligned)
    const bool vec4 = step % 4 == 0 && seg_len % 4 == 0 && last_len % 4 == 0 && S % 4 == 0 &&
                      (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(seg_main) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(seg_last) & 15) == 0;
    if (vec4) k_xfade<true><<<grid, 256, 0, st>>>(seg_main, seg_last, n_seg, seg_len, last_len, step, nch, (int)S, out);
    else k_xfade<false><<<grid, 256, 0, st>>>(seg_main, seg_last, n_seg, seg_len, last_len, step, nch, (int)S, out);
}

// ------------------------------------------------------------------------------------------
// k_argmax_columns  --  _periods on a caller-provided beat spectrum / spectrogram
//                                                                        repet.py:1249-1291
// beat[n_lags][n_columns] row-major float64; first maximum over lags [lo, hi) + 1 per column.
// ------------------------------------------------------------------------------------------
__global__ void k_argmax_columns(const double* __restrict__ beat, int n_columns, int lag_lo, int lag_hi,
                                 int* __restrict__ period) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= n_columns) return;
    double best = beat[(size_t)lag_lo * n_columns + col];
    int arg = lag_lo;
    for (int l = lag_lo + 1; l < lag_hi; ++l) {
        const double v = beat[(size_t)l * n_columns + col];
        if (v > best) {
            best = v;
            arg = l;
        }
    }
    period[col] = arg + 1;
}

void launch_argmax_columns(cudaStream_t st, const double* beat, int n_lags, int n_columns, int lag_lo, int lag_hi,
                           int* period) {
    (void)n_lags;
    k_argmax_columns<<<(n_columns + 127) / 128, 128, 0, st>>>(beat, n_columns, lag_lo, lag_hi, period);
}

// ------------------------------------------------------------------------------------------
// float64 (S, C) interleaved  <->  fp32 planar [C][S]: the reference API's NumPy convention
// (repet.py:73-77) converted on the device, so the host never touches the samples.
// ------------------------------------------------------------------------------------------
__global__ void k_f64_to_planar(const double* __restrict__ in, long long S, int C, float* __restrict__ out) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= S * C) return;
    const long long s = n / C;
    const int c = (int)(n - s * C);
    out[(long long)c * S + s] = (float)in[n];
}
__global__ void k_planar_to_f64(const float* __restrict__ in, long long S, int C, double* __restrict__ out) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= S * C) return;
    const long long s = n / C;
    const int c = (int)(n - s * C);
    out[n] = (double)in[(long long)c * S + s];
}
// int16 PCM in WAV order [clip][sample][channel] -> fp32 planar [clip][channel][sample] / 2^15 (repet.py:929)
__global__ void k_pcm16_to_planar(const int16_t* __restrict__ in, long long S, int C, float* __restrict__ out) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const long long clip = blockIdx.y;
    const int16_t* __restrict__ src = in + (clip * S + s) * C;
    for (int c = 0; c < C; ++c) out[(clip * C + c) * S + s] = (float)src[c] * (1.0f / 32768.0f);
}
void launch_pcm16_to_planar(cudaStream_t st, const int16_t* in, int n_clips, long long S, int C, float* out) {
    dim3 grid((unsigned)((S + 255) / 256), n_clips);
    k_pcm16_to_planar<<<grid, 256, 0, st>>>(in, S, C, out);
}

// fp32 planar [clip][channel][sample] -> int16 PCM in WAV order [clip][sample][channel]: round(y * 2^15) to nearest
// (ties to even), saturated -- the inverse of the normalisation above, what an int16 WAVE writer stores
__global__ void k_planar_to_pcm16(const float* __restrict__ in, long long S, int C, int16_t* __restrict__ out) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const long long clip = blockIdx.y;
    int16_t* __restrict__ dst = out + (clip * S + s) * C;
    for (int c = 0; c < C; ++c) {
        const int q = __float2int_rn(in[(clip * C + c) * S + s] * 32768.0f);
        dst[c] = (int16_t)max(-32768, min(32767, q));
    }
}
void launch_planar_to_pcm16(cudaStream_t st, const float* in, int n_clips, long long S, int C, int16_t* out) {
    dim3 grid((unsigned)((S + 255) / 256), n_clips);
    k_planar_to_pcm16<<<grid, 256, 0, st>>>(in, S, C, out);
}

// foreground = audio - background (README.md:68), 16 bytes per thread, tail by the last threads
__global__ void k_foreground(const float* __restrict__ audio, const float* __restrict__ background, long long n,
                             float* __restrict__ foreground) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n) {
        const float4 a = *reinterpret_cast<const float4*>(audio + i);
        const float4 b = *reinterpret_cast<const float4*>(background + i);
        *reinterpret_cast<float4*>(foreground + i) = make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
    } else {
        for (long long k = i; k < n; ++k) foreground[k] = audio[k] - background[k];
    }
}
void launch_foreground(cudaStream_t st, const float* audio, const float* background, long long n, float* foreground) {
    const long long threads = (n + 3) / 4;
    if (threads > 0) k_foreground<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(audio, background, n, foreground);
}

void launch_f64_interleaved_to_planar(cudaStream_t st, const double* in, long long S, int C, float* out) {
    const long long n = S * C;
    k_f64_to_planar<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, S, C, out);
}
void launch_planar_to_f64_interleaved(cudaStream_t st, const float* in, long long S, int C, double* out) {
    const long long n = S * C;
    k_planar_to_f64<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, S, C, out);
}

}  // namespace repet
