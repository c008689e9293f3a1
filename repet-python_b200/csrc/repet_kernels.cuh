// Launch-side declarations shared by repet_kernels.cu (device code) and repet_abi.cu (C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// Every kernel source is compiled once per supported window length (REPET_WIN_N = 512, 1024, 2048:
// sampling rates up to 12.8 / 25.6 / 51.2 kHz, repet.py:130) into its own namespace; repet_abi.cu
// dispatches on repet_params.window_length.  All sizes below are compile-time constants.
#ifndef REPET_WIN_N
#define REPET_WIN_N 2048
#endif
#define REPET_CAT2(a, b) a##b
#define REPET_CAT(a, b) REPET_CAT2(a, b)
#define repet REPET_CAT(repet_w, REPET_WIN_N)

// Launch-shape knobs (repet_set_tuning); defaults are the measured best on B200.  One object for
// every window-length instantiation (defined in repet_abi.cu).
struct repet_tuning {
    int stft_minb = 4;       // resident CTAs per SM the STFT kernel is compiled for (4, 5, 6)
    int mask_minb = 4;       // same for the mask+ISTFT kernel (3, 4, 5; shared memory allows 4)
    int frames_per_cta = 0;  // 0 = pick from the batch size
    int beat_parts = 0;      // 0 = pick from the batch size
    int cert_rel_ppm = 0;    // period certification window in ppm of the best value (0 = CERT_REL = 100 ppm)
    int simgemm_tc = 2;      // similarity fast pass: 2 = tcgen05 3xTF32 split, 1 = tcgen05 single TF32, 0 = fp32 CUDA cores
    int copy_chunk_mb = 128; // host-buffer entry points: megabytes per copy slot (pipeline granularity)
    int sim_frames64 = 1;    // similarity operand from the float64 front end (k_frames64); 0 = from k_stft's fp32 magnitudes
    int adaptive_vsq = 1;    // adaptive: k_stft also writes |X|^2 planes and the per-frame median gathers those
    int simgemm_bn = 256;    // tile width of the split similarity GEMM: 256 (128 x 256 tiles) or 128 (square tiles)
    int topk_force_exact = 0;  // test knob: every column of REPET-SIM goes through the exact float64 fallback
};
extern repet_tuning g_repet_tuning;

namespace repet {

constexpr int WIN_N = REPET_WIN_N;   // STFT window length of this compilation
constexpr int HOP = WIN_N / 2;       // step length H
constexpr int NBIN = WIN_N / 2 + 1;  // F magnitude bins (1025 at 44.1 kHz)
constexpr int XPITCH = WIN_N / 2;    // float2 per (frame, channel): bin 0 holds (DC.re, Nyquist.re)
constexpr int PPITCH = (NBIN + 7) / 8 * 8;  // floats per frame row of P / model (F rounded up to 32 B)
constexpr int BEAT_L = 2048;         // FFT length of the beat-spectrum transforms (time axis: any window)
constexpr int MAX_MEDIAN_REGS = 32;  // sorting-network path handles up to 32 gathered values
constexpr int KPAD = (NBIN + 31) / 32 * 32;  // K of the similarity GEMM operand: F zero-padded to 32 floats
constexpr int APITCH64 = PPITCH;     // doubles per row of the float64-normalised frames
constexpr int FRAME_THREADS = WIN_N / 16;  // threads of one frame transform

// A batch of equally long items cut out of planar audio [clip][channel][sample]:
// item = clip * seg_per_clip + seg starts at clip*clip_stride + seg*seg_stride (+ c*chan_stride).
// `original` uses seg_per_clip = 1; `extended` lays its 10 s segments out this way.
struct Geom {
    int n_items;
    int seg_per_clip;
    long long clip_stride;
    long long seg_stride;
    long long chan_stride;
    long long first_offset;  // added to every item start
    int S;                   // samples per item
    int T;                   // STFT frames per item
    int item0;               // global index of this launch's first item (workspace indices are local)
    // Online REPET-SIM frames are not centred (repet.py:781, 834-901): frame j covers samples
    // [j*H, j*H + N).  frame_shift = 1 maps the kernels' centred frame index jc to row jc - 1, and
    // rows below first_frame are never synthesised (quirk Q5).  Centred drivers use 0, 0.
    int frame_shift;
    int first_frame;
};

struct FftTables {
    const float2* tw1;    // frame transform: [15][N/16]   W_N^(m*k1)
    const float2* tw2;    //                  [R2][8]      W_(N/16)^(m2*k2)
    const float2* tw1_t;  // time-axis transform (2048): [15][128]
    const float2* tw2_t;  //                              [16][8]
    const float2* tw1_t1k;  // time-axis transform of short segments (1024): [15][64]
    const float2* tw2_t1k;  //                                               [8][8]
};

enum PMode { P_NONE = 0, P_POWER = 1, P_MAGNITUDE = 2, P_MIXDOWN = 3 };  // MIXDOWN: |STFT(mean_c x)| only, no X

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: remember what each device has been
// given (one handle per GPU in one process, INTEGRATION.md).  Returns false when the device refuses the size.
struct SmemOptIn {
    size_t bytes[64] = {0};
};
template <typename F>
inline bool smem_opt_in(F func, size_t smem, SmemOptIn& state) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if (smem <= state.bytes[dev]) return true;
    if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    state.bytes[dev] = smem;
    return true;
}

using Tuning = ::repet_tuning;
static Tuning& g_tuning = ::g_repet_tuning;

// k_stft: audio -> X (half spectra, both channels) [+ P = (mean_c |X|)^2 or mean_c |X|]
// Vsq (optional): also |X_c|^2 of every channel, [item][frame][channel][PPITCH]
void launch_stft(cudaStream_t st, const float* audio, Geom g, int nch, const float* window, FftTables tb, float2* X,
                 float* P, int pmode, int frames_per_cta, float* Vsq = nullptr);

// k_beat: P rows [t_first, t_first + t_len) of every item (zero outside [0, T)) -> partial PSD sums
// psd_part[item][part][2048]
void launch_beat(cudaStream_t st, const float* P, int n_items, int T, int t_first, int t_len, int seg_step, int n_seg,
                 FftTables tb, float* psd_part, int n_parts, int f_per_part, int L = BEAT_L);
// transform length for a beat item of `rows` frames and lags below `max_lag`: 1024 when it fits, else BEAT_L
inline int beat_transform_length(int rows, int max_lag) { return rows + max_lag - 1 <= 1024 ? 1024 : BEAT_L; }

// k_periods: partial PSDs -> beat spectrum b[l] (optional) and argmax period per beat item (fp64)
void launch_periods(cudaStream_t st, const float* psd_part, const float* psd_part_im, int n_beat_items, int n_parts,
                    int t_len, double norm_rows, int lag_lo, int lag_hi, int out_lo, int out_hi, double* beat_out,
                    int beat_pitch, int* period, double* stats, int* cert, int L = BEAT_L);
// near-tied period candidates re-decided in float64 (cert: [item][1 + CERT_MAX] ints written by k_periods)
constexpr int CERT_MAX = 8;
// k_period_certify splits each candidate's sum into CERT_TSPLIT time chunks (partial sums added in a fixed order):
// cert_val is [item][CERT_MAX][CERT_TSPLIT] doubles
constexpr int CERT_TSPLIT = 16;
constexpr double CERT_REL = 1e-4;
// n_items beat items = clips x n_seg segments of rows [t_first + seg*seg_step, ... + t_len) (original: 0, T, 0, 1)
void launch_period_certify(cudaStream_t st, const float* P, int n_items, int T, int t_first, int t_len, int seg_step,
                           int n_seg, const int* cert, double* cert_val, int* period);
// k_beat_blocked: clips longer than one transform, complex cross-spectrum partials
// g_re / g_im [item][block][fpart][2048]
void launch_beat_blocked(cudaStream_t st, const float* P, int n_items, int T, int Bk, int max_lag, FftTables tb,
                         float* g_re, float* g_im, int n_blocks, int n_fparts, int f_per_part);

// k_model: median over the period-strided frames of every phase -> model[item][c][q][PPITCH]
void launch_model(cudaStream_t st, const float2* X, int n_items, int T, int nch, const int* period, int pmax,
                  float* model);

// k_mask_istft: soft mask from the periodic model, high-pass, Hermitian pack, inverse FFT, overlap-add
void launch_mask_istft(cudaStream_t st, const float2* X, Geom g_out, int nch, const int* period, int pmax,
                       const float* model, int cutoff, float scale, FftTables tb, float* out, int blocks_per_cta);

// plain ISTFT of caller-provided half spectra (helper-level entry point)
void launch_istft(cudaStream_t st, const float2* X, Geom g_out, int nch, float scale, FftTables tb, float* out,
                  int blocks_per_cta);

// mask only (helper-level): writes M[item][c][T][PPITCH]
void launch_mask_only(cudaStream_t st, const float2* X, int n_items, int T, int nch, const int* period, int pmax,
                      const float* model, float* mask_out);

// adaptive: per-frame periods from per-segment periods (quirk Q3), per-frame median model
void launch_expand_periods(cudaStream_t st, const int* seg_period, int n_items, int n_seg, int T, int step, int lag_lo,
                           int* frame_period);
// Vsq (optional, from launch_stft): the taps are gathered from the 4-byte squared magnitudes instead of the spectra
void launch_adaptive_model(cudaStream_t st, const float2* X, int n_items, int T, int nch, const int* frame_period,
                           int order, float* model, const float* Vsq = nullptr);
// extended: triangular cross-fade of the separated segments
void launch_xfade(cudaStream_t st, const float* seg_main, const float* seg_last, int n_clips, int n_seg, int seg_len,
                  int last_len, int step, int nch, long long S, float* out);

// _periods on caller-provided float64 beat spectra
void launch_argmax_columns(cudaStream_t st, const double* beat, int n_lags, int n_columns, int lag_lo, int lag_hi,
                           int* period);

// REPET-SIM (repet_sim.cu)
void launch_normalize(cudaStream_t st, const float* V, int n_rows, double* An64, float* An32, float* An32lo,
                      int round_tf32);
// float64 analysis front end of REPET-SIM: audio (fp32 planar, or float64 interleaved of one clip) -> normalised
// frames An64 and the fast operands rounded from them
void launch_frames64(cudaStream_t st, const float* audio, const double* audio64, Geom g, int nch,
                     const double* window64, const double2* tw64, double* An64, float* An32, float* An32lo,
                     int round_tf32);
// tcgen05 / TMEM / TMA self-similarity GEMM (repet_simgemm.cu); returns 0 on success
int launch_selfsim_tc(cudaStream_t st, const float* hi, const float* lo, int n_items, int T, float* S, int sm_count);
void launch_selfsim_simt(cudaStream_t st, const float* An32, int n_items, int T, float* S);
// rows [r0, r0 + rows) of one item's S, row-major with pitch T (S_panel[r - r0][c])
int launch_selfsim_tc_panel(cudaStream_t st, const float* hi, const float* lo, int T, int r0, int rows, float* S_panel,
                            int sm_count);
void launch_selfsim_simt_panel(cudaStream_t st, const float* An32, int T, int r0, int rows, float* S_panel);
// The similar-frame selection in two launches.  k_topk settles columns [c0, c0 + n_cols) of every item from the rows
// S[(item * n_cols + c - c0) * T ...] (the whole matrix: c0 = 0, n_cols = T; a row panel of one item: its first row
// and height) and queues the columns it cannot settle; k_topk_exact then settles every queued column, once after the
// last panel.  overflow: [4] ints zeroed by the caller ([0] = columns queued for the exact fallback, [1..3]
// statistics); ovf_cols: [n_items * T] ints; scratch: topk_exact_scratch_bytes(T, sm_count) bytes.
int launch_topk_propose(cudaStream_t st, const float* S, int c0, int n_cols, const double* An64, int n_items, int T,
                        float tau, double thr, int d, int number, int* idx_out, int* cnt_out, int* overflow,
                        int* ovf_cols);
void launch_topk_exact(cudaStream_t st, const double* An64, int T, double thr, int d, int number, const int* overflow,
                       const int* ovf_cols, unsigned char* scratch, int* idx_out, int* cnt_out, int sm_count);
size_t topk_exact_scratch_bytes(int T, int sm_count);
// returns 0, or nonzero when the device refuses the shared memory / scratch the ring needs
int launch_online_select(cudaStream_t st, const double* An64, int n_items, int T, int B, int frame_base, double thr,
                         int d, int number, int* idx_out, int* cnt_out);
void launch_sqmag(cudaStream_t st, const float2* X, long long n_rows, float* Vsq);
// Vsq (squared magnitudes [item][T][nch][PPITCH]) is required when number > 32
int launch_simmodel(cudaStream_t st, const float2* X, const float* Vsq, int n_items, int T, int nch, const int* idx,
                    const int* cnt, int number, int first_frame, float* model);

// helper-level similarity kernels (exact float64)
void launch_cosine64(cudaStream_t st, const double* A1, int n1, const double* A2, int n2, double* out);
int launch_localmaxima64(cudaStream_t st, const double* data, int n, int n_columns, double thr, int d, int number,
                         int* idx_out, int* cnt_out, double* val_out);

// foreground = audio - background, any layout (n fp32 elements; 16-byte aligned pointers)
void launch_foreground(cudaStream_t st, const float* audio, const float* background, long long n, float* foreground);

// layout converters for the float64 (S, C) NumPy convention of the reference API
void launch_pcm16_to_planar(cudaStream_t st, const int16_t* in, int n_clips, long long S, int C, float* out);
void launch_planar_to_pcm16(cudaStream_t st, const float* in, int n_clips, long long S, int C, int16_t* out);
void launch_f64_interleaved_to_planar(cudaStream_t st, const double* in, long long S, int C, float* out);
void launch_planar_to_f64_interleaved(cudaStream_t st, const float* in, long long S, int C, double* out);

}  // namespace repet
