// REPET-SIM kernels: column normalisation, self-similarity, similar-frame selection with exact
// float64 certification, and the similar-frame median model.   Reference: repet.py:1209-1246
// (_selfsimilaritymatrix / _similaritymatrix), 1294-1383 (_localmaxima / _indices), 1511-1545
// (_simmask), 834-901 (the online loop).
#include "repet_kernels.cuh"
#include "fft_core.cuh"
#include "median_networks.cuh"
#include "median_networks_large.cuh"

#include <algorithm>

namespace repet {

// ------------------------------------------------------------------------------------------
// k_normalize  --  A[:, t] = V[:, t] / ||V[:, t]||_2                       repet.py:1220, 1240
// V = mean_c |X| comes from k_stft in fp32; the norm and the quotient are taken in float64.
// Outputs: An64[row][APITCH64] (exact dot products) and An32[row][KPAD] (fast GEMM operand,
// zero padded to a multiple of 32 floats = one 128-byte swizzle atom per K block).
// An all-zero frame gives 0/0 = NaN as in the reference (quirk Q18).   One warp per frame.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_normalize(const float* __restrict__ V, int n_rows, double* __restrict__ An64, float* __restrict__ An32,
            float* __restrict__ An32lo, int round_tf32) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_rows) return;
    const float* __restrict__ v = V + (size_t)warp * PPITCH;
    double sum = 0.0;
    for (int k = lane; k < NBIN; k += 32) {
        const double x = (double)v[k];
        sum = fma(x, x, sum);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const double norm = sqrt(sum);
    for (int k = lane; k < KPAD; k += 32) {
        const double a = k < NBIN ? (double)v[k] / norm : 0.0;
        if (An64 && k < APITCH64) An64[(size_t)warp * APITCH64 + k] = a;
        if (An32) {
            float f = (float)a;
            if (round_tf32) {  // round-to-nearest TF32 here, so the tensor core's operand truncation is exact
                uint32_t bits;
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(bits) : "f"(f));
                const float hi = __uint_as_float(bits);
                if (An32lo) {  // 3xTF32: the residual, itself rounded to TF32 (a ~ hi + lo to 2^-22)
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(bits) : "f"((float)(a - (double)hi)));
                    An32lo[(size_t)warp * KPAD + k] = __uint_as_float(bits);
                }
                f = hi;
            }
            An32[(size_t)warp * KPAD + k] = f;
        }
    }
}

void launch_normalize(cudaStream_t st, const float* V, int n_rows, double* An64, float* An32, float* An32lo,
                      int round_tf32) {
    k_normalize<<<(n_rows * 32 + 255) / 256, 256, 0, st>>>(V, n_rows, An64, An32, An32lo, round_tf32);
}

// ------------------------------------------------------------------------------------------
// k_frames64  --  float64 analysis front end of REPET-SIM       repet.py:633-667, 1001-1060, 1220
// A[:, t] = V[:, t] / ||V[:, t]||,  V = mean_c |STFT_c|, computed in float64 from the samples.
// The similar-frame lists are integers: every decision between two similarities (local-maximum
// test, threshold, rank) must come out as it does in the reference, which works in float64
// throughout.  The fp32 transforms of k_stft carry ~1e-7 of relative error into a similarity
// value -- enough to flip near-tied candidates on a long track -- so the operand of the similarity
// (An64, and the TF32 operands rounded from it) is rebuilt here with a float64 transform; the fp32
// spectra of k_stft are only used for the mask and the resynthesis (tolerance 1e-4).
// A CTA of N/16 threads walks 8 consecutive frames: both channels packed into one complex transform
// (z = w (xL + i xR)) run through the register-blocked 16 x R2 x 8 plan of fft_core.cuh instantiated for
// double2 (a thread ends up holding Z[k] and Z[N-k]: the Hermitian split needs no exchange), magnitudes,
// channel mean, float64 norm, and the three operand formats written from registers.
// An all-zero frame gives 0/0 = NaN as in the reference (quirk Q18).
// ------------------------------------------------------------------------------------------
using F64 = Fft<WIN_N, double2>;  // the frame transform of fft_core.cuh in float64: same plan, same ownership
constexpr int F64_FRAMES = 8;     // consecutive frames per CTA (twiddles stay in registers)

// one bin of the channel-mean magnitude from Z[k] and Z[N-k] of the packed transform (equal for k = 0, N/2)
template <int NCH>
__device__ __forceinline__ double mean_magnitude64(double2 zk, double2 zm) {
    // sqrt(re^2 + im^2): within 1.5 ulp of np.abs's hypot, no risk of overflow for audio-scale spectra
    if (NCH == 1) return sqrt(fma(zk.x, zk.x, zk.y * zk.y));
    const double lr = 0.5 * (zk.x + zm.x), li = 0.5 * (zk.y - zm.y), rr = 0.5 * (zk.x - zm.x), ri = 0.5 * (zk.y + zm.y);
    return 0.5 * (sqrt(fma(lr, lr, li * li)) + sqrt(fma(rr, rr, ri * ri)));
}

__device__ __forceinline__ void write_operands(size_t row, int k, double a, double* __restrict__ An64,
                                               float* __restrict__ An32, float* __restrict__ An32lo, int round_tf32) {
    An64[row * APITCH64 + k] = a;
    if (!An32) return;
    float f = (float)a;
    if (round_tf32) {  // round-to-nearest TF32 here, so the tensor core's operand truncation is exact
        uint32_t bits;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(bits) : "f"(f));
        const float hi = __uint_as_float(bits);
        if (An32lo) {  // 3xTF32: the residual, itself rounded to TF32 (a ~ hi + lo to 2^-22)
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(bits) : "f"((float)(a - (double)hi)));
            An32lo[row * KPAD + k] = __uint_as_float(bits);
        }
        f = hi;
    }
    An32[row * KPAD + k] = f;
}

template <int NCH>
__global__ void __launch_bounds__(F64::THREADS)
k_frames64(const float* __restrict__ audio, const double* __restrict__ audio64, Geom g,
           const double* __restrict__ window64, const double2* __restrict__ tw64, double* __restrict__ An64,
           float* __restrict__ An32, float* __restrict__ An32lo, int round_tf32) {
    extern __shared__ __align__(16) unsigned char s_raw64[];
    double2* bufA = reinterpret_cast<double2*>(s_raw64);
    double2* bufB = bufA + F64::BUF;
    double2* s_tw2 = bufB + F64::BUF;
    __shared__ double s_red[F64::THREADS / 32];
    const int t = threadIdx.x;
    const int item = blockIdx.y;
    const int j0 = blockIdx.x * F64_FRAMES, j1 = min(j0 + F64_FRAMES, g.T);
    // W_N^i for any i < N from the half table: W_N^(i + N/2) = -W_N^i
    auto twiddle = [&](int i) {
        const double2 w = tw64[i & (WIN_N / 2 - 1)];
        return (i & (WIN_N / 2)) ? make_double2(-w.x, -w.y) : w;
    };
    F64::Twiddle1 tw;  // W_N^(t k1), k1 = 1..15
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) tw.w[k1 - 1] = twiddle((t * k1) & (WIN_N - 1));
    if (t < F64::TW2) s_tw2[t] = twiddle((16 * (t >> 3) * (t & 7)) & (WIN_N - 1));  // W_T^(m2 k2) at [k2*8 + m2]
    const int gitem = g.item0 + item;
    const int clip = gitem / g.seg_per_clip, sg = gitem - clip * g.seg_per_clip;
    const long long start = g.first_offset + (long long)clip * g.clip_stride + (long long)sg * g.seg_stride;
    __syncthreads();
    for (int j = j0; j < j1; ++j) {
        double2 r[16];
        const long long base = (long long)(j - 1 + g.frame_shift) * HOP + t;
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const long long idx = base + n1 * F64::THREADS;
            double xl = 0.0, xr = 0.0;
            if (idx >= 0 && idx < g.S) {
                if (audio64) {  // float64 (samples, channels) of one clip: the reference's own input
                    xl = audio64[(start + idx) * NCH];
                    if (NCH == 2) xr = audio64[(start + idx) * NCH + 1];
                } else {
                    xl = (double)__ldg(audio + start + idx);
                    if (NCH == 2) xr = (double)__ldg(audio + start + g.chan_stride + idx);
                }
            }
            const double w = __ldg(window64 + n1 * F64::THREADS + t);
            r[n1] = make_double2(xl * w, xr * w);
        }
        F64::stage1(r, tw, bufA, t);
        __syncthreads();
        F64::stage2(r, bufA, bufB, s_tw2, t);
        __syncthreads();
        F64::stage3(r, bufB, t);
        // r[h*8 + k3] = Z[out_column(t, h) + 2T k3]; the mirror bin N - k sits in the other column at 7 - k3
        // (thread 0 owns the self-mirrored columns 0 and T).  Bins 0 .. N/2 of the thread:
        double mag[9];
        int bin[9];
        int nb = 8;
        if (t != 0) {
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
                for (int k3 = 0; k3 < 4; ++k3) {
                    bin[h * 4 + k3] = (h == 0 ? t : F64::CCOLS - t) + F64::CCOLS * k3;
                    mag[h * 4 + k3] = mean_magnitude64<NCH>(r[h * 8 + k3], r[(1 - h) * 8 + 7 - k3]);
                }
            bin[8] = 0;
            mag[8] = 0.0;
        } else {
            bin[0] = 0;
            mag[0] = mean_magnitude64<NCH>(r[0], r[0]);
#pragma unroll
            for (int k3 = 1; k3 < 4; ++k3) {
                bin[k3] = F64::CCOLS * k3;
                mag[k3] = mean_magnitude64<NCH>(r[k3], r[8 - k3]);
            }
#pragma unroll
            for (int k3 = 0; k3 < 4; ++k3) {
                bin[4 + k3] = F64::THREADS + F64::CCOLS * k3;
                mag[4 + k3] = mean_magnitude64<NCH>(r[8 + k3], r[8 + 7 - k3]);
            }
            bin[8] = WIN_N / 2;
            mag[8] = mean_magnitude64<NCH>(r[4], r[4]);
            nb = 9;
        }
        double sum = 0.0;
#pragma unroll
        for (int i = 0; i < 9; ++i) sum = fma(mag[i], mag[i], sum);  // mag[8] = 0 where unused
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if ((t & 31) == 0) s_red[t >> 5] = sum;
        __syncthreads();
        double total = 0.0;
#pragma unroll
        for (int i = 0; i < F64::THREADS / 32; ++i) total += s_red[i];
        const double inv_norm = 1.0 / sqrt(total);  // all-zero frame: 0 * inf = NaN, the reference's 0/0 (quirk Q18)
        const size_t row = (size_t)item * g.T + j;
#pragma unroll
        for (int i = 0; i < 9; ++i)
            if (i < nb) write_operands(row, bin[i], mag[i] * inv_norm, An64, An32, An32lo, round_tf32);
        // zero padding of the rows: bins NBIN .. APITCH64-1 (float64) and NBIN .. KPAD-1 (fp32 operands)
        if (NBIN + t < APITCH64) An64[row * APITCH64 + NBIN + t] = 0.0;
        if (An32 && NBIN + t < KPAD) {
            An32[row * KPAD + NBIN + t] = 0.f;
            if (round_tf32 && An32lo) An32lo[row * KPAD + NBIN + t] = 0.f;
        }
    }
}

void launch_frames64(cudaStream_t st, const float* audio, const double* audio64, Geom g, int nch,
                     const double* window64, const double2* tw64, double* An64, float* An32, float* An32lo,
                     int round_tf32) {
    const size_t smem = (size_t)(2 * F64::BUF + F64::TW2) * sizeof(double2);
    static SmemOptIn opt_in1, opt_in2;
    smem_opt_in(k_frames64<1>, smem, opt_in1);
    smem_opt_in(k_frames64<2>, smem, opt_in2);
    dim3 grid((g.T + F64_FRAMES - 1) / F64_FRAMES, g.n_items);
    if (nch == 2)
        k_frames64<2><<<grid, F64::THREADS, smem, st>>>(audio, audio64, g, window64, tw64, An64, An32, An32lo, round_tf32);
    else
        k_frames64<1><<<grid, F64::THREADS, smem, st>>>(audio, audio64, g, window64, tw64, An64, An32, An32lo, round_tf32);
}

// ------------------------------------------------------------------------------------------
// k_selfsim_simt  --  S = A^T A in fp32 on the CUDA cores (fast pass, error bound tau)
// 64x64 output tile per CTA, 16x16 threads x 4x4 accumulators, K in chunks of 16 through smem.
// The products are summed in the same k order for (i, j) and (j, i): S is bitwise symmetric.
// ------------------------------------------------------------------------------------------
// Output rows j in [r0, r0 + rows) (the whole matrix: r0 = 0, rows = T) at Sout[(j - r0) * T + i].
__global__ void __launch_bounds__(256)
k_selfsim_simt(const float* __restrict__ An32, int T, int r0, int rows, float* __restrict__ S) {
    __shared__ float sa[16][65];
    __shared__ float sb[16][65];
    const int item = blockIdx.z;
    const float* __restrict__ A = An32 + (size_t)item * T * KPAD;
    float* __restrict__ Sout = S + (size_t)item * rows * T;
    const int ti = threadIdx.x & 15, tj = threadIdx.x >> 4;
    const int i0 = blockIdx.y * 64, j0 = r0 + blockIdx.x * 64;
    const int j_end = r0 + rows;
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
    for (int k0 = 0; k0 < KPAD; k0 += 16) {
        // 64 rows x 16 k per operand: 1024 elements, 4 per thread
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int idx = threadIdx.x + 256 * e;
            const int row = idx >> 4, kk = idx & 15;
            const int ri = i0 + row, rj = j0 + row;
            sa[kk][row] = ri < T ? A[(size_t)ri * KPAD + k0 + kk] : 0.f;
            sb[kk][row] = rj < j_end ? A[(size_t)rj * KPAD + k0 + kk] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float av[4], bv[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) av[a] = sa[kk][ti + 16 * a];
#pragma unroll
            for (int b = 0; b < 4; ++b) bv[b] = sb[kk][tj + 16 * b];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int i = i0 + ti + 16 * a, j = j0 + tj + 16 * b;
            if (i < T && j < j_end) Sout[(size_t)(j - r0) * T + i] = acc[a][b];
        }
}

void launch_selfsim_simt(cudaStream_t st, const float* An32, int n_items, int T, float* S) {
    dim3 grid((T + 63) / 64, (T + 63) / 64, n_items);
    k_selfsim_simt<<<grid, 256, 0, st>>>(An32, T, 0, T, S);
}

// the same products as the whole matrix, so a panel holds exactly the whole matrix's rows
void launch_selfsim_simt_panel(cudaStream_t st, const float* An32, int T, int r0, int rows, float* S_panel) {
    dim3 grid((rows + 63) / 64, (T + 63) / 64, 1);
    k_selfsim_simt<<<grid, 256, 0, st>>>(An32, T, r0, rows, S_panel);
}

constexpr int DOTN = (NBIN + 31) / 32;  // elements of a frame per lane

// exact float64 dot product of two normalised frames, one warp (result in every lane).  All the loads
// of the global operand are issued before the first multiply so that their latencies overlap.
__device__ __forceinline__ double warp_dot64(const double* __restrict__ a, const double* __restrict__ b, int lane) {
    double bv[DOTN];
#pragma unroll
    for (int i = 0; i < DOTN; ++i) {
        const int k = lane + 32 * i;
        bv[i] = k < NBIN ? __ldg(b + k) : 0.0;
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < DOTN; ++i) {
        const int k = lane + 32 * i;
        if (k < NBIN) s = fma(a[k], bv[i], s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

// ------------------------------------------------------------------------------------------
// k_topk  --  _localmaxima / _indices with certification            repet.py:1294-1383
// One CTA per column c of the similarity matrix.  The fast values v~ (row c of the fp32 matrix,
// |v~ - v| <= tau) only PROPOSE candidates:
//   dropped for sure   : v~[i] < thr - tau, or some neighbour within +-d has v~[u] >= v~[i] + 2 tau
//   candidate          : otherwise; "certain" when no neighbour is within 2 tau and v~[i] >= thr + tau
// Every candidate's similarity is then recomputed EXACTLY (float64 dot of the float64-normalised
// frames), uncertain candidates are re-decided against the exact values of their near-tie
// neighbours, and the survivors are ranked by exact value (descending; ties by descending index,
// which is what argsort()[::-1] gives).  The first `number` indices are written.
// With tau = 0 this is the reference's rule verbatim (strict >, windows clipped at the ends,
// NaN never a maximum: quirk Q7).
// ------------------------------------------------------------------------------------------
// CTA shape, measured on the 10-minute track (scripts/gpu_topk_sweep.sh, profiles/r2e_topk_sweep.txt): the kernel is
// a chain of short phases separated by barriers (ncu: barrier stalls 9.4 per issue at 512 threads, 2 CTAs / SM), so
// smaller CTAs with a smaller shared-memory footprint (38 KB -> 5 CTAs / SM) hide them: 4.82 -> 3.35 ms.  Columns
// with more than TOPK_CAP candidates go to k_topk_exact.
#ifndef REPET_TOPK_THREADS
#define REPET_TOPK_THREADS 256
#endif
#ifndef REPET_TOPK_CAP
#define REPET_TOPK_CAP 768
#endif
#ifndef REPET_TOPK_CHUNK
#define REPET_TOPK_CHUNK 1536
#endif
constexpr int TOPK_THREADS = REPET_TOPK_THREADS;
constexpr int TOPK_CAP = REPET_TOPK_CAP;       // candidates per column held in shared memory
constexpr int TOPK_CHUNK = REPET_TOPK_CHUNK;   // elements of the fast row resident at a time (3 arrays)
constexpr int TOPK_BINS = 512;       // histogram of fast values over [-1, 1) for the top-`number` cut
// candidates held before the running prune cuts the buffer (checked at chunk boundaries: one chunk of a row proposes
// at most about payload / (d + 1) certain candidates, far below the remaining TOPK_CAP - TOPK_FILL for d of a second)
constexpr int TOPK_FILL = TOPK_CAP * 3 / 4;
__device__ __forceinline__ int topk_bin(float v) {
    return min(TOPK_BINS - 1, max(0, (int)floorf((v + 1.f) * (TOPK_BINS / 2.f))));
}

// ---- prune: only the `number` best survive the ranking -------------------------------------------
// Let c be a value that at least `number` CERTAIN candidates (kept whatever the exact values say) reach in the fast
// pass.  A candidate with v~ < c - 2 tau is exactly below all of them, so it can never be written; it needs no exact
// value and takes no part in the ranking.  c comes from a histogram of the certain candidates (bin width 2^-8),
// conservative by up to one bin.  REFINE (the running prune of long rows, whose maxima crowd the bins near the cut)
// splits that bin into TOPK_BINS sub-bins of 2^-17 with a second histogram, so c is conservative by 2^-17 instead.
// Compacts s_cand / s_vc to the candidates at or above the cut and returns their count; *s_cut is the cut (-inf:
// fewer than `number` certain candidates, nothing pruned).  Every thread of the CTA calls it with the same count;
// s_hist is TOPK_BINS ints of free shared memory, s_sel two ints.
template <bool REFINE>
__device__ int topk_prune(int count, int number, float two_tau, int* s_cand, float* s_vc, int* s_hist, float* s_cut,
                          int* s_count, int* s_sel) {
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int b = t; b < TOPK_BINS; b += blockDim.x) s_hist[b] = 0;
    __syncthreads();
    for (int q = t; q < count; q += blockDim.x)
        if (!(s_cand[q] & (1 << 30))) atomicAdd(&s_hist[topk_bin(s_vc[q])], 1);
    __syncthreads();
    if (warp == 0) {
        constexpr int PER_LANE = TOPK_BINS / 32;
        int mine = 0;
#pragma unroll
        for (int u = 0; u < PER_LANE; ++u) mine += s_hist[lane * PER_LANE + u];
        int above = 0;  // certain candidates in the bins of higher lanes
#pragma unroll
        for (int o = 0; o < 32; ++o) {
            const int other = __shfl_sync(0xffffffffu, mine, o);
            if (o > lane) above += other;
        }
        const bool holds = above < number && above + mine >= number;
        const unsigned who = __ballot_sync(0xffffffffu, holds);
        if (who == 0) {
            if (lane == 0) {
                *s_cut = -INFINITY;  // fewer than `number` certain candidates: nothing to prune
                if (REFINE) s_sel[0] = -1;
            }
        } else if (lane == __ffs(who) - 1) {
            int cum = above, b = lane * PER_LANE + PER_LANE - 1;
            for (; b > lane * PER_LANE; --b) {
                cum += s_hist[b];
                if (cum >= number) break;
            }
            if (REFINE && b == lane * PER_LANE && cum < number) cum += s_hist[b];  // the loop stops before the lane's last bin
            *s_cut = (float)b * (2.f / TOPK_BINS) - 1.f - two_tau - 1e-6f;  // lower edge of the bin, minus 2 tau (and binning rounding)
            if (REFINE) {
                s_sel[0] = b;
                s_sel[1] = cum - s_hist[b];  // certain candidates above bin b
            }
        }
    }
    __syncthreads();
    if (REFINE && s_sel[0] >= 0) {  // the same value in every thread
        const int b = s_sel[0], base = s_sel[1];
        const float lo = (float)b * (2.f / TOPK_BINS) - 1.f;
        constexpr float SUB_SCALE = (float)TOPK_BINS * TOPK_BINS / 2.f;  // sub-bins per unit of v
        __syncthreads();  // every thread has read s_sel before the histogram is reused
        for (int u = t; u < TOPK_BINS; u += blockDim.x) s_hist[u] = 0;
        __syncthreads();
        for (int q = t; q < count; q += blockDim.x) {
            const float v = s_vc[q];
            if (!(s_cand[q] & (1 << 30)) && topk_bin(v) == b)
                atomicAdd(&s_hist[min(TOPK_BINS - 1, max(0, (int)floorf((v - lo) * SUB_SCALE)))], 1);
        }
        __syncthreads();
        if (warp == 0) {
            constexpr int PER_LANE = TOPK_BINS / 32;
            int mine = 0;
#pragma unroll
            for (int u = 0; u < PER_LANE; ++u) mine += s_hist[lane * PER_LANE + u];
            int above = base;
#pragma unroll
            for (int o = 0; o < 32; ++o) {
                const int other = __shfl_sync(0xffffffffu, mine, o);
                if (o > lane) above += other;
            }
            const bool holds = above < number && above + mine >= number;
            const unsigned who = __ballot_sync(0xffffffffu, holds);
            if (who != 0 && lane == __ffs(who) - 1) {  // none: keep the bin's own cut
                int cum = above, sb = lane * PER_LANE + PER_LANE - 1;
                for (; sb > lane * PER_LANE; --sb) {
                    cum += s_hist[sb];
                    if (cum >= number) break;
                }
                *s_cut = lo + (float)sb / SUB_SCALE - two_tau - 1e-6f;  // lower edge of the sub-bin, minus 2 tau
            }
        }
        __syncthreads();
    }
    const float cut = *s_cut;
    if (cut > -INFINITY) {
        // compact the survivors in place (one warp, chunks of 32 in order: writes never pass reads)
        if (warp == 0) {
            int kept = 0;
            for (int q0 = 0; q0 < count; q0 += 32) {
                const int q = q0 + lane;
                const int code = q < count ? s_cand[q] : 0;
                const float v = q < count ? s_vc[q] : 0.f;
                const bool keep = q < count && v >= cut;
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                __syncwarp();
                if (keep) {
                    const int pos = kept + __popc(m & ((1u << lane) - 1));
                    s_cand[pos] = code;
                    s_vc[pos] = v;
                }
                kept += __popc(m);
                __syncwarp();
            }
            if (lane == 0) *s_count = kept;
        }
        __syncthreads();
        count = *s_count;
    }
    return count;
}

// Column c = c0 + blockIdx.x reads its fast row at S + (item * gridDim.x + blockIdx.x) * T: the whole matrix
// (c0 = 0, gridDim.x = T) or a row panel of one item (c0 = its first row).  Outputs are indexed by the absolute column.
// RUNNING: the running prune below, compiled in for rows that can hold more than TOPK_CAP maxima.
template <bool RUNNING>
__global__ void __launch_bounds__(TOPK_THREADS)
k_topk(const float* __restrict__ S, int c0, const double* __restrict__ An64, int T, float tau, double thr, int d,
       int number, int nb, int* __restrict__ idx_out, int* __restrict__ cnt_out, int* __restrict__ overflow,
       int* __restrict__ ovf_cols, int force_exact) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* s_col = reinterpret_cast<double*>(smem);           // [APITCH64]   column c, float64
    double* s_exact = s_col + APITCH64;                        // [TOPK_CAP]   exact similarity of candidates
    int* s_cand = reinterpret_cast<int*>(s_exact + TOPK_CAP);  // [TOPK_CAP]   index | uncertain << 30
    float* s_vc = reinterpret_cast<float*>(s_cand + TOPK_CAP); // [TOPK_CAP]   fast value of candidates
    float* s_e = s_vc + TOPK_CAP;                              // [nb*d]       extended chunk of the fast row
    float* s_pm = s_e + TOPK_CHUNK;                            // prefix maxima within blocks of d
    float* s_sm = s_pm + TOPK_CHUNK;                           // suffix maxima within blocks of d
    __shared__ int s_count, s_kept, s_sel[2];
    __shared__ float s_cut;
    const int item = blockIdx.y, c = c0 + blockIdx.x;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarp = blockDim.x >> 5;
    const float* __restrict__ row = S + ((size_t)item * gridDim.x + blockIdx.x) * (size_t)T;
    const double* __restrict__ A = An64 + (size_t)item * T * APITCH64;
    if (force_exact) {  // test knob: every column goes through k_topk_exact
        if (t == 0) ovf_cols[atomicAdd(overflow, 1)] = item * T + c;
        return;
    }
    if (t == 0) {
        s_count = 0;
        s_kept = 0;
    }
    for (int k = t; k < APITCH64; k += blockDim.x) s_col[k] = A[(size_t)c * APITCH64 + k];
    const float thr_f = (float)thr;
    const float two_tau = 2.f * tau;
    // ---- propose: sliding-window maxima by van Herk / Gil-Werman on chunks of the row -----------
    // chunk = nb blocks of d elements: one halo block on each side, nb-2 payload blocks
    const int payload = d > 0 ? (nb - 2) * d : TOPK_CHUNK;
    const int ext = d > 0 ? nb * d : payload;     // elements staged per chunk (<= TOPK_CHUNK)
    const int halo = d > 0 ? d : 0;
    // the next chunk of the row is fetched into registers while the current one is examined
    constexpr int PER_THREAD = TOPK_CHUNK / TOPK_THREADS;
    float nxt[PER_THREAD];
    auto fetch = [&](int g0) {
#pragma unroll
        for (int u = 0; u < PER_THREAD; ++u) {
            const int x = t + u * TOPK_THREADS;
            const int g = g0 - halo + x;
            nxt[u] = (x < ext && g >= 0 && g < T) ? __ldg(row + g) : -INFINITY;
        }
    };
    // Running prune: a long row proposes more local maxima than the buffer holds (about one per 2 d frames).  When
    // the buffer passes TOPK_FILL at a chunk boundary, topk_prune cuts it down to what can still be among the
    // `number` best, and later proposals below that cut are dropped.  The cut only rises as certain candidates
    // arrive, so a dropped proposal stays exactly below `number` certain ones.  It is compiled in only for rows that
    // can hold more than TOPK_CAP maxima d + 1 frames apart (launch_topk_propose); shorter rows can overflow only
    // through near-ties, which is what k_topk_exact is for, and run exactly the kernel they ran before.
    float run_cut = -INFINITY;
    fetch(0);
    for (int g0 = 0; g0 < T; g0 += payload) {
        __syncthreads();
        if (RUNNING && g0 > 0) {  // every proposal of the previous chunk is in; s_pm / s_sm are free until the staging
            const int n = s_count;
            if (n > TOPK_FILL && n <= TOPK_CAP && n > number) {
                topk_prune<true>(n, number, two_tau, s_cand, s_vc, reinterpret_cast<int*>(s_pm), &s_cut, &s_count, s_sel);
                run_cut = fmaxf(run_cut, s_cut);
            }
        }
#pragma unroll
        for (int u = 0; u < PER_THREAD; ++u) {
            const int x = t + u * TOPK_THREADS;
            float v = nxt[u];
            if (v != v) v = INFINITY;  // NaN is never a maximum and blocks its neighbours (quirk Q7)
            if (x < ext) s_e[x] = v;
        }
        if (g0 + payload < T) fetch(g0 + payload);
        __syncthreads();
        if (d > 0) {
            for (int blk = t; blk < nb; blk += blockDim.x) {
                float m = -INFINITY;
                for (int x = blk * d; x < (blk + 1) * d; ++x) {
                    m = fmaxf(m, s_e[x]);
                    s_pm[x] = m;
                }
                m = -INFINITY;
                for (int x = (blk + 1) * d - 1; x >= blk * d; --x) {
                    m = fmaxf(m, s_e[x]);
                    s_sm[x] = m;
                }
            }
            __syncthreads();
        }
        for (int x = t; x < payload; x += blockDim.x) {
            const int i = g0 + x;
            if (i >= T) break;
            const int xe = d > 0 ? x + d : x;
            const float v = s_e[xe];
            if (!(v >= thr_f - tau) || !(v < INFINITY)) continue;
            if (RUNNING && v < run_cut) continue;  // below `number` certain candidates already held
            float m = -INFINITY;
            if (d > 0) {
                // left window [xe-d, xe-1] and right window [xe+1, xe+d]: each exactly one block long
                m = fmaxf(fmaxf(s_sm[xe - d], s_pm[xe - 1]), fmaxf(s_sm[xe + 1], s_pm[xe + d]));
            }
            if (!(m < v + two_tau)) continue;  // a neighbour is at least 2 tau above (or is NaN): not a maximum
            if (tau == 0.f && !(m < v)) continue;  // exact fast values: the strict rule decides ties here
            const bool uncertain = tau > 0.f && ((m > v - two_tau) || !(v >= thr_f + tau));
            const int slot = atomicAdd(&s_count, 1);
            if (slot < TOPK_CAP) {
                s_cand[slot] = i | (uncertain ? (1 << 30) : 0);
                s_vc[slot] = v;
            }
        }
    }
    __syncthreads();
    int count = s_count;
    if (count > TOPK_CAP) {
        // more near-tied candidates than the certification budget holds (a stationary or exactly looped stretch:
        // thousands of similarities within 2 tau of each other): the column is handed to k_topk_exact, which
        // applies the reference's rule to an exact float64 row
        if (t == 0) ovf_cols[atomicAdd(overflow, 1)] = item * T + c;
        return;
    }
    if (t == 0) atomicAdd(overflow + 1, count);  // statistics: candidates proposed
    // ---- prune: only the `number` best survive the ranking (topk_prune) -------------------------
    if (count > number)
        count = topk_prune<false>(count, number, two_tau, s_cand, s_vc, reinterpret_cast<int*>(s_pm), &s_cut, &s_count, s_sel);
    // ---- which candidates need their exact value? ---------------------------------------------
    // the uncertain ones (local-maximum test within 2 tau) and every pair whose fast values are within
    // 2 tau of each other (their ORDER is not decided by the fast pass); bit 29 marks them
    for (int q = t; q < count; q += blockDim.x) {
        int code = s_cand[q];
        bool need = (code & (1 << 30)) != 0;
        const float v = s_vc[q];
        for (int r = 0; r < count && !need; ++r)
            if (r != q && fabsf(s_vc[r] - v) <= two_tau) need = true;
        if (need) s_cand[q] = code | (1 << 29);
    }
    __syncthreads();
    for (int q = warp; q < count; q += nwarp) {
        const int code = s_cand[q];
        if (!(code & (1 << 29))) continue;
        const int i = code & 0x1fffffff;
        const double e = warp_dot64(s_col, A + (size_t)i * APITCH64, lane);
        if (lane == 0) s_exact[q] = e;
    }
    __syncthreads();
    // ---- re-decide the uncertain ones against exact neighbour values ---------------------------
    for (int q = warp; q < count; q += nwarp) {
        const int code = s_cand[q];
        if (!(code & (1 << 30))) continue;
        const int i = code & 0x1fffffff;
        const double e = s_exact[q];
        const float v = s_vc[q];
        bool keep = e >= thr;
        if (lane == 0) atomicAdd(overflow + 2, 1);  // statistics: uncertain candidates
        const int lo = max(i - d, 0), hi = min(i + d, T - 1);
        for (int u0 = lo; u0 <= hi && keep; u0 += 32) {
            const int u = u0 + lane;
            const bool near_tie = u <= hi && u != i && (row[u] > v - two_tau);
            unsigned mask = __ballot_sync(0xffffffffu, near_tie);
            while (mask && keep) {
                const int src = __ffs(mask) - 1;
                mask &= mask - 1;
                const double eu = warp_dot64(s_col, A + (size_t)(u0 + src) * APITCH64, lane);
                if (lane == 0) atomicAdd(overflow + 3, 1);  // statistics: near-tie neighbour dots
                if (!(e > eu)) keep = false;  // strict >, NaN never passes
            }
        }
        if (lane == 0 && !keep) s_cand[q] = -1;
    }
    __syncthreads();
    // ---- rank the survivors: fast values decide when they differ by more than 2 tau, exact values
    // (both are available then) otherwise; ties by descending index -----------------------------
    for (int q = t; q < count; q += blockDim.x) {
        const int code = s_cand[q];
        if (code < 0) continue;
        const int i = code & 0x1fffffff;
        const float v = s_vc[q];
        const double e = s_exact[q];
        int rank = 0;
        for (int r = 0; r < count; ++r) {
            const int other = s_cand[r];
            if (other < 0 || r == q) continue;
            const float vo = s_vc[r];
            if (fabsf(vo - v) > two_tau) {
                rank += vo > v;
            } else {
                const double eo = s_exact[r];
                const int io = other & 0x1fffffff;
                rank += (eo > e) || (eo == e && io > i);
            }
        }
        atomicAdd(&s_kept, 1);
        if (rank < number) idx_out[((size_t)item * T + c) * (size_t)number + rank] = i;
    }
    __syncthreads();
    if (t == 0) cnt_out[(size_t)item * T + c] = min(s_kept, number);
}

// ------------------------------------------------------------------------------------------
// k_topk_exact  --  _localmaxima on an exact float64 similarity row           repet.py:1294-1345
// The columns k_topk could not settle within its candidate budget.  A persistent CTA walks the list: the whole
// row <A[c], A[u]>, u < T, as exact float64 dots (global scratch), then the reference's rule verbatim -- v >= thr,
// strictly above every neighbour within +-d (windows clipped, NaN never wins), survivors ranked by value
// descending (ties: descending index) -- with no tolerance anywhere.
// ------------------------------------------------------------------------------------------
constexpr int TOPK_EXACT_CTAS_PER_SM = 2;

__global__ void __launch_bounds__(TOPK_THREADS)
k_topk_exact(const double* __restrict__ An64, int T, double thr, int d, int number, const int* __restrict__ overflow,
             const int* __restrict__ ovf_cols, unsigned char* __restrict__ scratch, size_t per_cta,
             int* __restrict__ idx_out, int* __restrict__ cnt_out) {
    __shared__ double s_col[APITCH64];
    __shared__ int s_kept;
    const int n_cols = overflow[0];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarp = blockDim.x >> 5;
    double* __restrict__ row = reinterpret_cast<double*>(scratch + (size_t)blockIdx.x * per_cta);  // [T]
    int* __restrict__ kept = reinterpret_cast<int*>(row + T);                                     // [T]
    for (int e = blockIdx.x; e < n_cols; e += gridDim.x) {
        const int col = ovf_cols[e];
        const int item = col / T, c = col - item * T;
        const double* __restrict__ A = An64 + (size_t)item * T * APITCH64;
        __syncthreads();  // the previous column's ranking has finished with row / kept / s_col
        if (t == 0) s_kept = 0;
        for (int k = t; k < APITCH64; k += blockDim.x) s_col[k] = A[(size_t)c * APITCH64 + k];
        __syncthreads();
        for (int u = warp; u < T; u += nwarp) {
            const double v = warp_dot64(s_col, A + (size_t)u * APITCH64, lane);
            if (lane == 0) row[u] = v;
        }
        __syncthreads();
        for (int i = t; i < T; i += blockDim.x) {
            const double v = row[i];
            bool keep = v >= thr;
            const int lo = max(i - d, 0), hi = min(i + d, T - 1);
            for (int u = lo; u <= hi && keep; ++u)
                if (u != i && !(v > row[u])) keep = false;
            if (keep) kept[atomicAdd(&s_kept, 1)] = i;
        }
        __syncthreads();
        const int K = s_kept;
        for (int q = t; q < K; q += blockDim.x) {
            const int i = kept[q];
            const double v = row[i];
            int rank = 0;
            for (int r = 0; r < K; ++r) {
                const int io = kept[r];
                const double vo = row[io];
                rank += (vo > v) || (vo == v && io > i);
            }
            if (rank < number) idx_out[((size_t)item * T + c) * (size_t)number + rank] = i;
        }
        if (t == 0) cnt_out[(size_t)item * T + c] = min(K, number);
    }
}

size_t topk_exact_scratch_bytes(int T, int sm_count) {
    const size_t per_cta = ((size_t)T * 12 + 255) / 256 * 256;
    return per_cta * (size_t)(sm_count * TOPK_EXACT_CTAS_PER_SM);
}

int launch_topk_propose(cudaStream_t st, const float* S, int c0, int n_cols, const double* An64, int n_items, int T,
                        float tau, double thr, int d, int number, int* idx_out, int* cnt_out, int* overflow,
                        int* ovf_cols) {
    // blocks of d elements per chunk: as many as fit, at least halo + one payload block
    int nb = 3;
    if (d > 0) {
        nb = std::min(TOPK_THREADS, TOPK_CHUNK / d);
        if (nb < 3) return -1;  // similarity_distance too large for the shared-memory window
    }
    const size_t smem = (size_t)APITCH64 * 8 + (size_t)TOPK_CAP * 16 + 3 * (size_t)TOPK_CHUNK * 4;
    dim3 grid(n_cols, n_items);
    // the running prune pays for rows that can hold more than TOPK_CAP maxima (strict maxima within +-d are more
    // than d frames apart): at similarity_distance 1 s, tracks above about 13 minutes
    if ((long long)T > (long long)(d + 1) * TOPK_CAP) {
        static SmemOptIn opt_in;
        smem_opt_in(k_topk<true>, smem, opt_in);
        k_topk<true><<<grid, TOPK_THREADS, smem, st>>>(S, c0, An64, T, tau, thr, d, number, nb, idx_out, cnt_out,
                                                       overflow, ovf_cols, g_tuning.topk_force_exact);
    } else {
        static SmemOptIn opt_in;
        smem_opt_in(k_topk<false>, smem, opt_in);
        k_topk<false><<<grid, TOPK_THREADS, smem, st>>>(S, c0, An64, T, tau, thr, d, number, nb, idx_out, cnt_out,
                                                        overflow, ovf_cols, g_tuning.topk_force_exact);
    }
    return 0;
}

void launch_topk_exact(cudaStream_t st, const double* An64, int T, double thr, int d, int number, const int* overflow,
                       const int* ovf_cols, unsigned char* scratch, int* idx_out, int* cnt_out, int sm_count) {
    const size_t per_cta = ((size_t)T * 12 + 255) / 256 * 256;
    k_topk_exact<<<sm_count * TOPK_EXACT_CTAS_PER_SM, TOPK_THREADS, 0, st>>>(An64, T, thr, d, number, overflow, ovf_cols,
                                                                            scratch, per_cta, idx_out, cnt_out);
}

// ------------------------------------------------------------------------------------------
// k_online_select  --  the per-frame selection of the online REPET-SIM     repet.py:834-866
// Frame j (>= B-1) is compared with the B frames in its ring buffer, visited in SLOT order:
// slot b holds frame j-(j0-b) for b <= j0 and j-(j0-b)-B for b > j0, j0 = j mod B (quirk Q6).
// Similarities are exact float64 dots of the float64-normalised frames (float64 tensor-core MMAs,
// mma.sync m8n8k4), so the local-maximum rule and the ranking need no certification.  Writes FRAME indices.
// ------------------------------------------------------------------------------------------
constexpr int ONLINE_FB = 16;                  // target frames per CTA: two 8-row A blocks of the float64 MMA
constexpr int TGT_PITCH = APITCH64 + 10;       // doubles per target row in shared memory; pitch % 16 == 2 keeps the
                                               // 16-byte A-fragment loads of a quarter warp on disjoint banks
static_assert(TGT_PITCH % 16 == 2, "target row pitch");

// D (8x8) += A (8x4, row major) * B (4x8, column major), float64 tensor-core MMA.  Lane l holds
// A[l/4][l%4], B[l%4][l/4] and D[l/4][2*(l%4) + {0, 1}].
__device__ __forceinline__ void dmma884(double (&d)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(d[0]), "+d"(d[1])
                 : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(512)
k_online_select(const double* __restrict__ An64, int T, int B, int frame_base, double thr, int d, int number,
                int* __restrict__ idx_out, int* __restrict__ cnt_out, int item0, int cta0, unsigned char* scratch,
                size_t scratch_per_cta) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* s_tgt = reinterpret_cast<double*>(smem);          // [ONLINE_FB][TGT_PITCH]  target frames
    // similarity by ring slot [ONLINE_FB][B] and keep flags [ONLINE_FB][B]: shared memory, or -- for rings too long
    // for it (buffer_length above ~16 s at 44.1 kHz) -- this CTA's slice of a global scratch buffer (L2 resident)
    double* s_sim = scratch ? reinterpret_cast<double*>(scratch + (size_t)blockIdx.x * scratch_per_cta)
                            : s_tgt + ONLINE_FB * TGT_PITCH;
    unsigned char* s_keep = reinterpret_cast<unsigned char*>(s_sim + ONLINE_FB * B);
    __shared__ int s_kept[ONLINE_FB];
    const int item = item0 + blockIdx.y;
    // rows are frames frame_base .. frame_base + T - 1 of the stream; the first synthesised row is the
    // one whose absolute index is B - 1
    const int row_first = max(0, B - 1 - frame_base);
    const int j_first = (cta0 + blockIdx.x) * ONLINE_FB + row_first;
    const int nf = min(ONLINE_FB, T - j_first);  // target frames of this CTA
    if (nf <= 0) return;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarp = blockDim.x >> 5;
    const double* __restrict__ A = An64 + (size_t)item * T * APITCH64;
    if (t < ONLINE_FB) s_kept[t] = 0;
    for (int f = 0; f < ONLINE_FB; ++f)
        for (int k = t; k < APITCH64; k += blockDim.x)
            s_tgt[f * TGT_PITCH + k] = f < nf ? __ldg(A + (size_t)(j_first + f) * APITCH64 + k) : 0.0;
    // slots whose frame lies before the window (a stream window with partial history) can never be maxima
    for (int e = t; e < nf * B; e += blockDim.x) s_sim[e] = -INFINITY;
    __syncthreads();
    // Frame u sits in ring slot u mod B.  The similarities of the block's 16 targets with every buffer frame
    // u in [j_first - B + 1, j_first + nf - 1] are exact float64 dot products on the float64 tensor cores:
    // a warp takes 8 buffer frames at a time (B operand, streamed once from L2 in 128-byte row pieces) against
    // both 8-target blocks (A operand, shared memory).  The bins are visited in a lane-permuted order (lane
    // quad member q owns bins 16 c + 4 q .. + 3 of chunk c, one per MMA) so that every lane loads 32 contiguous
    // bytes; a sum does not care about the order of its terms.
    const int u_lo = max(0, j_first - (B - 1)), u_hi = j_first + nf - 1;
    const int n_blocks = (u_hi - u_lo + 8) >> 3;
    const int fr = lane >> 2, q = lane & 3;
    for (int nb = warp; nb < n_blocks; nb += nwarp) {
        const int u0 = u_lo + 8 * nb;
        const double* __restrict__ brow = A + (size_t)min(u0 + fr, u_hi) * APITCH64 + 4 * q;
        const double* __restrict__ arow0 = s_tgt + fr * TGT_PITCH + 4 * q;
        const double* __restrict__ arow1 = arow0 + 8 * TGT_PITCH;
        double c0[2] = {0.0, 0.0}, c1[2] = {0.0, 0.0};
        // groups of 4 chunks (64 bins): the B fragments of the next group are in flight (8 x 16-byte loads per
        // lane) while the 32 MMAs of the current one run -- without this every chunk waits out an L2 round trip
        constexpr int GROUP = 4, N_GROUPS = (NBIN - 1) / (16 * GROUP);
        static_assert((NBIN - 1) % (16 * GROUP) == 0, "bins - 1 must be a multiple of 64");
        double2 bn[2 * GROUP];
#pragma unroll
        for (int i = 0; i < GROUP; ++i) {
            bn[2 * i] = __ldg(reinterpret_cast<const double2*>(brow + 16 * i));
            bn[2 * i + 1] = __ldg(reinterpret_cast<const double2*>(brow + 16 * i + 2));
        }
#pragma unroll 1
        for (int g = 0; g < N_GROUPS; ++g) {
            double2 bc[2 * GROUP];
#pragma unroll
            for (int i = 0; i < 2 * GROUP; ++i) bc[i] = bn[i];
            if (g + 1 < N_GROUPS) {
                const double* __restrict__ nxt = brow + 16 * GROUP * (g + 1);
#pragma unroll
                for (int i = 0; i < GROUP; ++i) {
                    bn[2 * i] = __ldg(reinterpret_cast<const double2*>(nxt + 16 * i));
                    bn[2 * i + 1] = __ldg(reinterpret_cast<const double2*>(nxt + 16 * i + 2));
                }
            }
#pragma unroll
            for (int i = 0; i < GROUP; ++i) {
                const int k0 = 16 * (GROUP * g + i);
                const double2 x01 = *reinterpret_cast<const double2*>(arow0 + k0);
                const double2 x23 = *reinterpret_cast<const double2*>(arow0 + k0 + 2);
                const double2 y01 = *reinterpret_cast<const double2*>(arow1 + k0);
                const double2 y23 = *reinterpret_cast<const double2*>(arow1 + k0 + 2);
                dmma884(c0, x01.x, bc[2 * i].x);
                dmma884(c1, y01.x, bc[2 * i].x);
                dmma884(c0, x01.y, bc[2 * i].y);
                dmma884(c1, y01.y, bc[2 * i].y);
                dmma884(c0, x23.x, bc[2 * i + 1].x);
                dmma884(c1, y23.x, bc[2 * i + 1].x);
                dmma884(c0, x23.y, bc[2 * i + 1].y);
                dmma884(c1, y23.y, bc[2 * i + 1].y);
            }
        }
        // lane holds the sums of targets fr and fr + 8 with frames u0 + 2 q and u0 + 2 q + 1; the last bin
        // (NBIN - 1, the Nyquist row) is the one left over by the chunks of 16
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int u = u0 + 2 * q + e;
            if (u > u_hi) continue;
            const double last = __ldg(A + (size_t)u * APITCH64 + (NBIN - 1));
            const int slot = (u + frame_base) % B;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int f = fr + 8 * half;
                const int j = j_first + f;
                if (f >= nf || u > j || u < j - (B - 1)) continue;
                const double sum = half ? c1[e] : c0[e];
                s_sim[f * B + slot] = fma(s_tgt[f * TGT_PITCH + (NBIN - 1)], last, sum);
            }
        }
    }
    __syncthreads();
    // strict local maxima in slot order, windows clipped at slots 0 and B-1 (not circular), quirk Q6.
    // Both passes are warp-cooperative: a warp looks at 32 consecutive entries, compacts the few that matter
    // with a ballot (entries above both direct neighbours; then the kept ones) and spreads each one's window /
    // ranking loop over its lanes -- per-thread loops left 31 lanes waiting for the one that held a maximum.
    const int chunks = (B + 31) >> 5;  // 32-slot pieces per target
    for (int w = warp; w < nf * chunks; w += nwarp) {
        const int f = w / chunks, b0 = (w - f * chunks) << 5;
        const double* __restrict__ sim = s_sim + f * B;
        unsigned char* __restrict__ keepf = s_keep + f * B;
        const int b = b0 + lane;
        bool cand = false;
        if (b < B) {
            const double v = sim[b];
            cand = v >= thr;
            // cheap pre-filter on the four nearest slots of each side before the full window
            const int near = min(d, 4);
            for (int o = 1; o <= near && cand; ++o)
                cand = (b - o < 0 || v > sim[b - o]) && (b + o > B - 1 || v > sim[b + o]);
            keepf[b] = (d <= 4 && cand) ? 1 : 0;
        }
        unsigned todo = d > 4 ? __ballot_sync(0xffffffffu, cand) : 0u;
        while (todo) {
            const int bc = b0 + __ffs(todo) - 1;
            todo &= todo - 1;
            const double v = sim[bc];
            const int lo = max(bc - d, 0), hi = min(bc + d, B - 1);
            bool bad = false;
            for (int x = lo + lane; x <= hi; x += 32) bad |= (x != bc && !(v > sim[x]));
            if (!__any_sync(0xffffffffu, bad) && lane == 0) keepf[bc] = 1;
        }
    }
    __syncthreads();
    for (int w = warp; w < nf * chunks; w += nwarp) {
        const int f = w / chunks, b0 = (w - f * chunks) << 5;
        const double* __restrict__ sim = s_sim + f * B;
        const unsigned char* __restrict__ keepf = s_keep + f * B;
        unsigned todo = __ballot_sync(0xffffffffu, b0 + lane < B && keepf[b0 + lane]);
        while (todo) {
            const int b = b0 + __ffs(todo) - 1;
            todo &= todo - 1;
            const double v = sim[b];
            int rank = 0;
            for (int x = lane; x < B; x += 32)
                if (x != b && keepf[x]) rank += (sim[x] > v) || (sim[x] == v && x > b);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
            if (lane == 0) {
                atomicAdd(&s_kept[f], 1);
                if (rank < number) {
                    const int j = j_first + f, j0 = (j + frame_base) % B;
                    const int frame = b <= j0 ? j - (j0 - b) : j - (j0 - b) - B;
                    idx_out[((size_t)item * T + j) * (size_t)number + rank] = frame;
                }
            }
        }
    }
    __syncthreads();
    if (t < nf) cnt_out[(size_t)item * T + j_first + t] = min(s_kept[t], number);
}

int launch_online_select(cudaStream_t st, const double* An64, int n_items, int T, int B, int frame_base, double thr,
                         int d, int number, int* idx_out, int* cnt_out) {
    const int row_first = std::max(0, B - 1 - frame_base);
    if (T <= row_first) return 0;
    const size_t tgt_bytes = (size_t)ONLINE_FB * TGT_PITCH * 8 + 16;
    const size_t sel_bytes = ((size_t)ONLINE_FB * B * 9 + 15) / 16 * 16;
    int dev = 0, max_optin = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    static SmemOptIn opt_in;
    const int n_targets = T - row_first;
    const int n_cta = (n_targets + ONLINE_FB - 1) / ONLINE_FB;
    if (tgt_bytes + sel_bytes <= (size_t)max_optin) {
        const size_t smem = tgt_bytes + sel_bytes;
        if (smem > 48 * 1024 && !smem_opt_in(k_online_select, smem, opt_in)) return -1;
        dim3 grid(n_cta, n_items);
        k_online_select<<<grid, 512, smem, st>>>(An64, T, B, frame_base, thr, d, number, idx_out, cnt_out, 0, 0, nullptr, 0);
        return 0;
    }
    // ring longer than shared memory holds: similarity rows in a stream-ordered global scratch buffer, at most
    // 256 MB of it in flight per launch
    if (!smem_opt_in(k_online_select, tgt_bytes, opt_in)) return -1;
    const int per_launch = (int)std::min<size_t>((size_t)n_cta, std::max<size_t>(1, ((size_t)256 << 20) / sel_bytes));
    unsigned char* scratch = nullptr;
    if (cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)per_launch * sel_bytes, st) != cudaSuccess) {
        (void)cudaGetLastError();
        return -2;
    }
    for (int item = 0; item < n_items; ++item)
        for (int cta0 = 0; cta0 < n_cta; cta0 += per_launch) {
            dim3 grid(std::min(per_launch, n_cta - cta0), 1);
            k_online_select<<<grid, 512, tgt_bytes, st>>>(An64, T, B, frame_base, thr, d, number, idx_out, cnt_out, item,
                                                          cta0, scratch, sel_bytes);
        }
    cudaFreeAsync(scratch, st);
    return 0;
}

// ------------------------------------------------------------------------------------------
// k_simmodel  --  the similar-frame median of _simmask               repet.py:1529-1535, 872
// model[j][c][bin] = median over u in list(j) of |X_c[u][bin]| (an empty list gives NaN, as
// np.median of an empty selection does).  One CTA per (frame, item*channel).  Lists of up to 32
// frames go through the register selection networks on bin pairs; longer lists are staged as
// squared magnitudes in shared memory [n][256 bins] and selected by an in-place quickselect.
// ------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ float2 gather_median_pair(const float2* __restrict__ chan, size_t row, const int* __restrict__ list,
                                                     int k, bool first_is_dc) {
    float v0[N], v1[N];
#pragma unroll
    for (int s = 0; s < N; ++s) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(chan + (size_t)list[s] * row + k));
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
__device__ __forceinline__ void simmodel_small(const float2* __restrict__ chan, size_t row, const int* __restrict__ list,
                                               float* __restrict__ out, int t) {
#pragma unroll 1
    for (int k = 2 * t; k < XPITCH; k += 256)
        *reinterpret_cast<float2*>(out + k) = gather_median_pair<N>(chan, row, list, k, k == 0);
    // the Nyquist bin (bin 0's imaginary slot) of every frame is done by k_simmodel_nyquist
}

// median of column `col` of a [n][pitch] shared-memory tile of squared magnitudes: in-place Hoare
// quickselect of the upper middle element (expected ~3n compares instead of the n^2 of rank counting),
// then the lower middle = max of what ended up left of it.  The column is private to the thread.
__device__ __forceinline__ float tile_median(float* __restrict__ tile, int n, int pitch, int col) {
    float* __restrict__ v = tile + col;
    const int k = n >> 1;
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const float a = v[lo * pitch], b = v[((lo + hi) >> 1) * pitch], c = v[hi * pitch];
        const float pivot = fmaxf(fminf(a, b), fminf(fmaxf(a, b), c));  // median of three
        int i = lo, j = hi;
        while (i <= j) {
            while (v[i * pitch] < pivot) ++i;
            while (v[j * pitch] > pivot) --j;
            if (i <= j) {
                const float x = v[i * pitch];
                v[i * pitch] = v[j * pitch];
                v[j * pitch] = x;
                ++i;
                --j;
            }
        }
        if (k <= j) hi = j;
        else if (k >= i) lo = i;
        else break;
    }
    const float v_hi = v[k * pitch];
    if (n & 1) return fast_sqrt(v_hi);
    float v_lo = -INFINITY;
    for (int s = 0; s < k; ++s) v_lo = fmaxf(v_lo, v[s * pitch]);
    return 0.5f * (fast_sqrt(v_lo) + fast_sqrt(v_hi));
}

constexpr int SIMMODEL_THREADS = 256;

// squared magnitudes of every (frame, channel) row, [rows][PPITCH]: bin 0 = DC^2, bin N/2 = Nyquist^2.
// Long similar-frame lists gather these 4-byte values instead of the 8-byte spectra.
__global__ void __launch_bounds__(256)
k_sqmag(const float2* __restrict__ X, long long n_rows, float* __restrict__ Vsq) {
    const long long row = blockIdx.x;  // rows on grid.x: there can be more than 65535 of them
    const int k = blockIdx.y * 256 + threadIdx.x;
    if (row >= n_rows || k > XPITCH) return;
    const float2* __restrict__ x = X + row * XPITCH;
    float v;
    if (k == 0) {
        const float a = __ldg(&x[0]).x;
        v = __fmul_rn(a, a);
    } else if (k == XPITCH) {
        const float a = __ldg(&x[0]).y;
        v = __fmul_rn(a, a);
    } else {
        v = cmag2(__ldg(&x[k]));
    }
    Vsq[row * PPITCH + k] = v;
}

void launch_sqmag(cudaStream_t st, const float2* X, long long n_rows, float* Vsq) {
    dim3 grid((unsigned)n_rows, (XPITCH + 256) / 256);
    k_sqmag<<<grid, 256, 0, st>>>(X, n_rows, Vsq);
}

// median of n (<= NS) squared magnitudes gathered straight into registers: slots 0..n-1 hold data,
// the rest is padded with floor((NS-n)/2) times -inf and the remainder +inf, so that the median sits
// at sorted positions NS/2-1 (odd n) or NS/2-1, NS/2 (even n) whatever n is.
template <int NS>
__device__ __forceinline__ float gather_median_large(const float* __restrict__ vchan, size_t vrow,
                                                     const int* __restrict__ list, int n, int k) {
    float v[NS];
    const int lo = (NS - n) >> 1;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        if (s < n) v[s] = __ldg(vchan + (size_t)list[s] * vrow + k);
        else v[s] = (s - n) < lo ? -INFINITY : INFINITY;
    }
    median_select<NS>(v);
    return (n & 1) ? fast_sqrt(v[NS / 2 - 1]) : 0.5f * (fast_sqrt(v[NS / 2 - 1]) + fast_sqrt(v[NS / 2]));
}

template <int NS>
__device__ __forceinline__ void simmodel_large(const float* __restrict__ vchan, size_t vrow, const int* __restrict__ list,
                                               int n, float* __restrict__ out, int t) {
#pragma unroll 1
    for (int k = t; k < XPITCH; k += 128) out[k] = gather_median_large<NS>(vchan, vrow, list, n, k);
}

// k_simmodel_large: lists of 33..128 similar frames.  One CTA of 128 threads per (frame, channel); a
// thread gathers the n squared magnitudes of a bin (4-byte coalesced loads from Vsq) into registers and
// runs a pruned selection network -- no shared-memory tile, no data-dependent control flow.
__global__ void __launch_bounds__(128, 3)
k_simmodel_large(const float* __restrict__ Vsq, int T, int nch, const int* __restrict__ idx, const int* __restrict__ cnt,
                 int number, int first_frame, float* __restrict__ model) {
    __shared__ int s_list[128];
    const int j = blockIdx.x + first_frame;
    const int item = blockIdx.y / nch, c = blockIdx.y - item * nch;
    const int t = threadIdx.x;
    const int n = cnt[(size_t)item * T + j];
    if (n <= 32 || n > 128) return;  // k_simmodel handles those
    if (t < n) s_list[t] = idx[((size_t)item * T + j) * (size_t)number + t];
    __syncthreads();
    const float* __restrict__ vchan = Vsq + ((size_t)item * T * nch + c) * PPITCH;
    const size_t vrow = (size_t)nch * PPITCH;
    float* __restrict__ out = model + (((size_t)item * nch + c) * (size_t)T + j) * PPITCH;
    if (n <= 48) simmodel_large<48>(vchan, vrow, s_list, n, out, t);
    else if (n <= 64) simmodel_large<64>(vchan, vrow, s_list, n, out, t);
    else if (n <= 100) simmodel_large<100>(vchan, vrow, s_list, n, out, t);
    else simmodel_large<128>(vchan, vrow, s_list, n, out, t);
}

// k_simmodel_nyquist: the median of the Nyquist bin (the 1025th of a row) for lists of 1..128 frames, one THREAD
// per (frame, channel).  Inside the per-frame CTAs that bin cost a whole extra pass of a selection network with a
// single active lane (1/9 of the long-list kernel, 1/5 of the short-list one); here 32 frames share the pass.
template <int N>
__device__ __forceinline__ float nyquist_median_small(const float2* __restrict__ chan, size_t row,
                                                      const int* __restrict__ list) {
    float v[N];
#pragma unroll
    for (int s = 0; s < N; ++s) {
        const float y = __ldg(&chan[(size_t)__ldg(list + s) * row]).y;
        v[s] = __fmul_rn(y, y);
    }
    median_select<N>(v);
    return (N & 1) ? fast_sqrt(v[(N - 1) / 2]) : 0.5f * (fast_sqrt(v[(N - 1) / 2]) + fast_sqrt(v[N / 2]));
}
template <int NS>
__device__ __forceinline__ float nyquist_median_large(const float* __restrict__ vchan, size_t vrow,
                                                      const int* __restrict__ list, int n) {
    float v[NS];
    const int lo = (NS - n) >> 1;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        if (s < n) v[s] = __ldg(vchan + (size_t)__ldg(list + s) * vrow + XPITCH);
        else v[s] = (s - n) < lo ? -INFINITY : INFINITY;
    }
    median_select<NS>(v);
    return (n & 1) ? fast_sqrt(v[NS / 2 - 1]) : 0.5f * (fast_sqrt(v[NS / 2 - 1]) + fast_sqrt(v[NS / 2]));
}

__global__ void __launch_bounds__(128)
k_simmodel_nyquist(const float2* __restrict__ X, const float* __restrict__ Vsq, int T, int nch, const int* __restrict__ idx,
                   const int* __restrict__ cnt, int number, int first_frame, float* __restrict__ model) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x + first_frame;
    if (j >= T) return;
    const int item = blockIdx.y / nch, c = blockIdx.y - item * nch;
    const int n = cnt[(size_t)item * T + j];
    if (n < 1 || n > 128) return;  // empty lists are NaN rows already; longer ones take the shared-memory path
    const int* __restrict__ list = idx + ((size_t)item * T + j) * (size_t)number;
    float* __restrict__ out = model + (((size_t)item * nch + c) * (size_t)T + j) * PPITCH + XPITCH;
    if (n <= 32) {
        const size_t row = (size_t)nch * XPITCH;
        const float2* __restrict__ chan = X + (size_t)item * T * row + (size_t)c * XPITCH;
        switch (n) {
#define REPET_CASE(N) case N: *out = nyquist_median_small<N>(chan, row, list); break;
            REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
            REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
            REPET_CASE(15) REPET_CASE(16) REPET_CASE(17) REPET_CASE(18) REPET_CASE(19) REPET_CASE(20) REPET_CASE(21)
            REPET_CASE(22) REPET_CASE(23) REPET_CASE(24) REPET_CASE(25) REPET_CASE(26) REPET_CASE(27) REPET_CASE(28)
            REPET_CASE(29) REPET_CASE(30) REPET_CASE(31) REPET_CASE(32)
#undef REPET_CASE
        }
        return;
    }
    const float* __restrict__ vchan = Vsq + ((size_t)item * T * nch + c) * PPITCH;
    const size_t vrow = (size_t)nch * PPITCH;
    if (n <= 48) *out = nyquist_median_large<48>(vchan, vrow, list, n);
    else if (n <= 64) *out = nyquist_median_large<64>(vchan, vrow, list, n);
    else if (n <= 100) *out = nyquist_median_large<100>(vchan, vrow, list, n);
    else *out = nyquist_median_large<128>(vchan, vrow, list, n);
}

__global__ void __launch_bounds__(SIMMODEL_THREADS)
k_simmodel(const float2* __restrict__ X, const float* __restrict__ Vsq, int T, int nch, const int* __restrict__ idx,
           const int* __restrict__ cnt, int number, int first_frame, float* __restrict__ model) {
    extern __shared__ __align__(16) unsigned char smem[];
    int* s_list = reinterpret_cast<int*>(smem);                              // [number]
    float* s_tile = reinterpret_cast<float*>(s_list + ((number + 3) & ~3));  // [n][256] when n > 32
    const int j = blockIdx.x + first_frame;
    const int item = blockIdx.y / nch, c = blockIdx.y - item * nch;
    const int t = threadIdx.x;
    const size_t row = (size_t)nch * XPITCH;
    const float2* __restrict__ chan = X + (size_t)item * T * row + (size_t)c * XPITCH;
    float* __restrict__ out = model + (((size_t)item * nch + c) * (size_t)T + j) * PPITCH;
    const int n = cnt[(size_t)item * T + j];
    for (int s = t; s < n; s += SIMMODEL_THREADS) s_list[s] = idx[((size_t)item * T + j) * (size_t)number + s];
    __syncthreads();
    if (n == 0) {
        for (int k = t; k <= XPITCH; k += SIMMODEL_THREADS) out[k] = nanf("");
        return;
    }
    if (n > 32 && n <= 128) return;  // k_simmodel_large
    if (n <= 32) {
        // short lists: register selection networks on bin pairs, 128 threads x 256 bins per pass
        if (t < 128) {
            switch (n) {
#define REPET_CASE(N) case N: simmodel_small<N>(chan, row, s_list, out, t); break;
                REPET_CASE(1) REPET_CASE(2) REPET_CASE(3) REPET_CASE(4) REPET_CASE(5) REPET_CASE(6) REPET_CASE(7)
                REPET_CASE(8) REPET_CASE(9) REPET_CASE(10) REPET_CASE(11) REPET_CASE(12) REPET_CASE(13) REPET_CASE(14)
                REPET_CASE(15) REPET_CASE(16) REPET_CASE(17) REPET_CASE(18) REPET_CASE(19) REPET_CASE(20) REPET_CASE(21)
                REPET_CASE(22) REPET_CASE(23) REPET_CASE(24) REPET_CASE(25) REPET_CASE(26) REPET_CASE(27) REPET_CASE(28)
                REPET_CASE(29) REPET_CASE(30) REPET_CASE(31) REPET_CASE(32)
#undef REPET_CASE
            }
        }
        return;
    }
    // long lists: passes of 256 bins.  The CTA gathers the [n][256] tile of squared magnitudes with
    // 16-byte loads (4 rows per sweep, 8 sweeps in flight per thread), then every thread selects the
    // median of its own column (bank = lane: conflict free) by quickselect.
    const float* __restrict__ vchan = Vsq + ((size_t)item * T * nch + c) * PPITCH;
    const size_t vrow = (size_t)nch * PPITCH;
    const int sub = t >> 6, quad = (t & 63) * 4;  // this thread gathers row (4 s' + sub), bins quad..quad+3
    for (int pass = 0; pass < XPITCH / 256; ++pass) {
        const int k0 = 256 * pass;
        for (int s0 = 0; s0 < n; s0 += 32) {
            float4 x[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int s = min(s0 + 4 * u + sub, n - 1);
                x[u] = __ldg(reinterpret_cast<const float4*>(vchan + (size_t)s_list[s] * vrow + k0 + quad));
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int s = s0 + 4 * u + sub;
                if (s < n) *reinterpret_cast<float4*>(s_tile + s * 256 + quad) = x[u];
            }
        }
        __syncthreads();
        out[k0 + t] = tile_median(s_tile, n, 256, t);
        __syncthreads();
    }
    if (t == 0) {
        // Nyquist^2 sits at bin N/2 of the Vsq rows
        for (int s = 0; s < n; ++s) s_tile[s * 256] = __ldg(vchan + (size_t)s_list[s] * vrow + XPITCH);
        out[XPITCH] = tile_median(s_tile, n, 256, 0);
    }
}

int launch_simmodel(cudaStream_t st, const float2* X, const float* Vsq, int n_items, int T, int nch, const int* idx,
                    const int* cnt, int number, int first_frame, float* model) {
    const size_t smem = (size_t)((number + 3) & ~3) * 4 + (number > 32 ? (size_t)number * 256 * 4 : 0);
    if (smem > 220 * 1024) return -1;
    if (number > 32 && !Vsq) return -2;
    static SmemOptIn opt_in;
    if (smem > 48 * 1024 && !smem_opt_in(k_simmodel, smem, opt_in)) return -1;
    if (T <= first_frame) return 0;
    dim3 grid(T - first_frame, n_items * nch);
    k_simmodel<<<grid, SIMMODEL_THREADS, smem, st>>>(X, Vsq, T, nch, idx, cnt, number, first_frame, model);
    if (number > 32) k_simmodel_large<<<grid, 128, 0, st>>>(Vsq, T, nch, idx, cnt, number, first_frame, model);
    k_simmodel_nyquist<<<dim3((T - first_frame + 127) / 128, n_items * nch), 128, 0, st>>>(X, Vsq, T, nch, idx, cnt, number,
                                                                                          first_frame, model);
    return 0;
}

// ------------------------------------------------------------------------------------------
// k_cosine64  --  _similaritymatrix / _selfsimilaritymatrix as helpers     repet.py:1209-1246
// Exact float64 cosine similarity of float64-normalised frames: out[i][j] = <A1[i], A2[j]>.
// One warp per output element (helper sizes only; the drivers use the tensor-core pass).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_cosine64(const double* __restrict__ A1, int n1, const double* __restrict__ A2, int n2, double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= (long long)n1 * n2) return;
    const int i = (int)(w / n2), j = (int)(w - (long long)i * n2);
    const double e = warp_dot64(A1 + (size_t)i * APITCH64, A2 + (size_t)j * APITCH64, lane);
    if (lane == 0) out[(size_t)i * n2 + j] = e;
}

void launch_cosine64(cudaStream_t st, const double* A1, int n1, const double* A2, int n2, double* out) {
    const long long threads = (long long)n1 * n2 * 32;
    k_cosine64<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(A1, n1, A2, n2, out);
}

// ------------------------------------------------------------------------------------------
// k_localmaxima64  --  _localmaxima / _indices on caller-provided float64 data
//                                                                       repet.py:1294-1383
// Column c of a row-major [n][n_columns] matrix (n_columns = 1: a vector).  The reference's rule
// verbatim: v[i] >= thr and v[i] > every neighbour within +-d (windows clipped, NaN never wins),
// survivors ranked by value descending (ties: descending index), first `number` kept.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_localmaxima64(const double* __restrict__ data, int n, int n_columns, double thr, int d, int number,
                int* __restrict__ idx_out, int* __restrict__ cnt_out, double* __restrict__ val_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* s_v = reinterpret_cast<double*>(smem);          // [n]
    unsigned char* s_keep = reinterpret_cast<unsigned char*>(s_v + n);  // [n]
    __shared__ int s_kept;
    const int c = blockIdx.x, t = threadIdx.x;
    if (t == 0) s_kept = 0;
    for (int i = t; i < n; i += blockDim.x) s_v[i] = data[(size_t)i * n_columns + c];
    __syncthreads();
    for (int i = t; i < n; i += blockDim.x) {
        const double v = s_v[i];
        bool keep = v >= thr;
        const int lo = max(i - d, 0), hi = min(i + d, n - 1);
        for (int u = lo; u <= hi && keep; ++u)
            if (u != i && !(v > s_v[u])) keep = false;
        s_keep[i] = keep ? 1 : 0;
    }
    __syncthreads();
    for (int i = t; i < n; i += blockDim.x) {
        if (!s_keep[i]) continue;
        const double v = s_v[i];
        int rank = 0;
        for (int u = 0; u < n; ++u)
            if (u != i && s_keep[u]) rank += (s_v[u] > v) || (s_v[u] == v && u > i);
        atomicAdd(&s_kept, 1);
        if (rank < number) {
            idx_out[(size_t)c * number + rank] = i;
            if (val_out) val_out[(size_t)c * number + rank] = v;
        }
    }
    __syncthreads();
    if (t == 0) cnt_out[c] = min(s_kept, number);
}

int launch_localmaxima64(cudaStream_t st, const double* data, int n, int n_columns, double thr, int d, int number,
                         int* idx_out, int* cnt_out, double* val_out) {
    const size_t smem = (size_t)n * 9 + 16;
    if (smem > 220 * 1024) return -1;
    static SmemOptIn opt_in;
    if (smem > 48 * 1024 && !smem_opt_in(k_localmaxima64, smem, opt_in)) return -1;
    k_localmaxima64<<<n_columns, 256, smem, st>>>(data, n, n_columns, thr, d, number, idx_out, cnt_out, val_out);
    return 0;
}

}  // namespace repet
