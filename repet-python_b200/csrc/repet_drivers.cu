// Batch drivers behind the C ABI: repet.original / extended / adaptive (repet.py:67-568) over
// device-resident clips, their host-buffer variants (chunked, copy/compute overlapped) and the
// reference's float64 (samples, channels) calling convention.
#include "repet_internal.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <functional>

using namespace repet;

namespace {

enum Kind { KIND_ORIGINAL = 0, KIND_EXTENDED = 1, KIND_ADAPTIVE = 2, KIND_SIM = 3, KIND_SIMONLINE = 4 };

// rigorous bound on |fp32 similarity - exact|: sequential fp32 accumulation of 1025 products of unit
// vectors (gamma_n = n u ~ 6e-5) plus the fp32 rounding of the operands
constexpr float TAU_FP32_GEMM = 1e-4f;
// TF32 tensor-core pass: operands rounded to nearest TF32 (2^-11 each, products of unit vectors:
// <= 2 * 2^-11 ~ 9.8e-4) plus the fp32 accumulation of 1056 products inside the tensor core
constexpr float TAU_TF32_GEMM = 1.5e-3f;
// 3xTF32 split pass: dropped lo lo^T term and hi + lo representation error (3 * 2^-22 ~ 7e-7, products of unit
// vectors) plus the fp32 accumulation of 3 x 132 MMAs in the tensor core, each assumed to round the running sum
// (<= 1) once by at most one ulp (2^-23): 396 * 2^-23 ~ 4.7e-5 worst case.  tau = 6e-5 keeps a margin over that
// bound (round 1 used 1e-4); measured max |S~ - S| on 10-minute tracks: 1.8e-5 (tests/test_gpu_sim.py asserts the
// bound).  Halving tau halves the width of the near-tie windows k_topk has to settle with exact float64 dots.
constexpr float TAU_3XTF32_GEMM = 6.0e-5f;

// ---------------------------------------------------------------------------------------------
// the period pipeline shared by `original` and the segments of `extended`:
// STFT -> beat spectrum -> period -> median model -> mask + ISTFT
// ---------------------------------------------------------------------------------------------
struct PeriodShape {
    int T = 0, lag_hi = 0, pmax = 0, n_parts = 0, f_per_part = 0;
    // clips longer than one beat transform: blocks of `block_frames` frames, complex partials
    int n_blocks = 1, block_frames = 0;
    size_t bytes_per_item = 0;
};

// Workspace layouts.  Each carve is the single description of a pipeline's buffers for a chunk of g items: run on
// Bump(nullptr) with g = 1 it gives the bytes per item the chunk sizes are computed from, and the runner carves the
// same layout from its workspace.  Every take's count is affine in g with non-negative terms, so a layout for g
// items never needs more than g x (its size for one item): a chunk of G = ws_bytes / bytes_per_item items fits.
// A carve returns its buffers in a braced list, which is evaluated left to right: the members' order is the layout.
struct PeriodBuffers { float2* X; float *P, *psd, *psd_im, *model; int* cert; double* cert_val; };

PeriodBuffers carve_period(Bump& b, const PeriodShape& s, int nch, size_t g) {
    const size_t psd_floats = g * s.n_blocks * s.n_parts * BEAT_L;
    return {b.take<float2>(g * s.T * nch * XPITCH), b.take<float>(g * s.T * PPITCH), b.take<float>(psd_floats),
            s.n_blocks > 1 ? b.take<float>(psd_floats) : nullptr, b.take<float>(g * nch * s.pmax * PPITCH),
            b.take<int>(g * (CERT_MAX + 1)), b.take<double>(g * CERT_MAX * CERT_TSPLIT)};  // period certification
}

void pick_beat_parts(repet_handle* h, int chunk_hint, int floor_parts, int* n_parts, int* f_per_part) {
    // measured on B200 (profiles/r1_sweep2.txt): ~64 partitions of the 1025 rows per clip is the sweet spot
    int want = std::max(floor_parts, std::min(129, (h->sm_count * 6 + chunk_hint - 1) / std::max(1, chunk_hint)));
    if (g_tuning.beat_parts > 0) want = std::min(129, g_tuning.beat_parts);
    *f_per_part = ((NBIN + want - 1) / want + 7) / 8 * 8;
    *n_parts = (NBIN + *f_per_part - 1) / *f_per_part;
}

int period_shape(repet_handle* h, const repet_params* p, int nch, int64_t n_samples, int chunk_hint, PeriodShape* s) {
    const int T = frames_of(n_samples);
    const int lag_hi = std::min(p->period_hi, T / 3);  // repet.py:1265-1267 (quirk Q2)
    if (p->period_lo < 0 || lag_hi <= p->period_lo)
        return fail(h, REPET_E_TOO_SHORT,
                    "attempt to get argmax of an empty sequence (signal too short for the period range)");
    s->T = T;
    s->lag_hi = lag_hi;
    s->pmax = lag_hi;  // period = lag + 1 <= lag_hi
    s->n_blocks = 1;
    s->block_frames = 0;
    if (T + lag_hi - 1 > BEAT_L) {
        if (lag_hi > BEAT_L / 2)
            return fail(h, REPET_E_UNSUPPORTED, "period range above 1024 frames needs a longer beat transform");
        s->block_frames = BEAT_L - lag_hi + 1;
        s->n_blocks = (T + s->block_frames - 1) / s->block_frames;
    }
    pick_beat_parts(h, chunk_hint * s->n_blocks, s->n_blocks > 1 ? 16 : 64, &s->n_parts, &s->f_per_part);
    Bump measure(nullptr);
    carve_period(measure, *s, nch, 1);
    s->bytes_per_item = measure.off;
    return REPET_OK;
}

int pick_frames_per_cta(repet_handle* h, long long total_frames) {
    if (g_tuning.frames_per_cta > 0) return g_tuning.frames_per_cta;
    long long k = total_frames / ((long long)h->sm_count * 8);
    return (int)std::max(4LL, std::min(24LL, k));  // profiles/r1e_sweep.txt: 24 frames per CTA is the sweet spot
}

// gin / gout describe ALL items; the pipeline walks them in workspace-sized chunks.
int period_pipeline(repet_handle* h, const float* audio, Geom gin, float* out, Geom gout, int nch,
                    const repet_params* p, const PeriodShape& s, int32_t* periods_dev, unsigned char* ws,
                    size_t ws_bytes) {
    const int n_items = gin.n_items;
    // carve_period(g) <= g x bytes_per_item (see the layouts above)
    const int G = (int)std::min<size_t>(std::min<size_t>((size_t)n_items, MAX_ITEMS_PER_LAUNCH),
                                        std::max<size_t>(1, ws_bytes / s.bytes_per_item));
    const float scale = (float)(1.0 / ((double)WIN_N * p->cola_gain));
    cudaStream_t st = h->stream;
    const bool blocked = s.n_blocks > 1;
    const int beat_L = blocked ? BEAT_L : beat_transform_length(s.T, s.lag_hi);
    const int total_parts = s.n_blocks * s.n_parts;
    for (int first = 0; first < n_items; first += G) {
        const int g_items = std::min(G, n_items - first);
        Bump bump(ws, ws_bytes);
        const auto [X, P, psd, psd_im, model, cert, cert_val] = carve_period(bump, s, nch, g_items);
        if (!bump.fits()) return fail(h, REPET_E_CUDA, "period pipeline layout exceeds its workspace");
        gin.n_items = gout.n_items = g_items;
        gin.item0 = gout.item0 = first;
        const int K = pick_frames_per_cta(h, (long long)g_items * s.T);
        {
            Timed timed(h, REPET_K_STFT);
            launch_stft(st, audio, gin, nch, window_of(h), tables(h), X, P, P_POWER, K);
        }
        {
            Timed timed(h, REPET_K_BEAT);
            if (blocked)
                launch_beat_blocked(st, P, g_items, s.T, s.block_frames, s.lag_hi, tables(h), psd, psd_im, s.n_blocks,
                                    s.n_parts, s.f_per_part);
            else
                launch_beat(st, P, g_items, s.T, 0, s.T, 0, 1, tables(h), psd, s.n_parts, s.f_per_part, beat_L);
        }
        {
            Timed timed(h, REPET_K_PERIODS, 3);  // k_periods, k_period_certify, k_period_finalize
            launch_periods(st, psd, psd_im, g_items, total_parts, s.T, (double)NBIN, p->period_lo, s.lag_hi, 0, 0, nullptr,
                           0, periods_dev + first, nullptr, cert, beat_L);
            launch_period_certify(st, P, g_items, s.T, 0, s.T, 0, 1, cert, cert_val, periods_dev + first);
        }
        {
            Timed timed(h, REPET_K_MODEL);
            launch_model(st, X, g_items, s.T, nch, periods_dev + first, s.pmax, model);
        }
        {
            Timed timed(h, REPET_K_MASK_ISTFT);
            launch_mask_istft(st, X, gout, nch, periods_dev + first, s.pmax, model, p->cutoff_bins, scale, tables(h), out, K);
        }
    }
    CU(cudaGetLastError());
    return REPET_OK;
}

Geom clip_geom(int n_clips, int nch, int64_t n_samples, int T) {
    Geom g;
    g.n_items = n_clips;
    g.seg_per_clip = 1;
    g.clip_stride = (long long)nch * n_samples;
    g.seg_stride = 0;
    g.chan_stride = n_samples;
    g.first_offset = 0;
    g.S = (int)n_samples;
    g.T = T;
    g.item0 = 0;
    g.frame_shift = 0;
    g.first_frame = 0;
    return g;
}

// ---------------------------------------------------------------------------------------------
// per-kind plans: workspace per clip, integer outputs per clip, and the device-resident runner
// ---------------------------------------------------------------------------------------------
struct Plan {
    int kind = 0, nch = 0;
    int64_t S = 0;
    int T = 0;
    repet_params p;
    PeriodShape whole;  // original; extended when the signal is a single segment
    // extended (repet.py:266-281)
    int n_seg = 1, seg_len = 0, last_len = 0, step = 0;
    PeriodShape seg_main, seg_last;
    // adaptive (repet.py:519-520, 1174-1188)
    int seg_frames = 0, step_frames = 0, n_beat_seg = 0, left_pad = 0, lag_hi = 0, beat_parts = 0, beat_f_per_part = 0;
    // sim / simonline
    int number = 0, distance = 0, buffer_frames = 0;
    // sim: height of the row panels S is formed in (a multiple of 128), 0 = the whole matrix at once
    int panel_rows = 0;
    int ints_per_clip = 1;
    size_t bytes_per_clip = 0;
};

// extended: the segments' backgrounds and periods; the period pipeline of the segments runs in what follows them
struct ExtendedBuffers { float *seg_main, *seg_last; int32_t *per_main, *per_last; };

ExtendedBuffers carve_extended(Bump& b, const Plan& plan, size_t g) {
    const size_t n_main = plan.n_seg - 1;
    return {b.take<float>(g * n_main * plan.nch * plan.seg_len), b.take<float>(g * plan.nch * plan.last_len),
            b.take<int32_t>(g * n_main), b.take<int32_t>(g)};
}

struct AdaptiveBuffers { float2* X; float *P, *psd; int32_t* seg_period; float *model, *Vsq; int* cert; double* cert_val; };

AdaptiveBuffers carve_adaptive(Bump& b, const Plan& plan, size_t g) {
    const size_t T = plan.T, items = g * plan.n_beat_seg, planes = g * plan.nch * T * PPITCH;
    return {b.take<float2>(g * T * plan.nch * XPITCH), b.take<float>(g * T * PPITCH),
            b.take<float>(items * plan.beat_parts * BEAT_L), b.take<int32_t>(items),
            b.take<float>(planes), g_tuning.adaptive_vsq ? b.take<float>(planes) : nullptr,  // model, squared magnitudes
            b.take<int>(items * (CERT_MAX + 1)), b.take<double>(items * CERT_MAX * CERT_TSPLIT)};  // period certification
}

// sim / simonline; `s_floats` is the size of the similarity matrix S (sim only): g whole matrices or one row panel
struct SimBuffers {
    float2* X; float* V; double* An64; int32_t *idx, *cnt; float *model, *Vsq; int32_t* overflow;
    float *An32, *An32lo, *S; int32_t* ovf_cols; unsigned char* ovf_scratch;
};

SimBuffers carve_sim(Bump& b, const Plan& plan, size_t g, size_t s_floats, int sm_count) {
    const size_t T = plan.T, planes = g * plan.nch * T * PPITCH;
    const bool sim = plan.kind == KIND_SIM;
    return {b.take<float2>(g * T * plan.nch * XPITCH), b.take<float>(g * T * PPITCH), b.take<double>(g * T * APITCH64),
            b.take<int32_t>(g * T * plan.number), b.take<int32_t>(g * T),  // idx, cnt
            b.take<float>(planes), plan.number > 32 ? b.take<float>(planes) : nullptr,  // model, squared magnitudes
            b.take<int32_t>(4),  // [overflow flag, candidates, uncertain, neighbour dots]
            sim ? b.take<float>(g * T * KPAD) : nullptr, sim ? b.take<float>(g * T * KPAD) : nullptr,  // An32 hi, lo
            sim ? b.take<float>(s_floats) : nullptr,
            sim ? b.take<int32_t>(g * T) : nullptr,  // columns handed to the exact fallback
            sim ? b.take<unsigned char>(topk_exact_scratch_bytes(plan.T, sm_count)) : nullptr};
}

int make_plan(repet_handle* h, int kind, const repet_params* p, int nch, int64_t S, int chunk_hint, Plan* plan) {
    plan->kind = kind;
    plan->nch = nch;
    plan->S = S;
    plan->T = frames_of(S);
    plan->p = *p;
    int rc;
    if (S > 2147483647LL - 4096) return fail(h, REPET_E_UNSUPPORTED, "more than 2^31 samples per clip");
    if (kind == KIND_ORIGINAL) {
        if ((rc = period_shape(h, p, nch, S, chunk_hint, &plan->whole))) return rc;
        plan->ints_per_clip = 1;
        plan->bytes_per_clip = plan->whole.bytes_per_item;
        return REPET_OK;
    }
    if (kind == KIND_EXTENDED) {
        const int64_t seg_len = p->segment_length, step = p->segment_step;
        if (seg_len <= 0 || step <= 0 || seg_len <= step)
            return fail(h, REPET_E_INVALID_ARG, "segment_length must exceed segment_step (both positive)");
        if (S < seg_len + step) {  // repet.py:271-274: a single segment, i.e. the original REPET
            plan->n_seg = 1;
            if ((rc = period_shape(h, p, nch, S, chunk_hint, &plan->whole))) return rc;
            plan->ints_per_clip = 1;
            plan->bytes_per_clip = plan->whole.bytes_per_item;
            return REPET_OK;
        }
        plan->n_seg = 1 + (int)((S - seg_len) / step);  // repet.py:279-281
        plan->seg_len = (int)seg_len;
        plan->step = (int)step;
        plan->last_len = (int)(S - (int64_t)(plan->n_seg - 1) * step);  // repet.py:320-322
        const int main_hint = chunk_hint * std::max(1, plan->n_seg - 1);
        if ((rc = period_shape(h, p, nch, seg_len, main_hint, &plan->seg_main))) return rc;
        if ((rc = period_shape(h, p, nch, plan->last_len, chunk_hint, &plan->seg_last))) return rc;
        plan->ints_per_clip = plan->n_seg;
        Bump measure(nullptr);
        carve_extended(measure, *plan, 1);
        plan->bytes_per_clip = measure.off + (size_t)(plan->n_seg - 1) * plan->seg_main.bytes_per_item +
                               plan->seg_last.bytes_per_item;
        return REPET_OK;
    }
    if (kind == KIND_ADAPTIVE) {
        const int L = p->segment_length, step = p->segment_step;
        if (L <= 0 || step <= 0) return fail(h, REPET_E_INVALID_ARG, "segment length and step must be positive");
        if (p->filter_order < 1) return fail(h, REPET_E_INVALID_ARG, "filter_order must be at least 1");
        const int lag_hi = std::min(p->period_hi, L / 3);  // n_lags of the beat spectrogram = segment length
        if (p->period_lo < 0 || lag_hi <= p->period_lo)
            return fail(h, REPET_E_TOO_SHORT, "attempt to get argmax of an empty sequence (segment too short for the period range)");
        if (L + lag_hi - 1 > BEAT_L)
            return fail(h, REPET_E_UNSUPPORTED, "segment longer than the single-block beat transform");
        plan->seg_frames = L;
        plan->step_frames = step;
        plan->lag_hi = lag_hi;
        plan->left_pad = (L - 1 + 1) / 2;  // ceil((L-1)/2), repet.py:1182
        plan->n_beat_seg = (plan->T + step - 1) / step;
        pick_beat_parts(h, chunk_hint * plan->n_beat_seg, 4, &plan->beat_parts, &plan->beat_f_per_part);
        plan->ints_per_clip = plan->T;
        Bump measure(nullptr);
        carve_adaptive(measure, *plan, 1);
        plan->bytes_per_clip = measure.off;
        return REPET_OK;
    }
    if (kind == KIND_SIM || kind == KIND_SIMONLINE) {
        if (p->similarity_number < 1) return fail(h, REPET_E_INVALID_ARG, "similarity_number must be at least 1");
        if (p->similarity_distance < 0) return fail(h, REPET_E_INVALID_ARG, "similarity_distance must not be negative");
        plan->number = p->similarity_number;
        plan->distance = p->similarity_distance;
        int T = plan->T;
        if (kind == KIND_SIMONLINE) {
            const int B = p->buffer_frames;
            if (B < 1) return fail(h, REPET_E_INVALID_ARG, "buffer_length must cover at least one frame");
            if (p->online_frame_base < 0) return fail(h, REPET_E_INVALID_ARG, "online_frame_base must not be negative");
            // the reference's warm-up loop multiplies a truncated slice by the window (repet.py:801-804);
            // a window of a longer stream (online_frame_base > 0) has had its warm-up earlier
            if (S < WIN_N || (p->online_frame_base == 0 && (int64_t)(B - 2) * HOP + WIN_N > S))
                return fail(h, REPET_E_INVALID_ARG,
                            "operands could not be broadcast together (signal shorter than the buffer)");
            T = (int)((S - WIN_N + HOP - 1) / HOP) + 1;  // repet.py:781, frames are not centred
            plan->T = T;
            plan->buffer_frames = B;
        }
        plan->ints_per_clip = T * (plan->number + 1);
        auto clip_bytes = [&](size_t s_floats) { Bump m(nullptr); carve_sim(m, *plan, 1, s_floats, h->sm_count); return m.off; };
        size_t s_floats = 0;  // simonline forms no S
        if (kind == KIND_SIM) {
            // S: the whole matrix when it fits the workspace limit beside the linear part; otherwise row panels of
            // as many rows as the limit leaves room for (128 when the linear part alone exceeds it), one track per
            // chunk
            const size_t linear = clip_bytes(0), row_bytes = (size_t)T * sizeof(float);
            const size_t limit = default_ws_limit(h);
            plan->panel_rows = 0;
            if (clip_bytes((size_t)T * T) > limit) {
                const size_t room = limit > linear + 256 ? (limit - linear - 256) / row_bytes : 0;  // 256: alignment
                const int P = (int)std::max<size_t>(128, std::min<size_t>(room, (size_t)T) / 128 * 128);
                if (P < T) plan->panel_rows = P;
            }
            s_floats = (size_t)(plan->panel_rows ? plan->panel_rows : T) * T;
        }
        plan->bytes_per_clip = clip_bytes(s_floats);
        return REPET_OK;
    }
    return fail(h, REPET_E_INVALID_ARG, "unknown driver kind");
}

// idx/cnt (item-major workspace arrays) -> the ABI's per-clip layout [cnt T][idx T*number]
int scatter_lists(repet_handle* h, const Plan& plan, int g, const int32_t* idx, const int32_t* cnt, int32_t* ints) {
    const int T = plan.T;
    const size_t ipc = (size_t)plan.ints_per_clip * sizeof(int32_t);
    CU(cudaMemcpy2DAsync(ints, ipc, cnt, (size_t)T * sizeof(int32_t), (size_t)T * sizeof(int32_t), g,
                         cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaMemcpy2DAsync(ints + T, ipc, idx, (size_t)T * plan.number * sizeof(int32_t),
                         (size_t)T * plan.number * sizeof(int32_t), g, cudaMemcpyDeviceToDevice, h->stream));
    return REPET_OK;
}

int run_sim(repet_handle* h, const Plan& plan, const float* audio, int n_clips, float* out, int32_t* ints,
            unsigned char* ws, size_t ws_bytes) {
    const int nch = plan.nch, T = plan.T;
    const bool online = plan.kind == KIND_SIMONLINE;
    const int P = online ? 0 : plan.panel_rows;  // row panels: one track per chunk
    // carve_sim(g) <= g x bytes_per_clip (see the layouts above)
    const int G = P ? 1 : (int)std::min<size_t>(std::min<size_t>((size_t)n_clips, MAX_ITEMS_PER_LAUNCH / 2),
                                                std::max<size_t>(1, ws_bytes / plan.bytes_per_clip));
    const float scale = (float)(1.0 / ((double)WIN_N * plan.p.cola_gain));
    const int fast = g_tuning.simgemm_tc;
    cudaStream_t st = h->stream;
    for (int clip0 = 0; clip0 < n_clips; clip0 += G) {
        const int g = std::min(G, n_clips - clip0);
        Bump bump(ws, ws_bytes);
        const auto [X, V, An64, idx, cnt, model, Vsq, overflow, An32, An32lo, S, ovf_cols, ovf_scratch] =
            carve_sim(bump, plan, g, (P ? (size_t)P : (size_t)g * T) * T, h->sm_count);
        if (!bump.fits()) return fail(h, REPET_E_CUDA, "sim layout exceeds its workspace");
        Geom geom = clip_geom(g, nch, plan.S, T);
        geom.first_offset = (long long)clip0 * geom.clip_stride;
        if (online) {
            geom.frame_shift = 1;
            geom.first_frame = std::max(0, plan.buffer_frames - 1 - plan.p.online_frame_base);
        }
        const int K = pick_frames_per_cta(h, (long long)g * T);
        const bool frames64 = g_tuning.sim_frames64 != 0;
        {
            Timed timed(h, REPET_K_STFT);
            // long lists gather squared magnitudes: k_stft writes that plane itself (round 1 ran a separate k_sqmag pass)
            launch_stft(st, audio, geom, nch, window_of(h), tables(h), X, frames64 ? nullptr : V, P_MAGNITUDE, K, Vsq);
        }
        {
            Timed timed(h, REPET_K_NORMALIZE);
            if (frames64)
                // the similarity operand comes from a float64 transform of the samples (of the float64 samples
                // themselves when a *_f64 entry point holds them): integer decisions as in the reference
                launch_frames64(st, audio, n_clips == 1 ? h->f64_audio : nullptr, geom, nch, h->win[WIN_SLOT].window64,
                                h->win[WIN_SLOT].tw64, An64, An32, fast >= 2 ? An32lo : nullptr, fast ? 1 : 0);
            else
                launch_normalize(st, V, g * T, An64, An32, fast >= 2 ? An32lo : nullptr, fast ? 1 : 0);
        }
        CU(cudaMemsetAsync(cnt, 0, (size_t)g * T * sizeof(int32_t), st));
        if (online) {
            Timed timed(h, REPET_K_TOPK);
            if (launch_online_select(st, An64, g, T, plan.buffer_frames, plan.p.online_frame_base,
                                     plan.p.similarity_threshold, plan.distance, plan.number, idx, cnt))
                return fail(h, REPET_E_UNSUPPORTED, "buffer_length too long for the online selection kernel on this device");
        } else {
            const float tau = fast >= 2 ? TAU_3XTF32_GEMM : (fast ? TAU_TF32_GEMM : TAU_FP32_GEMM);
            const double thr = plan.p.similarity_threshold;
            const float* lo = fast >= 2 ? An32lo : nullptr;
            // rows [r0, r0 + rows) of S, then the columns they settle: one range covers the whole matrices of the g
            // tracks (the GEMM forms their upper triangles), or ranges of P rows cover one track panel by panel.  The
            // columns k_topk queues for the exact fallback accumulate over the ranges and are settled once at the end
            CU(cudaMemsetAsync(overflow, 0, 4 * sizeof(int32_t), st));
            const int range = P ? P : T;
            for (int r0 = 0; r0 < T; r0 += range) {
                const int rows = std::min(range, T - r0);
                {
                    Timed timed(h, REPET_K_SIMGEMM);
                    if (!fast)
                        P ? launch_selfsim_simt_panel(st, An32, T, r0, rows, S) : launch_selfsim_simt(st, An32, g, T, S);
                    else if (P ? launch_selfsim_tc_panel(st, An32, lo, T, r0, rows, S, h->sm_count)
                               : launch_selfsim_tc(st, An32, lo, g, T, S, h->sm_count))
                        return fail(h, REPET_E_CUDA, "tensor-map encode failed for the similarity GEMM");
                }
                Timed timed(h, REPET_K_TOPK);
                if (launch_topk_propose(st, S, r0, rows, An64, g, T, tau, thr, plan.distance, plan.number, idx, cnt,
                                        overflow, ovf_cols))
                    return fail(h, REPET_E_UNSUPPORTED, "similarity_distance too large for the in-shared-memory similarity row");
            }
            Timed timed(h, REPET_K_TOPK);
            launch_topk_exact(st, An64, T, thr, plan.distance, plan.number, overflow, ovf_cols, ovf_scratch, idx, cnt,
                              h->sm_count);
        }
        {
            Timed timed(h, REPET_K_MODEL, Vsq ? 3 : 2);  // k_simmodel, [k_simmodel_large,] k_simmodel_nyquist
            if (launch_simmodel(st, X, Vsq, g, T, nch, idx, cnt, plan.number, geom.first_frame, model))
                return fail(h, REPET_E_UNSUPPORTED, "similarity_number too large for the shared-memory median");
        }
        {
            Timed timed(h, REPET_K_MASK_ISTFT);
            launch_mask_istft(st, X, geom, nch, nullptr, T, model, plan.p.cutoff_bins, scale, tables(h), out, K);
        }
        int rc = scatter_lists(h, plan, g, idx, cnt, ints + (size_t)clip0 * plan.ints_per_clip);
        if (rc) return rc;
        if (!online && getenv("REPET_DEBUG_TOPK")) {  // statistics only: the stream is not synchronised otherwise
            int32_t flag[4] = {0, 0, 0, 0};
            CU(cudaMemcpyAsync(flag, overflow, sizeof(flag), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            fprintf(stderr, "k_topk: %d columns (%d through the exact fallback), %d candidates, %d uncertain, %d near-tie "
                            "neighbour dots; %d row panels of %d\n", g * T, flag[0], flag[1], flag[2], flag[3],
                    P ? (T + P - 1) / P : 1, P ? P : T);
        }
    }
    CU(cudaGetLastError());
    return REPET_OK;
}

int run_extended(repet_handle* h, const Plan& plan, const float* audio, int n_clips, float* out, int32_t* ints,
                 unsigned char* ws, size_t ws_bytes) {
    const int nch = plan.nch;
    const int n_main = plan.n_seg - 1;
    // carve_extended(g) plus the period layouts of its g x n_seg segments <= g x bytes_per_clip (see the layouts above)
    const int G = (int)std::min<size_t>((size_t)n_clips, std::max<size_t>(1, ws_bytes / plan.bytes_per_clip));
    cudaStream_t st = h->stream;
    for (int clip0 = 0; clip0 < n_clips; clip0 += G) {
        const int g = std::min(G, n_clips - clip0);
        Bump bump(ws, ws_bytes);
        const auto [seg_main, seg_last, per_main, per_last] = carve_extended(bump, plan, g);
        if (!bump.fits()) return fail(h, REPET_E_CUDA, "extended layout exceeds its workspace");
        unsigned char* pws = ws + bump.off;
        const size_t pws_bytes = ws_bytes - bump.off;
        const float* a = audio + (size_t)clip0 * nch * plan.S;
        // equally long segments j < n_seg-1 (repet.py:318-319)
        Geom gin = clip_geom(g * n_main, nch, plan.S, plan.seg_main.T);
        gin.seg_per_clip = n_main;
        gin.seg_stride = plan.step;
        gin.S = plan.seg_len;
        Geom gout = clip_geom(g * n_main, nch, plan.seg_len, plan.seg_main.T);
        int rc = period_pipeline(h, a, gin, seg_main, gout, nch, &plan.p, plan.seg_main, per_main, pws, pws_bytes);
        if (rc) return rc;
        // the last segment takes the remainder (repet.py:320-322)
        gin = clip_geom(g, nch, plan.S, plan.seg_last.T);
        gin.first_offset = (long long)n_main * plan.step;
        gin.S = plan.last_len;
        gout = clip_geom(g, nch, plan.last_len, plan.seg_last.T);
        rc = period_pipeline(h, a, gin, seg_last, gout, nch, &plan.p, plan.seg_last, per_last, pws, pws_bytes);
        if (rc) return rc;
        {
            Timed timed(h, REPET_K_XFADE);
            launch_xfade(st, seg_main, seg_last, g, plan.n_seg, plan.seg_len, plan.last_len, plan.step, nch, plan.S,
                         out + (size_t)clip0 * nch * plan.S);
        }
        int32_t* dst = ints + (size_t)clip0 * plan.n_seg;
        CU(cudaMemcpy2DAsync(dst, plan.n_seg * sizeof(int32_t), per_main, n_main * sizeof(int32_t),
                             n_main * sizeof(int32_t), g, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpy2DAsync(dst + n_main, plan.n_seg * sizeof(int32_t), per_last, sizeof(int32_t), sizeof(int32_t), g,
                             cudaMemcpyDeviceToDevice, st));
    }
    CU(cudaGetLastError());
    return REPET_OK;
}

int run_adaptive(repet_handle* h, const Plan& plan, const float* audio, int n_clips, float* out, int32_t* ints,
                 unsigned char* ws, size_t ws_bytes) {
    const int nch = plan.nch, T = plan.T;
    // grid.y carries clips x beat segments in k_beat: keep it below 65535
    const size_t grid_cap = std::max<size_t>(1, 60000 / (size_t)std::max(1, plan.n_beat_seg));
    // carve_adaptive(g) <= g x bytes_per_clip (see the layouts above)
    const int G = (int)std::min<size_t>(std::min<size_t>((size_t)n_clips, std::min<size_t>(MAX_ITEMS_PER_LAUNCH / 2, grid_cap)),
                                        std::max<size_t>(1, ws_bytes / plan.bytes_per_clip));
    const float scale = (float)(1.0 / ((double)WIN_N * plan.p.cola_gain));
    cudaStream_t st = h->stream;
    for (int clip0 = 0; clip0 < n_clips; clip0 += G) {
        const int g = std::min(G, n_clips - clip0);
        Bump bump(ws, ws_bytes);
        const auto [X, P, psd, seg_period, model, Vsq, cert, cert_val] = carve_adaptive(bump, plan, g);
        if (!bump.fits()) return fail(h, REPET_E_CUDA, "adaptive layout exceeds its workspace");
        int32_t* frame_period = ints + (size_t)clip0 * T;
        Geom geom = clip_geom(g, nch, plan.S, T);
        geom.first_offset = (long long)clip0 * geom.clip_stride;
        const int K = pick_frames_per_cta(h, (long long)g * T);
        const int beat_L = beat_transform_length(plan.seg_frames, plan.lag_hi);
        {
            Timed timed(h, REPET_K_STFT);
            launch_stft(st, audio, geom, nch, window_of(h), tables(h), X, P, P_POWER, K, Vsq);
        }
        {
            // segment i spans frames [i - left_pad, i - left_pad + L) (zero outside), repet.py:1177-1198
            Timed timed(h, REPET_K_BEAT);
            launch_beat(st, P, g, T, -plan.left_pad, plan.seg_frames, plan.step_frames, plan.n_beat_seg, tables(h), psd,
                        plan.beat_parts, plan.beat_f_per_part, beat_L);
        }
        {
            Timed timed(h, REPET_K_PERIODS, 3);
            launch_periods(st, psd, nullptr, g * plan.n_beat_seg, plan.beat_parts, plan.seg_frames, (double)NBIN, plan.p.period_lo,
                           plan.lag_hi, 0, 0, nullptr, 0, seg_period, nullptr, cert, beat_L);
            launch_period_certify(st, P, g * plan.n_beat_seg, T, -plan.left_pad, plan.seg_frames, plan.step_frames,
                                  plan.n_beat_seg, cert, cert_val, seg_period);
        }
        {
            Timed timed(h, REPET_K_MODEL, 2);
            launch_expand_periods(st, seg_period, g, plan.n_beat_seg, T, plan.step_frames, plan.p.period_lo, frame_period);
            launch_adaptive_model(st, X, g, T, nch, frame_period, plan.p.filter_order, model, Vsq);
        }
        {
            Timed timed(h, REPET_K_MASK_ISTFT);
            launch_mask_istft(st, X, geom, nch, nullptr, T, model, plan.p.cutoff_bins, scale, tables(h), out, K);
        }
    }
    CU(cudaGetLastError());
    return REPET_OK;
}

// device-resident run of `n_clips` clips starting at `audio` / `out` / `ints`
int run_plan(repet_handle* h, const Plan& plan, const float* audio, int n_clips, float* out, int32_t* ints,
             unsigned char* ws, size_t ws_bytes) {
    if (plan.kind == KIND_ORIGINAL || (plan.kind == KIND_EXTENDED && plan.n_seg == 1)) {
        Geom g = clip_geom(n_clips, plan.nch, plan.S, plan.whole.T);
        return period_pipeline(h, audio, g, out, g, plan.nch, &plan.p, plan.whole, ints, ws, ws_bytes);
    }
    if (plan.kind == KIND_EXTENDED) return run_extended(h, plan, audio, n_clips, out, ints, ws, ws_bytes);
    if (plan.kind == KIND_ADAPTIVE) return run_adaptive(h, plan, audio, n_clips, out, ints, ws, ws_bytes);
    return run_sim(h, plan, audio, n_clips, out, ints, ws, ws_bytes);
}

int chunk_clips(repet_handle* h, const Plan& plan, int n_clips) {
    if (plan.panel_rows) return std::min(n_clips, 1);  // a track in row panels runs alone
    const size_t limit = default_ws_limit(h);
    return (int)std::min<size_t>((size_t)n_clips, std::max<size_t>(1, limit / plan.bytes_per_clip));
}

// ---------------------------------------------------------------------------------------------
// the three calling conventions
// ---------------------------------------------------------------------------------------------
int batch_dev(repet_handle* h, int kind, const float* audio, int n_clips, int nch, int64_t S, const repet_params* p,
              float* background, int32_t* ints_dev, int32_t* ints_host, int* ints_per_clip_out) {
    int rc = check_common(h, p, nch);
    if (rc) return rc;
    if (!audio || !background || n_clips < 0 || S < 0) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    Plan plan;
    if ((rc = make_plan(h, kind, p, nch, S, std::max(1, std::min(n_clips, 64)), &plan))) return rc;
    int G = chunk_clips(h, plan, n_clips);
    if ((rc = make_plan(h, kind, p, nch, S, std::max(1, G), &plan))) return rc;
    if (ints_per_clip_out) *ints_per_clip_out = plan.ints_per_clip;
    if (n_clips == 0) return REPET_OK;
    G = chunk_clips(h, plan, n_clips);
    const size_t ws_bytes = (size_t)G * plan.bytes_per_clip;
    int32_t* ints = ints_dev; unsigned char* ws;
    rc = carve_arena(h, [&](Bump& b) {
        if (!ints_dev) ints = b.take<int32_t>((size_t)n_clips * plan.ints_per_clip);
        ws = b.take<unsigned char>(ws_bytes);
    });
    if (rc) return rc;
    rc = run_plan(h, plan, audio, n_clips, background, ints, ws, ws_bytes);
    if (rc) return rc;
    if (ints_host) {
        CU(cudaMemcpyAsync(ints_host, ints, (size_t)n_clips * plan.ints_per_clip * sizeof(int32_t), cudaMemcpyDeviceToHost,
                           h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return REPET_OK;
}

// Host buffers in, host buffers out: copies chunked and overlapped with the compute on three streams.
// Formats (include/repet_b200.h): REPET_FMT_F32_PLANAR [clip][channel][sample] fp32, or REPET_FMT_PCM16, int16 PCM
// in WAV order [clip][sample][channel] (2 bytes per sample over PCIe instead of 4).  PCM input is normalised by
// 2^15 as repet.wavread does (repet.py:929) and made planar on the device; PCM output is round(y * 2^15)
// saturated to int16, interleaved on the device.
int batch_host(repet_handle* h, int kind, const void* audio_any, int in_fmt, int n_clips, int nch, int64_t S,
               const repet_params* p, void* background_any, int out_fmt, int32_t* ints_host) {
    int rc = check_common(h, p, nch);
    if (rc) return rc;
    if (!audio_any || !background_any || n_clips < 0 || S < 0) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    if ((in_fmt != REPET_FMT_F32_PLANAR && in_fmt != REPET_FMT_PCM16) ||
        (out_fmt != REPET_FMT_F32_PLANAR && out_fmt != REPET_FMT_PCM16))
        return fail(h, REPET_E_INVALID_ARG, "unknown sample format");
    if (n_clips == 0) return REPET_OK;
    CU(cudaSetDevice(h->device));
    const bool pcm_in = in_fmt == REPET_FMT_PCM16, pcm_out = out_fmt == REPET_FMT_PCM16;
    const unsigned char* audio = static_cast<const unsigned char*>(audio_any);
    unsigned char* background = static_cast<unsigned char*>(background_any);
    const size_t clip_elems = (size_t)nch * (size_t)S;
    const size_t clip_bytes = clip_elems * sizeof(float);
    const size_t in_clip_bytes = clip_elems * (pcm_in ? sizeof(int16_t) : sizeof(float));
    const size_t out_clip_bytes = clip_elems * (pcm_out ? sizeof(int16_t) : sizeof(float));
    // copy granularity: about copy_chunk_mb of fp32 samples per slot, two slots in flight in each direction.  Small
    // slots shorten the fill and drain of the H2D -> compute -> D2H pipeline (the first upload and the last download
    // overlap nothing); the kernels have ~10x headroom over PCIe, so their efficiency on small chunks does not matter
    const size_t slot_target = (size_t)std::max(8, g_tuning.copy_chunk_mb) << 20;
    int Gc = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_clips, slot_target / std::max<size_t>(1, clip_bytes)));
    Plan plan;
    if ((rc = make_plan(h, kind, p, nch, S, Gc, &plan))) return rc;
    const int Gw = std::min(Gc, chunk_clips(h, plan, Gc));
    const size_t ws_bytes = (size_t)Gw * plan.bytes_per_clip;
    int32_t* ints; unsigned char *in_slot[2], *out_slot[2], *ws; float *in32 = nullptr, *out32 = nullptr;
    rc = carve_arena(h, [&](Bump& b) {
        ints = b.take<int32_t>((size_t)n_clips * plan.ints_per_clip);
        for (unsigned char*& slot : in_slot) slot = b.take<unsigned char>((size_t)Gc * in_clip_bytes);
        for (unsigned char*& slot : out_slot) slot = b.take<unsigned char>((size_t)Gc * out_clip_bytes);
        if (pcm_in) in32 = b.take<float>((size_t)Gc * clip_elems);
        if (pcm_out) out32 = b.take<float>((size_t)Gc * clip_elems);
        ws = b.take<unsigned char>(ws_bytes);
    });
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));  // the arena must be idle before the copy streams touch it
    auto pipeline = [&]() -> int {
        int n_chunks = 0;
        for (int first = 0; first < n_clips; first += Gc, ++n_chunks) {
            const int s = n_chunks & 1;
            const int g = std::min(Gc, n_clips - first);
            if (n_chunks >= 2) CU(cudaStreamWaitEvent(h->h2d_stream, h->ev_compute[s], 0));  // slot's input consumed
            CU(cudaMemcpyAsync(in_slot[s], audio + (size_t)first * in_clip_bytes, (size_t)g * in_clip_bytes,
                               cudaMemcpyHostToDevice, h->h2d_stream));
            CU(cudaEventRecord(h->ev_h2d[s], h->h2d_stream));
            CU(cudaStreamWaitEvent(h->stream, h->ev_h2d[s], 0));
            if (n_chunks >= 2) CU(cudaStreamWaitEvent(h->stream, h->ev_d2h[s], 0));  // slot's output drained
            const float* chunk_in = reinterpret_cast<const float*>(in_slot[s]);
            if (pcm_in) {
                Timed timed(h, REPET_K_CONVERT);
                launch_pcm16_to_planar(h->stream, reinterpret_cast<const int16_t*>(in_slot[s]), g, S, nch, in32);
                chunk_in = in32;
            }
            float* chunk_out = pcm_out ? out32 : reinterpret_cast<float*>(out_slot[s]);
            int rc2 = run_plan(h, plan, chunk_in, g, chunk_out, ints + (size_t)first * plan.ints_per_clip, ws, ws_bytes);
            if (rc2) return rc2;
            if (pcm_out) {
                Timed timed(h, REPET_K_CONVERT);
                launch_planar_to_pcm16(h->stream, out32, g, S, nch, reinterpret_cast<int16_t*>(out_slot[s]));
            }
            CU(cudaEventRecord(h->ev_compute[s], h->stream));
            CU(cudaStreamWaitEvent(h->d2h_stream, h->ev_compute[s], 0));
            CU(cudaMemcpyAsync(background + (size_t)first * out_clip_bytes, out_slot[s], (size_t)g * out_clip_bytes,
                               cudaMemcpyDeviceToHost, h->d2h_stream));
            CU(cudaEventRecord(h->ev_d2h[s], h->d2h_stream));
        }
        if (ints_host)
            CU(cudaMemcpyAsync(ints_host, ints, (size_t)n_clips * plan.ints_per_clip * sizeof(int32_t),
                               cudaMemcpyDeviceToHost, h->stream));
        return REPET_OK;
    };
    rc = pipeline();
    // also on the error path: copies from / into the caller's buffers may still be in flight, and the caller is
    // free to release them as soon as this returns
    const cudaError_t e1 = cudaStreamSynchronize(h->h2d_stream), e2 = cudaStreamSynchronize(h->stream),
                      e3 = cudaStreamSynchronize(h->d2h_stream);
    if (rc) return rc;
    CU(e1);
    CU(e2);
    CU(e3);
    return REPET_OK;
}

// |STFT(mean_c x)|[0:F] of every clip (the display spectrogram of README.md:79-81), device resident:
// spectrogram [n_clips][T][PPITCH] fp32
int spectrogram_dev(repet_handle* h, const float* audio, int n_clips, int nch, int64_t S, const repet_params* p,
                    float* spectrogram) {
    int rc = check_common(h, p, nch);
    if (rc) return rc;
    if (!audio || !spectrogram || n_clips < 0 || S < 1) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    if (S > 2147483647LL - 4096) return fail(h, REPET_E_UNSUPPORTED, "more than 2^31 samples per clip");
    CU(cudaSetDevice(h->device));
    const int T = frames_of(S);
    for (int first = 0; first < n_clips; first += MAX_ITEMS_PER_LAUNCH) {
        Geom g = clip_geom(std::min(MAX_ITEMS_PER_LAUNCH, n_clips - first), nch, S, T);
        g.first_offset = (long long)first * g.clip_stride;
        Timed timed(h, REPET_K_STFT);
        launch_stft(h->stream, audio, g, nch, window_of(h), tables(h), nullptr, spectrogram + (size_t)first * T * PPITCH,
                    P_MIXDOWN, pick_frames_per_cta(h, (long long)g.n_items * T));
    }
    CU(cudaGetLastError());
    return REPET_OK;
}

// float64 (samples, channels) in and out -- the reference's own convention (repet.py:73-77).
// Optional by-products of the buffers already resident (README.md:64-81): the foreground
// (audio - background) and the display spectrograms of mixture, background and foreground,
// spectrograms [3][T][PPITCH] fp32 on the host.
int single_f64(repet_handle* h, int kind, const double* audio, int64_t S, int nch, const repet_params* p,
               double* background, int32_t* ints_host, int ints_capacity, double* foreground = nullptr,
               float* spectrograms = nullptr) {
    int rc = check_common(h, p, nch);
    if (rc) return rc;
    if (!audio || !background || S < 0) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    Plan plan;
    if ((rc = make_plan(h, kind, p, nch, S, 1, &plan))) return rc;
    if (ints_host && ints_capacity < plan.ints_per_clip)
        return fail(h, REPET_E_INVALID_ARG, "integer output buffer too small");
    const size_t n = (size_t)S * nch;
    const int T_spec = frames_of(S);
    const size_t spec_elems = spectrograms ? (size_t)3 * T_spec * PPITCH : 0;
    int32_t* ints; double* d64; float *in32, *out32, *fg32, *spec; unsigned char* ws;
    rc = carve_arena(h, [&](Bump& b) {
        ints = b.take<int32_t>(plan.ints_per_clip);
        d64 = b.take<double>(n);
        in32 = b.take<float>(n);
        out32 = b.take<float>(n);
        fg32 = b.take<float>(n);
        spec = b.take<float>(spec_elems);
        ws = b.take<unsigned char>(plan.bytes_per_clip);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(d64, audio, n * sizeof(double), cudaMemcpyHostToDevice, st));
    {
        Timed timed(h, REPET_K_CONVERT);
        launch_f64_interleaved_to_planar(st, d64, S, nch, in32);
    }
    h->f64_audio = d64;
    rc = run_plan(h, plan, in32, 1, out32, ints, ws, plan.bytes_per_clip);
    h->f64_audio = nullptr;
    if (rc) return rc;
    if (foreground || spectrograms) {
        Timed timed(h, REPET_K_CONVERT);
        launch_foreground(st, in32, out32, (long long)n, fg32);
    }
    if (spectrograms) {
        const float* sources[3] = {in32, out32, fg32};
        for (int i = 0; i < 3; ++i)
            if ((rc = spectrogram_dev(h, sources[i], 1, nch, S, p, spec + (size_t)i * T_spec * PPITCH))) return rc;
        CU(cudaMemcpyAsync(spectrograms, spec, spec_elems * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    {
        Timed timed(h, REPET_K_CONVERT);
        launch_planar_to_f64_interleaved(st, out32, S, nch, d64);
    }
    CU(cudaMemcpyAsync(background, d64, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (foreground) {
        // stream order: the copy above has read d64 before it is overwritten
        Timed timed(h, REPET_K_CONVERT);
        launch_planar_to_f64_interleaved(st, fg32, S, nch, d64);
        CU(cudaMemcpyAsync(foreground, d64, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    if (ints_host)
        CU(cudaMemcpyAsync(ints_host, ints, (size_t)plan.ints_per_clip * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return REPET_OK;
}

// float64 (samples, channels) in and out, both already on the DEVICE; stream-ordered, no synchronisation.
// The stateful simonline stream keeps its sample history in device memory and runs its windows through here.
int single_f64_dev(repet_handle* h, int kind, const double* d_audio, int64_t S, int nch, const repet_params* p,
                   double* d_background) {
    int rc = check_common(h, p, nch);
    if (rc) return rc;
    if (!d_audio || !d_background || S < 0) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    CU(cudaSetDevice(h->device));
    Plan plan;
    if ((rc = make_plan(h, kind, p, nch, S, 1, &plan))) return rc;
    const size_t n = (size_t)S * nch;
    int32_t* ints; float *in32, *out32; unsigned char* ws;
    rc = carve_arena(h, [&](Bump& b) {
        ints = b.take<int32_t>(plan.ints_per_clip);
        in32 = b.take<float>(n);
        out32 = b.take<float>(n);
        ws = b.take<unsigned char>(plan.bytes_per_clip);
    });
    if (rc) return rc;
    cudaStream_t st = h->stream;
    {
        Timed timed(h, REPET_K_CONVERT);
        launch_f64_interleaved_to_planar(st, d_audio, S, nch, in32);
    }
    h->f64_audio = d_audio;
    rc = run_plan(h, plan, in32, 1, out32, ints, ws, plan.bytes_per_clip);
    h->f64_audio = nullptr;
    if (rc) return rc;
    {
        Timed timed(h, REPET_K_CONVERT);
        launch_planar_to_f64_interleaved(st, out32, S, nch, d_background);
    }
    CU(cudaGetLastError());
    return REPET_OK;
}

}  // namespace

namespace repet {

int drv_single_f64_dev(repet_handle* h, int kind, const double* d_audio, int64_t n_samples, int n_channels,
                       const repet_params* p, double* d_background) {
    return single_f64_dev(h, kind, d_audio, n_samples, n_channels, p, d_background);
}
int drv_batch_dev(repet_handle* h, int kind, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                  const repet_params* p, float* background, int32_t* ints_dev, int32_t* ints_host) {
    return batch_dev(h, kind, audio, n_clips, n_channels, n_samples, p, background, ints_dev, ints_host, nullptr);
}
int drv_batch_host(repet_handle* h, int kind, const void* audio, int in_format, int n_clips, int n_channels,
                   int64_t n_samples, const repet_params* p, void* background, int out_format, int32_t* ints) {
    return batch_host(h, kind, audio, in_format, n_clips, n_channels, n_samples, p, background, out_format, ints);
}
int drv_single_f64(repet_handle* h, int kind, const double* audio, int64_t n_samples, int n_channels,
                   const repet_params* p, double* background, int32_t* ints, int64_t ints_capacity) {
    return single_f64(h, kind, audio, n_samples, n_channels, p, background, ints,
                      (int)std::min<int64_t>(ints_capacity, INT32_MAX));
}
int drv_separate_f64(repet_handle* h, int kind, const double* audio, int64_t n_samples, int n_channels,
                     const repet_params* p, double* background, double* foreground, float* spectrograms, int32_t* ints,
                     int64_t ints_capacity) {
    return single_f64(h, kind, audio, n_samples, n_channels, p, background, ints,
                      (int)std::min<int64_t>(ints_capacity, INT32_MAX), foreground, spectrograms);
}
int drv_spectrogram_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                        const repet_params* p, float* spectrogram) {
    return spectrogram_dev(h, audio, n_clips, n_channels, n_samples, p, spectrogram);
}
int drv_foreground_dev(repet_handle* h, const float* audio, const float* background, int64_t n, float* foreground) {
    if (!h || !audio || !background || !foreground || n < 0) return fail(h, REPET_E_INVALID_ARG, "bad buffer or size");
    if (((uintptr_t)audio | (uintptr_t)background | (uintptr_t)foreground) & 15)
        return fail(h, REPET_E_INVALID_ARG, "buffers must be 16-byte aligned");
    CU(cudaSetDevice(h->device));
    Timed timed(h, REPET_K_CONVERT);
    launch_foreground(h->stream, audio, background, (long long)n, foreground);
    CU(cudaGetLastError());
    return REPET_OK;
}

}  // namespace repet
