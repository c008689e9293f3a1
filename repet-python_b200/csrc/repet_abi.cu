// C ABI of librepet_b200.so (declared in include/repet_b200.h): handle lifetime, transform tables,
// profiling, and the dispatch of every driver / helper entry point to the instantiation compiled
// for the window length in use (repet_drivers.cu, repet_helpers.cu; 512, 1024 and 2048 points).
// This file is compiled once; it uses nothing of repet_kernels.cuh that depends on the length.
#include "repet_internal.h"

#include <cmath>
#include <cstdio>
#include <cstring>

using repet::fail;

namespace {

const double kPi = 3.14159265358979323846264338327950288;
const int kWindowLengths[3] = {512, 1024, 2048};

const char* kKernelNames[REPET_NUM_KERNELS] = {"k_stft",    "k_beat",  "k_periods",   "k_model",   "k_mask_istft", "k_convert",
                                               "k_xfade",   "k_normalize", "k_simgemm", "k_topk",       "k_other10", "k_other11"};

}  // namespace

repet_tuning g_repet_tuning;

namespace repet_w512 { const repet_entry* entry_table(); }
namespace repet_w1024 { const repet_entry* entry_table(); }
namespace repet_w2048 { const repet_entry* entry_table(); }

namespace {

int slot_of(int window_n) { return window_n == 512 ? 0 : (window_n == 1024 ? 1 : (window_n == 2048 ? 2 : -1)); }

const repet_entry* entry_of_slot(int slot) {
    switch (slot) {
        case 0: return repet_w512::entry_table();
        case 1: return repet_w1024::entry_table();
        case 2: return repet_w2048::entry_table();
    }
    return nullptr;
}

// drivers: the instantiation follows repet_params.window_length
const repet_entry* entry_for(repet_handle* h, const repet_params* p) {
    if (!h) return nullptr;
    if (!p) {
        h->err = "params is null";
        return nullptr;
    }
    const repet_entry* e = entry_of_slot(slot_of(p->window_length));
    if (!e) h->err = "window_length must be 512, 1024 or 2048 (sampling frequencies up to 51.2 kHz)";
    return e;
}

// helpers that transform or consume half spectra: the window set last decides
const repet_entry* entry_current(repet_handle* h) {
    if (!h) return nullptr;
    const repet_entry* e = entry_of_slot(slot_of(h->window_n));
    if (!e) h->err = "repet_set_window has not been called";
    return e;
}

// helpers on zero-padded rows (beat spectra, similarities): the smallest instantiation that holds n_rows
const repet_entry* entry_rows(repet_handle* h, int n_rows) {
    if (!h) return nullptr;
    return entry_of_slot(n_rows <= 257 ? 0 : (n_rows <= 513 ? 1 : 2));
}

enum Kind { KIND_ORIGINAL = 0, KIND_EXTENDED = 1, KIND_ADAPTIVE = 2, KIND_SIM = 3, KIND_SIMONLINE = 4 };

}  // namespace


extern "C" {

const char* repet_version(void) { return "repet_b200 0.1 (sm_100a)"; }

int repet_create(int device, repet_handle** out) {
    if (!out) return REPET_E_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return REPET_E_CUDA;
    repet_handle* h = new repet_handle();
    h->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_compute[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_d2h[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0)
            h->sm_count = sms;
    }
    // transform tables in double precision, rounded once to fp32 (fft_core.cuh: N = 16 x R2 x 8)
    for (int s = 0; s < 3 && e == cudaSuccess; ++s) {
        const int n = kWindowLengths[s], threads = n / 16, r2 = threads / 8;
        std::vector<float2> tw1((size_t)15 * threads), tw2((size_t)r2 * 8);
        for (int k1 = 1; k1 < 16; ++k1)
            for (int m = 0; m < threads; ++m) {
                const double a = -2.0 * kPi * (double)((m * k1) % n) / (double)n;
                tw1[(size_t)(k1 - 1) * threads + m] = make_float2((float)std::cos(a), (float)std::sin(a));
            }
        for (int k2 = 0; k2 < r2; ++k2)
            for (int m2 = 0; m2 < 8; ++m2) {
                const double a = -2.0 * kPi * (double)((m2 * k2) % threads) / (double)threads;
                tw2[(size_t)k2 * 8 + m2] = make_float2((float)std::cos(a), (float)std::sin(a));
            }
        repet_handle::WindowSlot& w = h->win[s];
        e = cudaMalloc(&w.tw1, tw1.size() * sizeof(float2));
        if (e == cudaSuccess) e = cudaMalloc(&w.tw2, tw2.size() * sizeof(float2));
        if (e == cudaSuccess) e = cudaMalloc(&w.window, n * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&w.window64, n * sizeof(double));
        if (e == cudaSuccess) e = cudaMalloc(&w.tw64, (n / 2) * sizeof(double2));
        if (e == cudaSuccess) {
            std::vector<double2> tw64(n / 2);
            for (int i = 0; i < n / 2; ++i) {
                // exact octant symmetries keep cos/sin of the table consistent to the last bit
                const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)i / (long double)n;
                tw64[i] = make_double2((double)cosl(a), (double)sinl(a));
            }
            e = cudaMemcpy(w.tw64, tw64.data(), tw64.size() * sizeof(double2), cudaMemcpyHostToDevice);
        }
        if (e == cudaSuccess) e = cudaMemcpy(w.tw1, tw1.data(), tw1.size() * sizeof(float2), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(w.tw2, tw2.data(), tw2.size() * sizeof(float2), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        repet_destroy(h);
        return REPET_E_CUDA;
    }
    h->stream = h->own_stream;
    *out = h;
    return REPET_OK;
}

int repet_destroy(repet_handle* h) {
    if (!h) return REPET_OK;
    cudaSetDevice(h->device);
    if (h->own_stream) cudaStreamSynchronize(h->own_stream);
    cudaFree(h->arena);
    for (int s = 0; s < 3; ++s) {
        cudaFree(h->win[s].tw1);
        cudaFree(h->win[s].tw2);
        cudaFree(h->win[s].window);
        cudaFree(h->win[s].window64);
        cudaFree(h->win[s].tw64);
    }
    for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
    for (int i = 0; i < 2; ++i) {
        if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
        if (h->ev_compute[i]) cudaEventDestroy(h->ev_compute[i]);
        if (h->ev_d2h[i]) cudaEventDestroy(h->ev_d2h[i]);
    }
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->h2d_stream) cudaStreamDestroy(h->h2d_stream);
    if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
    delete h;
    return REPET_OK;
}

const char* repet_last_error(repet_handle* h) { return h ? h->err.c_str() : "null handle"; }

int repet_set_stream(repet_handle* h, void* cuda_stream) {
    if (!h) return REPET_E_INVALID_ARG;
    h->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : h->own_stream;
    return REPET_OK;
}

int repet_set_window(repet_handle* h, const double* window, int n) {
    if (!h || !window) return REPET_E_INVALID_ARG;
    const int slot = slot_of(n);
    if (slot < 0)
        return fail(h, REPET_E_UNSUPPORTED, "window_length must be 512, 1024 or 2048 (sampling frequencies up to 51.2 kHz)");
    CU(cudaSetDevice(h->device));
    std::vector<float> w(n);
    for (int i = 0; i < n; ++i) w[i] = (float)window[i];
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(h->win[slot].window, w.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->win[slot].window64, window, n * sizeof(double), cudaMemcpyHostToDevice));
    h->win[slot].window_set = true;
    h->window_n = n;
    return REPET_OK;
}

int repet_set_workspace_limit(repet_handle* h, uint64_t bytes) {
    if (!h) return REPET_E_INVALID_ARG;
    h->ws_limit = bytes;
    return REPET_OK;
}

uint64_t repet_workspace_bytes(repet_handle* h) { return h ? (uint64_t)h->arena_bytes : 0; }

int repet_synchronize(repet_handle* h) {
    if (!h) return REPET_E_INVALID_ARG;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    return REPET_OK;
}

uint64_t repet_launch_count(repet_handle* h) { return h ? h->launches : 0; }

int repet_set_tuning(const char* name, int value) {
    if (!name) return REPET_E_INVALID_ARG;
    const std::string key(name);
    if (key == "stft_minb") g_repet_tuning.stft_minb = value;
    else if (key == "mask_minb") g_repet_tuning.mask_minb = value;
    else if (key == "frames_per_cta") g_repet_tuning.frames_per_cta = value;
    else if (key == "beat_parts") g_repet_tuning.beat_parts = value;
    else if (key == "simgemm_tc") g_repet_tuning.simgemm_tc = value;
    else if (key == "sim_frames64") g_repet_tuning.sim_frames64 = value;
    else if (key == "copy_chunk_mb") g_repet_tuning.copy_chunk_mb = value;
    else if (key == "cert_rel_ppm") g_repet_tuning.cert_rel_ppm = value;
    else if (key == "topk_force_exact") g_repet_tuning.topk_force_exact = value;
    else if (key == "simgemm_bn") g_repet_tuning.simgemm_bn = value;
    else if (key == "adaptive_vsq") g_repet_tuning.adaptive_vsq = value;
    else return REPET_E_INVALID_ARG;
    return REPET_OK;
}

int repet_set_profiling(repet_handle* h, int on) {
    if (!h) return REPET_E_INVALID_ARG;
    h->profiling = on != 0;
    return REPET_OK;
}

int repet_profile_read(repet_handle* h, double* ms, uint64_t* counts, int reset) {
    if (!h) return REPET_E_INVALID_ARG;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
        float t = 0.f;
        CU(cudaEventElapsedTime(&t, h->prof_events[i], h->prof_events[i + 1]));
        const int id = h->prof_ids[i / 2];
        h->prof_ms[id] += (double)t;
        h->prof_count[id] += 1;
    }
    h->prof_used = 0;
    h->prof_ids.clear();
    for (int k = 0; k < REPET_NUM_KERNELS; ++k) {
        if (ms) ms[k] = h->prof_ms[k];
        if (counts) counts[k] = h->prof_count[k];
        if (reset) {
            h->prof_ms[k] = 0.0;
            h->prof_count[k] = 0;
        }
    }
    return REPET_OK;
}

const char* repet_kernel_name(int id) { return (id >= 0 && id < REPET_NUM_KERNELS) ? kKernelNames[id] : ""; }

// ---------------------------------------------------------------------------------------------
// drivers (repet.py:67-911): one template per calling convention
// ---------------------------------------------------------------------------------------------
#define REPET_DRIVER(name, KIND)                                                                                       \
    int repet_##name##_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,  \
                                 const repet_params* p, float* background, int32_t* ints_dev, int32_t* ints_host) {    \
        const repet_entry* e = entry_for(h, p);                                                                        \
        if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;                      \
        return e->batch_dev(h, KIND, audio, n_clips, n_channels, n_samples, p, background, ints_dev, ints_host);       \
    }                                                                                                                  \
    int repet_##name##_batch(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,      \
                             const repet_params* p, float* background, int32_t* ints_host) {                           \
        const repet_entry* e = entry_for(h, p);                                                                        \
        if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;                      \
        return e->batch_host(h, KIND, audio, REPET_FMT_F32_PLANAR, n_clips, n_channels, n_samples, p, background,     \
                             REPET_FMT_F32_PLANAR, ints_host);                                                         \
    }

REPET_DRIVER(original, KIND_ORIGINAL)
REPET_DRIVER(extended, KIND_EXTENDED)
REPET_DRIVER(adaptive, KIND_ADAPTIVE)
REPET_DRIVER(sim, KIND_SIM)
REPET_DRIVER(simonline, KIND_SIMONLINE)
#undef REPET_DRIVER

static int dispatch_f64(repet_handle* h, int kind, const double* audio, int64_t n_samples, int n_channels,
                        const repet_params* p, double* background, int32_t* ints, int64_t capacity) {
    const repet_entry* e = entry_for(h, p);
    if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;
    return e->single_f64(h, kind, audio, n_samples, n_channels, p, background, ints, capacity);
}

int repet_original_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                       double* background, int32_t* period_host) {
    return dispatch_f64(h, KIND_ORIGINAL, audio, n_samples, n_channels, p, background, period_host, 1);
}
int repet_extended_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                       double* background, int32_t* periods_host, int periods_capacity) {
    return dispatch_f64(h, KIND_EXTENDED, audio, n_samples, n_channels, p, background, periods_host, periods_capacity);
}
int repet_adaptive_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                       double* background, int32_t* periods_host, int periods_capacity) {
    return dispatch_f64(h, KIND_ADAPTIVE, audio, n_samples, n_channels, p, background, periods_host, periods_capacity);
}
int repet_sim_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                  double* background, int32_t* lists_host, int lists_capacity) {
    return dispatch_f64(h, KIND_SIM, audio, n_samples, n_channels, p, background, lists_host, lists_capacity);
}
int repet_simonline_f64(repet_handle* h, const double* audio, int64_t n_samples, int n_channels, const repet_params* p,
                        double* background, int32_t* lists_host, int lists_capacity) {
    return dispatch_f64(h, KIND_SIMONLINE, audio, n_samples, n_channels, p, background, lists_host, lists_capacity);
}

/* ---- stateful online REPET-SIM stream (SURVEY.md 8(b): repet_simonline_block) -------------------------- */
}  // extern "C"

struct repet_stream {
    repet_handle* h = nullptr;
    repet_params p;
    int channels = 0;
    int64_t received = 0;       // samples taken so far
    int64_t emitted = 0;        // background samples handed out so far
    int64_t frame0 = 0;         // first frame whose samples are still held (sample frame0 * H)
    int64_t held = 0;           // samples held in d_hist (from sample frame0 * H on)
    int64_t capacity = 0;       // samples d_hist / d_out can hold
    double* d_hist = nullptr;   // device: the sample history, float64 (samples, channels)
    double* d_out = nullptr;    // device: the background of the window analysed last / scratch for compaction
};

namespace {

int stream_reserve(repet_stream* s, int64_t samples) {
    repet_handle* h = s->h;
    if (samples <= s->capacity) return REPET_OK;
    const int64_t cap = std::max<int64_t>(samples + samples / 2, 1 << 16);
    double *hist = nullptr, *out = nullptr;
    CU(cudaMalloc(&hist, (size_t)cap * s->channels * sizeof(double)));
    if (cudaMalloc(&out, (size_t)cap * s->channels * sizeof(double)) != cudaSuccess) {
        cudaFree(hist);
        return fail(h, REPET_E_OOM, "out of device memory for the stream history");
    }
    if (s->held > 0)
        CU(cudaMemcpyAsync(hist, s->d_hist, (size_t)s->held * s->channels * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(s->d_hist);
    cudaFree(s->d_out);
    s->d_hist = hist;
    s->d_out = out;
    s->capacity = cap;
    return REPET_OK;
}

// Emit background samples [emitted, final_until): analyse the window of frames that cover them together with
// their similarity history (buffer_frames - 1 frames back), with the ring-slot order of the whole stream
// (online_frame_base, quirk Q6).  `window_end` = one past the last sample the window may read.
int stream_advance(repet_stream* s, int64_t final_until, int64_t window_end, double* background, int64_t capacity,
                   int64_t* n_out) {
    repet_handle* h = s->h;
    *n_out = 0;
    if (final_until <= s->emitted) return REPET_OK;
    const int64_t H = s->p.step_length, B = s->p.buffer_frames;
    const int64_t count = final_until - s->emitted;
    if (count > capacity) return fail(h, REPET_E_INVALID_ARG, "background buffer too small for the samples that became final");
    const int64_t first_block = s->emitted / H;
    const int64_t first_needed = std::max<int64_t>(0, first_block - 1);  // block b mixes frames b-1 and b
    int64_t first_frame = std::max<int64_t>(0, first_needed - (B - 1));   // ... and their similarity history
    first_frame = std::max(first_frame, s->frame0);
    const int64_t lo = (first_frame - s->frame0) * H;
    const int64_t window = window_end - first_frame * H;
    const repet_entry* e = entry_for(h, &s->p);
    if (!e) return REPET_E_UNSUPPORTED;
    repet_params p = s->p;
    p.online_frame_base = (int32_t)first_frame;
    int rc = e->single_f64_dev(h, KIND_SIMONLINE, s->d_hist + lo * s->channels, window, s->channels, &p, s->d_out);
    if (rc) return rc;
    CU(cudaMemcpyAsync(background, s->d_out + (s->emitted - first_frame * H) * s->channels,
                       (size_t)count * s->channels * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    s->emitted = final_until;
    *n_out = count;
    // drop the samples no later window will need (compaction through the scratch buffer: the ranges overlap)
    const int64_t keep_frame = std::max<int64_t>(0, s->emitted / H - 1 - (B - 1));
    if (keep_frame > s->frame0) {
        const int64_t drop = (keep_frame - s->frame0) * H;
        const int64_t rest = s->held - drop;
        if (rest > 0) {
            CU(cudaMemcpyAsync(s->d_out, s->d_hist + drop * s->channels, (size_t)rest * s->channels * sizeof(double),
                               cudaMemcpyDeviceToDevice, h->stream));
            std::swap(s->d_hist, s->d_out);
        }
        s->held = std::max<int64_t>(rest, 0);
        s->frame0 = keep_frame;
    }
    return REPET_OK;
}

}  // namespace

extern "C" {

int repet_simonline_open(repet_handle* h, const repet_params* p, int n_channels, repet_stream** out) {
    if (!h || !out) return REPET_E_INVALID_ARG;
    *out = nullptr;
    if (!p) return fail(h, REPET_E_INVALID_ARG, "params is null");
    if (!entry_for(h, p)) return REPET_E_UNSUPPORTED;
    if (n_channels < 1 || n_channels > 2) return fail(h, REPET_E_UNSUPPORTED, "1 or 2 channels supported");
    if (p->buffer_frames < 1) return fail(h, REPET_E_INVALID_ARG, "buffer_length must cover at least one frame");
    repet_stream* s = new repet_stream();
    s->h = h;
    s->p = *p;
    s->p.online_frame_base = 0;
    s->channels = n_channels;
    *out = s;
    return REPET_OK;
}

int repet_simonline_block(repet_stream* s, const double* block, int64_t n_samples, double* background, int64_t capacity,
                          int64_t* n_out) {
    if (!s || !n_out) return REPET_E_INVALID_ARG;
    repet_handle* h = s->h;
    *n_out = 0;
    if (n_samples < 0 || (n_samples > 0 && !block)) return fail(h, REPET_E_INVALID_ARG, "bad block");
    CU(cudaSetDevice(h->device));
    int rc = stream_reserve(s, s->held + n_samples);
    if (rc) return rc;
    if (n_samples > 0) {
        CU(cudaMemcpyAsync(s->d_hist + s->held * s->channels, block, (size_t)n_samples * s->channels * sizeof(double),
                           cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));  // the caller may reuse `block` as soon as this returns
    }
    s->held += n_samples;
    s->received += n_samples;
    const int64_t N = s->p.window_length, H = s->p.step_length, B = s->p.buffer_frames;
    if (s->received < N) return REPET_OK;
    const int64_t last_complete = (s->received - N) / H;
    const int64_t final_until = (last_complete + 1) * H;
    if (last_complete < B - 1) {
        // nothing is synthesised before frame buffer_frames - 1 (quirk Q5): the final samples are zeros
        const int64_t count = std::max<int64_t>(0, final_until - s->emitted);
        if (count > capacity) return fail(h, REPET_E_INVALID_ARG, "background buffer too small for the samples that became final");
        if (count > 0) std::memset(background, 0, (size_t)count * s->channels * sizeof(double));
        s->emitted = std::max(s->emitted, final_until);
        *n_out = count;
        return REPET_OK;
    }
    return stream_advance(s, final_until, last_complete * H + N, background, capacity, n_out);
}

int repet_simonline_flush(repet_stream* s, double* background, int64_t capacity, int64_t* n_out) {
    if (!s || !n_out) return REPET_E_INVALID_ARG;
    repet_handle* h = s->h;
    *n_out = 0;
    if (s->received <= s->emitted) return REPET_OK;
    const int64_t N = s->p.window_length, H = s->p.step_length, B = s->p.buffer_frames;
    if (s->received < (B - 2) * H + N)
        return fail(h, REPET_E_INVALID_ARG, "operands could not be broadcast together (signal shorter than the buffer)");
    CU(cudaSetDevice(h->device));
    return stream_advance(s, s->received, s->received, background, capacity, n_out);
}

int repet_simonline_close(repet_stream* s) {
    if (!s) return REPET_OK;
    cudaSetDevice(s->h->device);
    cudaStreamSynchronize(s->h->stream);
    cudaFree(s->d_hist);
    cudaFree(s->d_out);
    delete s;
    return REPET_OK;
}

int repet_separate_f64(repet_handle* h, int method, const double* audio, int64_t n_samples, int n_channels,
                       const repet_params* p, double* background, double* foreground, float* spectrograms,
                       int32_t* ints_host, int ints_capacity) {
    const repet_entry* e = entry_for(h, p);
    if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;
    if (method < KIND_ORIGINAL || method > KIND_SIMONLINE) return fail(h, REPET_E_INVALID_ARG, "unknown method");
    return e->separate_f64(h, method, audio, n_samples, n_channels, p, background, foreground, spectrograms, ints_host,
                           ints_capacity);
}
int repet_spectrogram_pitch(const repet_params* p) { return p ? (p->window_length / 2 + 1 + 7) / 8 * 8 : 0; }
int repet_spectrogram_frames(const repet_params* p, int64_t n_samples) {
    return (p && p->step_length > 0) ? (int)((n_samples + p->step_length - 1) / p->step_length) + 1 : 0;
}
int repet_spectrogram_batch_dev(repet_handle* h, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                                const repet_params* p, float* spectrogram) {
    const repet_entry* e = entry_for(h, p);
    if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;
    return e->spectrogram_dev(h, audio, n_clips, n_channels, n_samples, p, spectrogram);
}
int repet_foreground_dev(repet_handle* h, const float* audio, const float* background, int64_t n_elements,
                         float* foreground) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_of_slot(2)->foreground_dev(h, audio, background, n_elements, foreground);
}

// int16 PCM in WAV order [clip][sample][channel] (repet.py:914-947)
int repet_original_batch_pcm16(repet_handle* h, const int16_t* audio, int n_clips, int n_channels, int64_t n_samples,
                               const repet_params* p, float* background, int32_t* periods_host) {
    const repet_entry* e = entry_for(h, p);
    if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;
    return e->batch_host(h, KIND_ORIGINAL, audio, REPET_FMT_PCM16, n_clips, n_channels, n_samples, p, background,
                         REPET_FMT_F32_PLANAR, periods_host);
}

// any driver, any of the two sample formats on either side (repet.py:914-946 either side of the separation)
int repet_separate_batch(repet_handle* h, int method, const void* audio, int in_format, int n_clips, int n_channels,
                         int64_t n_samples, const repet_params* p, void* background, int out_format, int32_t* ints_host) {
    const repet_entry* e = entry_for(h, p);
    if (!e) return h ? (p ? REPET_E_UNSUPPORTED : REPET_E_INVALID_ARG) : REPET_E_INVALID_ARG;
    if (method < KIND_ORIGINAL || method > KIND_SIMONLINE) return fail(h, REPET_E_INVALID_ARG, "unknown method");
    return e->batch_host(h, method, audio, in_format, n_clips, n_channels, n_samples, p, background, out_format, ints_host);
}

// integer outputs per clip of a driver (the size of `ints_host` per clip for repet_separate_batch)
int64_t repet_ints_per_clip(int method, const repet_params* p, int64_t n_samples) {
    if (!p || p->step_length <= 0) return 0;
    const int64_t T = (n_samples + p->step_length - 1) / p->step_length + 1;
    switch (method) {
        case KIND_ORIGINAL: return 1;
        case KIND_EXTENDED: return repet_extended_segments(p, n_samples);
        case KIND_ADAPTIVE: return T;
        case KIND_SIM: return T * ((int64_t)p->similarity_number + 1);
        case KIND_SIMONLINE: return (int64_t)repet_simonline_frames(p, n_samples) * ((int64_t)p->similarity_number + 1);
    }
    return 0;
}

// page-locked host memory for the host-buffer entry points (pageable buffers are staged by the driver at a
// fraction of the link rate)
int repet_host_alloc(void** out, uint64_t bytes) {
    if (!out) return REPET_E_INVALID_ARG;
    *out = nullptr;
    const cudaError_t e = cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? REPET_E_OOM : REPET_E_CUDA;
    }
    return REPET_OK;
}
int repet_host_free(void* ptr) {
    if (!ptr) return REPET_OK;
    return cudaFreeHost(ptr) == cudaSuccess ? REPET_OK : REPET_E_CUDA;
}
int repet_host_register(void* ptr, uint64_t bytes) {
    if (!ptr) return REPET_E_INVALID_ARG;
    const cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return REPET_E_CUDA;
    }
    return REPET_OK;
}
int repet_host_unregister(void* ptr) {
    if (!ptr) return REPET_OK;
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) (void)cudaGetLastError();
    return e == cudaSuccess ? REPET_OK : REPET_E_CUDA;
}
int repet_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

// number of 10 s segments of repet.extended (repet.py:270-283)
int repet_extended_segments(const repet_params* p, int64_t n_samples) {
    if (!p || p->segment_length <= 0 || p->segment_step <= 0) return 0;
    if (n_samples < (int64_t)p->segment_length + p->segment_step) return 1;
    return 1 + (int)((n_samples - p->segment_length) / p->segment_step);
}

// number of uncentred frames of repet.simonline (repet.py:781)
int repet_simonline_frames(const repet_params* p, int64_t n_samples) {
    if (!p || n_samples < p->window_length) return 0;
    return (int)((n_samples - p->window_length + p->step_length - 1) / p->step_length) + 1;
}

// ---------------------------------------------------------------------------------------------
// helpers (repet.py:1001-1545)
// ---------------------------------------------------------------------------------------------
#define REPET_CURRENT(h)                            \
    const repet_entry* e = entry_current(h);        \
    if (!e) return REPET_E_INVALID_ARG

int repet_stft(repet_handle* h, const float* signal, int n_channels, int64_t n_samples, float* spectrum, float* power,
               int32_t* n_frames_out) {
    REPET_CURRENT(h);
    return e->stft(h, signal, n_channels, n_samples, spectrum, power, n_frames_out);
}
int repet_istft(repet_handle* h, const float* spectrum, int n_channels, int n_frames, double cola_gain, float* signal) {
    REPET_CURRENT(h);
    return e->istft(h, spectrum, n_channels, n_frames, cola_gain, signal);
}
int repet_mask(repet_handle* h, const float* magnitude, int n_frames, int period, float* mask) {
    REPET_CURRENT(h);
    return e->mask(h, magnitude, n_frames, period, mask);
}
int repet_adaptivemask(repet_handle* h, const float* magnitude, int n_frames, const int32_t* periods, int filter_order,
                       float* mask) {
    REPET_CURRENT(h);
    return e->adaptivemask(h, magnitude, n_frames, periods, filter_order, mask);
}
int repet_simmask(repet_handle* h, const float* magnitude, int n_frames, const int32_t* indices, const int32_t* counts,
                  int number, float* mask) {
    REPET_CURRENT(h);
    return e->simmask(h, magnitude, n_frames, indices, counts, number, mask);
}
#undef REPET_CURRENT

int repet_beatspectrum(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, double* beat) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!beat) return fail(h, REPET_E_INVALID_ARG, "beat is null");
    return entry_rows(h, n_rows)->beat_common(h, spectrogram, n_frames, n_rows, 0, 0, beat, nullptr);
}
int repet_period(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, int period_lo, int period_hi,
                 int32_t* period) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!period) return fail(h, REPET_E_INVALID_ARG, "period is null");
    const int lag_hi = std::min(period_hi, n_frames / 3);  // repet.py:1265-1267
    if (period_lo < 0 || lag_hi <= period_lo)
        return fail(h, REPET_E_TOO_SHORT, "attempt to get argmax of an empty sequence");
    return entry_rows(h, n_rows)->beat_common(h, spectrogram, n_frames, n_rows, period_lo, lag_hi, nullptr, period);
}
int repet_beatspectrogram(repet_handle* h, const float* spectrogram, int n_frames, int n_rows, int segment_length,
                          int segment_step, double* beat, int32_t* n_segments_out) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_rows(h, n_rows)->beatspectrogram(h, spectrogram, n_frames, n_rows, segment_length, segment_step, beat,
                                                  n_segments_out);
}
int repet_selfsimilarity(repet_handle* h, const float* magnitude, int n_frames, int n_rows, float* similarity) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_rows(h, n_rows)->selfsimilarity(h, magnitude, n_frames, n_rows, similarity);
}
int repet_similarity(repet_handle* h, const float* magnitude1, int n_frames1, const float* magnitude2, int n_frames2,
                     int n_rows, double* similarity) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_rows(h, n_rows)->similarity(h, magnitude1, n_frames1, magnitude2, n_frames2, n_rows, similarity);
}
int repet_periods(repet_handle* h, const double* beat, int n_lags, int n_columns, int period_lo, int period_hi,
                  int32_t* periods) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_of_slot(2)->periods(h, beat, n_lags, n_columns, period_lo, period_hi, periods);
}
int repet_localmaxima(repet_handle* h, const double* data, int n, int n_columns, double minimum_value,
                      int minimum_distance, int number_values, int32_t* indices, int32_t* counts, double* values) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_of_slot(2)->localmaxima(h, data, n, n_columns, minimum_value, minimum_distance, number_values, indices,
                                         counts, values);
}
int repet_acorr(repet_handle* h, const float* data, int n_rows, int n_columns, double* autocorrelation) {
    if (!h) return REPET_E_INVALID_ARG;
    return entry_of_slot(2)->acorr(h, data, n_rows, n_columns, autocorrelation);
}

}  // extern "C"
