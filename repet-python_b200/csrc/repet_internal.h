// Internals shared by repet_abi.cu (handle, dispatch), repet_helpers.cu (helper entry points) and
// repet_drivers.cu (batch drivers).  The last two are compiled once per window length.
#pragma once
#include "../../include/repet_b200.h"
#include "repet_kernels.cuh"

#include <algorithm>
#include <string>
#include <vector>

struct repet_handle {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t h2d_stream = nullptr;
    cudaStream_t d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr};
    cudaEvent_t ev_compute[2] = {nullptr, nullptr};
    cudaEvent_t ev_d2h[2] = {nullptr, nullptr};
    std::string err;
    // per window length (slot 0, 1, 2 = 512, 1024, 2048): frame-transform tables and analysis window
    struct WindowSlot {
        float2* tw1 = nullptr;
        float2* tw2 = nullptr;
        float* window = nullptr;
        double* window64 = nullptr;  // the same window as given (float64): k_frames64
        double2* tw64 = nullptr;     // W_N^i, i < N/2, float64: k_frames64
        bool window_set = false;
    } win[3];
    int window_n = 0;  // length of the window set last: what the helper entry points transform with
    unsigned char* arena = nullptr;
    size_t arena_bytes = 0;
    uint64_t ws_limit = 0;
    size_t ws_auto = 0;  // cached automatic workspace limit
    uint64_t launches = 0;
    // float64 (samples, channels) copy of the clip being separated by a *_f64 entry point, device memory;
    // the float64 front end of REPET-SIM reads the samples from here instead of their fp32 rounding
    const double* f64_audio = nullptr;
    int sm_count = 148;
    // optional per-kernel timing (bench.py's roofline): one event pair per launch
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;
    std::vector<int> prof_ids;
    size_t prof_used = 0;
    double prof_ms[REPET_NUM_KERNELS] = {0};
    uint64_t prof_count[REPET_NUM_KERNELS] = {0};
};

// One table of entry points per compiled window length.
struct repet_entry {
    int window_n;
    // drivers: kind = 0 original, 1 extended, 2 adaptive, 3 sim, 4 simonline
    int (*batch_dev)(repet_handle*, int kind, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                     const repet_params* p, float* background, int32_t* ints_dev, int32_t* ints_host);
    int (*batch_host)(repet_handle*, int kind, const void* audio, int in_format, int n_clips, int n_channels,
                      int64_t n_samples, const repet_params* p, void* background, int out_format, int32_t* ints);
    int (*single_f64)(repet_handle*, int kind, const double* audio, int64_t n_samples, int n_channels,
                      const repet_params* p, double* background, int32_t* ints, int64_t ints_capacity);
    // helpers
    int (*stft)(repet_handle*, const float*, int, int64_t, float*, float*, int32_t*);
    int (*istft)(repet_handle*, const float*, int, int, double, float*);
    int (*beat_common)(repet_handle*, const float*, int, int, int, int, double*, int32_t*);
    int (*mask)(repet_handle*, const float*, int, int, float*);
    int (*adaptivemask)(repet_handle*, const float*, int, const int32_t*, int, float*);
    int (*beatspectrogram)(repet_handle*, const float*, int, int, int, int, double*, int32_t*);
    int (*selfsimilarity)(repet_handle*, const float*, int, int, float*);
    int (*periods)(repet_handle*, const double*, int, int, int, int, int32_t*);
    int (*similarity)(repet_handle*, const float*, int, const float*, int, int, double*);
    int (*localmaxima)(repet_handle*, const double*, int, int, double, int, int, int32_t*, int32_t*, double*);
    int (*simmask)(repet_handle*, const float*, int, const int32_t*, const int32_t*, int, float*);
    int (*acorr)(repet_handle*, const float*, int, int, double*);
    // by-products (README.md:64-81)
    int (*separate_f64)(repet_handle*, int kind, const double* audio, int64_t n_samples, int n_channels,
                        const repet_params* p, double* background, double* foreground, float* spectrograms,
                        int32_t* ints, int64_t ints_capacity);
    int (*spectrogram_dev)(repet_handle*, const float* audio, int n_clips, int n_channels, int64_t n_samples,
                           const repet_params* p, float* spectrogram);
    int (*foreground_dev)(repet_handle*, const float* audio, const float* background, int64_t n, float* foreground);
    // float64 (samples, channels) device in / device out, stream-ordered (the stateful simonline stream)
    int (*single_f64_dev)(repet_handle*, int kind, const double* d_audio, int64_t n_samples, int n_channels,
                          const repet_params* p, double* d_background);
};

namespace repet {

inline int fail(repet_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return repet::fail(h, e__ == cudaErrorMemoryAllocation ? REPET_E_OOM : REPET_E_CUDA,   \
                               std::string(#call) + ": " + cudaGetErrorString(e__));               \
    } while (0)

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Lays buffers out one after the other, each 256-byte aligned.  A layout is written once, as a sequence of takes,
// and run twice: on Bump(nullptr), where take returns nullptr and only advances `off`, to measure it, and on the
// memory it was measured for, to carve it.  `cap` is the size of that memory: a runner that carves from a
// workspace it was handed checks `fits()` before it launches anything.
struct Bump {
    unsigned char* base;
    size_t cap;
    size_t off = 0;
    explicit Bump(unsigned char* b, size_t capacity = SIZE_MAX) : base(b), cap(capacity) {}
    template <typename T>
    T* take(size_t count) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off = align_up(off + count * sizeof(T));
        return p;
    }
    bool fits() const { return off <= cap; }
};

// Brackets the launches of one pipeline step with an event pair when profiling is on; always counts the
// kernels launched inside (`kernels`, default one).
struct Timed {
    repet_handle* h;
    Timed(repet_handle* handle, int id, int kernels = 1) : h(handle) {
        h->launches += kernels;
        if (!h->profiling) return;
        if (h->prof_used + 2 > h->prof_events.size()) {
            for (int i = 0; i < 2; ++i) {
                cudaEvent_t e = nullptr;
                cudaEventCreate(&e);
                h->prof_events.push_back(e);
            }
        }
        h->prof_ids.push_back(id);
        cudaEventRecord(h->prof_events[h->prof_used], h->stream);
    }
    ~Timed() {
        if (!h->profiling) return;
        cudaEventRecord(h->prof_events[h->prof_used + 1], h->stream);
        h->prof_used += 2;
    }
};

constexpr int MAX_ITEMS_PER_LAUNCH = 16384;  // grid.y / grid.z stay far below 65535

constexpr int WIN_SLOT = WIN_N == 512 ? 0 : (WIN_N == 1024 ? 1 : 2);

inline int ensure_arena(repet_handle* h, size_t bytes) {
    if (bytes <= h->arena_bytes) return REPET_OK;
    CU(cudaStreamSynchronize(h->stream));
    if (h->arena) CU(cudaFree(h->arena));
    h->arena = nullptr;
    h->arena_bytes = 0;
    CU(cudaMalloc(&h->arena, bytes));
    h->arena_bytes = bytes;
    return REPET_OK;
}

// Measures `layout` (a callable taking Bump&), grows the arena to its size and carves it from the arena.
template <typename Layout>
int carve_arena(repet_handle* h, Layout&& layout) {
    Bump measure(nullptr);
    layout(measure);
    const int rc = ensure_arena(h, measure.off);
    if (rc) return rc;
    Bump bump(h->arena);
    layout(bump);
    return REPET_OK;
}

inline size_t default_ws_limit(repet_handle* h) {
    if (h->ws_limit) return (size_t)h->ws_limit;
    if (h->ws_auto) return h->ws_auto;  // cudaMemGetInfo is a slow driver call: ask once per handle
    // big chunks win (launch tails and the per-clip period kernel amortise): up to 24 GB, but never
    // more than 40 % of what is free on the device
    size_t free_b = 0, total_b = 0;
    size_t limit = (size_t)24 << 30;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
        limit = std::min(limit, (size_t)((double)(free_b + h->arena_bytes) * 0.4));
    h->ws_auto = std::max(limit, (size_t)256 << 20);
    return h->ws_auto;
}

inline int frames_of(int64_t n_samples) {  // repet.py:1018-1028 with N = 2H
    return (int)((n_samples + HOP - 1) / HOP) + 1;
}
inline const float* window_of(repet_handle* h) { return h->win[WIN_SLOT].window; }
inline FftTables tables(repet_handle* h) {
    return FftTables{h->win[WIN_SLOT].tw1, h->win[WIN_SLOT].tw2, h->win[2].tw1, h->win[2].tw2, h->win[1].tw1, h->win[1].tw2};
}

inline int check_common(repet_handle* h, const repet_params* p, int n_channels) {
    if (!h) return REPET_E_INVALID_ARG;
    if (!p) return fail(h, REPET_E_INVALID_ARG, "params is null");
    if (p->window_length != WIN_N || p->step_length != HOP)
        return fail(h, REPET_E_UNSUPPORTED, "window_length / step_length do not match this instantiation");
    if (n_channels < 1 || n_channels > 2)
        return fail(h, REPET_E_UNSUPPORTED, "1 or 2 channels supported");
    if (!h->win[WIN_SLOT].window_set)
        return fail(h, REPET_E_INVALID_ARG, "repet_set_window has not been called for this window length");
    return REPET_OK;
}

// Entry points of this window-length instantiation (repet_drivers.cu, repet_helpers.cu); the
// extern "C" functions in repet_abi.cu pick the table from repet_params.window_length (drivers) or
// from the window set last (helpers).
const repet_entry* entry_table();

}  // namespace repet
