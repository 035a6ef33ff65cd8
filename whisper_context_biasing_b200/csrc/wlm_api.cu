// libwlm.so -- C ABI (include/wlm.h) over the sm_100a log-mel kernels.
//
// Host side only: plan construction (mel table -> sparse form, constant tables), argument
// validation, launch sequencing, the pinned-ring H2D pipeline of wlm_logmel_host.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "logmel_fused.cuh"
#include "wlm_common.cuh"

using namespace wlm;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define WLM_CUDA(expr)                                                                      \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail(WLM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                \
    } while (0)

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
struct wlm_plan {
    int device = -1;
    int n_mels = 0;
    int sm_count = 0;
    std::atomic<int64_t> launches{0};
    int out_format = WLM_OUT_F32;
    int flat_override = -1;        // clips for the flat kernel (dense batches); -1 = the library's split

    // constant tables: the sparse mel form travels in the constant bank (kernel argument), the window on the device
    MelSparse h_sparse;
    fused::Tables* d_fused_tables = nullptr;
    fused::Tables h_fused_tables;
    ClipQueue* d_queue = nullptr;  // clip counter the two kernels of a launch pull from (self-resetting)
    int max_clusters = 0;          // co-resident clusters of the fused kernel (occupancy query)
    int flat_ctas = 0;             // SMs the clusters cannot cover: they run the flat kernel (programmatic dependent launch)
    int variant = 0;               // 80 / 128: unrolled mel stage (Whisper banks); 0: table-driven

    // wlm_logmel_host pipeline
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_slot_free[2] = {nullptr, nullptr};
    cudaEvent_t ev_kernels_done = nullptr;
    bool kernels_done_valid = false;
    void* d_stage = nullptr;  // packed PCM
    size_t d_stage_bytes = 0;
    void* h_ring[2] = {nullptr, nullptr};
    size_t h_ring_bytes = 0;
    int64_t* d_offsets = nullptr;
    int32_t* d_lengths = nullptr;
    int64_t* h_offsets = nullptr;  // pinned
    int32_t* h_lengths = nullptr;  // pinned
    int meta_cap = 0;
    void* d_ws = nullptr;
    size_t d_ws_bytes = 0;
};

extern "C" int wlm_version(void) { return WLM_VERSION; }
extern "C" const char* wlm_last_error(void) { return g_last_error.c_str(); }

static int build_sparse(const float* dense, int n_mels, MelSparse* sp, std::vector<int16_t>* klo,
                        std::vector<int16_t>* khi) {
    klo->assign(n_mels, 0);
    khi->assign(n_mels, -1);
    std::vector<int> seen(n_mels, 0);
    memset(sp, 0, sizeof(*sp));
    for (int k = 0; k < kNFreq + 3; ++k) sp->lo[k] = -1;  // -1 = "filter before the first" (dummy)
    int prev_lo = -1;
    for (int k = 0; k < kNFreq; ++k) {
        int idx[3], n = 0;
        for (int m = 0; m < n_mels; ++m) {
            const float w = dense[k * n_mels + m];
            if (!(w == w) || std::isinf(w)) return fail(WLM_ERR_BAD_ARG, "mel table has a non-finite entry at [%d][%d]", k, m);
            if (w != 0.0f) {
                if (n == 2) return fail(WLM_ERR_UNSUPPORTED, "mel table: FFT bin %d feeds more than two filters", k);
                idx[n++] = m;
                if (!seen[m]) { (*klo)[m] = (int16_t)k; seen[m] = 1; }
                if ((*khi)[m] >= 0 && (*khi)[m] != k - 1)
                    return fail(WLM_ERR_UNSUPPORTED, "mel table: filter %d has non-contiguous support at bin %d", m, k);
                (*khi)[m] = (int16_t)k;
            }
        }
        if (n == 2 && idx[1] != idx[0] + 1)
            return fail(WLM_ERR_UNSUPPORTED, "mel table: FFT bin %d feeds non-adjacent filters %d,%d", k, idx[0], idx[1]);
        if (n == 0) {
            sp->lo[k] = (int16_t)prev_lo;  // both weights 0
        } else if (n == 2) {
            sp->lo[k] = (int16_t)idx[0];
            sp->w_lo[k] = dense[k * n_mels + idx[0]];
            sp->w_hi[k] = dense[k * n_mels + idx[1]];
        } else if (idx[0] == 0 && prev_lo == -1) {
            // first interval [f0, f1): only the rising side of filter 0 -> "hi" weight of the pair (-1, 0)
            sp->lo[k] = -1;
            sp->w_hi[k] = dense[k * n_mels + 0];
        } else {
            // single filter m elsewhere: filter m-1 is exactly zero here, i.e. the bin sits on the
            // centre of m or on its falling side with m+1 not started -> "lo" weight of the pair (m, m+1)
            sp->lo[k] = (int16_t)idx[0];
            sp->w_lo[k] = dense[k * n_mels + idx[0]];
        }
        if (sp->lo[k] < prev_lo) return fail(WLM_ERR_UNSUPPORTED, "mel table: filter order not monotone at bin %d", k);
        prev_lo = sp->lo[k];
    }
    for (int m = 0; m < n_mels; ++m)
        if (!seen[m]) { (*klo)[m] = 0; (*khi)[m] = -1; }  // empty filter: contributes 0 -> log10(1e-10)
    return WLM_OK;
}

extern "C" int wlm_plan_create(int device, int n_mels, const float* mel_dense_host, wlm_plan** out) {
    if (!out) return fail(WLM_ERR_BAD_ARG, "out is NULL");
    *out = nullptr;
    if (!mel_dense_host) return fail(WLM_ERR_BAD_ARG, "mel_dense_host is NULL");
    if (n_mels < 1 || n_mels > kMaxMels) return fail(WLM_ERR_UNSUPPORTED, "n_mels=%d outside [1,%d]", n_mels, kMaxMels);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(WLM_ERR_NO_DEVICE, "no CUDA device (%s); libwlm has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(WLM_ERR_BAD_ARG, "device %d out of range [0,%d)", device, ndev);
    cudaDeviceProp prop;
    WLM_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(WLM_ERR_NO_DEVICE, "device %d is sm_%d%d; libwlm is built for sm_100a only", device, prop.major, prop.minor);
    WLM_CUDA(cudaSetDevice(device));

    wlm_plan* p = new wlm_plan();
    p->device = device;
    p->n_mels = n_mels;
    p->sm_count = prop.multiProcessorCount;
    std::vector<int16_t> klo, khi;
    int rc = build_sparse(mel_dense_host, n_mels, &p->h_sparse, &klo, &khi);
    if (rc != WLM_OK) { delete p; return rc; }

#define WLM_CUDA_P(expr)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            wlm_plan_destroy(p);                                                                  \
            return fail(WLM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                         \
    } while (0)

    {
        if (fused::build_tables(p->h_sparse, n_mels, &p->h_fused_tables, &p->variant) != 0) {
            wlm_plan_destroy(p);
            return fail(WLM_ERR_UNSUPPORTED, "mel table: a filter has no FFT bin (num_mel_filters too high for 201 bins)");
        }
        WLM_CUDA_P(cudaMalloc(&p->d_fused_tables, sizeof(fused::Tables)));
        WLM_CUDA_P(cudaMemcpy(p->d_fused_tables, &p->h_fused_tables, sizeof(fused::Tables), cudaMemcpyHostToDevice));
        WLM_CUDA_P(cudaMalloc(&p->d_queue, sizeof(ClipQueue)));
        WLM_CUDA_P(cudaMemset(p->d_queue, 0, sizeof(ClipQueue)));
        cudaError_t fe = fused::configure(p->variant, &p->max_clusters);
        if (fe != cudaSuccess) {
            wlm_plan_destroy(p);
            return fail(WLM_ERR_CUDA, "fused kernel configuration failed: %s", cudaGetErrorString(fe));
        }
        // the SMs that whole clusters cannot cover run the flat kernel (WLM_FLAT=0 turns that off)
        const char* fl = getenv("WLM_FLAT");
        p->flat_ctas = (fl && atoi(fl) == 0) ? 0 : std::max(0, p->sm_count - fused::kCluster * p->max_clusters);
        // read ONCE (not per launch); clamped to [0, B - 1] when used
        if (const char* fc = getenv("WLM_FLAT_CLIPS")) p->flat_override = std::max(-1, atoi(fc));
    }

    WLM_CUDA_P(cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
    for (auto& ev : p->ev_chunk) WLM_CUDA_P(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    for (auto& ev : p->ev_slot_free) WLM_CUDA_P(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    WLM_CUDA_P(cudaEventCreateWithFlags(&p->ev_kernels_done, cudaEventDisableTiming));
#undef WLM_CUDA_P
    *out = p;
    return WLM_OK;
}

extern "C" int wlm_plan_destroy(wlm_plan* p) {
    if (!p) return WLM_OK;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    cudaFree(p->d_fused_tables);
    cudaFree(p->d_queue);
    cudaFree(p->d_stage); cudaFree(p->d_offsets); cudaFree(p->d_lengths); cudaFree(p->d_ws);
    for (auto& r : p->h_ring) if (r) cudaFreeHost(r);
    if (p->h_offsets) cudaFreeHost(p->h_offsets);
    if (p->h_lengths) cudaFreeHost(p->h_lengths);
    for (auto& ev : p->ev_chunk) if (ev) cudaEventDestroy(ev);
    for (auto& ev : p->ev_slot_free) if (ev) cudaEventDestroy(ev);
    if (p->ev_kernels_done) cudaEventDestroy(p->ev_kernels_done);
    if (p->copy_stream) cudaStreamDestroy(p->copy_stream);
    delete p;
    return WLM_OK;
}

extern "C" int wlm_plan_n_mels(const wlm_plan* p) { return p ? p->n_mels : fail(WLM_ERR_BAD_ARG, "plan is NULL"); }
extern "C" int wlm_plan_device(const wlm_plan* p) { return p ? p->device : fail(WLM_ERR_BAD_ARG, "plan is NULL"); }
extern "C" int wlm_plan_sm_count(const wlm_plan* p) { return p ? p->sm_count : fail(WLM_ERR_BAD_ARG, "plan is NULL"); }
extern "C" int wlm_plan_kernel_variant(const wlm_plan* p) { return p ? p->variant : fail(WLM_ERR_BAD_ARG, "plan is NULL"); }
extern "C" int wlm_plan_max_clusters(const wlm_plan* p) { return p ? p->max_clusters : fail(WLM_ERR_BAD_ARG, "plan is NULL"); }
extern "C" int64_t wlm_plan_launch_count(const wlm_plan* p) { return p ? p->launches.load() : -1; }
extern "C" int wlm_plan_output_format(const wlm_plan* p) { return p ? p->out_format : fail(WLM_ERR_BAD_ARG, "plan is NULL"); }
extern "C" int wlm_plan_set_output_format(wlm_plan* p, int out_format) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (out_format != WLM_OUT_F32 && out_format != WLM_OUT_BF16 && out_format != WLM_OUT_F16)
        return fail(WLM_ERR_BAD_ARG, "unknown out_format %d", out_format);
    p->out_format = out_format;
    return WLM_OK;
}
extern "C" int wlm_plan_set_flat_clips(wlm_plan* p, int n_flat) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    p->flat_override = n_flat < 0 ? -1 : n_flat;
    return WLM_OK;
}
static size_t out_elem_size(const wlm_plan* p) { return p->out_format == WLM_OUT_F32 ? 4 : 2; }

extern "C" size_t wlm_workspace_bytes(const wlm_plan* p, int B) {
    if (!p || B <= 0) return 0;
    return ((size_t)B * sizeof(float) + 255) / 256 * 256;  // per-clip gmax when the caller passes none
}

// ------------------------------------------------------------------------------------------
// launch
// ------------------------------------------------------------------------------------------
// the per-call fields of a launch; fused::launch fills in the work split (clip_first, n_workers, ...), launch_logmel the queue
static ClipArgs clip_args(const wlm_plan* p, const void* pcm, int pcm_format, const int64_t* offsets, const int32_t* lengths,
                          int64_t row_stride, int B, void* out, float* gmax) {
    ClipArgs a{};
    a.pcm = pcm;
    a.offsets = offsets;
    a.lengths = lengths;
    a.row_stride = row_stride;
    a.dense_len = (int32_t)std::min<int64_t>(row_stride > 0 ? row_stride : 0, kNSamples);
    a.pcm_format = pcm_format;
    a.n_mels = p->n_mels;
    a.B = B;
    a.out = out;
    a.gmax = gmax;
    a.out_format = p->out_format;
    return a;
}

static int launch_logmel(wlm_plan* p, const ClipArgs& a0, cudaStream_t st) {
    int n_launches = 0;
    bool flat_broken = false;
    ClipArgs a = a0;
    a.queue = p->d_queue;
    cudaError_t e = fused::launch(a, p->d_fused_tables, p->h_fused_tables, p->variant, p->max_clusters, st, &n_launches,
                                  p->flat_ctas, p->flat_override, &flat_broken);
    if (flat_broken) p->flat_ctas = 0;
    if (e != cudaSuccess) {
        cudaMemsetAsync(p->d_queue, 0, sizeof(ClipQueue), st);      // whatever was launched has left: start clean next time
        return fail(WLM_ERR_CUDA, "fused launch failed: %s", cudaGetErrorString(e));
    }
    p->launches += n_launches;
    WLM_CUDA(cudaGetLastError());
    return WLM_OK;
}

extern "C" int wlm_logmel(wlm_plan* p, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                          const int32_t* lengths_dev, int64_t row_stride, int B, void* out_dev,
                          float* gmax_dev, void* workspace, size_t workspace_bytes, void* stream) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (B == 0) return WLM_OK;
    if (!pcm_dev || !out_dev) return fail(WLM_ERR_BAD_ARG, "pcm_dev/out_dev is NULL");
    if (pcm_format != WLM_PCM_F32 && pcm_format != WLM_PCM_I16) return fail(WLM_ERR_BAD_ARG, "unknown pcm_format %d", pcm_format);
    if ((reinterpret_cast<uintptr_t>(pcm_dev) & 15) || (reinterpret_cast<uintptr_t>(out_dev) & 15))
        return fail(WLM_ERR_BAD_ARG, "pcm_dev and out_dev must be 16-byte aligned");
    if (!offsets_dev) {
        if (row_stride <= 0) return fail(WLM_ERR_BAD_ARG, "dense layout needs row_stride > 0 (got %lld)", (long long)row_stride);
        const int gran = pcm_format == WLM_PCM_I16 ? 8 : 4;
        if (row_stride % gran)
            return fail(WLM_ERR_BAD_ARG, "dense row_stride must be a multiple of %d elements (16 bytes), got %lld", gran, (long long)row_stride);
    } else if (!lengths_dev) {
        return fail(WLM_ERR_BAD_ARG, "ragged layout (offsets_dev) needs lengths_dev");
    }
    float* gmax = gmax_dev;
    if (!gmax) {
        const size_t need = wlm_workspace_bytes(p, B);
        if (!workspace || workspace_bytes < need)
            return fail(WLM_ERR_WORKSPACE, "workspace %zu B < required %zu B", workspace_bytes, need);
        gmax = static_cast<float*>(workspace);
    }
    WLM_CUDA(cudaSetDevice(p->device));
    const ClipArgs a = clip_args(p, pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, B, out_dev, gmax);
    return launch_logmel(p, a, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------
// attention mask (TF-FE:328-337)
// ------------------------------------------------------------------------------------------
__global__ void frame_mask_kernel(const int32_t* __restrict__ lengths, int B, int32_t* __restrict__ mask) {
    const int64_t total = (int64_t)B * kNFrames;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / kNFrames), t = (int)(i - (int64_t)b * kNFrames);
        const int len = max(0, min(lengths[b], kNSamples));
        mask[i] = (t * kHop < len) ? 1 : 0;
    }
}

extern "C" int wlm_frame_mask(wlm_plan* p, const int32_t* lengths_dev, int B, int32_t* mask_dev, void* stream) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (B == 0) return WLM_OK;
    if (!lengths_dev || !mask_dev) return fail(WLM_ERR_BAD_ARG, "lengths_dev/mask_dev is NULL");
    WLM_CUDA(cudaSetDevice(p->device));
    const int64_t total = (int64_t)B * kNFrames;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)p->sm_count * 8);
    frame_mask_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(lengths_dev, B, mask_dev);
    p->launches += 1;
    WLM_CUDA(cudaGetLastError());
    return WLM_OK;
}

// ------------------------------------------------------------------------------------------
// host-buffer end-to-end path
// ------------------------------------------------------------------------------------------
static bool is_pinned_host(const void* ptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

extern "C" int wlm_logmel_host(wlm_plan* p, const void* const* clips_host, const int32_t* lengths_host,
                               int pcm_format, int B, void* out_dev, void* out_host, void* stream) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (B == 0) return WLM_OK;
    if (!clips_host || !lengths_host || !out_dev) return fail(WLM_ERR_BAD_ARG, "clips_host/lengths_host/out_dev is NULL");
    if (pcm_format != WLM_PCM_F32 && pcm_format != WLM_PCM_I16) return fail(WLM_ERR_BAD_ARG, "unknown pcm_format %d", pcm_format);
    if (reinterpret_cast<uintptr_t>(out_dev) & 15) return fail(WLM_ERR_BAD_ARG, "out_dev must be 16-byte aligned");
    WLM_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t esz = pcm_format == WLM_PCM_I16 ? 2 : 4;
    const int64_t align_el = 16 / esz * 2;  // clip starts at 32-byte boundaries of the packed buffer

    // metadata
    if (B > p->meta_cap) {
        cudaFree(p->d_offsets); cudaFree(p->d_lengths);
        if (p->h_offsets) cudaFreeHost(p->h_offsets);
        if (p->h_lengths) cudaFreeHost(p->h_lengths);
        p->d_offsets = nullptr; p->d_lengths = nullptr; p->h_offsets = nullptr; p->h_lengths = nullptr;
        p->meta_cap = 0;
        const int cap = std::max(B, 256);
        WLM_CUDA(cudaMalloc(&p->d_offsets, sizeof(int64_t) * cap));
        WLM_CUDA(cudaMalloc(&p->d_lengths, sizeof(int32_t) * cap));
        WLM_CUDA(cudaMallocHost(&p->h_offsets, sizeof(int64_t) * cap));
        WLM_CUDA(cudaMallocHost(&p->h_lengths, sizeof(int32_t) * cap));
        p->meta_cap = cap;
    }
    // a previous call's kernels may still be reading the staging buffers / metadata
    if (p->kernels_done_valid) WLM_CUDA(cudaEventSynchronize(p->ev_kernels_done));

    int64_t total_el = 0;
    for (int b = 0; b < B; ++b) {
        if (lengths_host[b] < 0) return fail(WLM_ERR_BAD_ARG, "lengths_host[%d]=%d is negative", b, lengths_host[b]);
        if (lengths_host[b] > 0 && !clips_host[b]) return fail(WLM_ERR_BAD_ARG, "clips_host[%d] is NULL", b);
        const int32_t len = std::min<int32_t>(lengths_host[b], kNSamples);
        p->h_offsets[b] = total_el;
        p->h_lengths[b] = len;
        total_el += (len + align_el - 1) / align_el * align_el;
    }
    const size_t total_bytes = std::max<size_t>((size_t)total_el * esz, 256);
    if (total_bytes > p->d_stage_bytes) {
        cudaFree(p->d_stage);
        p->d_stage = nullptr; p->d_stage_bytes = 0;
        WLM_CUDA(cudaMalloc(&p->d_stage, total_bytes));
        p->d_stage_bytes = total_bytes;
    }
    const size_t ws_need = wlm_workspace_bytes(p, B);
    if (ws_need > p->d_ws_bytes) {
        cudaFree(p->d_ws);
        p->d_ws = nullptr; p->d_ws_bytes = 0;
        WLM_CUDA(cudaMalloc(&p->d_ws, ws_need));
        p->d_ws_bytes = ws_need;
    }
    // Small pageable batches -- the reference's own call shape, ONE clip per call (REF/data_utils/data_loader.py:171):
    // no ring bounce, no copy stream, no events.  cudaMemcpyAsync from pageable memory returns once the source has been
    // staged by the driver, so the host buffers are reusable on return without any synchronisation here.
    bool small_pageable = (size_t)total_el * esz <= (4u << 20);
    for (int b = 0; small_pageable && b < B; ++b)
        if (p->h_lengths[b] > 0 && is_pinned_host(clips_host[b])) small_pageable = false;
    if (small_pageable) {
        for (int b = 0; b < B; ++b)
            if (p->h_lengths[b] > 0)
                WLM_CUDA(cudaMemcpyAsync(static_cast<char*>(p->d_stage) + p->h_offsets[b] * esz, clips_host[b],
                                         (size_t)p->h_lengths[b] * esz, cudaMemcpyHostToDevice, st));
        WLM_CUDA(cudaMemcpyAsync(p->d_offsets, p->h_offsets, sizeof(int64_t) * B, cudaMemcpyHostToDevice, st));
        WLM_CUDA(cudaMemcpyAsync(p->d_lengths, p->h_lengths, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
        const ClipArgs a = clip_args(p, p->d_stage, pcm_format, p->d_offsets, p->d_lengths, 0, B, out_dev,
                                     static_cast<float*>(p->d_ws));
        int rc = launch_logmel(p, a, st);
        if (rc != WLM_OK) return rc;
        WLM_CUDA(cudaEventRecord(p->ev_kernels_done, st));
        p->kernels_done_valid = true;
        if (out_host) {
            WLM_CUDA(cudaMemcpyAsync(out_host, out_dev, out_elem_size(p) * (size_t)B * p->n_mels * kNFrames,
                                     cudaMemcpyDeviceToHost, st));
            WLM_CUDA(cudaStreamSynchronize(st));
        }
        return WLM_OK;
    }
    WLM_CUDA(cudaMemcpyAsync(p->d_offsets, p->h_offsets, sizeof(int64_t) * B, cudaMemcpyHostToDevice, p->copy_stream));
    WLM_CUDA(cudaMemcpyAsync(p->d_lengths, p->h_lengths, sizeof(int32_t) * B, cudaMemcpyHostToDevice, p->copy_stream));

    // chunks of ~48 MB of PCM: copy chunk c+1 while the kernels of chunk c run
    const size_t kChunkBytes = 48u << 20;
    const size_t kRingBytes = 64u << 20;
    int b0 = 0, chunk = 0, slot_uses[2] = {0, 0};
    while (b0 < B) {
        int b1 = b0;
        size_t bytes = 0;
        while (b1 < B && (b1 == b0 || bytes + (size_t)p->h_lengths[b1] * esz <= kChunkBytes)) {
            bytes += (size_t)p->h_lengths[b1] * esz;
            ++b1;
        }
        // copy clips [b0,b1): merge host-contiguous pinned runs into single copies
        int b = b0;
        while (b < b1) {
            const int32_t len = p->h_lengths[b];
            if (len == 0) { ++b; continue; }
            const char* src = static_cast<const char*>(clips_host[b]);
            char* dst = static_cast<char*>(p->d_stage) + p->h_offsets[b] * esz;
            if (is_pinned_host(src)) {
                size_t run = (size_t)len * esz;
                int e = b + 1;
                while (e < b1 && p->h_lengths[e] > 0 &&
                       static_cast<const char*>(clips_host[e]) == src + run &&
                       (size_t)(p->h_offsets[e] * esz) == (size_t)(p->h_offsets[b] * esz) + run)
                { run += (size_t)p->h_lengths[e] * esz; ++e; }
                WLM_CUDA(cudaMemcpyAsync(dst, src, run, cudaMemcpyHostToDevice, p->copy_stream));
                b = e;
            } else {
                // pageable source: bounce through the pinned ring, as many clips as fit
                if (!p->h_ring[0]) {
                    WLM_CUDA(cudaMallocHost(&p->h_ring[0], kRingBytes));
                    WLM_CUDA(cudaMallocHost(&p->h_ring[1], kRingBytes));
                    p->h_ring_bytes = kRingBytes;
                }
                const int slot = (slot_uses[0] + slot_uses[1]) & 1;
                if (slot_uses[slot]) WLM_CUDA(cudaEventSynchronize(p->ev_slot_free[slot]));
                char* ring = static_cast<char*>(p->h_ring[slot]);
                size_t used = 0;
                int e = b;
                const int64_t first_off = p->h_offsets[b];
                while (e < b1 && !is_pinned_host(clips_host[e] ? clips_host[e] : ring)) {
                    const size_t rel = (size_t)(p->h_offsets[e] - first_off) * esz;
                    const size_t nbytes = (size_t)p->h_lengths[e] * esz;
                    if (rel + nbytes > p->h_ring_bytes) break;
                    if (nbytes) memcpy(ring + rel, clips_host[e], nbytes);
                    used = rel + nbytes;
                    ++e;
                }
                if (e == b) return fail(WLM_ERR_BAD_ARG, "clip %d does not fit the staging ring", b);
                WLM_CUDA(cudaMemcpyAsync(dst, ring, used, cudaMemcpyHostToDevice, p->copy_stream));
                WLM_CUDA(cudaEventRecord(p->ev_slot_free[slot], p->copy_stream));
                slot_uses[slot]++;
                b = e;
            }
        }
        cudaEvent_t ev = p->ev_chunk[chunk & 3];
        WLM_CUDA(cudaEventRecord(ev, p->copy_stream));
        WLM_CUDA(cudaStreamWaitEvent(st, ev, 0));
        const ClipArgs a = clip_args(p, p->d_stage, pcm_format, p->d_offsets + b0, p->d_lengths + b0, 0, b1 - b0,
                                     static_cast<char*>(out_dev) + (size_t)b0 * p->n_mels * kNFrames * out_elem_size(p),
                                     static_cast<float*>(p->d_ws) + b0);
        int rc = launch_logmel(p, a, st);
        if (rc != WLM_OK) return rc;
        b0 = b1;
        ++chunk;
    }
    WLM_CUDA(cudaEventRecord(p->ev_kernels_done, st));
    p->kernels_done_valid = true;
    if (out_host) {
        WLM_CUDA(cudaMemcpyAsync(out_host, out_dev, out_elem_size(p) * (size_t)B * p->n_mels * kNFrames,
                                 cudaMemcpyDeviceToHost, st));
        WLM_CUDA(cudaStreamSynchronize(st));
    }
    // host buffers must be reusable on return
    WLM_CUDA(cudaStreamSynchronize(p->copy_stream));
    return WLM_OK;
}

