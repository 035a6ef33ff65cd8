// libwlm.so -- C ABI (include/wlm.h) over the sm_100a log-mel kernels.
//
// Host side only: plan construction (mel table -> sparse form, constant tables), argument
// validation, the launch policy (which kernel instance, how the clips split between the cluster
// kernel and its flat twin), the pinned-ring H2D pipeline of wlm_logmel_host.
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
#include "logmel_long.cuh"
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
// kernel instances
// ------------------------------------------------------------------------------------------
typedef void (*KernelFn)(const ClipArgs, const fused::KernelTables, const float*);

// variant: 80 / 128 when the table's structure equals the baked one (and the partition was taken from it)
template <class OutT, bool DYN>
static KernelFn kernel_for_t(int variant, bool flat) {
    using fused::logmel_cluster_kernel;
    if (flat) {
        if (variant == 80) return logmel_cluster_kernel<80, true, OutT, DYN>;
        if (variant == 128) return logmel_cluster_kernel<128, true, OutT, DYN>;
        return logmel_cluster_kernel<0, true, OutT, DYN>;
    }
    if (variant == 80) return logmel_cluster_kernel<80, false, OutT, DYN>;
    if (variant == 128) return logmel_cluster_kernel<128, false, OutT, DYN>;
    return logmel_cluster_kernel<0, false, OutT, DYN>;
}
static KernelFn kernel_for(int variant, bool flat, int out_format, bool dyn) {
    if (dyn) {
        if (out_format == WLM_OUT_BF16) return kernel_for_t<__nv_bfloat16, true>(variant, flat);
        if (out_format == WLM_OUT_F16) return kernel_for_t<__half, true>(variant, flat);
        return kernel_for_t<float, true>(variant, flat);
    }
    if (out_format == WLM_OUT_BF16) return kernel_for_t<__nv_bfloat16, false>(variant, flat);
    if (out_format == WLM_OUT_F16) return kernel_for_t<__half, false>(variant, flat);
    return kernel_for_t<float, false>(variant, flat);
}

typedef void (*LongKernelFn)(const longform::LongArgs, const fused::KernelTables, const float*);
typedef void (*ClampKernelFn)(const longform::LongArgs);

template <class OutT>
static LongKernelFn long_kernel_for_t(int variant) {
    using longform::logmel_long_kernel;
    if (variant == 80) return logmel_long_kernel<80, OutT>;
    if (variant == 128) return logmel_long_kernel<128, OutT>;
    return logmel_long_kernel<0, OutT>;
}
static LongKernelFn long_kernel_for(int variant, int out_format) {
    if (out_format == WLM_OUT_BF16) return long_kernel_for_t<__nv_bfloat16>(variant);
    if (out_format == WLM_OUT_F16) return long_kernel_for_t<__half>(variant);
    return long_kernel_for_t<float>(variant);
}

typedef void (*CondKernelFn)(const longform::LongArgs, const fused::KernelTables, const float*, const longform::CondArgs);

template <class OutT>
static CondKernelFn cond_kernel_for_t(int variant) {
    using longform::logmel_long_cond_kernel;
    if (variant == 80) return logmel_long_cond_kernel<80, OutT>;
    if (variant == 128) return logmel_long_cond_kernel<128, OutT>;
    return logmel_long_cond_kernel<0, OutT>;
}
static CondKernelFn cond_kernel_for(int variant, int out_format) {
    if (out_format == WLM_OUT_BF16) return cond_kernel_for_t<__nv_bfloat16>(variant);
    if (out_format == WLM_OUT_F16) return cond_kernel_for_t<__half>(variant);
    return cond_kernel_for_t<float>(variant);
}
static ClampKernelFn clamp_kernel_for(int out_format) {
    if (out_format == WLM_OUT_BF16) return longform::logmel_long_clamp_kernel<__nv_bfloat16>;
    if (out_format == WLM_OUT_F16) return longform::logmel_long_clamp_kernel<__half>;
    return longform::logmel_long_clamp_kernel<float>;
}

// launch configuration of the cluster kernel; the flat kernel uses the same one without the cluster dimension (at[0])
static void fill_launch_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* at, int n_clusters, cudaStream_t st) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->gridDim = dim3(fused::kCluster * n_clusters);
    cfg->blockDim = dim3(fused::kThreads);
    cfg->dynamicSmemBytes = fused::kSmemBytes;
    cfg->stream = st;
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = fused::kCluster;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    // the cluster kernel waits (griddepcontrol.wait) for its predecessor in the stream itself, after its prologue
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg->attrs = at;
    cfg->numAttrs = 2;
}

static cudaError_t configure(int variant, int* max_clusters) {
    cudaError_t e = cudaSuccess;
    for (int fmt : {WLM_OUT_F32, WLM_OUT_BF16, WLM_OUT_F16})
        for (int k = 0; k < 4; ++k) {
            e = cudaFuncSetAttribute(kernel_for(variant, (k & 1) != 0, fmt, (k & 2) != 0),
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, fused::kSmemBytes);
            if (e != cudaSuccess) return e;
        }
    for (int fmt : {WLM_OUT_F32, WLM_OUT_BF16, WLM_OUT_F16}) {
        e = cudaFuncSetAttribute(long_kernel_for(variant, fmt), cudaFuncAttributeMaxDynamicSharedMemorySize, fused::kSmemBytes);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(cond_kernel_for(variant, fmt), cudaFuncAttributeMaxDynamicSharedMemorySize, fused::kSmemBytes);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[2];
    fill_launch_config(&cfg, at, 148, nullptr);
    int n = 0;
    e = cudaOccupancyMaxActiveClusters(&n, kernel_for(variant, false, WLM_OUT_F32, false), &cfg);
    if (e != cudaSuccess) return e;
    if (n < 1) return cudaErrorLaunchOutOfResources;
    *max_clusters = n;
    return cudaSuccess;
}

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
    fused::KernelTables mel;
    float* d_win_lane = nullptr;
    ClipQueue* d_queue = nullptr;  // clip counter the two kernels of a launch pull from (self-resetting)
    int max_clusters = 0;          // co-resident clusters of the fused kernel (occupancy query)
    int flat_ctas = 0;             // SMs the clusters cannot cover: they run the flat kernel (programmatic dependent launch)
    int variant = 0;               // 80 / 128: unrolled mel stage (Whisper banks); 0: table-driven

    // wlm_logmel_host pipeline; its buffers only grow (grow_buffer), each *_bytes is the size allocated
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_slot_free[2] = {nullptr, nullptr};
    cudaEvent_t ev_kernels_done = nullptr;
    bool kernels_done_valid = false;
    void* d_stage = nullptr;  // packed PCM
    size_t d_stage_bytes = 0;
    void* h_ring[2] = {nullptr, nullptr};  // pinned
    size_t h_ring_bytes[2] = {0, 0};
    int64_t* d_offsets = nullptr;
    size_t d_offsets_bytes = 0;
    int32_t* d_lengths = nullptr;
    size_t d_lengths_bytes = 0;
    int64_t* h_offsets = nullptr;  // pinned
    size_t h_offsets_bytes = 0;
    int32_t* h_lengths = nullptr;  // pinned
    size_t h_lengths_bytes = 0;
    void* d_ws = nullptr;
    size_t d_ws_bytes = 0;
};

extern "C" int wlm_version(void) { return WLM_VERSION; }
extern "C" const char* wlm_last_error(void) { return g_last_error.c_str(); }

static int build_sparse(const float* dense, int n_mels, MelSparse* sp) {
    std::vector<int16_t> khi(n_mels, -1);  // last bin of filter m so far: its support must be contiguous
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
                if (khi[m] >= 0 && khi[m] != k - 1)
                    return fail(WLM_ERR_UNSUPPORTED, "mel table: filter %d has non-contiguous support at bin %d", m, k);
                khi[m] = (int16_t)k;
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

    MelSparse sparse;
    const int rc = build_sparse(mel_dense_host, n_mels, &sparse);
    if (rc != WLM_OK) return rc;
    fused::Tables tables;
    int variant = 0;
    if (fused::build_tables(sparse, n_mels, &tables, &variant) != 0)
        return fail(WLM_ERR_UNSUPPORTED, "mel table: a filter has no FFT bin (num_mel_filters too high for 201 bins)");

    wlm_plan* p = new wlm_plan();
    p->device = device;
    p->n_mels = n_mels;
    p->sm_count = prop.multiProcessorCount;
    p->variant = variant;
    p->mel = tables.mel;

#define WLM_CUDA_P(expr)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            wlm_plan_destroy(p);                                                                  \
            return fail(WLM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                         \
    } while (0)

    WLM_CUDA_P(cudaMalloc(&p->d_win_lane, sizeof(tables.win_lane)));
    WLM_CUDA_P(cudaMemcpy(p->d_win_lane, tables.win_lane, sizeof(tables.win_lane), cudaMemcpyHostToDevice));
    WLM_CUDA_P(cudaMalloc(&p->d_queue, sizeof(ClipQueue)));
    WLM_CUDA_P(cudaMemset(p->d_queue, 0, sizeof(ClipQueue)));
    cudaError_t fe = configure(p->variant, &p->max_clusters);
    if (fe != cudaSuccess) {
        wlm_plan_destroy(p);
        return fail(WLM_ERR_CUDA, "fused kernel configuration failed: %s", cudaGetErrorString(fe));
    }
    // the SMs that whole clusters cannot cover run the flat kernel (WLM_FLAT=0 turns that off)
    const char* fl = getenv("WLM_FLAT");
    p->flat_ctas = (fl && atoi(fl) == 0) ? 0 : std::max(0, p->sm_count - fused::kCluster * p->max_clusters);
    // read ONCE (not per launch); clamped to [0, B - 1] when used
    if (const char* fc = getenv("WLM_FLAT_CLIPS")) p->flat_override = std::max(-1, atoi(fc));

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
    cudaFree(p->d_win_lane);
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
// the per-call fields of a launch; launch_logmel fills in the queue and the work split (clip_first, n_workers, ...)
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

// The flat kernel runs on the `flat_ctas` SMs the clusters leave idle.  Next to a running cluster kernel a flat CTA needs
// about `rounds_per_clip` cluster rounds (one clip per co-resident cluster) for a clip (tools/flat_time.py), so it is only
// worth starting -- and, in a dynamic launch, only worth taking another clip -- while the clusters still have at least that
// many rounds of clips ahead of them; otherwise the whole GPU would wait for 16 SMs at the end of the batch.
static double flat_rounds_per_clip(int n_mels) { return 6.5 + 0.00625 * n_mels; }
static int flat_reserve_clips(int n_mels, int n_clusters) {
    return static_cast<int>(flat_rounds_per_clip(n_mels) * n_clusters + 0.999);
}
// static split of a dense batch: the largest number of whole flat rounds (one clip per flat CTA) that finish no later
// than the cluster kernel does with the rest
static int flat_clip_count(int B, int n_mels, int max_clusters, int flat_ctas) {
    if (flat_ctas <= 0 || B < 2 * max_clusters) return 0;
    const double rounds_per_clip = flat_rounds_per_clip(n_mels);
    int k = 0;
    while ((k + 1) * flat_ctas < B &&
           (k + 1) * rounds_per_clip <= (B - (k + 1) * flat_ctas + max_clusters - 1) / max_clusters) ++k;
    return k * flat_ctas;
}

// Which clips the cluster kernel and its flat twin take:
//   dense batch (no per-clip lengths), flat_override < 0:  STATIC -- clips [0, B - n_flat) round-robin over the clusters,
//       the last n_flat over the flat CTAs (every clip costs the same, so the split is known up front and the kernels carry
//       no queue code: the dynamic variant measured 6 % slower on dense batches);
//   everything else:  DYNAMIC -- both kernels pull clips from the plan's queue.
// flat_override: -1 = the rules above; 0 = no flat kernel; n > 0 = dynamic, the flat kernel may take up to n clips, no
// reserve (tests: any assignment must give bit-identical features).
struct Split {
    struct Part { int B, clip_first, n_workers, worker_base; };   // the ClipArgs fields that differ between the kernels
    bool dyn;
    int n_clusters;               // grid of the cluster kernel, in clusters
    int n_flat;                   // grid of the flat kernel, in CTAs; 0 = the cluster kernel runs alone
    int flat_reserve, flat_cap;   // ClipArgs fields, the same for both kernels
    Part cluster, flat;
};

static Split split_clips(int B, bool dense, int n_mels, int max_clusters, int flat_ctas, int flat_override) {
    Split s{};
    s.dyn = !(dense && flat_override < 0);
    s.flat_cap = 0x7fffffff;
    if (!s.dyn) {
        const int n_flat = flat_clip_count(B, n_mels, max_clusters, flat_ctas);
        s.n_clusters = std::min(B - n_flat, max_clusters);
        s.n_flat = std::min(n_flat, flat_ctas);
        s.cluster = {B - n_flat, 0, s.n_clusters, 0};
        s.flat = {B, B - n_flat, s.n_flat, 0};
        return s;
    }
    const int nc = std::min(B, max_clusters);
    int nf = 0;
    s.flat_reserve = flat_reserve_clips(n_mels, nc);
    if (flat_ctas > 0 && flat_override != 0) {
        if (flat_override > 0) {
            nf = std::min(std::min(flat_override, flat_ctas), B - nc);
            s.flat_reserve = 0;
            s.flat_cap = nf > 0 ? (flat_override + nf - 1) / nf : 0;
        } else {
            nf = std::min(B - s.flat_reserve, flat_ctas);
        }
        nf = std::max(nf, 0);
    }
    s.n_clusters = nc;
    s.n_flat = nf;
    s.cluster = {B, 0, nc + nf, 0};
    s.flat = {B, 0, nc + nf, nc};
    return s;
}

// One launch = the cluster kernel plus, when it pays, its flat twin, as a PROGRAMMATIC DEPENDENT launch: the flat kernel
// becomes schedulable when every CTA of the cluster kernel has executed griddepcontrol.launch_dependents, i.e. is resident --
// its CTAs can then only land on the SMs the clusters left free.  (Submitted as an independent kernel on a second stream it
// sometimes got SMs first and kept clusters from being placed.)  It consumes nothing the cluster kernel produces; it
// executes griddepcontrol.wait just before it exits, so the last kernel in the stream completes after both have written
// everything and later work in the stream is ordered behind both.
static int launch_logmel(wlm_plan* p, ClipArgs a, cudaStream_t st) {
    const Split s = split_clips(a.B, a.lengths == nullptr, a.n_mels, p->max_clusters, p->flat_ctas, p->flat_override);
    a.queue = p->d_queue;
    a.flat_reserve = s.flat_reserve;
    a.flat_cap = s.flat_cap;
    auto args = [&](const Split::Part& k) {
        ClipArgs r = a;
        r.B = k.B;
        r.clip_first = k.clip_first;
        r.n_workers = k.n_workers;
        r.worker_base = k.worker_base;
        return r;
    };
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[2];
    fill_launch_config(&cfg, at, s.n_clusters, st);
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel_for(p->variant, false, a.out_format, s.dyn), args(s.cluster), p->mel,
                                       p->d_win_lane);
    if (e == cudaSuccess && s.n_flat > 0) {
        const KernelFn flat_fn = kernel_for(p->variant, true, a.out_format, s.dyn);
        cfg.gridDim = dim3(s.n_flat);
        cfg.attrs = at + 1;   // programmatic stream serialisation only
        cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, flat_fn, args(s.flat), p->mel, p->d_win_lane);
        if (e != cudaSuccess) {
            // the dependent launch was refused (driver without programmatic launches?): the flat CTAs' clips are already
            // theirs, so the same kernel goes out as an ordinary launch (it then runs after the cluster kernel) and the
            // plan stops using it
            (void)cudaGetLastError();
            p->flat_ctas = 0;
            cfg.attrs = nullptr;
            cfg.numAttrs = 0;
            e = cudaLaunchKernelEx(&cfg, flat_fn, args(s.flat), p->mel, p->d_win_lane);
        }
    }
    if (e != cudaSuccess) {
        cudaMemsetAsync(p->d_queue, 0, sizeof(ClipQueue), st);      // whatever was launched has left: start clean next time
        return fail(WLM_ERR_CUDA, "fused launch failed: %s", cudaGetErrorString(e));
    }
    p->launches += s.n_flat > 0 ? 2 : 1;
    WLM_CUDA(cudaGetLastError());
    return WLM_OK;
}

// the batch arguments of every device-buffer entry point (B > 0): pointers, PCM format, alignment and layout
static int check_batch(const void* pcm_dev, int pcm_format, const int64_t* offsets_dev, const int32_t* lengths_dev,
                       int64_t row_stride, const void* out_dev) {
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
    return WLM_OK;
}

extern "C" int wlm_logmel(wlm_plan* p, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                          const int32_t* lengths_dev, int64_t row_stride, int B, void* out_dev,
                          float* gmax_dev, void* workspace, size_t workspace_bytes, void* stream) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (B == 0) return WLM_OK;
    const int rc = check_batch(pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, out_dev);
    if (rc != WLM_OK) return rc;
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
// [B][n_frames] of clips padded (or trimmed) to n_samples: 1 where 160 t < min(len, n_samples)
__global__ void frame_mask_kernel(const int32_t* __restrict__ lengths, int B, int n_frames, int n_samples,
                                  int32_t* __restrict__ mask) {
    const int64_t total = (int64_t)B * n_frames;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(i / n_frames), t = (int)(i - (int64_t)b * n_frames);
        const int len = max(0, min(lengths[b], n_samples));
        mask[i] = (t * kHop < len) ? 1 : 0;
    }
}

static int launch_frame_mask(wlm_plan* p, const int32_t* lengths_dev, int B, int n_frames, int n_samples, int32_t* mask_dev,
                             void* stream) {
    if (!lengths_dev || !mask_dev) return fail(WLM_ERR_BAD_ARG, "lengths_dev/mask_dev is NULL");
    WLM_CUDA(cudaSetDevice(p->device));
    const int64_t total = (int64_t)B * n_frames;
    const int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)p->sm_count * 8);
    frame_mask_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(lengths_dev, B, n_frames, n_samples, mask_dev);
    p->launches += 1;
    WLM_CUDA(cudaGetLastError());
    return WLM_OK;
}

extern "C" int wlm_frame_mask(wlm_plan* p, const int32_t* lengths_dev, int B, int32_t* mask_dev, void* stream) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (B == 0) return WLM_OK;
    return launch_frame_mask(p, lengths_dev, B, kNFrames, kNSamples, mask_dev, stream);
}

// torch.stft(center=True) needs more than n_fft / 2 samples to reflect; the frame index 160 t stays in int32
static int check_padded_len(int64_t padded_len) {
    if (padded_len <= kNfft / 2 || padded_len > INT32_MAX)
        return fail(WLM_ERR_BAD_ARG, "padded_len=%lld outside [%d, %d]", (long long)padded_len, kNfft / 2 + 1, INT32_MAX);
    return WLM_OK;
}

extern "C" int wlm_frame_mask_padded(wlm_plan* p, const int32_t* lengths_dev, int B, int64_t padded_len, int32_t* mask_dev,
                                     void* stream) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (check_padded_len(padded_len) != WLM_OK) return WLM_ERR_BAD_ARG;
    if (B == 0) return WLM_OK;
    return launch_frame_mask(p, lengths_dev, B, (int)(padded_len / kHop), (int)padded_len, mask_dev, stream);
}

// ------------------------------------------------------------------------------------------
// long-form features: any padded length (logmel_long.cuh)
// ------------------------------------------------------------------------------------------
// workspace: the per-clip maximum of the mel power, then the unit counter
static size_t padded_max_bytes(int B) { return ((size_t)B * sizeof(int) + 255) / 256 * 256; }

extern "C" size_t wlm_padded_workspace_bytes(const wlm_plan* p, int B) {
    if (!p || B <= 0) return 0;
    return padded_max_bytes(B) + 256;
}

// the checks of wlm_logmel_padded and wlm_logmel_conditioned before the workspace
static int check_padded_call(const wlm_plan* p, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                             const int32_t* lengths_dev, int64_t row_stride, int64_t padded_len, int B, const void* out_dev) {
    if (!p) return fail(WLM_ERR_BAD_ARG, "plan is NULL");
    if (B < 0) return fail(WLM_ERR_BAD_ARG, "B=%d is negative", B);
    if (check_padded_len(padded_len) != WLM_OK) return WLM_ERR_BAD_ARG;
    if (B == 0) return WLM_OK;
    return check_batch(pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, out_dev);
}

static int check_workspace(const void* workspace, size_t workspace_bytes, size_t need) {
    if (!workspace || workspace_bytes < need)
        return fail(WLM_ERR_WORKSPACE, "workspace %zu B < required %zu B", workspace_bytes, need);
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return fail(WLM_ERR_BAD_ARG, "workspace must be 16-byte aligned");
    return WLM_OK;
}

// pass-1 arguments; the workspace starts with the per-clip maxima and the unit counter (wlm_padded_workspace_bytes)
static longform::LongArgs long_args(const wlm_plan* p, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                                    const int32_t* lengths_dev, int64_t row_stride, int64_t padded_len, int B, void* out_dev,
                                    float* gmax_dev, void* workspace) {
    longform::LongArgs a{};
    a.pcm = pcm_dev;
    a.offsets = offsets_dev;
    a.lengths = lengths_dev;
    a.row_stride = offsets_dev ? 0 : row_stride;
    a.padded_len = (int32_t)padded_len;
    a.n_frames = (int32_t)(padded_len / kHop);
    a.n_tiles = (a.n_frames + fused::kTile - 1) / fused::kTile;
    a.units_per_clip = (a.n_tiles + longform::kLongRun - 1) / longform::kLongRun;
    a.pcm_format = pcm_format;
    a.n_mels = p->n_mels;
    a.B = B;
    a.out = out_dev;
    a.gmax = gmax_dev;
    a.pmax = static_cast<int*>(workspace);
    a.next_unit = reinterpret_cast<unsigned long long*>(static_cast<char*>(workspace) + padded_max_bytes(B));
    return a;
}

static int64_t long_ctas(const wlm_plan* p, const longform::LongArgs& a) {
    const int64_t units = (int64_t)a.B * a.units_per_clip;
    return std::min<int64_t>(p->sm_count, (units + fused::kGroups - 1) / fused::kGroups);
}

// pass 2; `a` says which half-tiles pass 1 wrote (long_clip's n_act)
static void launch_clamp(const wlm_plan* p, const longform::LongArgs& a, cudaStream_t st) {
    const int64_t vecs = ((int64_t)a.n_mels * a.n_frames * (int64_t)out_elem_size(p) + 15) / 16;
    const int gy = std::min(a.B, 65535);
    const int gx = (int)std::max<int64_t>(1, std::min<int64_t>((vecs + 1023) / 1024, std::max(1, 8 * p->sm_count / gy)));
    clamp_kernel_for(p->out_format)<<<dim3(gx, gy), 256, 0, st>>>(a);
}

// conditioned calls (do_normalize, dither); workspace: that of wlm_logmel_padded, then the per-clip moments [B] float2,
// then the moments partials [B][n_chunks] double2
static int64_t moment_chunks(int64_t padded_len) { return (padded_len + longform::kMomChunk - 1) / longform::kMomChunk; }
static size_t moments_bytes(int B) { return ((size_t)B * sizeof(float2) + 255) / 256 * 256; }

extern "C" size_t wlm_conditioned_workspace_bytes(const wlm_plan* p, int B, int64_t padded_len) {
    if (!p || B <= 0 || padded_len <= kNfft / 2 || padded_len > INT32_MAX) return 0;
    return wlm_padded_workspace_bytes(p, B) + moments_bytes(B) + (size_t)B * moment_chunks(padded_len) * sizeof(double2);
}

// The launches of a checked long-form call, plain and in stream order: pass 1 starts after everything before it, pass 2
// after pass 1.  With nothing to condition, pass 1 is logmel_long_kernel and only wlm_logmel_padded's workspace is used.
static int launch_long(wlm_plan* p, const longform::LongArgs& a, int do_normalize, float dither, uint64_t seed,
                       void* workspace, cudaStream_t st) {
    const size_t padded_bytes = wlm_padded_workspace_bytes(p, a.B);
    WLM_CUDA(cudaMemsetAsync(workspace, 0, padded_bytes, st));
    int launches = 2;
    longform::CondArgs c{};
    if (do_normalize) {
        char* ws = static_cast<char*>(workspace) + padded_bytes;
        float2* moments = reinterpret_cast<float2*>(ws);
        double2* partial = reinterpret_cast<double2*>(ws + moments_bytes(a.B));
        const int n_chunks = (int)moment_chunks(a.padded_len);
        longform::logmel_moments_kernel<<<dim3(n_chunks, std::min(a.B, 65535)), longform::kMomThreads, 0, st>>>(a, partial, n_chunks);
        WLM_CUDA(cudaGetLastError());
        const int blocks = (int)std::min<int64_t>(((int64_t)a.B * 32 + 255) / 256, (int64_t)p->sm_count * 8);
        longform::logmel_moments_merge_kernel<<<blocks, 256, 0, st>>>(a, partial, n_chunks, moments);
        WLM_CUDA(cudaGetLastError());
        c.moments = moments;
        launches += 2;
    }
    const int ctas = (int)long_ctas(p, a);
    if (!do_normalize && dither == 0.0f) {
        long_kernel_for(p->variant, p->out_format)<<<ctas, fused::kThreads, fused::kSmemBytes, st>>>(a, p->mel, p->d_win_lane);
    } else {
        c.dither = dither;
        c.key0 = (uint32_t)seed;
        c.key1 = (uint32_t)(seed >> 32);
        cond_kernel_for(p->variant, p->out_format)<<<ctas, fused::kThreads, fused::kSmemBytes, st>>>(a, p->mel, p->d_win_lane, c);
    }
    WLM_CUDA(cudaGetLastError());
    longform::LongArgs a2 = a;
    if (dither != 0.0f) {
        // pass 2 sees every clip as L samples long: every half-tile was written by pass 1
        a2.offsets = nullptr;
        a2.lengths = nullptr;
        a2.row_stride = a.padded_len;
    }
    launch_clamp(p, a2, st);
    p->launches += launches;
    WLM_CUDA(cudaGetLastError());
    return WLM_OK;
}

extern "C" int wlm_logmel_padded(wlm_plan* p, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                                 const int32_t* lengths_dev, int64_t row_stride, int64_t padded_len, int B, void* out_dev,
                                 float* gmax_dev, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_padded_call(p, pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, padded_len, B, out_dev);
    if (rc != WLM_OK || B == 0) return rc;
    if ((rc = check_workspace(workspace, workspace_bytes, wlm_padded_workspace_bytes(p, B))) != WLM_OK) return rc;
    WLM_CUDA(cudaSetDevice(p->device));
    return launch_long(p, long_args(p, pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, padded_len, B, out_dev, gmax_dev,
                                    workspace),
                       0, 0.0f, 0, workspace, static_cast<cudaStream_t>(stream));
}

extern "C" int wlm_logmel_conditioned(wlm_plan* p, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                                      const int32_t* lengths_dev, int64_t row_stride, int64_t padded_len, int B,
                                      int do_normalize, float dither, uint64_t seed, void* out_dev, float* gmax_dev,
                                      void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_padded_call(p, pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, padded_len, B, out_dev);
    if (rc != WLM_OK) return rc;
    if (!std::isfinite(dither)) return fail(WLM_ERR_BAD_ARG, "dither=%g is not finite", (double)dither);
    if (B == 0) return WLM_OK;
    if ((rc = check_workspace(workspace, workspace_bytes, wlm_conditioned_workspace_bytes(p, B, padded_len))) != WLM_OK) return rc;
    WLM_CUDA(cudaSetDevice(p->device));
    return launch_long(p, long_args(p, pcm_dev, pcm_format, offsets_dev, lengths_dev, row_stride, padded_len, B, out_dev, gmax_dev,
                                    workspace),
                       do_normalize, dither, seed, workspace, static_cast<cudaStream_t>(stream));
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

// Grows a buffer of the plan (device memory, or pinned host memory) to at least `bytes`; *cap is its allocated size.
template <class T>
static cudaError_t grow_buffer(T** buf, size_t* cap, size_t bytes, bool pinned) {
    if (bytes <= *cap) return cudaSuccess;
    void** b = reinterpret_cast<void**>(buf);
    if (*b) {
        if (pinned) cudaFreeHost(*b);
        else cudaFree(*b);
    }
    *b = nullptr;
    *cap = 0;
    const cudaError_t e = pinned ? cudaMallocHost(b, bytes) : cudaMalloc(b, bytes);
    if (e == cudaSuccess) *cap = bytes;
    return e;
}

static constexpr size_t kRingBytes = 64u << 20;   // each of the two pinned slots pageable clips bounce through

// wlm_logmel_host for all but small pageable batches: the PCM goes over on the plan's copy stream, chunk by chunk, and
// every chunk's kernels wait for its copies only.  h_offsets / h_lengths hold the batch's layout already.
static int launch_chunked(wlm_plan* p, const void* const* clips_host, int pcm_format, size_t esz, int B, void* out_dev,
                          cudaStream_t st) {
    WLM_CUDA(cudaMemcpyAsync(p->d_offsets, p->h_offsets, sizeof(int64_t) * B, cudaMemcpyHostToDevice, p->copy_stream));
    WLM_CUDA(cudaMemcpyAsync(p->d_lengths, p->h_lengths, sizeof(int32_t) * B, cudaMemcpyHostToDevice, p->copy_stream));

    // chunks of ~48 MB of PCM: copy chunk c+1 while the kernels of chunk c run
    const size_t kChunkBytes = 48u << 20;
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
                for (int r = 0; r < 2; ++r) WLM_CUDA(grow_buffer(&p->h_ring[r], &p->h_ring_bytes[r], kRingBytes, true));
                const int slot = (slot_uses[0] + slot_uses[1]) & 1;
                if (slot_uses[slot]) WLM_CUDA(cudaEventSynchronize(p->ev_slot_free[slot]));
                char* ring = static_cast<char*>(p->h_ring[slot]);
                size_t used = 0;
                int e = b;
                const int64_t first_off = p->h_offsets[b];
                while (e < b1 && !is_pinned_host(clips_host[e] ? clips_host[e] : ring)) {
                    const size_t rel = (size_t)(p->h_offsets[e] - first_off) * esz;
                    const size_t nbytes = (size_t)p->h_lengths[e] * esz;
                    if (rel + nbytes > kRingBytes) break;
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
    return WLM_OK;
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

    // a previous call's kernels may still be reading the staging buffers / metadata: wait before reusing or replacing them
    if (p->kernels_done_valid) WLM_CUDA(cudaEventSynchronize(p->ev_kernels_done));
    const size_t meta_n = std::max(B, 256);
    WLM_CUDA(grow_buffer(&p->d_offsets, &p->d_offsets_bytes, sizeof(int64_t) * meta_n, false));
    WLM_CUDA(grow_buffer(&p->d_lengths, &p->d_lengths_bytes, sizeof(int32_t) * meta_n, false));
    WLM_CUDA(grow_buffer(&p->h_offsets, &p->h_offsets_bytes, sizeof(int64_t) * meta_n, true));
    WLM_CUDA(grow_buffer(&p->h_lengths, &p->h_lengths_bytes, sizeof(int32_t) * meta_n, true));

    int64_t total_el = 0;
    for (int b = 0; b < B; ++b) {
        if (lengths_host[b] < 0) return fail(WLM_ERR_BAD_ARG, "lengths_host[%d]=%d is negative", b, lengths_host[b]);
        if (lengths_host[b] > 0 && !clips_host[b]) return fail(WLM_ERR_BAD_ARG, "clips_host[%d] is NULL", b);
        const int32_t len = std::min<int32_t>(lengths_host[b], kNSamples);
        p->h_offsets[b] = total_el;
        p->h_lengths[b] = len;
        total_el += (len + align_el - 1) / align_el * align_el;
    }
    WLM_CUDA(grow_buffer(&p->d_stage, &p->d_stage_bytes, std::max<size_t>((size_t)total_el * esz, 256), false));
    WLM_CUDA(grow_buffer(&p->d_ws, &p->d_ws_bytes, wlm_workspace_bytes(p, B), false));
    // Small pageable batches -- the reference's own call shape, ONE clip per call (REF/data_utils/data_loader.py:171):
    // no ring bounce, no copy stream, no events.  cudaMemcpyAsync from pageable memory returns once the source has been
    // staged by the driver, so the host buffers are reusable on return without any synchronisation here.
    bool small_pageable = (size_t)total_el * esz <= (4u << 20);
    for (int b = 0; small_pageable && b < B; ++b)
        if (p->h_lengths[b] > 0 && is_pinned_host(clips_host[b])) small_pageable = false;
    int rc;
    if (small_pageable) {
        for (int b = 0; b < B; ++b)
            if (p->h_lengths[b] > 0)
                WLM_CUDA(cudaMemcpyAsync(static_cast<char*>(p->d_stage) + p->h_offsets[b] * esz, clips_host[b],
                                         (size_t)p->h_lengths[b] * esz, cudaMemcpyHostToDevice, st));
        WLM_CUDA(cudaMemcpyAsync(p->d_offsets, p->h_offsets, sizeof(int64_t) * B, cudaMemcpyHostToDevice, st));
        WLM_CUDA(cudaMemcpyAsync(p->d_lengths, p->h_lengths, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
        rc = launch_logmel(p, clip_args(p, p->d_stage, pcm_format, p->d_offsets, p->d_lengths, 0, B, out_dev,
                                        static_cast<float*>(p->d_ws)), st);
    } else {
        rc = launch_chunked(p, clips_host, pcm_format, esz, B, out_dev, st);
    }
    if (rc != WLM_OK) return rc;
    WLM_CUDA(cudaEventRecord(p->ev_kernels_done, st));
    p->kernels_done_valid = true;
    if (out_host) {
        WLM_CUDA(cudaMemcpyAsync(out_host, out_dev, out_elem_size(p) * (size_t)B * p->n_mels * kNFrames,
                                 cudaMemcpyDeviceToHost, st));
        WLM_CUDA(cudaStreamSynchronize(st));
    }
    // host buffers must be reusable on return: the chunked path's copies may still be in flight
    if (!small_pageable) WLM_CUDA(cudaStreamSynchronize(p->copy_stream));
    return WLM_OK;
}
