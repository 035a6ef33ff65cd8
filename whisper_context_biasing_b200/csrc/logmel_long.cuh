// Long-form log-mel kernels for sm_100a: features of clips padded to ANY common length L (HF's
// `truncation=False, padding="longest"`), [B][n_mels][T] with T = L / 160.
//
// Every frame of a clip depends on the clip's maximum over ALL its frames (the max - 8 clamp), and a
// clip of 20 minutes does not fit on chip, so the work is split in two passes:
//
//   pass 1  logmel_long_kernel: a persistent grid of one CTA per SM, two independent groups of 8 warps,
//           the same pipeline stages and shared-memory layout as logmel_fused.cuh.  A group pulls UNITS
//           -- a run of kLongRun consecutive half-tiles of one clip -- from a counter in the workspace and
//           writes (max(log10 p, -10) + 4) / 4 straight to HBM (as the flat twin of the fused kernel does),
//           keeping the running maximum of the mel POWER in registers.  At the end of a unit the group's
//           maximum goes to the clip's slot with ONE atomicMax (non-negative floats order like their bit
//           patterns).  Half-tiles with no real sample are not computed.
//   pass 2  logmel_long_clamp_kernel: clip b owns [b M T, (b+1) M T) of the output; every element becomes
//           max(x, thr_b) with thr_b = (max(log10 pmax_b - 8, -10) + 4) / 4 rounded to the output type
//           (max(round x, round t) = round max(x, t): the 16-bit formats stay exact).  Frames of half-tiles
//           pass 1 skipped are written as thr_b without being read.
//
// At L = 480000 both passes reproduce wlm_logmel bit for bit: the raw buffer holds the same values (same
// reflection and zero fill), stages 1/2 and the mel stage are the same code, and the clamp is the flat
// kernel's.
//
// A conditioned call (wlm_logmel_conditioned: do_normalize, dither) runs logmel_long_cond_kernel, the same pass 1
// with cond_fixup on every half-tile, and, for do_normalize, the per-clip moments kernels before it.  Pass 2 is
// unchanged.
#pragma once
#include "logmel_fused.cuh"

namespace wlm {
namespace longform {

using fused::kGroups; using fused::kGroupWarps; using fused::kGroupThreads; using fused::kThreads;
using fused::kTile; using fused::kSubLen; using fused::kSubStep; using fused::kTileSamples; using fused::kRawShift;
using fused::kSmemRaw; using fused::kSmemY; using fused::kSmemGroup; using fused::kYWarpFloat2; using fused::kYN1;
using fused::kYLanes; using fused::kMaxFiltersPerWarp; using fused::KernelTables;

// half-tiles per unit of work.  Long enough that the per-unit costs (one counter atomic, one atomicMax on the
// clip's maximum, the pipeline bubble of the unit's first copy) stay small, short enough that the last units of a
// batch do not leave most groups idle.
constexpr int kLongRun = 8;

struct LongArgs {
    const void* pcm;                 // f32 or i16
    const int64_t* offsets;          // nullptr -> b * row_stride
    const int32_t* lengths;          // nullptr -> row_stride valid samples (dense)
    int64_t row_stride;
    int32_t padded_len;              // L: every clip is zero-padded to L, reflected at 0 and at L
    int32_t n_frames;                // T = L / 160
    int32_t n_tiles;                 // ceil(T / 32) half-tiles per clip
    int32_t units_per_clip;          // ceil(n_tiles / kLongRun)
    int32_t pcm_format;              // WLM_PCM_*
    int32_t n_mels;
    int32_t B;
    void* out;                       // [B][n_mels][T], element type OutT
    float* gmax;                     // optional [B]
    int* pmax;                       // [B] workspace: max mel power of clip b (float bits, zeroed before pass 1)
    unsigned long long* next_unit;   // workspace: the unit counter (zeroed before pass 1)
};

struct LongClip {
    int64_t base;   // element offset of the clip in the PCM buffer
    int64_t len;    // valid samples, <= L
    int n_act;      // half-tiles that contain any real sample
};

__device__ __forceinline__ LongClip long_clip(const LongArgs& a, int b) {
    LongClip c;
    c.base = a.offsets ? a.offsets[b] : static_cast<int64_t>(b) * a.row_stride;
    int64_t len = a.lengths ? static_cast<int64_t>(a.lengths[b]) : a.row_stride;
    if (!a.offsets) len = min(len, a.row_stride);
    c.len = max(static_cast<int64_t>(0), min(len, static_cast<int64_t>(a.padded_len)));
    // half-tile t starts at sample 5120 t - 200: active iff that is < len
    c.n_act = static_cast<int>(min(static_cast<int64_t>(a.n_tiles), (c.len + kNfft / 2 + kTile * kHop - 1) / (kTile * kHop)));
    return c;
}
__device__ __forceinline__ int64_t long_s0(int tile) { return static_cast<int64_t>(tile) * (kTile * kHop) - kNfft / 2; }

// issued by one thread: both sub-regions of the half-tile, valid sample range only (fused::tile_issue_tma without
// the 480000 cap, with 64-bit sample positions)
__device__ __forceinline__ void long_issue_tma(const LongArgs& a, const LongClip& c, int tile, float* raw, uint32_t bar) {
    using fused::mbar_expect_tx; using fused::tma_bulk_g2s; using fused::smem_u32;
    const int64_t s0 = long_s0(tile);
    const int esz = a.pcm_format == WLM_PCM_I16 ? 2 : 4;
    const uint32_t dst0 = smem_u32(raw) + (esz == 4 ? 0u : static_cast<uint32_t>(kSubLen) * 4u);
    if (s0 >= 0 && s0 + kTileSamples <= c.len) {
        const uint32_t bytes = static_cast<uint32_t>(kSubLen * esz);
        mbar_expect_tx(bar, 2u * bytes);
        const char* src = static_cast<const char*>(a.pcm) + (c.base + s0) * esz;
        tma_bulk_g2s(dst0, src, bytes, bar);
        tma_bulk_g2s(dst0 + bytes, src + static_cast<int64_t>(kSubStep) * esz, bytes, bar);
        return;
    }
    const int64_t gmask = esz == 4 ? 3 : 7;      // copies are whole 16-byte units
    const int64_t len_up = (c.len + gmask) & ~gmask;
    uint32_t total = 0;
    int64_t lo[2];
    int n[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int64_t s_lo = s0 + r * kSubStep;
        lo[r] = max(s_lo, static_cast<int64_t>(0));
        const int64_t hi = min(s_lo + kSubLen, len_up);
        n[r] = static_cast<int>(max(hi - lo[r], static_cast<int64_t>(0)));
        total += static_cast<uint32_t>(n[r]) * esz;
    }
    mbar_expect_tx(bar, total);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        if (n[r] <= 0) continue;
        const int64_t s_lo = s0 + r * kSubStep;
        const char* src = static_cast<const char*>(a.pcm) + (c.base + lo[r]) * esz;
        const uint32_t dst = dst0 + static_cast<uint32_t>(r * kSubLen + (lo[r] - s_lo)) * static_cast<uint32_t>(esz);
        tma_bulk_g2s(dst, src, static_cast<uint32_t>(n[r]) * esz, bar);
    }
}

// int16 -> float32 expansion in place (as fused::tile_fixup).  Runs on the 256 threads of one group.
__device__ __forceinline__ void long_expand_i16(float* raw, int grp, int tg) {
    using fused::group_sync;
    const int16_t* st = reinterpret_cast<const int16_t*>(raw + kSubLen);
    constexpr float kScale = 1.0f / 32768.0f;
    constexpr int kPer = (kSubLen + kGroupThreads - 1) / kGroupThreads;
#pragma unroll 1
    for (int i = tg; i < kSubLen; i += kGroupThreads) raw[i] = static_cast<float>(st[i]) * kScale;
    float tmp[kPer];
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
        const int i = tg + j * kGroupThreads;
        tmp[j] = i < kSubLen ? static_cast<float>(st[kSubLen + i]) * kScale : 0.f;
    }
    group_sync(grp);
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
        const int i = tg + j * kGroupThreads;
        if (i < kSubLen) raw[kSubLen + i] = tmp[j];
    }
    group_sync(grp);
}

// int16 expansion, then every position outside [0, len) of the half-tile: reflection at sample 0 (s < 0 -> -s),
// reflection at L (s >= L -> 2 (L - 1) - s; torch.stft center=True pads the L-sample array at both ends), zero padding in
// [len, L).  A reflected position only reads samples inside [0, len), which nobody patches; positions whose reflection
// falls outside the half-tile belong to frames >= T (never stored).
// Runs on the 256 threads of one group; the condition for calling it is group-uniform.
__device__ __forceinline__ void long_fixup(int pcm_format, int64_t len, int64_t L, int tile, float* raw, int grp, int tg) {
    using fused::group_sync;
    const int64_t s0 = long_s0(tile);
    if (pcm_format == WLM_PCM_I16) long_expand_i16(raw, grp, tg);
    if (s0 < 0 || s0 + kTileSamples > len) {
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
            const int64_t s_lo = s0 + r * kSubStep;
#pragma unroll 1
            for (int i = tg; i < kSubLen; i += kGroupThreads) {
                const int64_t s = s_lo + i;
                if (s >= 0 && s < len) continue;
                const int64_t sr = s < 0 ? -s : (s >= L ? 2 * (L - 1) - s : -1);     // -1: zero padding
                float v = 0.f;
                if (sr >= 0 && sr < len) {
                    const int64_t u = sr - s0;
                    if (u >= 0 && u < kTileSamples) v = raw[u < kSubLen ? u : kSubLen + (u - kSubStep)];
                }
                raw[r * kSubLen + i] = v;
            }
        }
        group_sync(grp);
    }
}

// ---- conditioning: do_normalize and dither (wlm_logmel_conditioned) ----------------------------------------------
struct CondArgs {
    const float2* moments;   // [B] (mean, 1 / sqrt(var + 1e-7)) of x[:len]; nullptr: no normalisation
    float dither;            // 0: no noise
    uint32_t key0, key1;     // Philox key: lo32 / hi32 of the seed
};

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants) of counter (c0, c1, 0, 0), then Box-Muller on (u0, u1) and
// (u2, u3) with u = ((r >> 8) + 0.5) 2^-24: four standard normal values.  The stream of include/wlm.h.
__device__ __forceinline__ void philox_normal4(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, float (&z)[4]) {
    uint32_t x0 = c0, x1 = c1, x2 = 0u, x3 = 0u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
        x0 = hi1 ^ x1 ^ k0; x1 = lo1; x2 = hi0 ^ x3 ^ k1; x3 = lo0;
    }
    const uint32_t w[4] = {x0, x1, x2, x3};
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        const float ua = fmaf(static_cast<float>(w[2 * p] >> 8), 0x1p-24f, 0x1p-25f);
        const float ub = fmaf(static_cast<float>(w[2 * p + 1] >> 8), 0x1p-24f, 0x1p-25f);
        const float rad = sqrtf(-2.0f * logf(ua));
        float sn, cs;
        sincospif(2.0f * ub, &sn, &cs);
        z[2 * p] = rad * cs;
        z[2 * p + 1] = rad * sn;
    }
}

// long_fixup for a conditioned call, on EVERY half-tile (also those the TMA filled completely), in HF's order:
//   1. every position with sample s in [0, L): (x - mean) scale on [0, len) (x when not normalising), 0 on [len, L), then
//      + dither z(seed, b, s).  A thread takes four consecutive samples: half-tiles and sub-regions start at multiples of
//      4, so one Philox call serves the quad;
//   2. then the positions outside [0, L) are reflected from the CONDITIONED values (a source may lie in the pad region,
//      which carries noise).
// The two sub-regions overlap by 240 samples; both copies get the same value, as z depends on (b, s) only.
__device__ __forceinline__ void cond_fixup(const CondArgs& cnd, int pcm_format, int b, float2 ms, int64_t len, int64_t L,
                                           int tile, float* raw, int grp, int tg) {
    using fused::group_sync;
    const int64_t s0 = long_s0(tile);
    if (pcm_format == WLM_PCM_I16) long_expand_i16(raw, grp, tg);
    constexpr int kQuads = kSubLen / 4;
    static_assert(kSubLen % 4 == 0 && kSubStep % 4 == 0 && (kTile * kHop) % 4 == 0 && (kNfft / 2) % 4 == 0,
                  "quads of the half-tile are quads of the noise stream");
#pragma unroll 1
    for (int q = tg; q < 2 * kQuads; q += kGroupThreads) {
        const int r = q >= kQuads ? 1 : 0;
        const int i = 4 * (q - r * kQuads);
        const int64_t s = s0 + r * kSubStep + i;         // a multiple of 4: the quad lies wholly below 0 or at/above 0
        if (s < 0 || s >= L) continue;
        float z[4] = {0.f, 0.f, 0.f, 0.f};
        if (cnd.dither != 0.f) philox_normal4(cnd.key0, cnd.key1, static_cast<uint32_t>(s >> 2), static_cast<uint32_t>(b), z);
        float* p = raw + r * kSubLen + i;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (s + e >= L) break;
            const float x = s + e < len ? (cnd.moments ? (p[e] - ms.x) * ms.y : p[e]) : 0.f;
            p[e] = fmaf(cnd.dither, z[e], x);
        }
    }
    group_sync(grp);
    if (s0 < 0 || s0 + kTileSamples > L) {
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
            const int64_t s_lo = s0 + r * kSubStep;
#pragma unroll 1
            for (int i = tg; i < kSubLen; i += kGroupThreads) {
                const int64_t s = s_lo + i;
                if (s >= 0 && s < L) continue;
                const int64_t sr = s < 0 ? -s : 2 * (L - 1) - s;
                const int64_t u = sr - s0;
                raw[r * kSubLen + i] = sr >= 0 && sr < L && u >= 0 && u < kTileSamples
                                             ? raw[u < kSubLen ? u : kSubLen + (u - kSubStep)] : 0.f;
            }
        }
        group_sync(grp);
    }
}

// ---- per-clip moments (do_normalize) -----------------------------------------------------------------------------
// Deterministic two-step reduction over x[:len] of every clip (len up to 2^31 - 1):
//   logmel_moments_kernel        CTA (chunk, clip): float64 sums of d and d^2 over the chunk's kMomChunk samples, with
//                                d = x - x[0] (the shift keeps a large DC offset from cancelling the variance away), in
//                                a fixed order -> partial[b][chunk];
//   logmel_moments_merge_kernel  one warp per clip: the partials in chunk order -> (mean, 1 / sqrt(var + 1e-7)), the
//                                population variance, as HF's zero_mean_unit_var_norm.
// No atomics: the result does not depend on scheduling.
constexpr int kMomChunk = 1 << 16;
constexpr int kMomThreads = 256;

__device__ __forceinline__ float pcm_at(const LongArgs& a, int64_t i) {
    return a.pcm_format == WLM_PCM_I16 ? static_cast<float>(static_cast<const int16_t*>(a.pcm)[i]) * (1.0f / 32768.0f)
                                       : static_cast<const float*>(a.pcm)[i];
}

__global__ void __launch_bounds__(kMomThreads) logmel_moments_kernel(const LongArgs a, double2* __restrict__ partial,
                                                                    int n_chunks) {
    __shared__ double2 red[kMomThreads / 32];
    const int tid = threadIdx.x;
    for (int b = blockIdx.y; b < a.B; b += gridDim.y) {
        const LongClip c = long_clip(a, b);
        const int64_t lo = static_cast<int64_t>(blockIdx.x) * kMomChunk;
        if (lo >= c.len) continue;                                        // CTA-uniform
        const int64_t hi = min(lo + kMomChunk, c.len);
        const double k = pcm_at(a, c.base);
        double s1 = 0.0, s2 = 0.0;
        // quads: the clip start is 16-byte aligned and so is every chunk start (f32: 16 B, i16: 8 B per quad)
        const int64_t q_hi = lo / 4 + (hi - lo) / 4;
        for (int64_t q = lo / 4 + tid; q < q_hi; q += kMomThreads) {
            float x[4];
            if (a.pcm_format == WLM_PCM_I16) {
                const short4 v = reinterpret_cast<const short4*>(static_cast<const int16_t*>(a.pcm) + c.base)[q];
                x[0] = v.x * (1.0f / 32768.0f); x[1] = v.y * (1.0f / 32768.0f);
                x[2] = v.z * (1.0f / 32768.0f); x[3] = v.w * (1.0f / 32768.0f);
            } else {
                const float4 v = __ldcs(reinterpret_cast<const float4*>(static_cast<const float*>(a.pcm) + c.base) + q);
                x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const double d = static_cast<double>(x[e]) - k;
                s1 += d;
                s2 = fma(d, d, s2);
            }
        }
        for (int64_t i = 4 * q_hi + tid; i < hi; i += kMomThreads) {
            const double d = static_cast<double>(pcm_at(a, c.base + i)) - k;
            s1 += d;
            s2 = fma(d, d, s2);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if ((tid & 31) == 0) red[tid >> 5] = make_double2(s1, s2);
        __syncthreads();
        if (tid == 0) {
            double2 t = red[0];
            for (int w = 1; w < kMomThreads / 32; ++w) { t.x += red[w].x; t.y += red[w].y; }
            partial[static_cast<int64_t>(b) * n_chunks + blockIdx.x] = t;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) logmel_moments_merge_kernel(const LongArgs a, const double2* __restrict__ partial,
                                                                  int n_chunks, float2* __restrict__ moments) {
    const int lane = threadIdx.x & 31;
    const int w0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (int b = w0; b < a.B; b += nw) {
        const LongClip c = long_clip(a, b);
        const int nc = static_cast<int>((c.len + kMomChunk - 1) / kMomChunk);
        double s1 = 0.0, s2 = 0.0;
        for (int j = lane; j < nc; j += 32) {
            const double2 t = partial[static_cast<int64_t>(b) * n_chunks + j];
            s1 += t.x;
            s2 += t.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if (lane == 0) {
            float2 m = make_float2(0.f, 0.f);             // an empty clip is all padding: nothing is normalised
            if (c.len > 0) {
                const double n = static_cast<double>(c.len), d1 = s1 / n;
                const double var = fmax(s2 / n - d1 * d1, 0.0);
                m = make_float2(static_cast<float>(static_cast<double>(pcm_at(a, c.base)) + d1),
                                static_cast<float>(1.0 / sqrt(var + 1e-7)));
            }
            moments[b] = m;
        }
    }
}

// ---- pass 1 ------------------------------------------------------------------------------------------------------
// NMELS = 80 / 128: unrolled mel stage of that Whisper bank; 0: table-driven.
// COND: a conditioned call (cond_fixup on every half-tile; with dither every half-tile of every clip is active).
template <int NMELS, class OutT, bool COND>
__device__ __forceinline__ void long_pass1(const LongArgs& a, const KernelTables& kt, const float* __restrict__ win_lane,
                                           const CondArgs& cnd) {
    using namespace fused;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = warp / kGroupWarps, wg = warp % kGroupWarps, tg = tid & (kGroupThreads - 1);
    unsigned char* gbase = smem + grp * kSmemGroup;
    float* raw = reinterpret_cast<float*>(gbase) + kRawShift;
    float2* Y = reinterpret_cast<float2*>(gbase + kSmemRaw) + wg * kYWarpFloat2;      // this WARP's stage-1 output
    float* P = reinterpret_cast<float*>(gbase + kSmemRaw + kSmemY);
    unsigned char* gm = smem + kGroups * kSmemGroup + grp * 64;
    const uint32_t bar_raw = smem_u32(gm);                                   // TMA landed the half-tile's PCM
    volatile long long* unit_slot = reinterpret_cast<volatile long long*>(gm + 16);   // [2] the group's units by parity
    int* grp_max = reinterpret_cast<int*>(gm + 32);                         // the unit's max over the group's warps
    if (tg == 0) {
        mbar_init(bar_raw, 1);
        *grp_max = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // the imaginary part of slot 0 in the warp's Y: zeros, written once (stage 1 never stores there)
    Y[(lane >> 1) * kYN1 + kYLanes + (lane & 1)] = make_float2(0.f, 0.f);
    const uint32_t s1_base = stage1_base(raw, wg, lane);
    float wv[25];
#pragma unroll
    for (int t = 0; t < 25; ++t) wv[t] = win_lane[(lane & 15) * 25 + t];
    const int nf = kt.nf[wg];
    const int m0 = kt.m0[wg];
    const int U = a.units_per_clip;
    const long long n_units = static_cast<long long>(a.B) * U;
    auto clip = [&](int b) {
        LongClip c = long_clip(a, b);
        if (COND && cnd.dither != 0.f) c.n_act = a.n_tiles;       // the noise reaches every half-tile
        return c;
    };

    // (thread 0 of the group) the next unit that holds an active half-tile, or -1.  The units of a clip are handed out
    // in order, so the first empty one ends the clip: the counter then skips the clip's remaining units.
    auto fetch = [&]() -> long long {
        while (true) {
            const unsigned long long u = atomicAdd(a.next_unit, 1ull);
            if (u >= static_cast<unsigned long long>(n_units)) return -1;
            const int b = static_cast<int>(u / U), j = static_cast<int>(u % U);
            if (j * kLongRun < clip(b).n_act) return static_cast<long long>(u);
            atomicMax(a.next_unit, static_cast<unsigned long long>(b + 1) * U);
        }
    };
    if (tg == 0) {
        const long long u = fetch();
        unit_slot[0] = u;
        if (u >= 0) long_issue_tma(a, clip(static_cast<int>(u / U)), static_cast<int>(u % U) * kLongRun, raw, bar_raw);
    }
    __syncthreads();

    int tnum = 0;           // half-tiles this group has processed: phase of bar_raw
    for (int k = 0;; ++k) {
        const long long u = unit_slot[k & 1];
        if (u < 0) break;
        const int b = static_cast<int>(u / U);
        const int t0 = static_cast<int>(u % U) * kLongRun;
        const LongClip c = clip(b);
        const int t1 = min(t0 + kLongRun, c.n_act);
        float2 ms = make_float2(0.f, 1.f);
        if (COND && cnd.moments) ms = cnd.moments[b];
        // the following unit: fetched now, so that its first copy can go out while this unit's last half-tile runs
        long long un = -1;
        if (tg == 0) {
            un = fetch();
            unit_slot[(k + 1) & 1] = un;
        }
        float mx = 0.f;                                  // running max of the mel power of this lane's frames
#pragma unroll 1
        for (int t = t0; t < t1; ++t, ++tnum) {
            mbar_wait(bar_raw, tnum & 1);
            const int64_t s0 = long_s0(t);
            if (COND)
                cond_fixup(cnd, a.pcm_format, b, ms, c.len, a.padded_len, t, raw, grp, tg);
            else if (a.pcm_format == WLM_PCM_I16 || s0 < 0 || s0 + kTileSamples > c.len)
                long_fixup(a.pcm_format, c.len, a.padded_len, t, raw, grp, tg);
            stage1(s1_base, Y, wv, wg, lane, [&]() {}, [&]() {});
            group_sync(grp);     // every warp is done with raw (and, from the previous half-tile, with P)
            if (tg == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                if (t + 1 < t1) long_issue_tma(a, c, t + 1, raw, bar_raw);
                else if (un >= 0)
                    long_issue_tma(a, clip(static_cast<int>(un / U)), static_cast<int>(un % U) * kLongRun, raw, bar_raw);
            }
            stage2(Y, P, wg, lane, [&]() {});
            group_sync(grp);     // P holds the half-tile's power
            // frames past T (the last lanes of the clip's last half-tile) are neither stored nor counted
            const int frame = t * kTile + lane;
            const bool keep = frame < a.n_frames;
            const int64_t e0 = (static_cast<int64_t>(b) * a.n_mels + m0) * a.n_frames + frame;
            auto sink = [&](const float (&o)[kMaxFiltersPerWarp]) {
                // (max(log10 p, -10) + 4) / 4 with the arithmetic of fused::output_block; rows are T apart
                constexpr float kLog10_2_4 = 0.30102999566398120f * 0.25f;
                OutT* of = static_cast<OutT*>(a.out) + e0;
#pragma unroll
                for (int q = 0; q < kMaxFiltersPerWarp; ++q)
                    if (q < nf && keep)
                        of[static_cast<int64_t>(q) * a.n_frames] = to_out<OutT>(fmaxf(fmaf(lg2_approx(o[q]), kLog10_2_4, 1.0f), -1.5f));
            };
            const float m1 = NMELS == 0 ? mel_stage(kt, P, wg, lane, sink) : mel_fixed<NMELS == 0 ? 80 : NMELS>(kt, P, wg, lane, sink);
            if (keep) mx = fmaxf(mx, m1);
        }
        // the unit's max: warps -> group (shared) -> clip (one global atomic)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) atomicMax(grp_max, __float_as_int(mx));
        group_sync(grp);
        if (tg == 0) atomicMax(a.pmax + b, atomicExch(grp_max, 0));
    }
}

template <int NMELS, class OutT>
__global__ void __launch_bounds__(kThreads, 1)
logmel_long_kernel(const LongArgs a, const __grid_constant__ KernelTables kt, const float* __restrict__ win_lane) {
    long_pass1<NMELS, OutT, false>(a, kt, win_lane, CondArgs{});
}

// pass 1 of wlm_logmel_conditioned
template <int NMELS, class OutT>
__global__ void __launch_bounds__(kThreads, 1)
logmel_long_cond_kernel(const LongArgs a, const __grid_constant__ KernelTables kt, const float* __restrict__ win_lane,
                        const CondArgs cnd) {
    long_pass1<NMELS, OutT, true>(a, kt, win_lane, cnd);
}

// ---- pass 2 ------------------------------------------------------------------------------------------------------
// grid (x: blocks per clip, y: clips, strided).  M T < 2^31 for every clip (T <= INT32_MAX / 160, M <= 128), so the
// in-clip element index is 32-bit; the clip's base is 64-bit.
template <class OutT>
__global__ void __launch_bounds__(256) logmel_long_clamp_kernel(const LongArgs a) {
    using namespace fused;
    constexpr int kPer = 16 / static_cast<int>(sizeof(OutT));
    struct alignas(16) Vec { OutT e[kPer]; };
    const int T = a.n_frames;
    const int n = a.n_mels * T;
    const int gt = blockIdx.x * blockDim.x + threadIdx.x, gs = gridDim.x * blockDim.x;
    for (int b = blockIdx.y; b < a.B; b += gridDim.y) {
        const float gmax = log10_floor(__int_as_float(a.pmax[b]));              // TF-FE:157
        const float thr = (fmaxf(gmax - 8.0f, -10.0f) + 4.0f) * 0.25f;            // TF-FE:158,161
        if (a.gmax && gt == 0) a.gmax[b] = gmax;
        const OutT thr_t = to_out<OutT>(thr);       // rounded like the features: max(round x, round t) = round max(x, t)
        const float thr_f = from_out<OutT>(thr_t);
        const int n_valid = min(T, long_clip(a, b).n_act * kTile);              // frames pass 1 wrote
        OutT* p = static_cast<OutT*>(a.out) + static_cast<int64_t>(b) * n;
        const int head = min(n, static_cast<int>(((16u - (reinterpret_cast<uintptr_t>(p) & 15u)) & 15u) / sizeof(OutT)));
        const int nv = (n - head) / kPer;
        const int tail0 = head + nv * kPer;
        // scalar ends: [0, head) and [tail0, n)
        for (int e = gt; e < head + (n - tail0); e += gs) {
            const int i = e < head ? e : tail0 + (e - head);
            const OutT v = i % T < n_valid ? p[i] : thr_t;
            p[i] = from_out<OutT>(v) < thr_f ? thr_t : v;
        }
        // 16-byte vectors, four in flight per thread
        Vec* pv = reinterpret_cast<Vec*>(p + head);
        for (int i0 = gt; i0 < nv; i0 += 4 * gs) {
            Vec v[4];
            bool silent[4][kPer];
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const int i = i0 + w * gs;
                int f = (head + i * kPer) % T;
                bool any = false;
#pragma unroll
                for (int e = 0; e < kPer; ++e) {
                    silent[w][e] = f >= n_valid;
                    any |= !silent[w][e];
                    v[w].e[e] = thr_t;
                    if (++f == T) f = 0;
                }
                if (i < nv && any) {
                    const float4 x = __ldcs(reinterpret_cast<const float4*>(pv + i));
                    v[w] = *reinterpret_cast<const Vec*>(&x);
                }
            }
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const int i = i0 + w * gs;
#pragma unroll
                for (int e = 0; e < kPer; ++e)
                    if (silent[w][e] || from_out<OutT>(v[w].e[e]) < thr_f) v[w].e[e] = thr_t;
                if (i < nv) __stcs(reinterpret_cast<float4*>(pv + i), *reinterpret_cast<const float4*>(&v[w]));
            }
        }
    }
}

}  // namespace longform
}  // namespace wlm
