// Fused log-mel kernel for sm_100a.
//
// A thread-block CLUSTER of 6 CTAs owns one clip.  Every CTA runs TWO independent warp groups of 8
// warps ("virtual CTAs"); the clip's 3000 frames are 94 half-tiles of 32 frames and half-tile u goes
// to virtual CTA u mod 12 (= 2 * cluster rank + group).  A group walks its half-tiles through
//
//   TMA (cp.async.bulk, mbarrier)  raw PCM  ->  shared memory, two sub-regions 16 banks apart
//   stage 1  per warp: 4 frames x 16 sub-transforms; lane = (n1, sub-region); 25-point real DFT of
//            the Hann-windowed samples n = (25 n1 + 16 n2) mod 400, packed f32x2 over two frames
//   stage 2  the SAME warp, on its own two frame pairs: lane = (k2 slot, pair), 26 lanes; 16-point
//            complex DFT over n1, |X|^2.  The hand-over is a __syncwarp (Y is private to the warp).
//   mel      per warp: a run of <= 16 filters, lane = frame; sparse gather; mel POWER retained in
//            TENSOR MEMORY (tcgen05.st), running max in registers
//
// with the prime-factor index maps of fft_pfa.cuh (no twiddles between the stages).  The FFT
// arithmetic is FADD2 / FMUL2 / FFMA2 on (frame a, frame b) pairs with immediate constants.
// The two groups share nothing but the clip-end exchange.  When the clip is done the 12 virtual
// CTAs deliver their maxima to each other through distributed shared memory (st.async completing
// bytes on the receiver's mbarrier: nobody waits), and the retained mel power is read back
// (tcgen05.ld) one half-tile per step of the NEXT clip and written as
// (max(log10(max(p,1e-10)), gmax - 8) + 4) / 4 -- the features touch HBM exactly once.
//
// Shared memory (bytes):  raw 2 x 22,400 | Y 2 x 54,272 | P 2 x 26,752 | mbarriers + scratch 1024
//
// Template parameters of the kernel: NMELS (80 / 128: mel stage unrolled with the structure of that Whisper bank; 0: table-
// driven), FLAT (the cluster-less twin for the SMs clusters cannot cover), OutT (float / bfloat16 / half feature store), DYN
// (clips from the queue both kernels share -- ragged batches -- or a static split -- dense batches).
// Two restructurings of this kernel were built and measured in round 2 and are NOT used (DESIGN.md section 4):
// warp-specialised FFT / mel+output warps, and a streaming variant with multi-buffered raw and P.
#pragma once
#include <cooperative_groups.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "wlm_common.cuh"

namespace wlm {
namespace fused {

// ---- packed two-frame value --------------------------------------------------------------------
struct V2 {
    float2 v;
};
__device__ __forceinline__ V2 mk(float a, float b) { V2 r; r.v = make_float2(a, b); return r; }
__device__ __forceinline__ V2 vadd(V2 a, V2 b) { V2 r; r.v = __fadd2_rn(a.v, b.v); return r; }
__device__ __forceinline__ V2 vsub(V2 a, V2 b) { V2 r; r.v = __fadd2_rn(a.v, make_float2(-b.v.x, -b.v.y)); return r; }
__device__ __forceinline__ V2 vmul(V2 a, V2 b) { V2 r; r.v = __fmul2_rn(a.v, b.v); return r; }
__device__ __forceinline__ V2 vfma(V2 a, V2 b, V2 c) { V2 r; r.v = __ffma2_rn(a.v, b.v, c.v); return r; }
__device__ __forceinline__ V2 vmulc(V2 a, float s) { V2 r; r.v = __fmul2_rn(a.v, make_float2(s, s)); return r; }
__device__ __forceinline__ V2 vfmac(V2 a, float s, V2 c) { V2 r; r.v = __ffma2_rn(a.v, make_float2(s, s), c.v); return r; }

}  // namespace fused
namespace fft {
using fused::vadd; using fused::vsub; using fused::vmul; using fused::vfma; using fused::vmulc; using fused::vfmac;
}
}  // namespace wlm

#include "fft_pfa.cuh"
#include "mel_structure.inc"

namespace wlm {
namespace fused {

// Knock-outs for tools/fused_ko.cu (TIMING ONLY, results are wrong with any of them): 1 no raw wait / TMA re-arm, 2 no
// wait for "P full", 4 no wait for "P free", 8 no mel arithmetic, 16 no output pass.  0 in every product build.
#ifndef WLM_KO
#define WLM_KO 0
#endif
constexpr bool kKoRaw = (WLM_KO & 1) != 0, kKoPfull = (WLM_KO & 2) != 0, kKoPfree = (WLM_KO & 4) != 0,
               kKoMel = (WLM_KO & 8) != 0, kKoOut = (WLM_KO & 16) != 0;
// finer ones: 64 the copy moves 16 bytes per sub-region, 128 output stores predicated
// off, 256 no tensor-memory read-back (the output pass works on stale registers), 512 no tensor-memory store
constexpr bool kKoTinyTma = (WLM_KO & 64) != 0, kKoStg = (WLM_KO & 128) != 0,
               kKoTld = (WLM_KO & 256) != 0, kKoTst = (WLM_KO & 512) != 0;

// -DWLM_WAITSTAT (tools/fused_ko.cu only): every warp accumulates the cycles it spends in each kind of wait and leaves them
// in a.gmax[(cta * 16 + warp) * 8 + {0 raw, 1 P full, 2 P free, 3 clip maxima, 4 whole loop}]
#ifdef WLM_WAITSTAT
#define WLM_WS_BEGIN() const long long ws_t0 = clock64()
#define WLM_WS_END(k) ws_acc[k] += clock64() - ws_t0
#else
#define WLM_WS_BEGIN()
#define WLM_WS_END(k)
#endif
constexpr int kGroups = 2;                // independent warp groups per CTA
constexpr int kGroupWarps = 8;
constexpr int kGroupThreads = kGroupWarps * 32;
constexpr int kWarps = kGroups * kGroupWarps;
constexpr int kThreads = kWarps * 32;
constexpr int kTile = 4 * kGroupWarps;    // frames per half-tile (the unit of work of one group): 2 pairs per warp
constexpr int kPairs = kTile / 2;         // 16 frame pairs
constexpr int kTilesPerClip = (kNFrames + kTile - 1) / kTile;  // 94
constexpr int kSubFrames = kTile / 2;                          // frames per raw sub-region
constexpr int kSubLen = (kSubFrames - 1) * kHop + kNfft;       // 2800 samples (= 16 mod 32: sub-regions 16 banks apart)
constexpr int kSubStep = kSubFrames * kHop;                    // 2560: sub-region 1 starts 16 frames later
constexpr int kRawFloats = 2 * kSubLen;                        // 5600 per group
constexpr int kTileSamples = (kTile - 1) * kHop + kNfft;       // 5360
static_assert(kSubLen % 32 == 16, "the two sub-regions must sit 16 banks apart");
static_assert(kSubStep + kSubLen == kTileSamples, "sub-regions cover the half-tile");

// Y (stage 1 -> stage 2) is PRIVATE to a warp: the warp that transforms the frame pairs (wg, kGroupWarps + wg) in stage 1
// also runs all 13 slots of those two pairs in stage 2 (lane = 2 slot + q, 26 lanes), so the hand-over is a __syncwarp,
// not a barrier over the group.  Per warp: [n1][Re: 13 slots x 2 pairs | Im: 13 x 2] float2, rows of 53 (odd: the 16 n1
// lanes of a stage-1 store hit 16 different 8-byte banks; stage 2 reads 26 consecutive float2).  Im of slot 0 is zero.
constexpr int kYLanes = 2 * fft::kNumSlots;                    // 26 (slot, q) combinations = lanes of stage 2
constexpr int kYN1 = 2 * kYLanes + 1;                          // 53 float2 per n1 row
constexpr int kYWarpFloat2 = 16 * kYN1;                        // 848 float2 = 6,784 B per warp
constexpr int kYFloat2 = kGroupWarps * kYWarpFloat2;
// P (stage 2 -> mel), per group: [pair][kPPair] float2 with the power of (slot, FFT16 output position i) at 13 i + slot
constexpr int kPRows = fft::kNumSlots * 16;                    // 208 (201 distinct bins; slot 0 holds seven of its bins twice)
constexpr int kPPair = kPRows + (kPairs == 16 ? 1 : 2);        // 209 (= 1 mod 16) / 210 (8 pairs: 4 x 210 = 8 mod 16)
constexpr int kPFloats = 2 * kPairs * kPPair;

// The raw buffer starts kRawShift floats into its 128-byte-aligned slab: the TMA source of a half-tile of a dense batch
// sits at (5120 t - 200) * 4 = 96 mod 128 bytes, and a copy whose destination has the same offset inside a 128-byte line
// is cheaper (tools/fused_ko.cu, shifts of 0/8/16/24 floats: 7,530 / 7,445 / 7,530 / 7,445 cycles per 64 frames; the two
// sub-regions are 64 bytes apart modulo 128 for the bank layout, so only one of them can be co-aligned).
constexpr int kRawShift = 24;
constexpr int kSmemRaw = kRawFloats * 4 + 128;                          // 22,400 + 128
constexpr int kSmemY = kYFloat2 * 8;
constexpr int kSmemP = kPFloats * 4;
constexpr int kSmemGroup = kSmemRaw + kSmemY + kSmemP;
constexpr int kSmemMisc = 1024;
constexpr int kSmemBytes = kGroups * kSmemGroup + kSmemMisc;
static_assert(kSmemRaw % 128 == 0 && kSmemY % 128 == 0 && kSmemP % 128 == 0, "buffers stay 128-byte aligned");

constexpr int kCluster = 6;                     // CTAs per clip: 22 co-resident clusters = 132 of 148 SMs (size 8: 15 = 120)
constexpr int kVCluster = kCluster * kGroups;   // 12 virtual CTAs per clip
constexpr int kMaxTilesPerGroup = (kTilesPerClip + kVCluster - 1) / kVCluster;   // 8
constexpr int kMaxFiltersPerWarp = 16;          // 8 warps x 16 >= 128 mels
constexpr int kMaxGroupBins = 16;               // bins between two adjacent filter centres
constexpr int kTmemColsPerTile = kMaxFiltersPerWarp;                          // 16 (lane = frame)
constexpr int kTmemColsPerWarp = kMaxTilesPerGroup * kTmemColsPerTile;        // 128; 4 warps per lane quarter = 512 columns
static_assert(4 * kTmemColsPerWarp <= 512, "the retained mel power must fit the 512 TMEM columns");
static_assert(kVCluster <= 32, "max reduction over the cluster uses one warp");

// float2 index, inside a pair's row of P, of FFT bin k (stage 2 stores position i of slot s at 13 i + s)
__host__ __device__ __forceinline__ int p_index_of_bin(int k) {
    const int row = fft::row_of_bin(k);        // 16 slot + position
    return 13 * (row & 15) + (row >> 4);
}

// Everything the kernel reads with warp-uniform indices, passed by value (constant bank).
//
// Mel projection: FFT bin k adds w_lo[k] P[k] to filter lo[k] and w_hi[k] P[k] to filter lo[k]+1
// (host-built from the caller's dense table, weights bit-identical).  Bins with the same lo[k] form
// a "group" (the bins between two adjacent filter centres).  Warp w of a warp group owns filters
// [m0, m0+nf) and walks groups g = 0..nf, group g = bins [gb[g], gb[g+1]) with lo = m0-1+g:
//     filter m0+q  =  sum_{k in group q} w_hi[k] P[k]  +  sum_{k in group q+1} w_lo[k] P[k]
struct KernelTables {
    float2 w2[kNFreq + 3];                               // (w_lo, w_hi) per bin
    int16_t prow[kNFreq + 3];                            // row of P that holds bin k
    int16_t gb[kGroupWarps][kMaxFiltersPerWarp + 2];     // group boundaries (bin indices)
    int16_t m0[kGroupWarps];                             // first filter of warp w
    int16_t nf[kGroupWarps];                             // number of filters of warp w (<= 16)
    int16_t n_mels;
};

// Host-visible tables
struct Tables {
    float win_lane[16 * 25];     // Hann window at n = (25 n1 + 16 t) mod 400
    KernelTables mel;
};

// returns 0, or -1 if the table does not fit the fused path (a group longer than 16 bins)
// *variant receives 80 / 128 when the structure equals the baked Whisper bank (unrolled kernel), else 0
inline int build_tables(const MelSparse& sp, int n_mels, Tables* t, int* variant) {
    *variant = 0;
    for (int n1 = 0; n1 < 16; ++n1)
        for (int tt = 0; tt < 25; ++tt) {
            const int n = (25 * n1 + 16 * tt) % 400;
            t->win_lane[n1 * 25 + tt] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * n / 400.0));
        }
    KernelTables& mp = t->mel;
    memset(&mp, 0, sizeof(mp));
    mp.n_mels = (int16_t)n_mels;
    for (int k = 0; k < kNFreq; ++k) {
        mp.w2[k] = make_float2(sp.w_lo[k], sp.w_hi[k]);
        mp.prow[k] = (int16_t)p_index_of_bin(k);
    }
    // first bin of every group: gstart[v] = first k with lo[k] >= v - 1   (v = lo + 1 in 0..n_mels)
    int gstart[kMaxMels + 2];
    {
        int k = 0;
        for (int v = 0; v <= n_mels + 1; ++v) {
            while (k < kNFreq && sp.lo[k] + 1 < v) ++k;
            gstart[v] = k;
        }
    }
    for (int v = 0; v <= n_mels; ++v)
        if (gstart[v + 1] - gstart[v] > kMaxGroupBins) return -1;
    const short* baked_g = n_mels == 80 ? kMelGstartHost80 : (n_mels == 128 ? kMelGstartHost128 : nullptr);
    const short* baked_m0 = n_mels == 80 ? kMelM0Host80 : kMelM0Host128;
    const short* baked_nf = n_mels == 80 ? kMelNfHost80 : kMelNfHost128;
    bool same = baked_g != nullptr;
    for (int v = 0; same && v <= n_mels + 1; ++v) same = gstart[v] == baked_g[v];
    if (same) *variant = n_mels;
    // contiguous filter runs per warp, balanced on issue slots: ~3 per bin of the two groups a filter
    // touches (shared with its neighbour) + ~7 per filter
    auto cost = [&](int m) { return 7.0 + 1.5 * (gstart[m + 2] - gstart[m]); };
    double total = 0;
    for (int m = 0; m < n_mels; ++m) total += cost(m);
    int m = 0;
    double acc = 0;
    for (int w = 0; w < kGroupWarps; ++w) {
        const double target = total * (w + 1) / kGroupWarps;
        int cnt = 0;
        mp.m0[w] = (int16_t)m;
        if (same) {   // partition baked into the unrolled kernel
            mp.m0[w] = baked_m0[w];
            cnt = baked_nf[w];
            m = mp.m0[w] + cnt;
        }
        while (!same && m < n_mels && cnt < kMaxFiltersPerWarp) {
            const bool must_take = n_mels - m > (kGroupWarps - 1 - w) * kMaxFiltersPerWarp;   // the rest could not hold them
            if (!must_take && cnt > 0 && acc + 0.5 * cost(m) > target) break;
            acc += cost(m);
            ++m;
            ++cnt;
        }
        mp.nf[w] = (int16_t)cnt;
        // groups g = 0..cnt: lo = m0 - 1 + g  ->  v = m0 + g
        for (int g = 0; g <= kMaxFiltersPerWarp + 1; ++g) {
            const int v = mp.m0[w] + (g <= cnt + 1 ? g : cnt + 1);
            mp.gb[w][g] = (int16_t)gstart[v <= n_mels + 1 ? v : n_mels + 1];
        }
    }
    if (m < n_mels) return -1;
    return 0;
}

// ---- PTX helpers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// (operand %2 is unused, but it stays: without it the PTX registers are numbered differently and ptxas allocates the
// registers of logmel_cluster_kernel<0, false, float, true> differently)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity), "r"(0) : "memory");
}
// same, acquiring at cluster scope: the data the barrier guards was written by other CTAs of the cluster.  (The acquire
// costs a CCTL.IVALL after the wait; a CTA-scope wait measured the same launch time, so the documented form stays.)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAITC_%=:\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONEC_%=;\n"
        "bra WAITC_%=;\n"
        "DONEC_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// TMA 1-D bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// named barrier over the 256 threads of one warp group (id 1 / 2; 0 is __syncthreads)
__device__ __forceinline__ void group_sync(int grp) {
    asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(kGroupThreads) : "memory");
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- tensor memory (tcgen05) -------------------------------------------------------------------
// The retained mel power never needs a tensor core; TMEM is used as 256 KB of per-SM scratch so the
// clip's features can wait on-chip for the cluster-wide max.  Warp w may only touch TMEM lanes
// [32 (w & 3), +32): lane i of the warp <-> TMEM lane 32 (w & 3) + i, i.e. one frame per lane.
__device__ __forceinline__ void tmem_alloc_512(uint32_t smem_dst) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_dst) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const float (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
          "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, float (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7]),
          "=f"(r[8]), "=f"(r[9]), "=f"(r[10]), "=f"(r[11]), "=f"(r[12]), "=f"(r[13]), "=f"(r[14]), "=f"(r[15])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- clip / tile bookkeeping (all values group-uniform) -------------------------------------------
struct ClipCtx {
    int b, len, n_act;     // clip index, valid samples (<= 480000), half-tiles that contain any real sample
    int edge0;             // first half-tile that runs past the clip's samples (zero fill / reflection at the end)
    int64_t base;          // element offset of the clip in the PCM buffer
};

__device__ __forceinline__ ClipCtx clip_ctx(const ClipArgs& a, int b) {
    ClipCtx c;
    c.b = b;
    c.base = a.offsets ? a.offsets[b] : static_cast<int64_t>(b) * a.row_stride;
    int len = a.lengths ? a.lengths[b] : a.dense_len;
    if (!a.offsets) len = static_cast<int>(min(static_cast<int64_t>(len), a.row_stride));
    c.len = max(0, min(len, kNSamples));
    // half-tile t starts at sample 5120 t - 200: active iff that is < len
    c.n_act = min(kTilesPerClip, (c.len + kNfft / 2 + kTile * kHop - 1) / (kTile * kHop));
    // half-tile t covers samples [5120 t - 200, 5120 t + 5160): it runs past the clip iff 5120 t > len - 5160
    c.edge0 = c.len >= kTileSamples - kNfft / 2 ? (c.len - (kTileSamples - kNfft / 2)) / (kTile * kHop) + 1 : 0;
    return c;
}
// the same clip context for another clip of a STATIC launch: every clip has the same length, only the position differs
__device__ __forceinline__ ClipCtx clip_ctx_like(const ClipArgs& a, const ClipCtx& c0, int b) {
    ClipCtx c = c0;
    c.b = b;
    c.base = a.offsets ? a.offsets[b] : static_cast<int64_t>(b) * a.row_stride;
    return c;
}
__device__ __forceinline__ int tile_s0(int tile) { return tile * (kTile * kHop) - kNfft / 2; }

// issued by one thread: both sub-regions of the half-tile, valid sample range only
__device__ __forceinline__ void tile_issue_tma(const ClipArgs& a, const ClipCtx& c, int tile, float* raw, uint32_t bar) {
    const int s0 = tile_s0(tile);
    const int esz = a.pcm_format == WLM_PCM_I16 ? 2 : 4;
    if ((s0 >= 0 && s0 + kTileSamples <= c.len && !kKoTinyTma)) {       // interior half-tile: two full sub-regions
        const uint32_t bytes = static_cast<uint32_t>(kSubLen * esz);
        mbar_expect_tx(bar, 2u * bytes);
        const char* src = static_cast<const char*>(a.pcm) + (c.base + s0) * esz;
        const uint32_t dst = smem_u32(raw) + (esz == 4 ? 0u : static_cast<uint32_t>(kSubLen) * 4u);
        tma_bulk_g2s(dst, src, bytes, bar);
        tma_bulk_g2s(dst + bytes, src + static_cast<int64_t>(kSubStep) * esz, bytes, bar);
        return;
    }
    const int gmask = esz == 4 ? 3 : 7;      // copies are multiples of 16 bytes: 4 float32 / 8 int16 samples (a mask: the
                                             // division by 16 / esz compiled into a 40-instruction software divide)
    const int len_up = min((c.len + gmask) & ~gmask, kNSamples);
    uint32_t total = 0;
    int lo[2], n[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int s_lo = s0 + r * kSubStep;
        lo[r] = max(s_lo, 0);
        const int hi = min(s_lo + kSubLen, len_up);
        n[r] = max(hi - lo[r], 0);
        if constexpr (kKoTinyTma) n[r] = min(n[r], 4);
        total += static_cast<uint32_t>(n[r]) * esz;
    }
    mbar_expect_tx(bar, total);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        if (n[r] <= 0) continue;
        const int s_lo = s0 + r * kSubStep;
        const char* src = static_cast<const char*>(a.pcm) + (c.base + lo[r]) * esz;
        uint32_t dst;
        if (esz == 4) dst = smem_u32(raw) + static_cast<uint32_t>(r * kSubLen + (lo[r] - s_lo)) * 4u;
        else dst = smem_u32(raw) + static_cast<uint32_t>(kSubLen) * 4u + static_cast<uint32_t>(r * kSubLen + (lo[r] - s_lo)) * 2u;
        tma_bulk_g2s(dst, src, static_cast<uint32_t>(n[r]) * esz, bar);
    }
}

// int16 -> float32 expansion in place (staging sits in the byte range of sub-region 1) + reflect /
// zero-fill patching of every position outside [0, len).  Only edge tiles and int16 input pay.
// Runs on the 256 threads of one group (tg = thread index inside the group).
// (scalars, not the argument structs: measured 1 % faster; as a __noinline__ function -- ~190 instructions an interior
// half-tile never executes -- it measured 3 % SLOWER)
__device__ __forceinline__ void tile_fixup(int pcm_format, int clip_len, int tile, float* raw, int grp, int tg) {
    const int s0 = tile_s0(tile);
    if (pcm_format == WLM_PCM_I16) {
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
    // Only the positions outside [0, len) are touched (a scan of the whole buffer cost ~8k cycles on the first
    // half-tile of every clip, and the other 11 virtual CTAs of the cluster wait for that one at the clip's end).
    if (s0 < 0) {   // first half-tile: s = idx - 200 < 0 reflects to sample 200 - idx (torch.stft center=True, TF-FE:149)
#pragma unroll 1
        for (int idx = tg; idx < -s0; idx += kGroupThreads) {
            const int sr = -(s0 + idx);
            raw[idx] = sr < clip_len ? raw[sr - s0] : 0.f;       // (sr - s0 <= 400 < kSubLen: same sub-region)
        }
    }
    if (s0 + kTileSamples > clip_len) {   // the half-tile runs past the clip: zero padding, reflected at sample 480000
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int s_lo = s0 + r * kSubStep;
#pragma unroll 1
            for (int i = max(clip_len - s_lo, 0) + tg; i < kSubLen; i += kGroupThreads) {
                const int s = s_lo + i;
                float v = 0.f;
                if (s >= kNSamples) {
                    const int sr = 2 * (kNSamples - 1) - s;
                    const int u = sr - s0;
                    if (sr < clip_len && u >= 0) v = raw[u < kSubLen ? u : kSubLen + (u - kSubStep)];
                }
                raw[r * kSubLen + i] = v;
            }
        }
    }
    if (s0 < 0 || s0 + kTileSamples > clip_len) group_sync(grp);
}

// ---- stage 1 ----------------------------------------------------------------------------------
// warp wg of the group, lane (n1 = lane & 15, sub = lane >> 4): the two ADJACENT frames 16 sub + 2 wg, + 1 of the
// half-tile (pair index 8 sub + wg).  The sample index (25 n1 + 16 t) mod 400 wraps for t >= tw(n1); with
// wrap_thr(t) = the first n1 that wraps at t, the select is one compare against a compile-time constant.
__host__ __device__ constexpr int wrap_tw(int n1) { return n1 == 0 ? 25 : (kNfft - 25 * n1 + 15) / 16; }
__host__ __device__ constexpr int wrap_thr(int t) {
    for (int n1 = 0; n1 < 16; ++n1)
        if (wrap_tw(n1) <= t) return n1;
    return 16;
}
// `loaded()` runs once the warp no longer needs the raw buffer, `before_store()` just before Y is written.
template <int T>
struct S1Load {   // samples t = T .. 24 of both frames: one compare + select per distinct wrap threshold, then LDS [reg + imm]
    static __device__ __forceinline__ void run(uint32_t a0, uint32_t a1, uint32_t n1, const float (&wv)[25], V2 (&y)[25]) {
        constexpr int thr = wrap_thr(T);
        uint32_t at;
        if (thr >= 16) at = a0;
        else if (thr <= 0) at = a1;
        else asm("{\n.reg .pred p;\nsetp.ge.u32 p, %1, %2;\nselp.b32 %0, %3, %4, p;\n}" : "=r"(at) : "r"(n1), "n"(thr), "r"(a1), "r"(a0));
        float xa, xb;
        asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(xa) : "r"(at), "n"(64 * T));
        asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(xb) : "r"(at), "n"(64 * T + 4 * kHop));
        y[T] = mk(xa * wv[T], xb * wv[T]);
        S1Load<T + 1>::run(a0, a1, n1, wv, y);
    }
};
template <>
struct S1Load<25> {
    static __device__ __forceinline__ void run(uint32_t, uint32_t, uint32_t, const float (&)[25], V2 (&)[25]) {}
};

__device__ __forceinline__ uint32_t stage1_base(const float* raw, int wg, int lane) {
    const int n1 = lane & 15, sub = lane >> 4;
    return smem_u32(raw + sub * kSubLen + 2 * kHop * wg + 25 * n1);
}
template <class Loaded, class BeforeStore>
__device__ __forceinline__ void stage1(uint32_t a0, float2* Y, const float (&wv)[25], int wg, int lane,
                                       Loaded loaded, BeforeStore before_store) {
    const int n1 = lane & 15, sub = lane >> 4;
    V2 y[25];
    S1Load<0>::run(a0, a0 - 4u * kNfft, static_cast<uint32_t>(n1), wv, y);
    loaded();      // (fence inside: every LDS above has been performed)
    V2 out[25];
    fft::rfft25<V2>(y, out);
    before_store();
    float2* yo = Y + n1 * kYN1 + sub;             // (Y = this warp's private buffer; q = sub)
    yo[0] = out[0].v;                             // slot 0: Re only
#pragma unroll
    for (int sl = 1; sl < fft::kNumSlots; ++sl) {
        yo[2 * sl] = out[2 * sl - 1].v;           // Re of slot sl
        yo[kYLanes + 2 * sl] = out[2 * sl].v;     // Im
    }
}

// ---- stage 2 ----------------------------------------------------------------------------------
// lane = 2 slot + q (26 of 32 lanes; the last six repeat lane 25): the 16-point complex DFT over n1 of slot `slot` for
// the warp's own frame pair q, then |X|^2.  The slot only selects base addresses, so it varies inside the warp for free.
// The power of FFT16 output position i goes to float2 13 i + slot of the pair's row of P (p_index_of_bin inverts that
// for the mel stage).  `before_store()` runs just before P is written.
template <class BeforeStore>
__device__ __forceinline__ void stage2(const float2* Y, float* P, int wg, int lane, BeforeStore before_store) {
    const int sl = min(lane, kYLanes - 1);
    const int slot = sl >> 1, q = sl & 1;
    const float2* yl = Y + sl;
    V2 xr[16], xi[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) {
        xr[n1].v = yl[n1 * kYN1];
        xi[n1].v = yl[n1 * kYN1 + kYLanes];      // slot 0 (k2 = 0, purely real Y): zeros, written once
    }
    fft::cfft16<V2>(xr, xi);
    before_store();
    float2* pl = reinterpret_cast<float2*>(P) + (wg + kGroupWarps * q) * kPPair + slot;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const V2 pw = vfma(xr[i], xr[i], vmul(xi[i], xi[i]));
        pl[13 * i] = pw.v;
    }
}

// ---- mel stage ------------------------------------------------------------------------------------
// One warp, its run of <= 16 filters, lane = frame.  Groups of bins between adjacent filter centres
// are walked once: every P value is loaded once and feeds the falling side of one filter and the
// rising side of the next (two independent FFMA chains, weights straight from the constant bank).
// The POWER goes to tensor memory (16 columns = 16 filters); log10 is monotone, so the running max
// is kept on the power.
#define WLM_MEL_TERM(i)                                                            \
    case (i) + 1: {                                                                \
        const float2 w = ww[i];                                                    \
        const float pv = pl[2 * pr[i]];                                            \
        A = fmaf(pv, w.y, A);                                                      \
        Bq = fmaf(pv, w.x, Bq);                                                    \
    }

// table-driven variant (any bank that fits the sparse form)
template <class Sink>
__device__ __forceinline__ float mel_stage(const KernelTables& kt, const float* P, int wg, int lane, Sink sink) {
    const int nf = kt.nf[wg];
    const float* pl = P + (lane >> 1) * (2 * kPPair) + (lane & 1);      // this frame's row of P
    float out[kMaxFiltersPerWarp];
#pragma unroll
    for (int q = 0; q < kMaxFiltersPerWarp; ++q) out[q] = 0.f;
#pragma unroll
    for (int g = 0; g <= kMaxFiltersPerWarp; ++g) {
        if (g <= nf) {
            const int k0 = kt.gb[wg][g];
            const int n = kt.gb[wg][g + 1] - k0;
            const int16_t* pr = kt.prow + k0;
            const float2* ww = kt.w2 + k0;
            float A = 0.f, Bq = 0.f;
            switch (n) {
                WLM_MEL_TERM(15) WLM_MEL_TERM(14) WLM_MEL_TERM(13) WLM_MEL_TERM(12)
                WLM_MEL_TERM(11) WLM_MEL_TERM(10) WLM_MEL_TERM(9) WLM_MEL_TERM(8)
                WLM_MEL_TERM(7) WLM_MEL_TERM(6) WLM_MEL_TERM(5) WLM_MEL_TERM(4)
                WLM_MEL_TERM(3) WLM_MEL_TERM(2) WLM_MEL_TERM(1) WLM_MEL_TERM(0)
                default: break;
            }
            if (g < kMaxFiltersPerWarp) out[g] = A;          // rising side of filter m0+g
            if (g > 0) out[g - 1] += Bq;                     // falling side of filter m0+g-1
        }
    }
    sink(out);          // the 16 mel powers of this lane's frame: tensor memory (cluster kernel) or HBM (flat kernel)
    float mx = 0.f;
#pragma unroll
    for (int q = 0; q < kMaxFiltersPerWarp; ++q)
        if (q < nf) mx = fmaxf(mx, out[q]);
    return mx;
}
#undef WLM_MEL_TERM

// Unrolled variant for the two Whisper banks: group boundaries, the warp's filter run and the P row of
// every bin are compile-time constants (mel_structure.inc, fft::row_of_bin), so the stage is
// straight-line code -- one LDS and two FFMA with constant-bank weights per bin.
template <int NMELS> struct MelFixed;
template <> struct MelFixed<80> {
    static __device__ __forceinline__ constexpr int gstart(int v) { return kMelGstart80[v]; }
    static __device__ __forceinline__ constexpr int m0(int w) { return kMelM0_80[w]; }
    static __device__ __forceinline__ constexpr int nf(int w) { return kMelNf_80[w]; }
};
template <> struct MelFixed<128> {
    static __device__ __forceinline__ constexpr int gstart(int v) { return kMelGstart128[v]; }
    static __device__ __forceinline__ constexpr int m0(int w) { return kMelM0_128[w]; }
    static __device__ __forceinline__ constexpr int nf(int w) { return kMelNf_128[w]; }
};

template <int NMELS, int W, class Sink>
__device__ __forceinline__ float mel_fixed_warp(const KernelTables& kt, const float* P, int lane, Sink sink) {
    using S = MelFixed<NMELS>;
    constexpr int nf = S::nf(W), m0 = S::m0(W);
    const float* pl = P + (lane >> 1) * (2 * kPPair) + (lane & 1);      // this frame's row of P
    float out[kMaxFiltersPerWarp];
#pragma unroll
    for (int q = 0; q < kMaxFiltersPerWarp; ++q) out[q] = 0.f;
#pragma unroll
    for (int g = 0; g <= nf; ++g) {
#pragma unroll
        for (int k = S::gstart(m0 + g); k < S::gstart(m0 + g + 1); ++k) {
            const float2 w = kt.w2[k];
            const float pv = pl[2 * p_index_of_bin(k)];
            if (g < nf) out[g] = fmaf(pv, w.y, out[g]);            // rising side of m0+g
            if (g > 0) out[g - 1] = fmaf(pv, w.x, out[g - 1]);     // falling side of m0+g-1
        }
    }
    sink(out);          // the 16 mel powers of this lane's frame: tensor memory (cluster kernel) or HBM (flat kernel)
    float mx = 0.f;
#pragma unroll
    for (int q = 0; q < nf; ++q) mx = fmaxf(mx, out[q]);
    return mx;
}

template <int NMELS, class Sink>
__device__ __forceinline__ float mel_fixed(const KernelTables& kt, const float* P, int wg, int lane, Sink sink) {
    // a tree of direct branches, not a switch: that becomes an indirect branch through a jump table (BRX), measured 1 % slower
    if (wg < 4) {
        if (wg < 2) {
            if (wg == 0) return mel_fixed_warp<NMELS, 0>(kt, P, lane, sink);
            return mel_fixed_warp<NMELS, 1>(kt, P, lane, sink);
        }
        if (wg == 2) return mel_fixed_warp<NMELS, 2>(kt, P, lane, sink);
        return mel_fixed_warp<NMELS, 3>(kt, P, lane, sink);
    }
    if (wg < 6) {
        if (wg == 4) return mel_fixed_warp<NMELS, 4>(kt, P, lane, sink);
        return mel_fixed_warp<NMELS, 5>(kt, P, lane, sink);
    }
    if (wg == 6) return mel_fixed_warp<NMELS, 6>(kt, P, lane, sink);
    return mel_fixed_warp<NMELS, 7>(kt, P, lane, sink);
}

// log10(max(p, 1e-10)) == max(log10 p, -10): exactly -10 for silence (TF-FE:155); p = 0 -> -inf -> -10
__device__ __forceinline__ float log10_floor(float p) {
    constexpr float kLog10_2 = 0.30102999566398120f;
    return fmaxf(lg2_approx(p) * kLog10_2, -10.0f);
}

// ---- output element formats ----------------------------------------------------------------------
// The features leave the chip as float32 (the reference's dtype, TF-FE:326), or as bfloat16 / float16 for a model that
// runs under autocast (REF/scripts/train.py:250): round-to-nearest of the same float32 value.
template <class T> __device__ __forceinline__ T to_out(float v);
template <> __device__ __forceinline__ float to_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 to_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half to_out<__half>(float v) { return __float2half_rn(v); }
template <class T> __device__ __forceinline__ float from_out(T v);
template <> __device__ __forceinline__ float from_out<float>(float v) { return v; }
template <> __device__ __forceinline__ float from_out<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float from_out<__half>(__half v) { return __half2float(v); }

// The element type is a template parameter of the kernel (a run-time switch tripled the code of the output pass and
// cost 6 % through the instruction cache): f is called with a.out as OutT*.  A lambda, not a block with a typed pointer:
// the lambda's scope shapes ptxas's register allocation, and the block form changed the SASS of every kernel instance.
template <class OutT, class F>
__device__ __forceinline__ void with_out_type(const ClipArgs& a, F f) { f(static_cast<OutT*>(a.out)); }
// One base pointer, immediate row offsets and one compare per row: left to the compiler, every row carried its own
// predicated address computation (LDC + LEA + LEA.HI.X + two ISETP) -- the output pass was 180 instructions per half-tile.
// base[ELEM_OFF] = v if q < lim: one compare and one predicated store with an immediate offset
template <class T, int ELEM_OFF>
__device__ __forceinline__ void store_row(T* base, float v, int lim, int q) {
    if constexpr (sizeof(T) == 4) {
        asm volatile("{\n.reg .pred p;\nsetp.lt.s32 p, %3, %4;\n@p st.global.f32 [%0+%1], %2;\n}"
                     ::"l"(base), "n"(ELEM_OFF * 4), "f"(v), "r"(q), "r"(lim) : "memory");
    } else {
        const T t = to_out<T>(v);
        asm volatile("{\n.reg .pred p;\nsetp.lt.s32 p, %3, %4;\n@p st.global.b16 [%0+%1], %2;\n}"
                     ::"l"(base), "n"(ELEM_OFF * 2), "h"(*reinterpret_cast<const unsigned short*>(&t)), "r"(q), "r"(lim) : "memory");
    }
}

// N (1..4) consecutive rows at once when the lane stores all of them or none: one compare for the block
template <class T, int ELEM_OFF, int N>
__device__ __forceinline__ void store_rows(T* base, const float (&v)[4], int ok) {
    static_assert(N >= 1 && N <= 4, "1..4 rows");
    constexpr int kB = static_cast<int>(sizeof(T));
    if constexpr (sizeof(T) == 4) {
        if constexpr (N == 4)
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %5, 0;\n@p st.global.f32 [%0+%1], %6;\n@p st.global.f32 [%0+%2], %7;\n"
                         "@p st.global.f32 [%0+%3], %8;\n@p st.global.f32 [%0+%4], %9;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "n"((ELEM_OFF + kNFrames) * kB), "n"((ELEM_OFF + 2 * kNFrames) * kB),
                           "n"((ELEM_OFF + 3 * kNFrames) * kB), "r"(ok), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
        else if constexpr (N == 3)
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %4, 0;\n@p st.global.f32 [%0+%1], %5;\n@p st.global.f32 [%0+%2], %6;\n"
                         "@p st.global.f32 [%0+%3], %7;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "n"((ELEM_OFF + kNFrames) * kB), "n"((ELEM_OFF + 2 * kNFrames) * kB),
                           "r"(ok), "f"(v[0]), "f"(v[1]), "f"(v[2]) : "memory");
        else if constexpr (N == 2)
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %3, 0;\n@p st.global.f32 [%0+%1], %4;\n@p st.global.f32 [%0+%2], %5;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "n"((ELEM_OFF + kNFrames) * kB), "r"(ok), "f"(v[0]), "f"(v[1]) : "memory");
        else
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %2, 0;\n@p st.global.f32 [%0+%1], %3;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "r"(ok), "f"(v[0]) : "memory");
    } else {
        unsigned short h[4] = {0, 0, 0, 0};
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const T t = to_out<T>(v[i]);
            h[i] = *reinterpret_cast<const unsigned short*>(&t);
        }
        if constexpr (N == 4)
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %5, 0;\n@p st.global.b16 [%0+%1], %6;\n@p st.global.b16 [%0+%2], %7;\n"
                         "@p st.global.b16 [%0+%3], %8;\n@p st.global.b16 [%0+%4], %9;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "n"((ELEM_OFF + kNFrames) * kB), "n"((ELEM_OFF + 2 * kNFrames) * kB),
                           "n"((ELEM_OFF + 3 * kNFrames) * kB), "r"(ok), "h"(h[0]), "h"(h[1]), "h"(h[2]), "h"(h[3]) : "memory");
        else if constexpr (N == 3)
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %4, 0;\n@p st.global.b16 [%0+%1], %5;\n@p st.global.b16 [%0+%2], %6;\n"
                         "@p st.global.b16 [%0+%3], %7;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "n"((ELEM_OFF + kNFrames) * kB), "n"((ELEM_OFF + 2 * kNFrames) * kB),
                           "r"(ok), "h"(h[0]), "h"(h[1]), "h"(h[2]) : "memory");
        else if constexpr (N == 2)
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %3, 0;\n@p st.global.b16 [%0+%1], %4;\n@p st.global.b16 [%0+%2], %5;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "n"((ELEM_OFF + kNFrames) * kB), "r"(ok), "h"(h[0]), "h"(h[1]) : "memory");
        else
            asm volatile("{\n.reg .pred p;\nsetp.ne.s32 p, %2, 0;\n@p st.global.b16 [%0+%1], %3;\n}"
                         ::"l"(base), "n"(ELEM_OFF * kB), "r"(ok), "h"(h[0]) : "memory");
    }
}

// rows Q0 .. Q0+3 of one retained half-tile: max((log10 p + 4) / 4, floor4) with floor4 = (floor + 4) / 4  (TF-FE:155-161;
// the scale is folded into the logarithm's constant: lg2, one FFMA, one FMNMX per value).  `nf` (warp-uniform) = rows of
// this warp, `lim` = rows this LANE stores (nf, or 0 for a frame past 3000).  NFC >= 0: nf is known at compile time (the
// unrolled kernels), so is the length of the last block, and every block is stored under ONE compare.
template <class T, int Q0, int NFC = -1>
__device__ __forceinline__ void output_block(T* of, const float (&r)[16], float floor4, int lim, int nf) {
    constexpr float kLog10_2_4 = 0.30102999566398120f * 0.25f;
    constexpr int kRows = NFC < 0 ? 4 : (NFC - Q0 < 4 ? NFC - Q0 : 4);
    float lg[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < kRows; ++i) lg[i] = fmaxf(fmaf(lg2_approx(r[Q0 + i]), kLog10_2_4, 1.0f), floor4);
    if constexpr (NFC >= 0) {
        store_rows<T, Q0 * kNFrames, kRows>(of, lg, lim);
    } else if (Q0 + 4 <= nf) {   // (warp-uniform) a full block: the lane stores all four rows or none
        store_rows<T, Q0 * kNFrames, 4>(of, lg, lim);
    } else {
        store_row<T, (Q0 + 0) * kNFrames>(of, lg[0], lim, Q0 + 0);
        store_row<T, (Q0 + 1) * kNFrames>(of, lg[1], lim, Q0 + 1);
        store_row<T, (Q0 + 2) * kNFrames>(of, lg[2], lim, Q0 + 2);
        store_row<T, (Q0 + 3) * kNFrames>(of, lg[3], lim, Q0 + 3);
    }
}
// all rows of a warp whose run length is a compile-time constant
template <class T, int NFC>
__device__ __forceinline__ void output_rows(T* of, const float (&r)[16], float floor4, int lim) {
    if constexpr (0 < NFC) output_block<T, 0, NFC>(of, r, floor4, lim, NFC);
    if constexpr (4 < NFC) output_block<T, 4, NFC>(of, r, floor4, lim, NFC);
    if constexpr (8 < NFC) output_block<T, 8, NFC>(of, r, floor4, lim, NFC);
    if constexpr (12 < NFC) output_block<T, 12, NFC>(of, r, floor4, lim, NFC);
}
// all rows of a warp whose run length `nf` (warp-uniform) is only known at run time
template <class T>
__device__ __forceinline__ void output_rows(T* of, const float (&r)[16], float floor4, int lim, int nf) {
    if (0 < nf) output_block<T, 0>(of, r, floor4, lim, nf);
    if (4 < nf) output_block<T, 4>(of, r, floor4, lim, nf);
    if (8 < nf) output_block<T, 8>(of, r, floor4, lim, nf);
    if (12 < nf) output_block<T, 12>(of, r, floor4, lim, nf);
}

// ---- the clip queue -----------------------------------------------------------------------------------------------
// Clips are handed out dynamically: a worker (a cluster, or a CTA of the flat kernel) takes clip `worker` first (its
// ordinal 0) and every further one from the global counter, so ragged batches balance themselves and the flat CTAs can
// work next to the clusters whatever the clip lengths.  The worker's LEADER (lane 0 of warp 0 of its first CTA) fetches
// ahead of need, at the TOP of a loop iteration (before anything in the iteration can block), and publishes the clip of
// ordinal n in slot n & 7 of a ring that sits in the shared memory of EVERY CTA of the worker (remote stores through
// distributed shared memory), tagged with the ordinal; everybody else polls its local copy.
//   cluster  ordinals 1 and 2 in the prologue; the atomic for ordinal n + 3 is ISSUED at the top of the leader's first
//            iteration of clip n and its result PUBLISHED at the top of the following iteration (a global atomic takes
//            1-2 us to return: consumed at once it stalled the leader's warp, and through the hand-overs its whole
//            cluster, once per clip -- 6 % of the batch)
//   flat     ordinal n + 1 at the top of the iteration four steps before the end of clip n -- a flat CTA needs ~7x
//            longer per clip than a cluster, so it commits late, and only while `flat_reserve` clips are still
//            unassigned (the clusters would otherwise sit idle waiting for it at the end of the batch)
// Readers look at most two (flat: one) ordinals ahead of the clip they are working on, i.e. only at values the leader
// published in an EARLIER iteration of its own program order; the leader's progress never depends on a reader that is
// ahead of it (hand-overs inside a group only involve half-tiles the waiting warp has already finished), so no poll can
// wait for itself.  A slot is reused eight ordinals later; a warp in clip n has waited for the maxima of clip n - 2 of
// all virtual CTAs, so nobody can still be reading ordinal n - 6.
constexpr int kClipEnd = 0x7fffffff;
constexpr int kQueueRing = 8;
__device__ __forceinline__ int queue_get(const unsigned long long* ring, int ord, int first) {
    if (ord == 0) return first;
    const volatile unsigned long long* p = ring + (ord & (kQueueRing - 1));
    unsigned long long v;
    do { v = *p; } while (static_cast<uint32_t>(v >> 32) != static_cast<uint32_t>(ord + 1));
    return static_cast<int>(static_cast<uint32_t>(v));
}
template <bool FLAT, int NCTA>
__device__ __forceinline__ void queue_put(unsigned long long* ring, int ord, int clip) {
    const unsigned long long v = (static_cast<unsigned long long>(static_cast<uint32_t>(ord + 1)) << 32) | static_cast<uint32_t>(clip);
    if constexpr (FLAT) {
        *reinterpret_cast<volatile unsigned long long*>(ring + (ord & (kQueueRing - 1))) = v;
    } else {
        const uint32_t local = static_cast<uint32_t>(__cvta_generic_to_shared(ring + (ord & (kQueueRing - 1))));
#pragma unroll 1
        for (int r = 0; r < NCTA; ++r) {
            uint32_t remote;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(r));
            asm volatile("st.volatile.shared::cluster.u64 [%0], %1;" ::"r"(remote), "l"(v) : "memory");
        }
    }
}
template <bool FLAT>
__device__ __forceinline__ int queue_fetch(const ClipArgs& a, int taken) {
    unsigned int* next = &a.queue->next;
    if constexpr (!FLAT) {
        const unsigned int c = static_cast<unsigned int>(a.n_workers) + atomicAdd(next, 1u);
        return c < static_cast<unsigned int>(a.B) ? static_cast<int>(c) : kClipEnd;
    } else {
        if (taken >= a.flat_cap) return kClipEnd;
        unsigned int cur = *reinterpret_cast<volatile unsigned int*>(next);
        while (true) {
            const long long c = static_cast<long long>(a.n_workers) + cur;
            if (c >= a.B || a.B - c < a.flat_reserve) return kClipEnd;
            const unsigned int old = atomicCAS(next, cur, cur + 1u);
            if (old == cur) return static_cast<int>(c);
            cur = old;
        }
    }
}

// ================================================================================================
// The kernel: persistent clusters of 6 CTAs x 2 warp groups, one clip per cluster at a time.
// ================================================================================================
// NMELS = 80 / 128: unrolled mel stage for the Whisper banks; NMELS = 0: table-driven mel stage.
//
// FLAT = true is the same pipeline for the SMs that 6-CTA clusters cannot cover (clusters do not span GPCs: 22 of them fit,
// 16 SMs stay idle; tools/ubench_corun.cu shows that a second kernel runs there undisturbed).  One CTA per clip, no cluster
// and no tensor memory: the mel stage writes (log10 + 4) / 4 straight to HBM, and when the clip is done the CTA's 16 warps
// meet once, take the clip's max and re-read the clip's 0.96 MB from L2 to apply the max - 8 clamp.
// DYN = false: clips are assigned statically (worker w of W takes clip_first + w, + W, ...; dense batches, where every
// clip costs the same and the host can split the batch between the two kernels up front); DYN = true: from the clip queue.
template <int NMELS, bool FLAT, class OutT, bool DYN>
__global__ void __launch_bounds__(kThreads, 1)
logmel_cluster_kernel(const ClipArgs a, const __grid_constant__ KernelTables kt, const float* __restrict__ win_lane) {
    namespace cg = cooperative_groups;
    constexpr int kVC = FLAT ? kGroups : kVCluster;      // virtual CTAs (warp groups) that share a clip
    constexpr int kCl = FLAT ? 1 : kCluster;
    extern __shared__ __align__(128) unsigned char smem_sym[];
    // The shared-memory base and the thread index as OPAQUE register values: left alone, the compiler re-derives every
    // shared address from S2R SR_CgaCtaId and re-reads SR_TID.X wherever it is short of registers -- 13 S2R per warp and
    // step, each ~50 cycles of latency on the path (3 % of the stall samples).
    uint32_t smem_base_u32;
    asm volatile("mov.b32 %0, %1;" : "=r"(smem_base_u32) : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem_sym))));
    unsigned char* const smem = static_cast<unsigned char*>(__cvta_shared_to_generic(smem_base_u32));
    // (flat kernel) the NEXT launch's cluster kernel may be queued now: its CTAs become resident as the clusters of this
    // launch exit and run their prologue; they wait for this launch to complete before they read or write anything of the
    // caller's (griddepcontrol.wait below)
    if constexpr (FLAT) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // (a special-register read is rematerialised by ptxas wherever it is short of a register, volatile or not; the result
    // of a shuffle is not: the thread index goes through one)
    int tid;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
    tid = __shfl_sync(0xffffffffu, tid, tid & 31);
    const int lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler
    int tg;                                                   // thread index inside the warp group
    asm volatile("mov.b32 %0, %1;" : "=r"(tg) : "r"(tid & (kGroupThreads - 1)));
    const int grp = warp / kGroupWarps, wg = warp % kGroupWarps;   // warp group and warp inside the group (shift / mask instead measured 4 % SLOWER: a different register allocation)

    // this warp's run of filters: compile-time for the 128-mel bank (eight runs of 16), from the tables otherwise
    auto warp_nf = [&]() -> int { if constexpr (NMELS == 128) return kMaxFiltersPerWarp; else return kt.nf[wg]; };
    auto warp_m0 = [&]() -> int { if constexpr (NMELS == 128) return kMaxFiltersPerWarp * wg; else return kt.m0[wg]; };
    unsigned char* gbase = smem + grp * kSmemGroup;
    float* raw = reinterpret_cast<float*>(gbase) + kRawShift;
    float2* Y = reinterpret_cast<float2*>(gbase + kSmemRaw) + wg * kYWarpFloat2;      // this WARP's stage-1 output
    float* P = reinterpret_cast<float*>(gbase + kSmemRaw + kSmemY);
    unsigned char* misc = smem + kGroups * kSmemGroup;
    // mbarriers (8 B each), one set per group.  Inside a warp stage 1 hands over to stage 2 through the warp's own Y
    // (__syncwarp); between warps there are only these: the shared raw buffer and the shared P buffer of the group.
    unsigned char* gm = misc + grp * 64;
    const uint32_t bar_raw = smem_u32(gm);           // TMA landed the half-tile's PCM              (tx, 1 arrival)
    const uint32_t bar_pfull = smem_u32(gm + 24);    // all warps of the group stored the power of the half-tile
    const uint32_t bar_pfree = smem_u32(gm + 32);    // all 8 warps finished the mel stage          (8)
    uint32_t* raw_readers = reinterpret_cast<uint32_t*>(gm + 40);     // warps done with the raw buffer
    // clip-end max exchange (all indexed by clip parity): every virtual CTA of the cluster delivers its max into
    // clip_max of EVERY CTA (distributed shared memory, st.async) which completes bytes on that CTA's bar_max
    const uint32_t bar_max = smem_u32(misc + 256);                    // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(misc + 272);    // TMEM base address
    uint32_t* grp_cnt = reinterpret_cast<uint32_t*>(misc + 288);      // [2][kGroups] warps of the group that have contributed
    int* grp_max = reinterpret_cast<int*>(misc + 320);                // [2][kGroups] running max of the group (float bits, >= 0)
    float* clip_max = reinterpret_cast<float*>(misc + 352);           // [2][kVCluster] written by the peers
    unsigned long long* clipq = reinterpret_cast<unsigned long long*>(misc + 512);   // [8] the worker's clips by ordinal & 7

    cg::cluster_group cluster = cg::this_cluster();
    const int rank = FLAT ? 0 : static_cast<int>(cluster.block_rank());
    // virtual CTA inside the clip -- read back from shared memory for the same reason as the thread index: the cluster rank
    // is a special register, and ptxas sees through a shuffle of a warp-uniform value
    int vrank;
    {
        volatile int* pin = reinterpret_cast<volatile int*>(misc + 768) + warp;
        if (lane == 0) *pin = rank * kGroups + grp;
        __syncwarp();
        vrank = *pin;
    }
    // the worker's first clip is its index; the rest come from the queue (DYN) or follow at a stride of W workers
    const int worker = FLAT ? static_cast<int>(blockIdx.x) : static_cast<int>(blockIdx.x) / kCluster;
    const int n_static = FLAT ? static_cast<int>(gridDim.x) : static_cast<int>(gridDim.x) / kCluster;
    const int first_clip = DYN ? a.worker_base + worker : a.clip_first + worker;
    const bool leader = DYN && rank == 0 && tid == 0;
    // flat kernel: clip-end meeting of the CTA's 16 warps and the clip's max (ring of three: see D)
    const uint32_t bar_clip = smem_u32(misc + 640);
    int* flat_max = reinterpret_cast<int*>(misc + 656);

    if (tid == 0) {
        for (int g = 0; g < kGroups; ++g) {
            const uint32_t b = smem_u32(misc + g * 64);
            mbar_init(b, 1);
            mbar_init(b + 24, kGroupWarps);
            mbar_init(b + 32, kGroupWarps);
            *reinterpret_cast<uint32_t*>(misc + g * 64 + 40) = 0;
        }
        mbar_init(bar_max, 1);          // one arrival (this CTA's group 0, with the byte count) + 12 x 4 bytes from the peers
        mbar_init(bar_max + 8, 1);
        for (int i = 0; i < 2 * kGroups; ++i) { grp_cnt[i] = 0; grp_max[i] = 0; }
        for (int i = 0; i < kQueueRing; ++i) clipq[i] = 0ull;
        mbar_init(bar_clip, kWarps);
        flat_max[0] = flat_max[1] = flat_max[2] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    uint32_t tmem_base = 0;
    if constexpr (FLAT) {
        __syncthreads();
    } else {
        if (warp == 0) tmem_alloc_512(smem_u32(tmem_slot));
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        cluster.sync();     // (also a CTA barrier) every peer's mbarriers and queue ring exist before anyone writes them remotely
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tmem_base = *tmem_slot;
    }
    // the imaginary part of slot 0 in the warp's Y: zeros, written once (stage 1 never stores there)
    Y[(lane >> 1) * kYN1 + kYLanes + (lane & 1)] = make_float2(0.f, 0.f);
    __syncwarp();
    // this warp's TMEM window: lane quarter (warp & 3), 128 columns at (warp >> 2) * 128
    const uint32_t twin = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) +
                          static_cast<uint32_t>((warp >> 2) * kTmemColsPerWarp);

    // per-lane stage-1 constants; the lane's first sample address is held in a register: re-derived, it is 15 instructions a step
    // (through a shuffle with itself: ptxas re-derives anything it can trace back to special registers and parameters)
    const uint32_t s1_base = __shfl_sync(0xffffffffu, stage1_base(raw, wg, lane), lane);
    const int n1 = lane & 15;
    float wv[25];
#pragma unroll
    for (int t = 0; t < 25; ++t) wv[t] = win_lane[n1 * 25 + t];
    if constexpr (!FLAT) {
        // Launched as a programmatic dependent of whatever precedes it in the stream (normally the previous wlm_logmel
        // launch): the launch latency and the prologue above -- barrier and tensor-memory set-up, the cluster barrier, the
        // window table -- overlap the tail of that kernel.  Nothing of the caller's has been touched so far (not the PCM,
        // not the features, not the clip queue); from here on everything earlier in the stream has completed and is
        // visible.  Only then may this launch's own dependent (the flat kernel, which reads PCM at once) start.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (leader) {                                            // (DYN) ordinals 1 and 2 of this cluster: one atomic
            const unsigned int c = static_cast<unsigned int>(a.n_workers) + atomicAdd(&a.queue->next, 2u);
            queue_put<false, kCluster>(clipq, 1, c < static_cast<unsigned int>(a.B) ? static_cast<int>(c) : kClipEnd);
            queue_put<false, kCluster>(clipq, 2, c + 1 < static_cast<unsigned int>(a.B) ? static_cast<int>(c + 1) : kClipEnd);
        }
    }

    // The group's work is a stream of steps, one per half-tile it owns (a clip in which it owns no active
    // half-tile still contributes one empty step so that it takes part in that clip's max exchange).
    // Program order of every warp in step i (half-tile t_i):
    //   Q  (leader lane) fetch a clip ahead and publish it to the worker's CTAs
    //   A  stage 1 of t_i            wait raw | load | last warp re-arms TMA | FFT | store (warp-private Y) | __syncwarp
    //   F  output pass of the clip that ended one step ago   (wait for the 12 maxima, TMEM read-back, stores)
    //   B  mel stage of t_{i-1}      wait P full | ... | arrive P free
    //   D  if t_{i-1} ended a clip:  warp max -> group max (atomic); the last warp delivers it to all 6 CTAs
    //   C  stage 2 of t_i            load own Y | FFT | wait P free | store | arrive P full
    // `c*` = the step whose half-tile is in stage 1 / stage 2, `p*` = the previous step (mel stage).
    auto my_tiles = [&](int n_act) { return n_act > vrank ? (n_act - vrank + kVC - 1) / kVC : 0; };
    int cord = 0;                                                   // ordinal of the current clip among this worker's
    int cb = first_clip, cj = 0, cn_my = 0;                         // clip, step inside the clip, half-tiles of mine in the clip
    bool cvalid = cb < a.B;
    ClipCtx cc;
    cc.b = cb; cc.len = 0; cc.n_act = 0; cc.base = 0; cc.edge0 = 0;
    if (cvalid) {
        cc = clip_ctx(a, cb);
        cn_my = my_tiles(cc.n_act);
    }
    const int n_my_static = cn_my;
    bool pvalid = false, phas = false, plast = false;
    int pb = 0, pj = 0, ptile = 0, pn_my = 0, pn_act = 0;
    int clip_seq = 0;                        // (flat kernel) clips this warp has finished
    int taken = FLAT ? 1 : 2;                // (leader) clips this worker has been given so far
    bool q_end = false;                      // (leader) the queue has answered "no more"
    // TMA target after (clip ordinal ord0, step j0): the next half-tile of the same clip, else the first half-tile of one
    // of the next two (flat: one) clips of this worker in which this group owns one.  Executed by ONE lane (the last warp
    // to finish reading raw).  Returns false if the target is not known yet: the lane then OWES the copy and issues it when
    // its own warp arrives at that half-tile (rare: clips so short that the group idles anyway).
    auto issue_next_tile = [&](int ord0, const ClipCtx& c0, int n_my0, int j0) -> bool {
        if constexpr (!DYN) {
            // static: every clip has the same length, so the target is this clip's next half-tile or the first one of the
            // worker's next clip; it is decided first and the copy issued at ONE place (tile_issue_tma is ~150 instructions
            // inlined: three call sites made the loop body 250 instructions longer, 1.6 % of the step)
            ClipCtx ct = c0;
            int tt = vrank + (j0 + 1) * kVC;
            bool have = j0 + 1 < n_my0;
            if (!have) {
                const int nb = c0.b + n_static;
                tt = vrank;
                if (nb < a.B && c0.n_act > vrank) {
                    ct = clip_ctx_like(a, c0, nb);
                    have = true;
                }
            }
            if (have) tile_issue_tma(a, ct, tt, raw, bar_raw);
            return true;
        } else {
            if (j0 + 1 < n_my0) {
                tile_issue_tma(a, c0, vrank + (j0 + 1) * kVC, raw, bar_raw);
                return true;
            }
#pragma unroll 1
            for (int d = 1; d <= (FLAT ? 1 : 2); ++d) {
                const int nb = queue_get(clipq, ord0 + d, first_clip);
                if (nb >= a.B) return true;                     // end of this worker's stream: nothing to load
                const ClipCtx c2 = clip_ctx(a, nb);
                if (c2.n_act > vrank) {
                    tile_issue_tma(a, c2, vrank, raw, bar_raw);
                    return true;
                }
            }
            return false;
        }
    };

    // Phase bookkeeping: the n-th half-tile this group processes (n = 0, 1, ...) uses phase n of every barrier,
    // i.e. parity n & 1.  A wait for phase n is only issued by a warp that has already arrived on phase n
    // or whose own later work is needed to complete phase n+1, so the barrier is never more than one
    // phase ahead of a waiter.
    int fin_seq = 0;                         // clips whose output pass this warp has done; parity = slot of the exchange
    int tnum = 0;                            // ordinal of cur's half-tile among those of this group (the previous step's is tnum - 1)
    bool i_owe = false;                      // (lane 0) this warp must issue the copy of the half-tile it is about to wait for
    bool q_pending = false;                  // (cluster leader) an atomic is in flight: its result is published one iteration later
    unsigned int q_val = 0;
    int q_ord = 0;
    if (tg == 0 && cvalid && !kKoRaw) {
        if (cn_my > 0) tile_issue_tma(a, cc, vrank, raw, bar_raw);
        else i_owe = !issue_next_tile(0, cc, 0, 0);
    }
    // frames past 3000 do not exist: they are the last lanes of the clip's last half-tile
    const bool tail_lane = lane >= kNFrames - (kTilesPerClip - 1) * kTile;
    // ... as a step index: the step of this group whose half-tile is the clip's last one, for the lanes it matters to
    const int tail_j = (tail_lane && (kTilesPerClip - 1 - vrank) % kVC == 0) ? (kTilesPerClip - 1 - vrank) / kVC : -1;
    float mx = 0.f;                          // running max of the mel power of the clip in flight (>= 0)
    bool pend = false;                       // an output pass is owed (max delivered, not yet waited for)
    int pend_b = 0, pend_n_my = 0;
    int64_t pend_e0 = 0;                     // element index of (pending clip, this warp's first filter, frame = lane)
    int out_j = 0;                           // next retained half-tile of the pending clip to write out
    bool have_max = false;                   // the pending clip's max has arrived (floor4 valid)
    float floor4 = 0.f;                      // (max(gmax - 8, -10) + 4) / 4: the clip's lowest feature value

#ifdef WLM_WAITSTAT
    long long ws_acc[5] = {0, 0, 0, 0, 0};
    const long long ws_loop0 = clock64();
#endif
    while (cvalid || pvalid || pend) {
        const bool do_tile = cvalid && cj < cn_my;
        const int ctile = vrank + cj * kVC;
        // ---- Q: the leader fetches ahead (see "the clip queue") ------------------------------------------
        if (leader) {
            if (q_pending) {
                const unsigned int c = static_cast<unsigned int>(a.n_workers) + q_val;
                q_end = c >= static_cast<unsigned int>(a.B);
                queue_put<FLAT, kCl>(clipq, q_ord, q_end ? kClipEnd : static_cast<int>(c));
                q_pending = false;
            }
            if (cvalid && !q_end) {
                if constexpr (FLAT) {
                    const int steps_q = cn_my > 0 ? cn_my : 1;
                    if (cj == (steps_q > 4 ? steps_q - 4 : 0)) {
                        const int c = queue_fetch<true>(a, taken);
                        ++taken;
                        q_end = c == kClipEnd;
                        queue_put<true, 1>(clipq, cord + 1, c);
                    }
                } else if (cj == 0) {
                    q_val = atomicAdd(&a.queue->next, 1u);      // (not consumed in this iteration)
                    q_ord = cord + 3;
                    q_pending = true;
                }
            }
        }
        // ---- A: stage 1 ----------------------------------------------------------------------------
        if (do_tile) {
            if constexpr (DYN) {
                if (lane == 0 && i_owe) {
                    tile_issue_tma(a, cc, ctile, raw, bar_raw);
                    i_owe = false;
                }
            }
            { WLM_WS_BEGIN(); if constexpr (!kKoRaw) mbar_wait(bar_raw, tnum & 1); WLM_WS_END(0); }
            // interior half-tiles of float32 PCM need no patching (group-uniform condition: tile_fixup has group barriers)
            if ((a.pcm_format == WLM_PCM_I16 || ctile == 0 || ctile >= cc.edge0)) tile_fixup(a.pcm_format, cc.len, ctile, raw, grp, tg);
            // This warp is done with raw once the 25-point DFTs have consumed its samples (the loads have then completed by
            // data dependence, so no fence holds the warp up between its loads and its arithmetic); the last of the 8
            // re-arms the TMA for the next half-tile, which is not needed before the next step.
            stage1(s1_base, Y, wv, wg, lane, [&]() {},
                   [&]() {
                       __syncwarp();
                       if (lane == 0) {
                           uint32_t old;      // (atom.inc wraps to 0 by itself; atom.add is turned into warp-aggregated code)
                           asm volatile("atom.shared.inc.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(raw_readers)), "n"(kGroupWarps - 1) : "memory");
                           if (old == kGroupWarps - 1) {
                               asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                               if constexpr (!kKoRaw) i_owe = !issue_next_tile(cord, cc, cn_my, cj);
                           }
                       }
                   });
            __syncwarp();      // Y is private to the warp: this is the whole stage 1 -> stage 2 hand-over
        }
        // ---- F: output of the clip that ended one step ago, ONE retained half-tile per step ----------------------
        // (the slot the mel stage below is about to overwrite: tcgen05.ld is 64 B/clk per SM, so a whole-clip pass by
        // all 16 warps at once stalls everything for ~4k cycles; spread over the next clip's steps it hides under the FFTs)
        auto output_finish = [&](int j, const float (&r)[16]) {
            const int nf = warp_nf();
            const int otile = vrank + j * kVC;
            const int64_t e0 = pend_e0 + otile * kTile;
            const int lim = (j != tail_j && !(kKoStg && a.B > 0)) ? nf : 0;       // rows this lane stores
            with_out_type<OutT>(a, [&](OutT* outp) {
                OutT* of = outp + e0;
                // rows in blocks of four (output_block): straight-line code inside a block, so four MUFU.LG2 chains overlap
                if constexpr (NMELS == 128) {      // eight runs of 16: no run-length branches, one compare per block (-2 %)
                    output_rows<OutT, kMaxFiltersPerWarp>(of, r, floor4, lim);    // (the same per warp for the 80-mel bank, behind
                                                                                  // an 8-way dispatch: 500 more instructions, 4.5 % SLOWER)
                } else {
                    output_rows<OutT>(of, r, floor4, lim, nf);
                }
            });
        };
        auto output_slot = [&](int j) {
            float r[16];
            if constexpr (kKoTld) {
#pragma unroll
                for (int i = 0; i < 16; ++i) r[i] = floor4 + static_cast<float>(i + j);
            } else {
                tmem_wait_st();
                tmem_ld_x16(twin + j * kTmemColsPerTile, r);
            }
            output_finish(j, r);
        };
        if (!FLAT && pend) {
            if ((!have_max)) {    // first step after the clip ended: the 12 maxima
                const int fpar = fin_seq & 1;
                { WLM_WS_BEGIN(); mbar_wait_cluster(bar_max + fpar * 8, (fin_seq >> 1) & 1); WLM_WS_END(3); }
                float pmax = lane < kVCluster ? clip_max[fpar * kVCluster + lane] : 0.f;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
                ++fin_seq;
                have_max = true;
                const float gmax = log10_floor(pmax);                 // TF-FE:157
                floor4 = (fmaxf(gmax - 8.0f, -10.0f) + 4.0f) * 0.25f;      // TF-FE:158,161 (log-mel is never below -10)
                if (vrank == 0 && tg == 0 && a.gmax) a.gmax[pend_b] = gmax;
                // half-tiles of mine that hold no real sample: log-mel is exactly -10 everywhere
                const float silent = floor4;
                const int nf = warp_nf();
                const int64_t e0 = pend_e0;
                with_out_type<OutT>(a, [&](OutT* outp) {
                    // (left to the compiler's unrolling: ragged batches of short clips spend real time here)
                    for (int tile = vrank + pend_n_my * kVCluster; tile < kTilesPerClip; tile += kVCluster) {
                        OutT* of = outp + e0 + tile * kTile;
                        if (tile * kTile + lane < kNFrames)
                            for (int q = 0; q < nf; ++q) of[q * kNFrames] = to_out<OutT>(silent);
                    }
                });
            }
            if (out_j < pend_n_my) {
                if constexpr (!kKoOut) output_slot(out_j);
                ++out_j;
            }
            if (out_j >= pend_n_my) pend = false;
        }
        // ---- B: mel stage of the previous half-tile ---------------------------------------------------------
        const bool clip_ends = pvalid && plast;
        const bool mel_tile = pvalid && phas;
        const int cpar = fin_seq & 1;            // F has run: this is the parity of the clip ending now
        float wmax = 0.f;                        // this warp's max over the clip (valid when clip_ends)
        if (mel_tile) {
            { WLM_WS_BEGIN(); if constexpr (!kKoPfull) mbar_wait(bar_pfull, (tnum - 1) & 1); WLM_WS_END(1); }
            const uint32_t tcol = twin + pj * kTmemColsPerTile;
            float m1;
            if constexpr (FLAT) {
                // no retention: (max(log10 p, -10) + 4) / 4 goes to HBM now, the max - 8 clamp follows when the clip is done
                const int nf = warp_nf();
                const int64_t e0 = (static_cast<int64_t>(pb) * a.n_mels + warp_m0()) * kNFrames + ptile * kTile + lane;
                const int lim = pj != tail_j ? nf : 0;      // rows this lane stores
                auto sink = [&](const float (&o)[kMaxFiltersPerWarp]) {
                    with_out_type<OutT>(a, [&](OutT* outp) {
                        OutT* of = outp + e0;
                        output_rows<OutT>(of, o, -1.5f, lim, nf);      // floor (-10 + 4) / 4
                    });
                };
                m1 = NMELS == 0 ? mel_stage(kt, P, wg, lane, sink) : mel_fixed<NMELS == 0 ? 80 : NMELS>(kt, P, wg, lane, sink);
            } else {
                auto sink = [&](const float (&o)[kMaxFiltersPerWarp]) {
                    if constexpr (kKoTst) { if (o[3] == -1.0f) tmem_st_x16(tcol, o); }
                    else tmem_st_x16(tcol, o);
                };
                if constexpr (kKoMel) m1 = P[lane];
                else m1 = NMELS == 0 ? mel_stage(kt, P, wg, lane, sink) : mel_fixed<NMELS == 0 ? 80 : NMELS>(kt, P, wg, lane, sink);
            }
            if (pj != tail_j) mx = fmaxf(mx, m1);
            if (clip_ends) {
                wmax = mx;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
                mx = 0.f;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_pfree);   // phase tnum - 1
        }
        // ---- D: the clip ended: warp max -> group max; the LAST warp of the group to get here delivers the group's
        // max to all 6 CTAs (remote store + remote mbarrier arrive).  Nobody waits; the peers get a whole step of
        // slack before anyone needs the result (F, next step).
        if (FLAT && (clip_ends)) {
            // The CTA's 16 warps meet (once per clip), take the clip's max and clamp the clip's features in place:
            // they were written moments ago and come back from L2.  flat_max is a ring of three so that the slot of the
            // clip after next can be cleared here without racing with anybody (its last readers arrived above, its next
            // writers wait for this thread's next arrival).
            const int slot3 = clip_seq % 3;
            __threadfence();                                         // this lane's feature stores are visible device-wide
            __syncwarp();
            if (lane == 0) {
                if (mel_tile) atomicMax(flat_max + slot3, __float_as_int(wmax));
                mbar_arrive(bar_clip);
            }
            mbar_wait(bar_clip, clip_seq & 1);
            const float gmax = log10_floor(__int_as_float(*reinterpret_cast<volatile int*>(flat_max + slot3)));   // TF-FE:157
            const float thr = (fmaxf(gmax - 8.0f, -10.0f) + 4.0f) * 0.25f;                                        // TF-FE:158,161
            if (tid == 0) {
                flat_max[(clip_seq + 2) % 3] = 0;
                if (a.gmax) a.gmax[pb] = gmax;
            }
            const int n_valid = min(kNFrames, pn_act * kTile);          // frames of half-tiles that hold real samples
            with_out_type<OutT>(a, [&](OutT* outp) {
                constexpr int kPer = 16 / static_cast<int>(sizeof(OutT));   // elements per 16-byte vector (3000 % kPer == 0)
                struct alignas(16) Vec { OutT e[kPer]; };
                Vec* oc = reinterpret_cast<Vec*>(outp + static_cast<int64_t>(pb) * a.n_mels * kNFrames);
                const OutT thr_t = to_out<OutT>(thr);                       // rounded like the features: max(round x, round t) = round max(x, t)
                const float thr_f = from_out<OutT>(thr_t);
                // eight 16-byte loads in flight per thread: the clip may have left L2 by now (the cluster kernel streams through it)
                constexpr int kRow = kNFrames / kPer;
                const int nv = a.n_mels * kRow;
                for (int i0 = tid; i0 < nv; i0 += 8 * kThreads) {
                    Vec v[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int i = i0 + u * kThreads;
#pragma unroll
                        for (int e = 0; e < kPer; ++e) v[u].e[e] = thr_t;     // silent half-tiles: exactly -10 everywhere -> thr
                        if (i < nv && (i % kRow) * kPer < n_valid) {          // (n_valid: multiple of 32 or 3000)
                            const float4 w = __ldcg(reinterpret_cast<const float4*>(oc + i));
                            v[u] = *reinterpret_cast<const Vec*>(&w);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int i = i0 + u * kThreads;
#pragma unroll
                        for (int e = 0; e < kPer; ++e)
                            if (from_out<OutT>(v[u].e[e]) < thr_f) v[u].e[e] = thr_t;
                        if (i < nv) *reinterpret_cast<float4*>(oc + i) = *reinterpret_cast<const float4*>(&v[u]);
                    }
                }
            });
            ++clip_seq;
        }
        if (!FLAT && (clip_ends)) {
            while (pend) {      // (only when this clip had fewer half-tiles than the one before it: finish that one first;
                                // draining inside F instead, one copy of the output code, measured 3 % slower)
                if (out_j < pend_n_my) output_slot(out_j++);
                if (out_j >= pend_n_my) pend = false;
            }
            if (lane == 0) {
                int* gmx = grp_max + cpar * kGroups + grp;
                uint32_t* gct = grp_cnt + cpar * kGroups + grp;
                if (mel_tile) atomicMax(gmx, __float_as_int(wmax));     // non-negative floats order like their bit patterns
                __threadfence_block();
                if (atomicAdd(gct, 1u) == kGroupWarps - 1) {
                    __threadfence_block();
                    const float m = __int_as_float(atomicExch(gmx, 0));  // (reset for the clip after next)
                    atomicExch(gct, 0u);
                    // Fire-and-forget: st.async writes the value into the peer's clip_max and completes 4 bytes on the
                    // peer's bar_max (a remote store + release-arrive pair cost ~900 cycles EACH on the one warp the
                    // whole group was then waiting for).  Every CTA's group 0 posts the expectation of 12 x 4 bytes.
                    const uint32_t slot_l = smem_u32(clip_max + cpar * kVCluster + vrank), bar_l = bar_max + cpar * 8;
                    if (grp == 0) mbar_expect_tx(bar_l, 4u * kVCluster);
#pragma unroll 1      /* once per clip and group: kept a loop, the body of the step loop is short of instruction cache */
                    for (int r = 0; r < kCluster; ++r) {
                        uint32_t slot_r, bar_r;
                        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(slot_r) : "r"(slot_l), "r"(r));
                        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bar_r) : "r"(bar_l), "r"(r));
                        asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                                     ::"r"(slot_r), "r"(__float_as_uint(m)), "r"(bar_r) : "memory");
                    }
                }
            }
            pend = true;
            have_max = false;
            out_j = 0;
            // static assignment: every clip has the same length, and the clip that just ended is one stride back
            pend_b = DYN ? pb : cb - n_static;
            pend_e0 = (static_cast<int64_t>(pend_b) * a.n_mels + warp_m0()) * kNFrames + lane;
            pend_n_my = DYN ? pn_my : n_my_static;
        }
        // ---- C: stage 2 (every warp, on its own two frame pairs) ------------------------------------------
        if (do_tile) {
            stage2(Y, P, wg, lane, [&]() {
                // the mel stage of the previous half-tile must have read P (all warps of the group)
                WLM_WS_BEGIN();
                if constexpr (!kKoPfree) if (tnum > 0) mbar_wait(bar_pfree, (tnum - 1) & 1);
                WLM_WS_END(2);
            });
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_pfull);   // phase tnum
        }
        // this step becomes the previous one; advance to the next step of the stream
        const int steps = cn_my > 0 ? cn_my : 1;
        pvalid = cvalid; phas = do_tile; plast = cvalid && cj + 1 >= steps;
        pj = cj;
        if constexpr (DYN || FLAT) { pb = cb; pn_my = cn_my; }
        if constexpr (FLAT) { ptile = ctile; pn_act = cc.n_act; }
        if (do_tile) ++tnum;
        if (cvalid) {
            if (cj + 1 < steps) {
                ++cj;
            } else {
                ++cord;
                cb = DYN ? queue_get(clipq, cord, first_clip) : cb + n_static;
                cj = 0;
                cn_my = 0;
                cvalid = cb < a.B;
                if (cvalid) {
                    if constexpr (DYN) {
                        cc = clip_ctx(a, cb);
                        cn_my = my_tiles(cc.n_act);
                    } else {
                        cc = clip_ctx_like(a, cc, cb);
                        cn_my = n_my_static;
                    }
                }
            }
        }
    }
#ifdef WLM_WAITSTAT
    ws_acc[4] = clock64() - ws_loop0;
    if (lane == 0 && a.gmax)
        for (int k = 0; k < 5; ++k) a.gmax[(blockIdx.x * kWarps + warp) * 8 + k] = static_cast<float>(ws_acc[k]);
#endif
    if constexpr (FLAT) {
        __syncthreads();
        // A programmatic dependent of the cluster kernel and the LAST kernel of the launch in the stream: it must not
        // complete before the clusters have written everything, or later work in the stream (the copy of the features, the
        // next launch) could overtake them.  The price is a second completion hop at the end of every launch (+10 us:
        // round 1 lacked the wait and was that much faster per launch -- and wrong).  Measured alternatives: a completion
        // counter polled here (+1 % on top), the flat kernel launched FIRST as the primary of the pair (its CTAs then
        // take SMs the clusters need: +55 %).
        asm volatile("griddepcontrol.wait;" ::: "memory");
    } else {
        // all TMEM reads are complete (tcgen05.wait::ld inside tmem_ld_x16); release the allocation
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        cluster.sync();   // also keeps every CTA's shared memory alive until its peers have delivered their last max
        if (warp == 0) tmem_dealloc_512(tmem_base);
    }
    // (DYN) every warp of this worker is past its last fetch: the last worker of the launch leaves the queue at {0, 0}
    if (leader) {
        if (atomicAdd(&a.queue->done, 1u) == static_cast<unsigned int>(a.n_workers) - 1u) {
            a.queue->next = 0u;
            a.queue->done = 0u;
            __threadfence();
        }
    }
}

}  // namespace fused
}  // namespace wlm
