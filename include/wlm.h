/*
 * wlm.h -- C ABI of libwlm.so, the B200 (sm_100a) log-mel front-end.
 *
 * Drop-in boundary for ONE path of thanh-nt25/Whisper-context-biasing: the
 * `WhisperFeatureExtractor` call that turns 16 kHz PCM into
 * `input_features [B, n_mels, 3000] float32`.
 *
 * The reference has no FFI for this path -- it injects a Python object by constructor
 * argument (REF/data_utils/data_loader.py:59,75 ; REF/data_utils/data_collator.py:71) and calls
 *
 *     feature_extractor(audio, sampling_rate=16000).input_features      data_loader.py:171
 *     feature_extractor(audio["array"], sampling_rate=...)              data_collator.py:19-21
 *     processor.feature_extractor.pad(..., padding="longest", "pt")     data_collator.py:71-76
 *
 * whose arithmetic lives in the third-party `transformers` package
 * (models/whisper/feature_extraction_whisper.py, "TF-FE" below; audio_utils.py "TF-AU";
 * feature_extraction_sequence_utils.py "TF-SU").  Each entry point below names the piece of
 * that interface it replaces.  Plain pointers and sizes only; no torch types.
 *
 * Conventions
 *   - every function returns 0 (WLM_OK) or a negative WLM_ERR_* code; wlm_last_error() gives
 *     a thread-local human-readable string for the last failure.
 *   - the caller owns every buffer.  Device work is asynchronous on the caller's stream; no
 *     implicit synchronisation unless stated.
 *   - a wlm_plan is per process and per device, and may be used by one host thread at a time.
 *   - there is NO CPU fallback: without a CUDA device of compute capability 10.x the plan
 *     cannot be created.
 */
#ifndef WLM_H_
#define WLM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WLM_VERSION 10100 /* 1.01.00 */

#define WLM_SAMPLING_RATE 16000 /* TF-FE:72 */
#define WLM_N_FFT 400           /* TF-FE:75 */
#define WLM_HOP 160             /* TF-FE:73 */
#define WLM_N_SAMPLES 480000    /* TF-FE:91  chunk_length * sampling_rate */
#define WLM_N_FRAMES 3000       /* TF-FE:92  nb_max_frames */
#define WLM_N_FREQ 201          /* TF-FE:96  1 + n_fft/2 */

enum {
    WLM_OK = 0,
    WLM_ERR_BAD_ARG = -1,      /* null pointer, negative size, misaligned buffer          */
    WLM_ERR_UNSUPPORTED = -2,  /* n_mels not in [1,128]; mel table not two-adjacent-per-bin */
    WLM_ERR_CUDA = -3,         /* a CUDA call failed; see wlm_last_error()                  */
    WLM_ERR_NO_DEVICE = -4,    /* no sm_100 device: the library never falls back to the CPU */
    WLM_ERR_WORKSPACE = -5     /* workspace smaller than wlm_workspace_bytes()              */
};

/* PCM sample formats accepted by wlm_logmel / wlm_logmel_host. */
enum {
    WLM_PCM_F32 = 0, /* float32 in [-1,1]  (what librosa.load returns, data_loader.py:170)   */
    WLM_PCM_I16 = 1  /* int16; converted on the GPU as x/32768 (data_loader.py:48 load_wave) */
};

/* Output element formats (wlm_plan_set_output_format).  Layout is always [B, n_mels, 3000],
 * mel-major, frame-contiguous.  The 16-bit formats are the round-to-nearest of the float32 value:
 * the model of the reference runs under fp16 autocast (REF/scripts/train.py:250), so its first
 * convolution rounds the features to 16 bits anyway; storing them that way halves the write bytes. */
enum {
    WLM_OUT_F32 = 0, /* float32: what the reference returns (TF-FE:326) */
    WLM_OUT_BF16 = 1,
    WLM_OUT_F16 = 2
};

typedef struct wlm_plan wlm_plan;

/* Library version (WLM_VERSION of the build). */
int wlm_version(void);

/* Thread-local description of the last error returned on this thread ("" if none). */
const char* wlm_last_error(void);

/*
 * Replaces WhisperFeatureExtractor.__init__ (TF-FE:69-103): fixes n_fft=400, hop=160,
 * 30 s chunks, padding_value 0.0 (dither is an argument of wlm_logmel_conditioned) and takes the mel table the constructor builds.
 *
 *   device              CUDA ordinal
 *   n_mels              feature_size (80 whisper-base/small, 128 large-v3)
 *   mel_dense_host      float32 [201][n_mels] row-major = `mel_filters.astype(float32)` of
 *                       TF-FE:95-103 / TF-AU:453-544, so the weights are bit-identical to the
 *                       ones the reference multiplies with (TF-FE:152-153).  The table must have
 *                       at most two non-zeros per FFT bin, in adjacent filters (true for every
 *                       triangular bank); otherwise WLM_ERR_UNSUPPORTED.
 */
int wlm_plan_create(int device, int n_mels, const float* mel_dense_host, wlm_plan** out);
int wlm_plan_destroy(wlm_plan* plan);

/* Introspection (all return <0 on a null plan). */
int wlm_plan_n_mels(const wlm_plan* plan);
int wlm_plan_device(const wlm_plan* plan);
int wlm_plan_sm_count(const wlm_plan* plan);
/* 80 / 128: the mel stage runs unrolled with the structure of that Whisper bank baked in (the
 * caller's table has exactly that structure); 0: table-driven mel stage (any other valid table). */
int wlm_plan_kernel_variant(const wlm_plan* plan);
/* Thread-block clusters of the fused kernel that are co-resident on the device (persistent grid). */
int wlm_plan_max_clusters(const wlm_plan* plan);

/*
 * Element type of `out_dev` for every later wlm_logmel / wlm_logmel_host call of this plan
 * (default WLM_OUT_F32).  With a 16-bit format `out_dev` points to 2-byte elements and
 * `out_host` of wlm_logmel_host likewise.
 */
int wlm_plan_set_output_format(wlm_plan* plan, int out_format);
int wlm_plan_output_format(const wlm_plan* plan);

/*
 * Debug / measurement knob for the cluster-less twin of the kernel that runs on the SMs whole
 * clusters cannot cover (both kernels pull clips from one queue): -1 (default) = the library's
 * own rule; 0 = never launch it; n > 0 = it may take up to n clips of every batch, whatever
 * the batch.  The environment variable WLM_FLAT_CLIPS, read ONCE when the plan is created,
 * sets the initial value.
 */
int wlm_plan_set_flat_clips(wlm_plan* plan, int n_flat);

/*
 * Device scratch needed by wlm_logmel for a batch of B clips (bytes, 256-aligned).
 * May be 0.  The buffer is only used during the call's stream work.
 */
size_t wlm_workspace_bytes(const wlm_plan* plan, int B);

/*
 * THE HOT PATH.  Replaces, for a whole batch in one launch sequence:
 *   pad/trim to 480000        SequenceFeatureExtractor.pad/_truncate/_pad  TF-SU:51-219,293-334
 *   reflect-pad + framing     torch.stft(center=True)                     TF-FE:149
 *   Hann window + rFFT-400    torch.hann_window / torch.stft              TF-FE:141,149
 *   |X|^2, drop frame 3000    stft[..., :-1].abs() ** 2                   TF-FE:150
 *   mel projection            mel_filters.T @ magnitudes                  TF-FE:152-153
 *   log10(clamp 1e-10)        torch.clamp(...).log10()                    TF-FE:155
 *   per-clip max - 8 clamp    torch.maximum(log_spec, max - 8.0)          TF-FE:156-160
 *   (x + 4) / 4               TF-FE:161
 *
 *   pcm_dev       device pointer, element type `pcm_format`, 16-byte aligned.
 *   offsets_dev   NULL  -> clip b starts at element b*row_stride (dense [B,row_stride] layout;
 *                          row_stride must be a multiple of 4 elements);
 *                 else  -> device int64[B], clip b starts at element offsets_dev[b] (ragged).
 *                          Every start must be 16-byte aligned (a multiple of 4 float32 / 8 int16
 *                          elements), and the buffer must be readable up to the next 16-byte
 *                          boundary after the last sample of every clip: the bulk copies move whole
 *                          16-byte units (what lies between lengths[b] and that boundary is ignored).
 *   lengths_dev   NULL  -> every clip has min(row_stride, 480000) valid samples (dense only);
 *                 else  -> device int32[B], valid samples of clip b (any value >= 0; values
 *                          above 480000 are truncated, the rest is right-padded with zeros,
 *                          exactly as TF-SU:327-332 and :268-278 do on the host).
 *   out_dev       device [B][n_mels][3000] of the plan's output format (float32 unless
 *                 wlm_plan_set_output_format was called), 16-byte aligned.
 *   gmax_dev      optional device float32[B]: receives the per-clip max of log10(mel)
 *                 (the value TF-FE:157 computes); may be NULL.
 *   workspace     device scratch of at least wlm_workspace_bytes(plan,B) bytes (or NULL if 0).
 *   stream        cudaStream_t (as void*) the work is enqueued on.
 */
int wlm_logmel(wlm_plan* plan, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
               const int32_t* lengths_dev, int64_t row_stride, int B, void* out_dev,
               float* gmax_dev, void* workspace, size_t workspace_bytes, void* stream);

/*
 * return_attention_mask=True of TF-FE:328-337: int32 [B][3000], 1 where frame t starts inside
 * the valid samples (160*t < min(len,480000)).  lengths_dev as above (must not be NULL).
 */
int wlm_frame_mask(wlm_plan* plan, const int32_t* lengths_dev, int B, int32_t* mask_dev,
                   void* stream);

/*
 * Long-form features (`truncation=False, padding="longest"` of TF-FE:189-342): every clip is
 * zero-padded to ONE common length padded_len = L of any value (the longest clip of the batch,
 * possibly rounded up by pad_to_multiple_of), reflected by 200 samples at sample 0 and at L
 * (torch.stft center=True), and the last STFT frame is dropped: T = L / 160 frames.  The max - 8
 * clamp uses each clip's maximum over all its T frames.
 *
 *   pcm_dev ... stream  as wlm_logmel; clip b contributes min(lengths_dev[b], padded_len) samples
 *                       (dense layout without lengths: min(row_stride, padded_len)).
 *   padded_len          L, in [201, INT32_MAX]; otherwise WLM_ERR_BAD_ARG.
 *   out_dev             device [B][n_mels][L / 160] of the plan's output format, 16-byte aligned (rows
 *                       are L / 160 elements, so they need not be aligned).
 *   workspace           device scratch of at least wlm_padded_workspace_bytes(plan, B) bytes, 16-byte
 *                       aligned; always required (it holds the per-clip maxima and a work counter).
 * At padded_len = 480000 the features and gmax equal those of wlm_logmel bit for bit.
 */
size_t wlm_padded_workspace_bytes(const wlm_plan* plan, int B);
int wlm_logmel_padded(wlm_plan* plan, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                      const int32_t* lengths_dev, int64_t row_stride, int64_t padded_len, int B, void* out_dev,
                      float* gmax_dev, void* workspace, size_t workspace_bytes, void* stream);

/*
 * The two waveform steps HF runs between padding and the STFT, for the long-form geometry and (with
 * padded_len = 480000) the 30-s one: `do_normalize=True` of TF-FE:189-342 (zero_mean_unit_var_norm
 * with the pad's mask) and the constructor's `dither` (TF-FE:141-161 adds dither * randn to the
 * whole padded waveform before torch.stft reflects it).  For clip b with n_b = min(len_b, L) valid
 * samples, in this order:
 *   1. do_normalize != 0: y = (x - mean) / sqrt(var + 1e-7) on [0, n_b), mean and population
 *      variance of x[:n_b] (x = pcm, or int16 / 32768); an empty clip stays zero;
 *   2. y = 0 on [n_b, L);
 *   3. y[n] += dither * z(seed, b, n) on [0, L), the pad region included;
 *   4. reflection at 0 and at L of the conditioned y, then the STFT etc. as wlm_logmel_padded.
 * The noise z is not torch.randn's; it is this stream, independent of B, the layout, the formats
 * and the work split (b is the clip's index in the call):
 *   Philox4x32-10 (Random123) with key (lo32(seed), hi32(seed)) and counter (n >> 2, b, 0, 0)
 *   gives words r0..r3; u_i = ((r_i >> 8) + 0.5) * 2^-24;
 *   (z0, z1) = sqrt(-2 ln u0) * (cos 2 pi u1, sin 2 pi u1), (z2, z3) likewise from (u2, u3);
 *   sample n takes z_{n & 3}.
 * The per-clip moments are reduced in a fixed order: repeated calls give bit-identical results.
 *
 *   arguments and errors as wlm_logmel_padded; in addition a non-finite dither is WLM_ERR_BAD_ARG.
 *   workspace     at least wlm_conditioned_workspace_bytes(plan, B, padded_len) bytes, 16-byte aligned
 *                 (0 when padded_len is out of range).
 * With do_normalize = 0 and dither = 0 the results equal wlm_logmel_padded's bit for bit.
 */
size_t wlm_conditioned_workspace_bytes(const wlm_plan* plan, int B, int64_t padded_len);
int wlm_logmel_conditioned(wlm_plan* plan, const void* pcm_dev, int pcm_format, const int64_t* offsets_dev,
                           const int32_t* lengths_dev, int64_t row_stride, int64_t padded_len, int B,
                           int do_normalize, float dither, uint64_t seed,
                           void* out_dev, float* gmax_dev, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Attention mask of the long-form call: int32 [B][padded_len / 160], 1 where 160*t < min(len, padded_len)
 * (TF-FE:328-337, including the trim of the last column when padded_len % 160 != 0).
 */
int wlm_frame_mask_padded(wlm_plan* plan, const int32_t* lengths_dev, int B, int64_t padded_len,
                          int32_t* mask_dev, void* stream);

/*
 * End-to-end convenience with HOST buffers (what the reference-facing Python shim calls for
 * numpy inputs): stages the ragged host clips through the plan's pinned ring, copies H2D in
 * chunks on an internal copy stream overlapped with the kernels, and leaves the features on
 * the device in `out_dev` (they feed the model there).  Synchronous with respect to the host
 * buffers: they may be reused as soon as the call returns.  The features are complete when
 * `stream` reaches the point of return (the call records its internal dependencies on it).
 *
 *   clips_host    array of B host pointers (element type pcm_format), lengths_host[b] valid
 *                 samples each (any value >= 0; >480000 is truncated).
 *   out_host      optional host [B][n_mels][3000] (same element type as out_dev): if not NULL the features are also
 *                 copied back (D2H inside the call, which then blocks until they arrived).
 */
int wlm_logmel_host(wlm_plan* plan, const void* const* clips_host, const int32_t* lengths_host,
                    int pcm_format, int B, void* out_dev, void* out_host, void* stream);

/* Number of kernels the plan has launched so far (bench.py's gpu_launches evidence). */
int64_t wlm_plan_launch_count(const wlm_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* WLM_H_ */
