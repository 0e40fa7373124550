/*
 * logmel_b200.h -- C ABI of the B200-native (sm_100a) log-mel front end for the ICBHI
 * lung-sound classifier.
 *
 * The reference (AkZuza/audio-classification-icbhi) has no FFI layer: its boundary for this
 * path is a Python class contract.  Each entry point below states the reference interface it
 * replaces (R/ = the reference tree, TA/ = site-packages/torchaudio):
 *
 *   lm_plan_create   <- AudioPreprocessor.__init__            R/src/data/preprocessing.py:20-53
 *                       FlexibleAudioPreprocessor.__init__    R/data/preprocessing_flexible.py:14-54
 *                       (T.MelSpectrogram buffers `window`, `fb`: TA/transforms/_transforms.py:86-87,
 *                        :402-405; T.AmplitudeToDB constants: TA/transforms/_transforms.py:324-333)
 *   lm_forward       <- AudioPreprocessor.preprocess minus load_audio, batched:
 *                       pad_or_crop  R/src/data/preprocessing.py:70-83
 *                       add_noise / time_shift / augment_waveform   :85-103
 *                       mel_spectrogram -> amplitude_to_db          :139-142
 *                         (TA/functional/functional.py:106-145, TA/transforms/_transforms.py:407-419,
 *                          TA/functional/functional.py:390-391)
 *                       augment_spectrogram  :105-109  (TA/functional/functional.py:885-958)
 *                       normalize            :111-116
 *                       and, with window offsets into one recording, the preprocessing half of
 *                       process_segments_batch  R/realtime_analyzer_parallel.py:171-191
 *   lm_forward_host  <- the same call made the way the reference makes it: host buffers in,
 *                       host features out (Dataset.__getitem__ R/src/data/dataset.py:135-147
 *                       returns CPU tensors); host<->device copies are inside the call.
 *
 * Conventions
 *   - every function returns LM_OK (0) or a negative lm_status; nothing throws across the ABI.
 *   - lm_forward allocates nothing, enqueues on the caller's stream and does not synchronise.
 *   - a plan's tables are immutable after creation: concurrent lm_forward calls from any threads on any
 *     streams are safe.  Each launch takes the next of 1024 plan-owned scheduling slots (a work counter
 *     and the small-batch scratch); the kernel leaves its slot zeroed, so a launch needs no memset and
 *     launches on one stream can never collide.  Only more than 1024 launches of ONE plan in flight at
 *     the same time on different streams could share a slot.  A launch captured in a CUDA graph keeps
 *     its slot: do not replay one captured launch concurrently with itself.
 *   - lm_forward_host / lm_forward_host_pcm16 use plan-owned staging buffers and streams; concurrent
 *     callers on one plan are serialised inside the library (a mutex), so they are safe, not parallel:
 *     use one plan per thread to overlap host pipelines.
 *   - there is no CPU fallback anywhere: without a CUDA device lm_plan_create fails.
 */
#ifndef LOGMEL_B200_H
#define LOGMEL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LM_ABI_VERSION 1
#define LM_MAX_RESAMPLERS 8   /* rate pairs of one lm_forward_resampled call */

typedef enum lm_status {
    LM_OK = 0,
    LM_ERR_INVALID_ARG = -1,   /* NULL pointer, negative size, ...                         */
    LM_ERR_UNSUPPORTED = -2,   /* n_fft not in {256, 512, 1024, 2048}, odd hop, ...        */
    LM_ERR_FILTERBANK = -3,    /* fb support too wide for the on-chip table                */
    LM_ERR_CUDA = -4,          /* a CUDA runtime call failed (see lm_last_cuda_error)      */
    LM_ERR_NO_DEVICE = -5,     /* no CUDA device / wrong architecture                      */
    LM_ERR_TOO_SHORT = -6      /* target_len <= n_fft/2: reflect padding undefined         */
} lm_status;

/* Constants of one preprocessor.  `window` and `fb` are HOST pointers, read during
 * lm_plan_create only: build them with the same torch calls torchaudio uses so the bits match
 * (torch.hann_window(n_fft); torchaudio.functional.melscale_fbanks(n_fft/2+1, 0, sr/2, n_mels,
 * sr, None, "htk")). */
typedef struct lm_config {
    int32_t n_fft;        /* 2048, 1024, 512 or 256                                    */
    int32_t hop;          /* even, 1 <= hop <= n_fft/4                                 */
    int32_t n_mels;       /* 1..256                                                    */
    int32_t target_len;   /* int(sample_rate * duration): every clip is padded/cropped */
    const float* window;  /* [n_fft]                                                   */
    const float* fb;      /* [(n_fft/2+1) x n_mels] row-major                          */
    float db_multiplier;  /* 10 for power spectrograms (T.AmplitudeToDB stype="power") */
    float amin;           /* 1e-10                                                     */
    float db_offset;      /* multiplier * log10(max(amin, ref)) = 0 for ref = 1        */
    float norm_eps;       /* 1e-8: out = (x - mean) / (std + eps)                      */
} lm_config;

/* One per clip; a NULL array means "no augmentation".  40 bytes, no implicit padding. */
typedef struct lm_aug {
    int32_t shift;        /* torch.roll amount (out[i] = in[(i - shift) mod T]); 0 = none   */
    float noise_scale;    /* 0 = none; 0.005 in the reference                                */
    float gain;           /* 1 = none (not in the reference; multiplies the padded clip)     */
    int32_t f0, f1;       /* frequency mask rows [f0, f1); empty if f1 <= f0                 */
    int32_t t0, t1;       /* time mask frames [t0, t1)                                       */
    int32_t flags;        /* reserved, 0                                                     */
    uint64_t seed;        /* Philox key for on-device N(0,1) noise when `noise` is NULL      */
} lm_aug;

typedef struct lm_plan lm_plan;

typedef struct lm_info {
    int32_t abi_version;
    int32_t frames;            /* 1 + target_len / hop                                    */
    int32_t n_freqs;           /* n_fft/2 + 1                                             */
    int32_t sm_count;          /* CTAs of the persistent grid at full batch               */
    int32_t threads_per_cta;
    int32_t smem_bytes;        /* dynamic shared memory per CTA                           */
    int32_t fb_nnz;            /* non-zeros kept from fb                                  */
    int32_t tma_staging;       /* 1 if interior tiles are staged with cp.async.bulk       */
    int64_t bytes_per_clip;    /* algorithmic bytes: 4*target_len + 4*n_mels*frames        */
} lm_info;

int lm_abi_version(void);
const char* lm_strerror(int status);
/* Text of the last CUDA error seen by this thread inside the library ("" if none). */
const char* lm_last_cuda_error(void);

int lm_plan_create(const lm_config* cfg, int device, lm_plan** plan);
int lm_plan_destroy(lm_plan* plan);
int lm_plan_frames(const lm_plan* plan);
int lm_plan_info(const lm_plan* plan, lm_info* info);
/* Tuning knobs for experiments: key "tma" (0/1), "max_ctas" (0 = SM count), "split" (small-batch mode:
 * 0 = automatic, 1 = off, k = at most k tile ranges per clip), "host_chunk_clips", "stagger_ns". */
int lm_plan_set(lm_plan* plan, const char* key, int value);
/* Number of kernels this plan has launched since creation (lm_forward, lm_forward_resampled: 1 per call,
 * lm_forward_host / lm_forward_host_pcm16: 1 per chunk). */
int64_t lm_plan_launch_count(const lm_plan* plan);

/*
 * Device-resident forward.  All pointers are DEVICE pointers on the plan's device.
 *   wave      packed fp32 samples; clip i = wave[offset[i] .. offset[i] + length[i])
 *   offset    [B] int64, length [B] int32 (0 allowed: an all-zero clip)
 *   aug       [B] lm_aug or NULL
 *   noise     [B x target_len] fp32 N(0,1) draws (host-replayed torch.randn) or NULL
 *   out_norm  [B, 1, n_mels, frames] fp32; normalised features (dB if normalize == 0)
 *   out_db    optional, same shape: dB after masks, before normalisation
 *   out_melpow optional, same shape: mel power before the log
 */
int lm_forward(lm_plan* plan, const float* wave, const int64_t* offset, const int32_t* length,
               int32_t B, const lm_aug* aug, const float* noise, float* out_norm, float* out_db,
               float* out_melpow, int32_t normalize, void* cuda_stream);

/*
 * lm_forward on 16-bit PCM, the sample format of the ICBHI wav files (R/src/data/preprocessing.py:55-68:
 * torchaudio.load decodes them to x / 32768 before anything else happens).  `pcm` is a DEVICE pointer to packed
 * int16 samples; offset / length count samples.  The kernel stages the raw samples (2 bytes each across HBM) and
 * expands them in shared memory: results are bit-identical to lm_pcm16_decode followed by lm_forward, without the
 * decode kernel and the fp32 copy of the waveforms.  Clips whose first staged sample is 16-byte aligned
 * (offset + centre-crop start a multiple of 8 samples) take the bulk-copy path, others the gather path.
 */
int lm_forward_pcm16(lm_plan* plan, const int16_t* pcm, const int64_t* offset, const int32_t* length,
                     int32_t B, const lm_aug* aug, const float* noise, float* out_norm, int32_t normalize,
                     void* cuda_stream);

/*
 * lm_forward fused with the feature all-gather of the multi-GPU layout (SURVEY.md section 8e; the reference
 * has no multi-GPU path -- its consumer, R/src/training/trainer_fixed.py, is single-device).  Every rank owns
 * the same slice [rank*B, rank*B + B) of a gathered buffer [world*B, 1, n_mels, frames] that exists on every
 * GPU.  The kernel writes this rank's normalised features to
 *   out_slice              its slice of its OWN gathered buffer, and
 *   peer_slices[r], r < n_peers (<= 7)   the same slice of the OTHER ranks' buffers, mapped into this process
 *                          (CUDA IPC / symmetric memory) and reached over NVLink by plain 16-byte stores, or
 *   mc_slice (optional)    the slice's multicast address: ONE multimem.st per 16 bytes, replicated by the
 *                          NVSwitch into every rank's buffer (then peer_slices is ignored and may be NULL).
 * The stores ride on the clip-end normalisation pass, so the transfer overlaps the remaining clips' compute.
 * The caller synchronises the ranks (a barrier after the stream has drained) before reading foreign slices.
 * Needs n_mels*frames % 4 == 0 and 16-byte aligned slices.
 */
int lm_forward_gather(lm_plan* plan, const float* wave, const int64_t* offset, const int32_t* length,
                      int32_t B, const lm_aug* aug, const float* noise, float* out_slice,
                      float* const* peer_slices, int32_t n_peers, float* mc_slice, void* cuda_stream);

/*
 * Host-buffer forward: the call a reference user makes.  All pointers are HOST pointers
 * (pinned memory makes the copies asynchronous).  Clips are cut into chunks; the H2D copy of
 * chunk k+1, the kernel of chunk k and the D2H copy of chunk k-1 overlap on plan-owned
 * streams.  Returns after the last byte of `out` has landed.
 *   total_samples  number of floats in `wave` (offset[i] + length[i] <= total_samples)
 */
int lm_forward_host(lm_plan* plan, const float* wave, int64_t total_samples, const int64_t* offset,
                    const int32_t* length, int32_t B, const lm_aug* aug, const float* noise,
                    float* out, int32_t normalize);

/*
 * Polyphase sinc resampler on the device = torchaudio.transforms.Resample(orig_freq, new_freq) with its
 * defaults (sinc_interp_hann, lowpass_filter_width 6, rolloff 0.99), the resampler of
 * AudioPreprocessor.load_audio (R/src/data/preprocessing.py:63-65): ICBHI ships 4, 10 and 44.1 kHz
 * recordings.  Mono; `in` / `out` are device pointers; out holds lm_resampler_out_len(r, in_len) =
 * ceil(new_freq * in_len / orig_freq) samples.  Float arithmetic: agrees with torchaudio to ~1e-6 of
 * full scale (torchaudio sums the same products as a dense conv1d, in another order).  Each output is one fmaf
 * chain over its phase's taps, zero-padded to a multiple of four, whichever kernel runs (shared-memory tiles, or one
 * output per thread for rate pairs whose tile span is over 96 KB): the bits do not depend on the kernel, non-finite
 * input included (a zero padding tap over inf or NaN gives NaN).
 */
typedef struct lm_resampler lm_resampler;
int lm_resampler_create(int32_t orig_freq, int32_t new_freq, int device, lm_resampler** r);
int lm_resampler_destroy(lm_resampler* r);
int64_t lm_resampler_out_len(const lm_resampler* r, int64_t in_len);
int lm_resample(const lm_resampler* r, const float* in, int64_t in_len, float* out, void* cuda_stream);
/* n_rows waveforms of equal length (channels of a file, clips of a batch) in one launch; row i starts at
 * in + i * in_stride and goes to out + i * out_stride (strides in floats). */
int lm_resample_rows(const lm_resampler* r, const float* in, int64_t in_len, int64_t in_stride, int32_t n_rows,
                     float* out, int64_t out_stride, void* cuda_stream);

/*
 * lm_forward for clips recorded at other sample rates (ICBHI: 4, 10 and 44.1 kHz), resampled to the plan's rate
 * inside the log-mel kernel's staging: one launch for a batch that mixes rates, no resampled copy in memory.
 *   resamplers  HOST array of n_resamplers (0..LM_MAX_RESAMPLERS) handles from lm_resampler_create(clip_rate,
 *               plan_rate, plan_device), on the plan's device.  The caller guarantees that each one's new rate is
 *               the rate the plan's filterbank was built for: lm_config carries no rate, so the library cannot check.
 *               They must outlive the launch in stream order.
 *   wave        DEVICE pointer to packed samples: fp32 when pcm16 == 0, 16-bit PCM (x / 32768) when pcm16 == 1
 *   offset, length  [B] int64 / int32, in samples at the clip's OWN rate
 *   source      [B] int32 DEVICE array: index into `resamplers` of the clip's rate pair, -1 for a clip already at the
 *               plan's rate.  An index outside [-1, n_resamplers) makes the clip a zero-length clip (nothing is read).
 *   aug, noise, out_norm, normalize  as lm_forward (noise rows hold target_len draws at the plan's rate); there are no
 *               extra outputs.  normalize == 0 leaves dB (the input of lm_resize_finish).
 * Output is bit-identical to: y_i = lm_resample(resamplers[source[i]], clip i) (ceil(q len / o) samples), the y_i
 * packed, then lm_forward (fp32) with the same aug, noise and normalize -- pad or centre crop, roll, gain and noise
 * act on y_i -- for every rate pair and any samples, non-finite ones included: the staging runs lm_resample's chain.
 * A clip with source -1 gives exactly what lm_forward (fp32) or lm_forward_pcm16 (pcm16) gives.
 * Returns LM_ERR_INVALID_ARG for NULL pointers or handles, a bad n_resamplers or pcm16, or a resampler on
 * another device.
 */
int lm_forward_resampled(lm_plan* plan, const lm_resampler* const* resamplers, int32_t n_resamplers,
                         const void* wave, int32_t pcm16, const int64_t* offset, const int32_t* length,
                         const int32_t* source, int32_t B, const lm_aug* aug, const float* noise,
                         float* out_norm, int32_t normalize, void* cuda_stream);

/*
 * Training batches need not carry whole recordings: which native samples a clip's features read is fixed by its length,
 * its rate pair and target_len (roll, noise, gain, reflect padding and masks all act inside the crop).  A data-loading
 * worker asks lm_clip_span for that span, reads only those samples from the file and ships them; lm_forward_spans
 * turns a batch of such spans into the features lm_forward_resampled gives for the whole clips.
 *
 * lm_clip_span: the native-sample span [*first, *first + *count) that the features of a clip of `length` samples at
 * orig_freq read when the plan runs at new_freq with target_len (orig == new: the pad / centre-crop span).  Every index
 * the resampler's fmaf chain touches inside [0, length) counts, zero padding taps included, so the span covers
 * non-finite samples exactly as the full clip would.  A clip of length 0 gives (0, 0).  Pure host arithmetic: no
 * device, no CUDA call, safe in forked workers.  LM_ERR_INVALID_ARG for rates or target_len < 1, length < 0 or NULL
 * outputs.
 */
int lm_clip_span(int32_t orig_freq, int32_t new_freq, int32_t target_len, int64_t length, int64_t* first,
                 int64_t* count);

/*
 * lm_forward_resampled on clips of which only a span is stored: clip i has length[i] native samples, and samples
 * [first[i], first[i] + stored[i]) sit at wave[offset[i] ...].  first (int64) / stored (int32) are [B] DEVICE arrays.
 * When the stored span contains lm_clip_span's span, the output is bit-identical to lm_forward_resampled on the full
 * clips.  A clip whose stored span does not contain it becomes a zero-length clip: nothing outside the stored span is
 * ever read.  Argument checks and status codes are those of lm_forward_resampled, with first and stored checked
 * for NULL with the other arrays.
 */
int lm_forward_spans(lm_plan* plan, const lm_resampler* const* resamplers, int32_t n_resamplers,
                     const void* wave, int32_t pcm16, const int64_t* offset, const int64_t* first,
                     const int32_t* stored, const int32_t* length, const int32_t* source, int32_t B,
                     const lm_aug* aug, const float* noise, float* out_norm, int32_t normalize,
                     void* cuda_stream);

/*
 * T.AmplitudeToDB() as a stand-alone transform (R/src/data/preprocessing.py:46; torchaudio/functional/functional.py:390-391,
 * stype "power", top_db None): out = multiplier * log10(max(in, amin)) - db_offset, element-wise.  Device pointers, in == out
 * allowed.  Serves the `amplitude_to_db` attribute of the drop-in AudioPreprocessor.
 */
int lm_amplitude_to_db(const float* in, float* out, int64_t n, float multiplier, float amin, float db_offset, void* cuda_stream);

/*
 * 16-bit PCM -> fp32 in [-1, 1): x / 32768, what torchaudio.load(normalize=True) hands the reference for a
 * PCM_16 wav (R/src/data/preprocessing.py:57).  Device pointers, both 16-byte aligned.
 */
int lm_pcm16_decode(const int16_t* in, float* out, int64_t n, void* cuda_stream);

/*
 * lm_forward_host for clips that are still 16-bit PCM (the sample format of the ICBHI wav files and of
 * every temp wav the analyzers write): the int16 samples cross PCIe -- half the bytes of the fp32 call --
 * and are expanded inside the log-mel kernel's staging (lm_forward_pcm16): one kernel per chunk.  offset/length
 * count samples.  Features are bit-identical to lm_forward_host on pcm[i] / 32768.
 */
int lm_forward_host_pcm16(lm_plan* plan, const int16_t* pcm, int64_t total_samples, const int64_t* offset,
                          const int32_t* length, int32_t B, const lm_aug* aug, const float* noise, float* out,
                          int32_t normalize);

/*
 * FlexibleAudioPreprocessor's tail for durations whose frame count differs from ceil(T/hop)
 * (R/data/preprocessing_flexible.py:118-154 resize_spectrogram, then :106-110 masks, :112-116
 * normalize; order of :182-190).  in: dB [B,1,n_mels,frames_in] from lm_forward(normalize=0, no
 * masks); out: [B,1,n_mels,frames_out].  Device pointers; in != out; aug may be NULL (only
 * f0,f1,t0,t1 are read, t in output frames).
 */
int lm_resize_finish(const float* in, int32_t B, int32_t n_mels, int32_t frames_in, int32_t frames_out,
                     const lm_aug* aug, float* out, int32_t normalize, float norm_eps, void* cuda_stream);

/*
 * y = rint(clamp(x,-1,1) * 32767) / 32768: the PCM_16 temp-wav round trip the analyzers put every
 * window through (R/realtime_analyzer_parallel.py:181-184; soundfile + torchaudio.load, neither in
 * the reference tree: parity unpinned).  Device pointers; in-place allowed.
 */
int lm_pcm16_roundtrip(const float* in, float* out, int64_t n, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* LOGMEL_B200_H */
