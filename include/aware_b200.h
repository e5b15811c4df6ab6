/* aware_b200 -- C ABI of the B200-native AWARE hot path.
 *
 * The reference (deepmarkpy/aware) is pure Python; it has no FFI of its own.  Each
 * entry point below replaces the body of one reference function (cited as
 * file:line relative to the reference tree) for a whole BATCH of clips.  The
 * Python mirror of the reference API (aware_b200/service, aware_b200/utils/models,
 * aware_b200/metrics, aware_b200/attacks) binds these with ctypes; see
 * INTEGRATION.md for the stub a maintainer would add to the reference itself.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure;
 *     aw_last_error() returns a message for the calling thread.
 *   - all `d_` pointers are DEVICE pointers owned by the caller; audio is float32,
 *     one clip per row, `stride` elements between consecutive clips.
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); nothing
 *     synchronises unless stated.  A context is bound to one device and must be
 *     used by one host thread at a time.
 *   - there is no CPU fallback: without a CUDA device aw_ctx_create fails.
 */
#ifndef AWARE_B200_H
#define AWARE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct aw_ctx aw_ctx;

/* GEMM arithmetic for the detector's 1x1-conv stack. */
enum {
  AW_PREC_TF32 = 0, /* tcgen05 tensor cores, TF32 operands, fp32 accumulate (default) */
  AW_PREC_FP32 = 1, /* CUDA-core GEMMs with float64 accumulation (validation yardstick)       */
  AW_PREC_BF16 = 2, /* tcgen05, bf16 operands AND bf16 activation storage (embed loop speed) */
  AW_PREC_FP16 = 3  /* tcgen05 kind::f16 with fp16 operands and fp16 activation storage: the same
                       10-bit mantissa as TF32 at half the bytes; back-propagated gradients carry
                       a power-of-two loss scale proportional to the clip length */
};

/* Model description handed over once (reference: utils/models/load_model.py:6-76,
 * cards/config.yaml, detection/multibit_detector_net.py:58-80).  Host pointers. */
typedef struct aw_model {
  const float* w[4];      /* conv weights, (C_out, C_in) row-major: 512x128, 1024x512,
                             1024x1024, 40x1024 (multibit_detector_net.py:58-70)      */
  const float* mel_basis; /* 128 x 513 (detection/modules/mel.py:105-149)             */
  const float* window;    /* 1024, torch.hann_window (utils/audio/stft.py:17)         */
  float band_lo_hz, band_hi_hz; /* config.yaml:13 embedding_bands                     */
  float tolerance_db;     /* config.yaml:14                                           */
  float threshold;        /* config.yaml:46                                           */
} aw_model;

const char* aw_last_error(void);
const char* aw_version(void);

int aw_ctx_create(aw_ctx** out, int device, const aw_model* model);
int aw_ctx_destroy(aw_ctx* ctx);
int aw_ctx_set_precision(aw_ctx* ctx, int prec);
/* band bins for a sample rate (embedding/multibit_embedder.py:43-47) */
int aw_band_bins(aw_ctx* ctx, int sample_rate, int* bin0, int* nbins);
/* number of CUDA kernels launched by this context since creation */
int64_t aw_launch_count(aw_ctx* ctx);

/* Run-time knobs.  AW_OPT_THRESHOLD: decision threshold of aw_decide_and_count and of the
 * low-margin test (detector.threshold, service/detect.py:17; default = aw_model.threshold).
 * AW_OPT_EXACT_MARGIN: aw_detect_batch re-evaluates every clip with min_i |v_i - threshold| below
 * this margin through the exact fp32 GEMM path, so decoded bits equal the reference's fp32
 * arithmetic (default 1e-3; 0 switches the re-evaluation and its stream synchronisation off).
 * AW_OPT_TC_SPECTRAL (default 1): with fp16 loop GEMMs and a band of <= 96 bins (44.1 / 48 kHz) the
 * embed loop's band-limited STFT / iSTFT run as tcgen05 GEMMs over Toeplitz views of the frame rows
 * (csrc/spectc.cuh); 0 keeps the fp32 FFT kernels.  AW_OPT_TWO_PASS (default 1): the K <= 128 layers run
 * as a statistics pass + an apply pass instead of materialising their raw output.  AW_OPT_PAIR_GEMM
 * (default 1): the K >= 512 layers run on CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles, each CTA
 * staging half of the weight tile) when the batch has an even number of 128-row tiles; results are
 * bit-identical to the one-CTA kernel.  AW_OPT_BWD64_STREAM (default 1): in the 16-bit loops the backward
 * K = 64 layer runs on k_gemm_bwd64 (csrc/gemm64.cuh: activation tiles streamed through a TMA ring, output
 * through a TMA bulk store) instead of the generic GEMM's statistics / apply epilogues. */
enum { AW_OPT_THRESHOLD = 0, AW_OPT_EXACT_MARGIN = 1, AW_OPT_TC_SPECTRAL = 2, AW_OPT_TWO_PASS = 3,
       AW_OPT_PAIR_GEMM = 4, AW_OPT_BWD64_STREAM = 5 };
int aw_ctx_set_option(aw_ctx* ctx, int option, double value);
/* counters since context creation: clips seen by aw_detect_batch / clips it re-evaluated exactly */
enum { AW_STAT_DETECT_CLIPS = 0, AW_STAT_REEVAL_CLIPS = 1 };
int aw_ctx_get_stat(aw_ctx* ctx, int which, int64_t* out);
/* CUDA-event timing of the tensor-core GEMM launches, on the launching stream (bench.py's
 * roofline).  aw_profile_read sums the launches recorded since the last read by
 * (n, k, epilogue kind) and clears the record. */
int aw_profile_enable(aw_ctx* ctx, int on);
int aw_profile_read(aw_ctx* ctx, int max_classes, int* n_classes, int* cls_n, int* cls_k,
                    int* cls_epi, int64_t* cls_count, double* cls_ms);
/* Device time of every kernel launched since the last read, summed per kernel class
 * (events on the launching stream around each launch).  names: max_classes x 32 chars. */
int aw_profile_read_named(aw_ctx* ctx, int max_classes, int* n_classes, char* names,
                          int64_t* cls_count, double* cls_ms);

/* ---- detection: AWAREDetector.detect (detection/multibit_detector.py:28-42) for a batch.
 * d_values: [n_clips][20] float32 tanh outputs.  Tensor-core pass first; clips whose decision
 * margin is below AW_OPT_EXACT_MARGIN are evaluated again in exact fp32 (one 4-byte D2H copy and
 * a stream synchronisation per call; none with the margin at 0 or in AW_PREC_FP32 mode). */
int aw_detect_batch(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples,
                    int64_t stride, int sample_rate, float* d_values, void* stream);

/* ---- embedding: AWAREEmbedder.embed (embedding/multibit_embedder.py:141-197) for a batch.
 * d_pattern : [n_clips][20] int32 in {-1,+1} (utils/watermark/encoder.py:35-45)
 * d_scale   : optional [n_clips] float32; output is multiplied by it -- may be NULL
 * scale_mode: AW_SCALE_SIGNED_MAX multiplies every output clip by the SIGNED max of its input,
 *             computed on the device in the same pass as the peak (service/embed.py:69,73:
 *             `audio_mx = np.max(audio)`); exclusive with d_scale
 * d_out     : [n_clips][out_stride], each clip gets 256*(n_samples/256) samples
 * d_best_loss: optional [n_clips]; d_losses: optional [iters][n_clips]
 * wave_clips: clips processed together per optimisation wave (0 = all). */
enum { AW_SCALE_NONE = 0, AW_SCALE_SIGNED_MAX = 1 };
int aw_embed_batch(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples, int64_t stride,
                   int sample_rate, const int32_t* d_pattern, int iters, const float* d_scale,
                   int scale_mode, float* d_out, int64_t out_stride, float* d_best_loss,
                   float* d_losses, int wave_clips, void* stream);
/* per-clip status of the last aw_embed_batch call, int32 [n_clips]: 1 = the clip met a non-finite
 * gradient inside the loop (only possible with 16-bit loop GEMMs; that NAdam update was skipped) */
int aw_embed_status(aw_ctx* ctx, int32_t* d_flags, int n_clips, void* stream);
/* ---- frame-sharded long-form mode (BASELINE configs[4]: one long clip over the GPUs of a box).
 * The reference processes a clip whole and every statistic is whole-clip (utils/audio/waveform.py:19,
 * detection/modules/globalStandardize.py:17-19, multibit_detector_net.py:50,126, modules/BRH.py:18).
 * Here each rank passes a SEGMENT of the clip: its own frames [own_lo, own_hi) (local indices) plus
 * 8 halo frames per inner side; per-clip sums / maxima are reduced over the ranks and halo frames are
 * refreshed through the caller's two collectives, both operating on a caller-owned device arena:
 *   allreduce(user, offset, count, dtype, op, stream)  in place, `count` 8-byte elements at arena+offset
 *   allgather(user, send_offset, recv_offset, bytes, stream)  rank-major result at arena+recv_offset
 * (host callbacks: they ENQUEUE the collective behind the work already on `stream`; 0 = success).
 * Geometry (T = 1 + N/256 frames of the whole clip): a rank owns global frames [f0, f1), f0 even, f1
 * even except on the last rank (f1 = T); segment frames [e0, e1) = [max(0, f0-8), min(T, f1+8));
 * segment samples = global samples [256 e0, ...): 256 (e1-e0-1) + 1 of them, or all remaining ones on
 * the last rank.  Results equal the single-GPU run up to float64 summation order. */
enum { AW_COMM_F64 = 0, AW_COMM_I64 = 1 };
enum { AW_COMM_SUM = 0, AW_COMM_MAX = 1 };
typedef struct aw_comm {
  void* user;
  int (*allreduce)(void* user, int64_t offset, int64_t count, int dtype, int op, void* stream);
  int (*allgather)(void* user, int64_t send_offset, int64_t recv_offset, int64_t bytes, void* stream);
  void* d_arena;         /* device scratch, >= 64 KiB + world * 32 KiB */
  int64_t arena_bytes;
  int rank, world;
} aw_comm;
/* d_values [20]: identical on every rank */
int aw_detect_sharded(aw_ctx* ctx, const float* d_segment, int seg_samples, int seg_first_frame,
                      int own_lo, int own_hi, int total_frames, int sample_rate, const aw_comm* comm,
                      float* d_values, void* stream);
/* d_out_own: this rank's samples of the watermarked clip, global [256 f0, min(256 f1, 256 (T-1))).
 * d_losses: optional [iters] (identical on every rank); comm_counts: optional int64[2] = number of
 * all-reduces / all-gathers issued. */
int aw_embed_sharded(aw_ctx* ctx, const float* d_segment, int seg_samples, int seg_first_frame,
                     int own_lo, int own_hi, int total_frames, int sample_rate,
                     const int32_t* d_pattern, int iters, const aw_comm* comm, float* d_out_own,
                     int64_t out_capacity, float* d_best_loss, float* d_losses, int64_t* comm_counts,
                     void* stream);

/* debug/parity hooks: after aw_embed_batch, copy the optimisation state of the LAST wave.
 * which: 0 coeffs c, 1 best coeffs, 2 initial coeffs c0, 3 last gradient-free state m, 4 v
 * layout [clip][T][nbins] float32. */
int aw_embed_state(aw_ctx* ctx, int which, float* d_dst, int64_t capacity, void* stream);

/* ---- bit decision + BER counters (utils/watermark/decoder.py:51,63; metrics/audio.py:15)
 * d_ref_bits may be NULL (no counting). d_counters: uint64[3] += {errors, bits, clips}. */
int aw_decide_and_count(aw_ctx* ctx, const float* d_values, const int32_t* d_ref_bits,
                        int n_clips, int32_t* d_bits_out, int32_t* d_err_per_clip,
                        uint64_t* d_counters, void* stream);

/* ---- SNR (metrics/audio.py:68-89): d_snr [n_clips] float64 dB, d_snr_sum float64[1] += */
int aw_snr_batch(aw_ctx* ctx, const float* d_out, int64_t out_stride, const float* d_target,
                 int64_t tgt_stride, int n_clips, int n, double* d_snr, double* d_snr_sum,
                 void* stream);

/* ---- STOI (metrics/audio.py:43-64 `STOI.__call__` -> pystoi.stoi(target, output, 16000), extended=False;
 * scripts/test.py:86-88 keeps scores > 0.1).  Both signals already at pystoi's internal 10 kHz (the
 * caller resamples with aw_attack_upfirdn and pystoi's Octave-style window), n samples per clip.
 * d_stoi [n_clips] float64; d_sum (may be NULL) float64[2] += {sum of scores > keep_above, their count}.
 * Clips with fewer than 30 analysis frames after silence removal score 1e-5, as pystoi does. */
int aw_stoi_batch(aw_ctx* ctx, const float* d_clean, int64_t clean_stride, const float* d_proc,
                  int64_t proc_stride, int n_clips, int n, double* d_stoi, double* d_sum,
                  double keep_above, void* stream);

/* ---- stage-level entry points (used by the parity tests and by callers that
 * want the STFT/iSTFT alone; reference utils/audio/stft.py:28,48,55,62) */
int aw_stft_band(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples, int64_t stride,
                 int sample_rate, int normalize, float* d_mag, float* d_phasor, void* stream);
int aw_istft_band(aw_ctx* ctx, const float* d_mag, const float* d_phasor, int n_clips,
                  int n_frames, int sample_rate, float* d_wave, void* stream);

/* ---- full-band STFT / phase vocoder / iSTFT: the stages of the time-stretch and pitch-shift attacks
 * (parity unpinned to upstream's rubberband calls; the classical phase vocoder of
 * librosa.effects.time_stretch, defined in DESIGN.md section 7).  Spectra are complex64, frame-major:
 * float2 [n_clips][n_frames][513].  None of the three synchronises the stream.
 *
 * aw_stft_full: torch.stft(x, 1024, 256, window, center=True, pad_mode="reflect") of every clip, all 513
 * bins, the input as it is (no peak normalisation).  n_samples > 1024; n_frames = 1 + n_samples / 256. */
int aw_stft_full(aw_ctx* ctx, const float* d_audio, int n_clips, int n_samples, int64_t stride,
                 float* d_spec, void* stream);
/* aw_phase_vocoder: librosa.phase_vocoder(D, rate, hop_length=256) in float64, out rounded to complex64.
 * rate finite and in [0.25, 4]; n_frames_out must equal ceil(n_frames / rate) (= len(np.arange(0, n_frames,
 * rate))).  One thread per (clip, bin): results do not depend on the batch. */
int aw_phase_vocoder(aw_ctx* ctx, const float* d_spec, int n_clips, int n_frames, double rate,
                     int n_frames_out, float* d_out, void* stream);
/* aw_istft_full: torch.istft(D, 1024, 256, window, center=True, length=n_out) per clip into rows of
 * out_stride floats.  The imaginary parts of bins 0 and 512 are ignored (as irfft does); samples
 * [256 (n_frames-1), 256 (n_frames-1) + 512) are the tail of the last frame over its window envelope,
 * samples past that are 0.  n_out >= 1. */
int aw_istft_full(aw_ctx* ctx, const float* d_spec, int n_clips, int n_frames, int n_out, float* d_wave,
                  int64_t out_stride, void* stream);
/* D[rows][N] = A[rows][K] * B[N][K]^T ; rows % 128 == 0, K % 32 == 0, N in {64,128,256,512,1024} */
int aw_gemm(aw_ctx* ctx, const float* d_a, const float* d_b, float* d_d, int rows, int n, int k,
            int prec, void* stream);

/* ---- attacks (scripts/attacks.py); every one is batch-wise, out-of-place ---------- */
/* A1 PCMBitDepthConversion.apply (attacks.py:44-70); bits in {8,12,16,24} */
int aw_attack_pcm(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride, int bits,
                  float* d_out, int64_t out_stride, void* stream);
/* A2 Resample.apply, sr // target > 1 branch (attacks.py:276-287) */
int aw_attack_decimate_interp(aw_ctx* ctx, const float* d_in, int n_clips, int n,
                              int64_t in_stride, int factor, float* d_out, int64_t out_stride,
                              void* stream);
/* A2 Resample.apply, polyphase branch: one scipy.signal.upfirdn pass (attacks.py:289-294).
 * d_h_tf: transposed+flipped zero-padded taps [up][taps_per_phase] (host prepares). */
int aw_attack_upfirdn(aw_ctx* ctx, const float* d_in, int n_clips, int n_in, int64_t in_stride,
                      const float* d_h_tf, int taps_per_phase, int up, int down, int first_out,
                      int n_out, float* d_out, int64_t out_stride, void* stream);
/* A3/A4 LowPassFilter / HighPassFilter .apply: scipy.signal.lfilter(b, a, x) in float64
 * (attacks.py:413-416, 451-453).  order <= 8.  warm <= 0: sequential scan, one thread per clip,
 * bit-identical to scipy; warm > 0: chunk-parallel scan with `warm` look-back samples (faster,
 * agrees to the filter's own round-off noise). */
int aw_attack_lfilter(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                      const double* b, const double* a, int order, int warm, float* d_out,
                      int64_t out_stride, void* stream);
/* A5 RandomBandstop.apply: scipy.signal.filtfilt(b, a, x) (attacks.py:348-349), odd padding
 * 3*max(len(a),len(b)), zi = lfilter_zi(b, a) supplied by the host. */
int aw_attack_filtfilt(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                       const double* b, const double* a, const double* zi, int order, int warm,
                       float* d_out, int64_t out_stride, void* stream);
/* A6 DeleteSamples.apply (attacks.py:162-178): d_start [n_clips] int32, host-drawn */
int aw_attack_delete(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                     const int32_t* d_start, int n_delete, float* d_out, int64_t out_stride,
                     void* stream);
/* A7 SampleSupression.apply (attacks.py:370-385) */
int aw_attack_suppress(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                       const int32_t* d_start, int n_zero, float* d_out, int64_t out_stride,
                       void* stream);
/* A8 Cropout.apply (attacks.py:192-205): drop the first n_drop samples */
int aw_attack_cropout(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                      int n_drop, float* d_out, int64_t out_stride, void* stream);
/* extensions without a reference counterpart (parity unpinned): out = gain*x + sigma*noise */
int aw_attack_affine(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                     float gain, const float* d_noise, int64_t noise_stride, float sigma,
                     float* d_out, int64_t out_stride, void* stream);

/* "compression approximation" named by the build brief (parity unpinned: upstream's MP3 attack calls
 * ffmpeg, attacks.py:73-148).  Per frame of a band spectrum [n_clips][n_frames][nbins] (aw_stft_band,
 * normalize = 0): magnitudes below max * 10^(floor_db/20) are zeroed, the rest are rounded to a
 * step_db grid in log-magnitude.  d_dmag receives (quantised - original); the caller resynthesises it
 * with the original phasors (aw_istft_band) and adds it to the input (aw_attack_affine). */
int aw_attack_spectral_quantize(aw_ctx* ctx, const float* d_mag, int n_clips, int n_frames, int nbins,
                                float step_db, float floor_db, float* d_dmag, void* stream);

/* ---- reverberation / echo attacks (no upstream counterpart; DESIGN.md section 7).
 * out = causal convolution of every clip with its filter, truncated to n samples (DESIGN section 7):
 * y[t] = sum_{m < M} h[m] x[t - m], x[< 0] = 0, by uniformly partitioned overlap-save (512-sample
 * partitions, 1024-point transforms).
 * d_spec: complex64 [n_filters][n_parts][513], the rfft of each 512-tap partition zero-padded to 1024
 * (host-computed in float64, rounded to complex64); 1 <= n_parts <= 512.
 * filter_of_clip: HOST int32 [n_clips] in [0, n_filters), or NULL (every clip uses filter 0);
 * validated here and uploaded with cudaMemcpyAsync.  1 <= n <= INT_MAX - 2048, strides >= n, n_clips <= 65535.
 * Does not synchronise the stream; a clip's result does not depend on the rest of the batch. */
int aw_attack_convolve(aw_ctx* ctx, const float* d_in, int n_clips, int n, int64_t in_stride,
                       const float* d_spec, int n_filters, int n_parts, const int32_t* filter_of_clip,
                       float* d_out, int64_t out_stride, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AWARE_B200_H */
