/* b200vf.h - C ABI of libb200vf.so: the B200-native VoiceFixer inference hot path.
 *
 * The reference (haoheliu/voicefixer_main) has no FFI for this path; its boundary is the Python object
 * protocol that eval_gsr_voicefixer.py:handler() consumes (SURVEY.md 8(b)).  Each entry point below
 * replaces one reference interface and is what a ctypes / cgo / JNI binding of that interface would bind:
 *
 *   vf_create / vf_load_weights   Model(hp, ...).load_from_checkpoint(ckpt); model.eval(); model.to(device)
 *                                 eval_gsr_voicefixer.py:31-35,40; config keys config/vctk_base_voicefixer_unet.json:68-78
 *   vf_frontend                   VoiceFixer.pre  models/gsr_voicefixer.py:178-181
 *                                 = FDomainHelper.wav_to_spectrogram_phase tools/pytorch/modules/fDomainHelper.py:67-89
 *                                 + MelScale.forward tools/pytorch/mel_scale.py:52-64
 *   vf_unet_mel                   VoiceFixer.forward models/gsr_voicefixer.py:183-193 -> Generator.forward :86-91
 *                                 -> UNetResComplex_100Mb.forward models/components/unet.py:60-103
 *   vf_vocoder                    model.vocoder(mel) eval_gsr_voicefixer.py:66 (third-party voicefixer.Vocoder)
 *   vf_restore / vf_restore_host  one iteration of the segment loop of handler(), eval_gsr_voicefixer.py:49-74:
 *                                 pre -> model -> from_log -> vocoder -> peak normalise -> trim_center
 *   vf_restore_varlen             the same over a batch of clips of different lengths (each row as if restored alone)
 *   vf_to_log / vf_from_log       tools/pytorch/pytorch_util.py:157-163
 *   vf_to_pcm16                   the int16 conversion of save_wave, tools/file/wav.py:22-24 (SURVEY.md 8(f) row 3)
 *   vf_mel                        MelScale.forward on any spectrogram, tools/pytorch/mel_scale.py:52-64
 *   vf_finalize                   peak normalise + trim_center, eval_gsr_voicefixer.py:68-72, tools/utils.py:57-70
 *   vf_ssr_forward / vf_ssr_restore(_host) / vf_ssr_unet
 *                                 SSR_UNet / GSR_UNet inference (BASELINE config 3): models/ssr_unet.py:140-155 ->
 *                                 Generator.forward :51-54 -> unet_v2 UNetResComplex_100Mb.forward
 *                                 models/components/unet_v2.py:86-148 (magnitude net, input phase, ISTFT)
 *   vf_ssr_restore_varlen         vf_ssr_restore over a batch of clips of different lengths (each row as if restored alone)
 *   vf_istft                      FDomainHelper.istft tools/pytorch/modules/fDomainHelper.py:30-32,127 (torchlibrosa ISTFT)
 *   vf_resample_poly              load_wav's rate conversion, tools/utils.py:46-48
 *   vf_lsd / vf_sispec            AudioMetrics.lsd / .sispec evaluation_proc/metrics.py:83-95 (handler's mel metrics,
 *                                 eval_gsr_voicefixer.py:56-64)
 *
 * Conventions: every function returns 0 on success or a negative VF_E* code and never throws; the message is
 * available from vf_last_error().  All tensor arguments are contiguous fp32.  Unless a name ends in `_host`,
 * pointers are DEVICE pointers owned by the caller (e.g. PyTorch tensors); the library never frees or retains
 * them.  `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream); calls are
 * asynchronous with respect to the host and contain no hidden synchronisation, except where stated.  One
 * context per device; calls on one context must be serialised by the caller.  There is no CPU fallback: without
 * a CUDA device every call fails with VF_ENODEVICE.
 */
#ifndef B200VF_H_
#define B200VF_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define VF_API __attribute__((visibility("default")))
#else
#define VF_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define VF_OK 0
#define VF_EINVAL (-1)     /* bad argument / unsupported shape */
#define VF_ENODEVICE (-2)  /* no usable CUDA device */
#define VF_ECUDA (-3)      /* CUDA runtime / driver error */
#define VF_ESTATE (-4)     /* weights not loaded, missing tensor, ... */
#define VF_EDEVICE (-5)    /* sticky device-side error flag (fp16 range overflow, pipeline time-out) */
#define VF_EASSERT (-6)    /* reference assertion would have fired (to_log on negative input) */

typedef struct vf_ctx vf_ctx;

/* Geometry of the front end (reference config "model"/"data" keys) and of the vocoder restatement. */
typedef struct vf_config {
  int sample_rate;        /* 44100 */
  int n_fft;              /* 2048  (window_size) */
  int hop;                /* 441   (hop_size) */
  int n_mels;             /* 128   (mel_freq_bins) */
  /* vocoder generator (voicefixer_main_b200/arch.py:VocoderConfig) */
  int voc_cond_channels;  /* 512 */
  int voc_cond_layers;    /* 5 */
  int voc_channels;       /* 1024 */
  int voc_num_stages;     /* 4 */
  int voc_scales[8];      /* 7,7,3,3 */
  int voc_depth[8];       /* 8,8,8,8 */
  float voc_stage_slope;  /* 0.2 */
  float voc_res_slope;    /* 0.01 */
  float voc_min_db;       /* -115 */
  float voc_ref_db;       /* 20 */
  float voc_amp_floor;    /* 1e-5 */
  float voc_tail_value;   /* -4 */
  int voc_tail_base;      /* 4 */
  double voc_mel_weight_a;
  double voc_mel_weight_b;
  int voc_tail_tanh;      /* 1 (the generator ends in tanh); 0 leaves the tail linear - test configurations only */
} vf_config;

/* Fills *cfg with the reference defaults listed above. */
VF_API void vf_default_config(vf_config* cfg);

typedef struct vf_tensor_desc {
  const char* name;      /* reference state-dict key, e.g. "generator.analysis_module.encoder_block1.conv_block1.bn1.weight",
                            "mel.fb", or "vocoder.<key>" (arch.py:vocoder_keys) */
  const void* data;      /* fp32, contiguous */
  int ndim;
  int64_t shape[4];
  int on_device;         /* 0: host pointer, 1: device pointer */
} vf_tensor_desc;

VF_API int vf_create(vf_ctx** out, int device, const vf_config* cfg);
VF_API void vf_destroy(vf_ctx* ctx);
VF_API const char* vf_last_error(vf_ctx* ctx);   /* ctx may be NULL: error of the last failed vf_create */

/* Copies and packs the tensors (BN folded to per-channel affine, conv weights to K-major fp16 hi/lo
 * matrices, mel filterbank to its sparse form).  Synchronous.  "mel.fb" is required; of the three networks -
 * "generator.analysis_module.*" (VoiceFixer's mel UNet; unet.py and unet_small.py share its keys), "vocoder.*",
 * "generator.unet.*" (unet_v2 of SSR_UNet / GSR_UNet) - whichever are present are loaded, and a network that is
 * present must be complete (missing key -> VF_ESTATE).  Entry points that need an absent network fail with VF_ESTATE. */
VF_API int vf_load_weights(vf_ctx* ctx, const vf_tensor_desc* descs, int n);

/* wav [B,N] -> mel_out [B,T,128] linear mel (T = 1 + N/hop); optional sp/cos/sin [B,T,1025] (NULL to skip). */
VF_API int vf_frontend(vf_ctx* ctx, const float* wav, int batch, int64_t n_samples, float* mel_out, float* sp_out,
                float* cos_out, float* sin_out, void* stream);

/* mel_lin [B,T,128] (non-negative) -> logmel_out [B,T,128] = unet(log10 mel) + log10 mel.
 * Negative inputs are counted on the device; vf_check_errors() then reports VF_EASSERT (to_log's assert). */
VF_API int vf_unet_mel(vf_ctx* ctx, const float* mel_lin, int batch, int frames, float* logmel_out, void* stream);

/* mel_lin [B,T,128] -> wav_out [B,L], L = vf_vocoder_out_len(ctx, T). */
VF_API int vf_vocoder(vf_ctx* ctx, const float* mel_lin, int batch, int frames, float* wav_out, void* stream);
VF_API int64_t vf_vocoder_out_len(vf_ctx* ctx, int frames);

/* Fused stages A -> B -> C + peak normalise + centre trim: wav [B,N] -> wav_out [B,N] (device pointers). */
VF_API int vf_restore(vf_ctx* ctx, const float* wav, int batch, int64_t n_samples, float* wav_out, void* stream);
/* vf_restore with per-call behaviour flags (re-entrant: nothing is stored in the context). */
#define VF_RESTORE_UNIFY_ENERGY 1u   /* amp_to_original_f (tools/utils.py:50-55) as handler() applies it when
                                        meta["unify_energy"] is set, eval_gsr_voicefixer.py:54-55 */
VF_API int vf_restore_ex(vf_ctx* ctx, const float* wav, int batch, int64_t n_samples, float* wav_out, unsigned flags,
                         void* stream);
/* vf_restore_ex over clips of different lengths.  wav [B, n_max] device; row b holds n_samples[b] valid samples (the rest is
 * never read).  n_samples: HOST array of B lengths, 1024 < n_samples[b] <= n_max; checked before anything is launched
 * (VF_EINVAL), and free for reuse as soon as the call returns.  wav_out [B, n_max] device: row b is bit-identical to
 * vf_restore_ex of that clip alone with the same flags; samples past n_samples[b] are 0.  Plans are cached per (batch,
 * 64-frame bucket of the longest clip), so calls whose longest clip falls in the same 0.64 s bucket share one plan and its
 * CUDA graphs; batches above 128 clips (or above the plan budget) run as sub-batches. */
VF_API int vf_restore_varlen(vf_ctx* ctx, const float* wav, int batch, int64_t n_max, const int64_t* n_samples,
                             float* wav_out, unsigned flags, void* stream);
/* Same through HOST buffers (pinned for true asynchrony).  The copies and the compute run on library-owned streams with
 * two staging buffer pairs, so back-to-back calls overlap (the H2D of call i+1 and the D2H of call i-1 run under the
 * compute of call i); `stream` only receives a wait on this call's D2H.  Contract: wav_host holds its data when the
 * call is made (host-written; it is not ordered after work queued on `stream`), and the caller synchronises `stream`
 * before reading out_host or reusing wav_host.  Option "host_pipeline" = 0 restores the single-stream behaviour. */
VF_API int vf_restore_host(vf_ctx* ctx, const float* wav_host, int batch, int64_t n_samples, float* out_host, void* stream);
/* Copies the intermediate results of the last vf_restore of this (batch, n_samples) into caller buffers
 * [B,T,128] (either may be NULL): the linear mel of stage A and the restored log10 mel of stage B. */
VF_API int vf_restore_stages(vf_ctx* ctx, int batch, int64_t n_samples, float* mel_lin_out, float* log_mel_out,
                             void* stream);

/* ---- SSR_UNet / GSR_UNet (unet_v2) path.  vf_ssr_forward = model(sp, wav)['wav'] of models/ssr_unet.py:145-155:
 * sp [B,T,1025] is the network input (NULL: the STFT magnitude of wav itself, i.e. pre() fused in), wav [B,N] supplies
 * the phase (unet_v2.py:96) and the output length; wav_out [B,N].  vf_ssr_restore(wav) == vf_ssr_forward(NULL, wav). */
VF_API int vf_ssr_forward(vf_ctx* ctx, const float* sp, const float* wav, int batch, int64_t n_samples, float* wav_out,
                          void* stream);
VF_API int vf_ssr_restore(vf_ctx* ctx, const float* wav, int batch, int64_t n_samples, float* wav_out, void* stream);
VF_API int vf_ssr_restore_host(vf_ctx* ctx, const float* wav_host, int batch, int64_t n_samples, float* out_host,
                               void* stream);
/* vf_ssr_restore over clips of different lengths, with the contract of vf_restore_varlen: wav [B, n_max] device, row b
 * holds n_samples[b] valid samples (the rest is never read); n_samples is a HOST array, 1024 < n_samples[b] <= n_max,
 * checked before anything is launched (VF_EINVAL).  wav_out [B, n_max]: row b is bit-identical to vf_ssr_restore of that
 * clip alone; samples past n_samples[b] are 0.  Plans are cached per (batch, 64-frame bucket of the longest clip); batches
 * above 128 clips (or above the plan budget) run as sub-batches. */
VF_API int vf_ssr_restore_varlen(vf_ctx* ctx, const float* wav, int batch, int64_t n_max, const int64_t* n_samples,
                                 float* wav_out, void* stream);
/* The magnitude branch alone (unet_v2.py:99-132): sp [B,T,1025] -> out_mag [B,T,1025] (last bin 0, F.pad :128). */
VF_API int vf_ssr_unet(vf_ctx* ctx, const float* sp, int batch, int frames, float* mag_out, void* stream);
/* Intermediates of the last vf_ssr_* call of this shape: input magnitude and predicted magnitude [B,T,1025]. */
VF_API int vf_ssr_stages(vf_ctx* ctx, int batch, int64_t n_samples, float* sp_out, float* mag_out, void* stream);
/* FDomainHelper.istft(real, imag, length): real, imag [B,T,1025] -> wav_out [B,length]. */
VF_API int vf_istft(vf_ctx* ctx, const float* real, const float* imag, int batch, int frames, int64_t length,
                    float* wav_out, void* stream);

/* MelScale.forward on an arbitrary spectrogram view: mel_out[o, t, m] = sum_f specgram[o*stride_outer + f*stride_freq +
 * t*stride_time] * fb[f, m]; strides in elements, mel_out [n_outer, frames, 128] contiguous (n_outer <= 65535). */
VF_API int vf_mel(vf_ctx* ctx, const float* specgram, int64_t n_outer, int64_t frames, int64_t stride_outer,
                  int64_t stride_freq, int64_t stride_time, float* mel_out, void* stream);
/* eval_gsr_voicefixer.py:68-72 as one op: wav [B,len] -> per clip `if max|x| > 1: x /= max|x|`, then trim_center to n
 * samples -> wav_out [B,n].  (handler() sees batch 1, so "per clip" is its semantics.) */
VF_API int vf_finalize(vf_ctx* ctx, const float* wav, int batch, int64_t len, int64_t n_samples, float* wav_out,
                       void* stream);

/* ---- I/O edges of handler() (SURVEY.md 8(f) rows 3-4).
 * Polyphase resampling by up/down (load_wav -> librosa.load(sr=44100), tools/utils.py:46-48, with the arithmetic of
 * scipy.signal.resample_poly as the reference uses it in tools/dsp/lowpass.py:138-141): out[b,m] = sum_i taps[m*down -
 * i*up + n_taps/2] * wav[b,i]; taps = the caller's symmetric FIR (odd n_taps, device pointer), n_out = ceil(n*up/down). */
VF_API int vf_resample_poly(vf_ctx* ctx, const float* wav, int batch, int64_t n_samples, int up, int down, const float* taps,
                            int n_taps, float* out, int64_t n_out, void* stream);
/* amp_to_original_f (tools/utils.py:50-55; handler() applies it when meta["unify_energy"], eval_gsr_voicefixer.py:54-55) on
 * linear mels [B,T,128]: mel_out = mel_est * (mean of mel_target over bins 5..24 / mean of mel_est over bins 5..24), per clip.
 * vf_restore_ex fuses the same step into the restore chain (VF_RESTORE_UNIFY_ENERGY). */
VF_API int vf_amp_to_original_f(vf_ctx* ctx, const float* mel_est, const float* mel_target, int batch, int frames, float* mel_out,
                                void* stream);
/* AudioMetrics.lsd (evaluation_proc/metrics.py:83-87): est, target [images, frames, bins] (non-log) -> out [images]. */
VF_API int vf_lsd(vf_ctx* ctx, const float* est, const float* target, int images, int frames, int bins, float* out, void* stream);
/* AudioMetrics.sispec (metrics.py:89-95) per batch item over n values -> out [batch] (the reference then averages over
 * the batch).  est_map / target_map: 0 none, 1 to_log, 2 from_log applied on the fly (eval_gsr_voicefixer.py:60-62). */
VF_API int vf_sispec(vf_ctx* ctx, const float* est, const float* target, int batch, int64_t n, int est_map, int target_map,
                     float* out, void* stream);

VF_API int vf_to_log(vf_ctx* ctx, const float* in, float* out, int64_t n, void* stream);
VF_API int vf_from_log(vf_ctx* ctx, const float* in, float* out, int64_t n, void* stream);
/* fp32 samples -> 16-bit PCM exactly as save_wave does it: x * 2^15, truncation toward zero through a 32-bit integer,
 * low 16 bits kept (so +1.0 wraps to -32768 like numpy's astype(np.short) on the reference's hosts).  `out` is a
 * device buffer of n int16. */
VF_API int vf_to_pcm16(vf_ctx* ctx, const float* in, int16_t* out, int64_t n, void* stream);
/* saturate != 0: clamp to [-32768, 32767] first, so a peak-normalised +1.0 becomes 32767 instead of wrapping to -32768 (an
 * audible click the reference's cast produces; not bit-compatible with save_wave, hence opt-in). */
VF_API int vf_to_pcm16_ex(vf_ctx* ctx, const float* in, int16_t* out, int64_t n, int saturate, void* stream);

/* Device memory the plan for (batch, n_samples) holds (activations + packed weights). */
VF_API int vf_workspace_bytes(vf_ctx* ctx, int batch, int64_t n_samples, size_t* bytes);

/* Synchronises `stream`, reads and clears the sticky device flags.  VF_OK, VF_EDEVICE or VF_EASSERT. */
VF_API int vf_check_errors(vf_ctx* ctx, void* stream);

/* Options: "vocoder_terms" (1 or 3 fp16 split terms; "unet_terms" accepts only 3), "unify_energy" (default flag of
 * vf_restore / vf_restore_host; prefer vf_restore_ex's per-call flag), "plan_cache_mb" (cap on the device memory
 * held by cached per-shape plans, least recently used evicted first; 0 = half of the free device memory),
 * "graphs" (default 1: the fixed-pointer launch chain of a plan is captured on its second use and replayed as one CUDA graph from then on),
 * "host_pipeline" (default 1, see vf_restore_host),
 * "validate_simt" (1: run every GEMM on the SIMT validation kernel instead of tcgen05 - tests only). */
VF_API int vf_set_option(vf_ctx* ctx, const char* key, int value);
/* Plans are cached per (path, batch, frames) - frames rounded up to 64 for vf_restore_varlen and vf_ssr_restore_varlen; the cache is bounded (see "plan_cache_mb").  A batch whose plan would not fit
 * the budget is processed in sub-batches through a smaller plan (same results: rows are independent); the *_stages accessors
 * then only see the last sub-batch. */
VF_API int vf_plan_cache_info(vf_ctx* ctx, int* n_plans, size_t* bytes, size_t* budget, int64_t* evicted);
/* Number of kernels this context has launched since creation. */
VF_API int64_t vf_launch_count(vf_ctx* ctx);

/* Stage timing: wraps the stages of subsequent vf_restore calls in CUDA events on the call's stream.
 * vf_stage_times synchronises and returns milliseconds of the last vf_restore: [frontend, unet, vocoder, tail]. */
VF_API int vf_enable_stage_timing(vf_ctx* ctx, int enable);
VF_API int vf_stage_times(vf_ctx* ctx, float ms[4]);

/* Per-launch profile: with op timing enabled, the next vf_restore records a CUDA event before every kernel of
 * the UNet and vocoder launch chains.  vf_op_info(i) synchronises and returns the device time of launch i
 * together with its ALGORITHMIC flops / minimum HBM bytes (the reference op's own counts), the flops the tensor
 * cores actually executed for it (3 MMAs per product in 3-term mode, tile / phase padding, identity taps), the tcgen05 tile
 * (bn, bk, fp16 split terms; 0 for non-GEMM kernels) and a label such as "enc3.b2.conv1".  For roofline reporting only. */
VF_API int vf_enable_op_timing(vf_ctx* ctx, int enable);
VF_API int vf_op_count(vf_ctx* ctx);
VF_API int vf_op_info(vf_ctx* ctx, int i, float* ms, double* flops, double* bytes, int* bn, int* bk, int* terms,
                      char* label, int label_cap, double* exec_flops /* nullable: tensor-core flops actually issued */);

/* Self-test of one flat-shift GEMM configuration: random fp16 hi/lo planes through the tcgen05 kernel and
 * the SIMT validation kernel; returns max |difference| and max |value|.  Synchronous. */
VF_API int vf_selftest_gemm(vf_ctx* ctx, int n_img, int rows, int cin, int cout, int ntaps, int dilation, int terms,
                     double* max_abs_diff, double* max_abs_ref);

#ifdef __cplusplus
}
#endif
#endif /* B200VF_H_ */
