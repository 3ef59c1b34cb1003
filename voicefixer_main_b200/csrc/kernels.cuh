// Parameter blocks and launchers of the non-GEMM kernels on the hot path.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vf {

// Clips of different lengths in one batch (vf_restore_varlen, vf_ssr_restore_varlen).  A small kernel writes one record per clip at the start of
// every call; every later kernel of the call reads its clip's lengths from it in device memory, so a captured launch chain
// stays valid whatever the lengths are.  All rows at or past a clip's length in a plane a later conv reads are written as
// zeros: what an earlier call with longer clips left in the slot never matters.
constexpr int VF_VARLEN_MAX_CLIPS = 128;     // lengths travel by value in the setup kernel's parameter block
struct VarlenImage {
  int n;              // valid input samples
  int T;              // frames, 1 + n / hop
  int Tp;             // T padded to a multiple of 64 (the UNet's zero input rows, unet.py:75-77)
  int unet_rows[7];   // valid rows of UNet level l: (Tp >> l) * Wp_l
  int voc_len[9];     // vocoder lengths: [0] = Tv = T + T % 2 + tail base, [s + 1] = output length of up-sampling stage s
  int L;              // vocoder output samples
  int skip;           // centre-trim offset (L - n) / 2
  int pad_[3];
};
constexpr int VARLEN_STRIDE = (int)(sizeof(VarlenImage) / sizeof(int));
static_assert(sizeof(VarlenImage) % 16 == 0, "VarlenImage: keep records 16-byte aligned");
struct VarlenSetupParams {
  int batch, W0, hop, tail_base, num_stages;
  int scales[8];
  VarlenImage* out;    // [batch]
  long long n[VF_VARLEN_MAX_CLIPS];
};
cudaError_t launch_varlen_setup(const VarlenSetupParams& p, cudaStream_t stream);

struct FrontendParams {
  const float* wav;      // [batch, n]
  long n;
  int batch, T;          // T = 1 + n / 441
  const float* window;   // [2048] periodic hann
  const float2* tw1024;  // e^{-2 pi i j / 1024}
  const float2* tw2048;  // e^{-2 pi i k / 2048}, k = 0..1024
  const int* fb_f0;      // [128] first non-zero frequency bin of each mel filter
  const int* fb_len;     // [128]
  const int* fb_ofs;     // [128] offset into fb_val
  const float* fb_val;
  float* sp_out;         // [batch, T, 1025] or null
  float* cos_out;        // with sp_out, or null
  float* sin_out;
  float* mel_out;        // [batch, T, 128] linear mel or null
  float* logmel_out;     // [batch, T, 128] log10(clip(mel, 1e-8)) or null
  const VarlenImage* vl; // or null.  Set: n is the row stride of wav, clip b has vl[b].n samples and vl[b].T frames;
                         // frames past them are written as zeros in every output that is set (all 1025 bins of sp / cos / sin)
};
cudaError_t launch_frontend(const FrontendParams& p, cudaStream_t stream);

struct PlanePtr {
  __half* hi;
  __half* lo;
};

// encoder_block1.conv_block1: BN(1ch) -> LeakyReLU -> Conv3x3 1->32, then bn2 -> LeakyReLU of the same
// block fused in (the only consumer), plus the 1->32 1x1 shortcut of the raw input (modules.py:263-271).
struct UnetFirstParams {
  const float* logmel;   // [batch, T, in_ld]; bins 0..W-1 feed the UNet (unet.py:78: log-mel, W = 127 of 128;
                         // unet_v2.py:108: linear magnitude, W = 1024 of 1025)
  int batch, T, Tp;      // Tp = T padded to a multiple of 64 with zero *input* rows (unet.py:75-77)
  int W, in_ld;          // valid bins per frame / input row stride; the planes use row pitch Wp = W + 1
  float bn1_scale, bn1_shift;
  const float* w1;       // [32][9]
  const float* bn2_scale;  // [32]
  const float* bn2_shift;
  const float* w_sc;     // [32] shortcut weight
  const float* b_sc;     // [32] shortcut bias
  float slope;
  PlanePtr a2;           // [batch, Tp*Wp, 32] act(bn2(conv1(...))), pad column zero
  float* sc_raw;         // [batch, Tp*Wp, 32] fp32 shortcut(x), pad column zero
  int* err;
  const VarlenImage* vl; // or null.  Set: T is the row stride of logmel; clip b uses vl[b].T / vl[b].Tp, rows past Tp_b are 0
};
cudaError_t launch_unet_first(const UnetFirstParams& p, cudaStream_t stream);

// avg_pool2d(2,2) (modules.py:183) + the consumer's BN/LeakyReLU + hi/lo split.
struct PoolParams {
  const float* in;       // [batch, H*Wp, C] fp32
  int batch, H, Wp, C;
  int Wpo;               // output row pitch = (Wp - 1) / 2 + 1 (floor pooling of the W = Wp - 1 valid columns + pad column)
  PlanePtr out_r;        // [batch, (H/2)*Wpo, C] pooled raw
  PlanePtr out_a;        // act(scale*pooled+shift)
  float* out_raw;        // fp32 pooled or null
  const float* a_scale;
  const float* a_shift;
  float slope;
  int* err;
  const VarlenImage* vl; // or null.  Set: output rows at or past vl[b].unet_rows[vl_level] are written as zeros
  int vl_level;          // UNet level of the output
};
cudaError_t launch_pool(const PoolParams& p, cudaStream_t stream);

// to_log / from_log (tools/pytorch/pytorch_util.py:157-163) for the stage-level API.
cudaError_t launch_to_log(const float* in, float* out, size_t n, int* neg_count, cudaStream_t stream);
cudaError_t launch_from_log(const float* in, float* out, size_t n, cudaStream_t stream);

// Vocoder prologue: mel / w -> dB -> normalise -> [T + tail, 128] planes with the constant tail.
struct VocCondParams {
  const float* mel;      // [batch, T, 128]; linear mel, or log10 mel when is_log (from_log fused)
  int is_log;
  int batch, T, Tv;
  const float* weight;       // [128] per-bin mel weight (divided out)
  float amp_floor, ref_db, min_db, tail_value;
  const float* band_sums;    // [batch][2] (target, estimate) low-band sums from launch_band_energy, or null:
                             // amp_to_original_f (tools/utils.py:50-55) scales the estimate by target/estimate
  PlanePtr out;          // [batch, Tv, 128]
  const VarlenImage* vl; // or null.  Set: T is the row stride of mel; clip b: mel rows [0, T_b), the tail on [T_b, Tv_b), zeros after
};
cudaError_t launch_voc_condition(const VocCondParams& p, cudaStream_t stream);

// amp_to_original_f, reduction half: per clip, sums over frames and mel bins [5, int(128*0.2)) of the noisy
// linear mel (target) and of from_log(restored log-mel) (estimate).  sums must be zeroed before the launch.
cudaError_t launch_band_energy(const float* mel_target_lin, const float* logmel_est, int batch, int T, float* sums,
                               cudaStream_t stream, const VarlenImage* vl = nullptr);   // vl: T is the row stride, sums over T_b

// amp_to_original_f as a stand-alone op: out = est * (low-band mean of target / low-band mean of est), linear mels [batch, T, 128].
cudaError_t launch_amp_to_original(const float* est, const float* tgt, int batch, int T, float* out, cudaStream_t stream);

// nn.ReflectionPad1d(3): rows [3, L+3) of each image are already written; fill 3 + 3 mirrored rows.
// vl (or null): L is the row pitch less 2 * pad; clip b reflects at its own length vl[b].voc_len[vl_stage].
cudaError_t launch_reflect_fill(PlanePtr planes, int batch, int L, int C, int pad, cudaStream_t stream,
                                const VarlenImage* vl = nullptr, int vl_stage = 0);

// Tail: ReflectionPad(3) (pre-filled) + Conv1d(C -> 1, k7) + tanh, plus the per-clip peak |out|.
struct VocTailParams {
  PlanePtr in;           // [batch, L + 6, C]
  int batch, L, C, terms;
  int tanh_out;          // 1: tanh on the output (the generator's last op); 0: linear (test configurations that exceed |1|)
  const float* w;        // [7][C]
  float bias;
  float* wav;            // [batch, L]
  unsigned int* peak_bits;   // [batch] max |out| as float bits (non-negative floats order like uints)
  const VarlenImage* vl;     // or null.  Set: clip b has vl[b].L samples (peak over those only, zeros after them)
};
cudaError_t launch_voc_tail(const VocTailParams& p, cudaStream_t stream);

// eval_gsr_voicefixer.py:68-72: out /= max|out| if it exceeds 1; trim_center (tools/utils.py:57-70).
struct FinalizeParams {
  const float* wav;      // [batch, L]
  const unsigned int* peak_bits;
  int batch;
  long L, n, skip;       // out[b, i] = wav[b, skip + i], i < n
  float* out;            // [batch, out_ld]
  long out_ld, out_off;
  const VarlenImage* vl; // or null.  Set: clip b keeps vl[b].n samples from vl[b].skip; out[b, i] = 0 for vl[b].n <= i < n
};
cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t stream);
cudaError_t launch_pcm16(const float* in, int16_t* out, size_t n, int saturate, cudaStream_t stream);

// max |wav| per clip as float bits (atomicMax), for the stand-alone peak normalise + trim entry point.
cudaError_t launch_peak(const float* wav, int batch, long L, unsigned int* peak_bits, cudaStream_t stream);

// MelScale.forward (tools/pytorch/mel_scale.py:52-64) as a stand-alone op on any [..., freq, time] view:
// out[o, t, m] = sum_f in[o * so + f * sf + t * st] * fb[f, m] with the filterbank in its sparse form.
struct MelParams {
  const float* in;
  long n_outer, T;
  long so, sf, st;       // input strides (elements) of the outer, frequency and time axes
  float* out;            // [n_outer, T, 128] contiguous
  const int* fb_f0;
  const int* fb_len;
  const int* fb_ofs;
  const float* fb_val;
};
cudaError_t launch_mel(const MelParams& p, cudaStream_t stream);

// ISTFT (FDomainHelper.istft, fDomainHelper.py:30-32,127 -> torchlibrosa ISTFT: n_fft = win = 2048, hop 441, periodic
// hann, center): stage 1 writes the windowed inverse-DFT frames, stage 2 overlap-adds them in a fixed order and divides
// by the overlap-added squared window (clamped at 1e-11).  Stage 1 takes the spectrum either as (real, imag), or -
// unet_v2.py:96,136-139 fused - as a magnitude plus the waveform whose STFT phase it is to carry:
// real = mag * cos, imag = mag * sin with cos, sin = re/|X|, im/|X| of the input (fDomainHelper.py:62-64).
struct IstftFramesParams {
  const float* real;     // [batch, T, 1025] or null
  const float* imag;
  const float* mag;      // [batch, T, 1025] (with wav) or null
  const float* wav;      // [batch, n]
  long n;
  int batch, T;
  const float* window;   // [2048]
  const float2* tw1024;
  const float2* tw2048;
  float* frames;         // [batch, T, 2048]
  const VarlenImage* vl; // or null.  Set: n is the row stride of wav and T of mag / frames; clip b reflects at vl[b].n and
                         // only its frames t < vl[b].T are computed (later frames are left as they are: no kernel reads them)
};
cudaError_t launch_istft_frames(const IstftFramesParams& p, cudaStream_t stream);
struct IstftOlaParams {
  const float* frames;   // [batch, T, 2048]
  int batch, T;
  long length;           // output samples per clip: y[n_fft/2 : n_fft/2 + length]
  const float* window;
  float* out;            // [batch, out_ld]
  long out_ld;
  const VarlenImage* vl; // or null.  Set: T is the row stride of frames, length the output samples per row; clip b sums its
                         // frames t < vl[b].T only (numerator AND window-square sum, as if restored alone), writes vl[b].n
                         // samples and exact zeros on [vl[b].n, length)
};
cudaError_t launch_istft_ola(const IstftOlaParams& p, cudaStream_t stream);

// edges.cu: polyphase resampling (load_wav) and the handler's mel metrics
cudaError_t launch_resample_poly(const float* x, int batch, long n, int up, int down, const float* h, int half, float* out, long n_out,
                                 cudaStream_t stream);
cudaError_t launch_lsd(const float* est, const float* tgt, int images, int T, int F, float* out, cudaStream_t stream);
cudaError_t launch_sispec(const float* est, const float* tgt, int batch, long n, int est_map, int tgt_map, float* out, cudaStream_t stream);

}  // namespace vf
