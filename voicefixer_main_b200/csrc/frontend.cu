// Stage A: fused STFT magnitude + mel projection (+ log10).
//
// Replaces, per frame, the reference chain
//   FDomainHelper.wav_to_spectrogram_phase  tools/pytorch/modules/fDomainHelper.py:60-89
//     (torchlibrosa STFT: reflect pad 1024, periodic-hann windowed 2048-point DFT as two conv1d, hop 441)
//   MelScale.forward                        tools/pytorch/mel_scale.py:52-64 (gsr_voicefixer.py:180)
//   to_log                                  tools/pytorch/pytorch_util.py:157-159
// with one CTA per (frame, clip): windowed load straight from the un-padded waveform (reflection by index
// math), a 1024-point complex radix-4 Stockham FFT in shared memory on the even/odd-packed real frame,
// the real-FFT split, |.| with the 1e-8 power clamp, and the triangular mel filterbank applied in its
// sparse form (2018 non-zeros instead of a 1025x128 dense matmul).  The 1025-bin spectrogram is only
// written when the caller asks for it (the GSR path discards it, eval_gsr_voicefixer.py:51).
// HBM traffic on the GSR path: N*4 bytes in, T*128*4 bytes out per clip (2.277 MB for 10 s).
#include "fft.cuh"
#include "kernels.cuh"

namespace vf {

__global__ void __launch_bounds__(256) frontend_kernel(FrontendParams p) {
  __shared__ float2 buf0[1024];
  __shared__ float2 buf1[1024];
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const float* x = p.wav + (size_t)b * p.n;
  long n = p.n;
  if (p.vl) {                    // clip of its own length in a wider batch: reflect at its end, zeros past its frames
    n = p.vl[b].n;
    if (t >= p.vl[b].T) {
      const size_t frame = (size_t)b * p.T + t;
      if (tid < 128) {
        if (p.mel_out) p.mel_out[frame * 128 + tid] = 0.f;
        if (p.logmel_out) p.logmel_out[frame * 128 + tid] = 0.f;
      }
      if (p.sp_out)
        for (int k = tid; k <= 1024; k += 256) {
          p.sp_out[frame * 1025 + k] = 0.f;
          if (p.cos_out) { p.cos_out[frame * 1025 + k] = 0.f; p.sin_out[frame * 1025 + k] = 0.f; }
        }
      return;
    }
  }

  // windowed, reflect-padded frame packed as z[n] = x[2n] + i x[2n+1]; 1024-point FFT (fft.cuh)
  load_frame_packed(buf0, x, n, t, p.window, tid);
  __syncthreads();
  const float2* src = fft1024_forward(buf0, buf1, p.tw1024, tid);
  // src == buf1 now holds Z[0..1023]; buf0 is free and becomes the magnitude row
  float* mag = reinterpret_cast<float*>(buf0);
  const size_t frame = (size_t)b * p.T + t;
  for (int k = tid; k <= 1024; k += 256) {
    const float2 xk = rfft_split(src, p.tw2048, k);
    const float re = xk.x, im = xk.y;
    const float m = sqrtf(fmaxf(re * re + im * im, 1e-8f));       // fDomainHelper.py:62, eps = 1e-8
    mag[k] = m;
    if (p.sp_out) {
      p.sp_out[frame * 1025 + k] = m;
      if (p.cos_out) {
        p.cos_out[frame * 1025 + k] = re / m;
        p.sin_out[frame * 1025 + k] = im / m;
      }
    }
  }
  __syncthreads();
  if (tid < 128) {
    const int f0 = __ldg(p.fb_f0 + tid), len = __ldg(p.fb_len + tid);
    const float* w = p.fb_val + __ldg(p.fb_ofs + tid);
    float acc = 0.f;
    for (int j = 0; j < len; ++j) acc = fmaf(mag[f0 + j], __ldg(w + j), acc);
    if (p.mel_out) p.mel_out[frame * 128 + tid] = acc;
    if (p.logmel_out) p.logmel_out[frame * 128 + tid] = log10f(fmaxf(acc, 1e-8f));
  }
}

cudaError_t launch_frontend(const FrontendParams& p, cudaStream_t stream) {
  dim3 grid(p.T, p.batch);
  frontend_kernel<<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace vf
