// Back end of the SSR / GSR-UNet path (SURVEY.md 8(f) row 1, BASELINE config 3) and small stand-alone ops of the
// drop-in boundary: ISTFT (two kernels), MelScale.forward on an arbitrary spectrogram view, per-clip peak.
//
// ISTFT replaces FDomainHelper.istft (tools/pytorch/modules/fDomainHelper.py:30-32,127; torchlibrosa ISTFT:
// mirrored-spectrum inverse-DFT conv + window + overlap-add + window-sum divide).  The 2048-point real inverse
// transform of a frame is ONE 1024-point complex FFT in shared memory: Z[k] = E[k] + i O[k] with
// E = (X[k] + conj X[1024-k])/2, O = (X[k] - conj X[1024-k])/2 * e^{+2 pi i k/2048}; z = IDFT_1024(Z) gives
// x[2n] = Re z[n], x[2n+1] = Im z[n]; the inverse FFT runs as conj(FFT(conj Z))/1024 on the forward code.
// In the fused SSR mode the same CTA first recomputes the STFT of its input frame (as unet_v2.py:96 does) so
// that cos/sin never exist in HBM: per frame 2048*4 B in (L2-resident waveform) + 1025*4 B magnitude in,
// 2048*4 B out.
#include <algorithm>

#include "fft.cuh"
#include "kernels.cuh"

namespace vf {

__global__ void __launch_bounds__(256) istft_frames_kernel(IstftFramesParams p) {
  __shared__ float2 buf0[1024];
  __shared__ float2 buf1[1024];
  __shared__ float2 Y[1025];
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const size_t frame = (size_t)b * p.T + t;
  if (p.vl && t >= p.vl[b].T) return;       // past a varlen clip's frames: nothing to compute (uniform per CTA)
  if (p.mag) {
    const long n = p.vl ? (long)p.vl[b].n : p.n;     // a varlen clip reflects at its own end
    load_frame_packed(buf0, p.wav + (size_t)b * p.n, n, t, p.window, tid);
    __syncthreads();
    const float2* Z = fft1024_forward(buf0, buf1, p.tw1024, tid);
    for (int k = tid; k <= 1024; k += 256) {
      const float2 xk = rfft_split(Z, p.tw2048, k);
      const float m = sqrtf(fmaxf(xk.x * xk.x + xk.y * xk.y, 1e-8f));     // fDomainHelper.py:62
      const float cs = xk.x / m, sn = xk.y / m;                              // fDomainHelper.py:63-64
      const float om = __ldg(p.mag + frame * 1025 + k);
      Y[k] = make_float2(om * cs, om * sn);                                  // unet_v2.py:136-137
    }
  } else {
    for (int k = tid; k <= 1024; k += 256) Y[k] = make_float2(__ldg(p.real + frame * 1025 + k), __ldg(p.imag + frame * 1025 + k));
  }
  __syncthreads();
  // conj(Z) of the packed inverse; the imaginary parts of the DC and Nyquist bins do not reach a real signal
  for (int k = tid; k < 1024; k += 256) {
    float2 yk = Y[k], yr = Y[1024 - k];
    if (k == 0) { yk.y = 0.f; yr.y = 0.f; }
    const float2 e = make_float2(0.5f * (yk.x + yr.x), 0.5f * (yk.y - yr.y));     // (Yk + conj Yr)/2
    const float2 d = make_float2(0.5f * (yk.x - yr.x), 0.5f * (yk.y + yr.y));     // (Yk - conj Yr)/2
    const float2 w = __ldg(p.tw2048 + k);
    const float2 o = cmul(d, make_float2(w.x, -w.y));                              // * e^{+2 pi i k/2048}
    // Z = E + i O = (e.x - o.y) + i (e.y + o.x); store conj(Z)
    buf0[k] = make_float2(e.x - o.y, -(e.y + o.x));
  }
  __syncthreads();
  const float2* z = fft1024_forward(buf0, buf1, p.tw1024, tid);
  float2* out = reinterpret_cast<float2*>(p.frames + frame * 2048);
  const float2* win = reinterpret_cast<const float2*>(p.window);
  for (int j = tid; j < 1024; j += 256) {
    const float2 v = z[j];
    const float2 w = __ldg(win + j);
    out[j] = make_float2(v.x * (1.f / 1024.f) * w.x, -v.y * (1.f / 1024.f) * w.y);
  }
}
cudaError_t launch_istft_frames(const IstftFramesParams& p, cudaStream_t stream) {
  dim3 grid(p.T, p.batch);
  istft_frames_kernel<<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// y[p] = sum_t frames[t][p - 441 t] / clamp(sum_t win^2[p - 441 t], 1e-11), p = i + 1024; ascending t (deterministic).
// A varlen clip ends its sum at its own last frame T_b - 1: frame T_b starts at 441 T_b < 1024 + n_b, so it would
// overlap the clip's last samples, and its window would enter the denominator even with a zero numerator.
__global__ void __launch_bounds__(256) istft_ola_kernel(IstftOlaParams p) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (i >= p.length) return;
  long T = p.T;
  if (p.vl) {
    if (i >= p.vl[b].n) { p.out[(size_t)b * p.out_ld + i] = 0.f; return; }
    T = p.vl[b].T;
  }
  const long pos = i + 1024;
  long t_lo = (pos - 2047 + 440) / 441;       // ceil((pos - 2047) / 441), pos >= 1024 so the numerator may be negative
  if (pos - 2047 <= 0) t_lo = 0;
  long t_hi = pos / 441;
  if (t_hi > T - 1) t_hi = T - 1;
  float acc = 0.f, ws = 0.f;
  for (long t = t_lo; t <= t_hi; ++t) {
    const int off = (int)(pos - 441 * t);
    acc += __ldg(p.frames + ((size_t)b * p.T + t) * 2048 + off);
    const float w = __ldg(p.window + off);
    ws = fmaf(w, w, ws);
  }
  p.out[(size_t)b * p.out_ld + i] = acc / fmaxf(ws, 1e-11f);
}
cudaError_t launch_istft_ola(const IstftOlaParams& p, cudaStream_t stream) {
  dim3 grid((unsigned)((p.length + 255) / 256), p.batch);
  istft_ola_kernel<<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// MelScale.forward: one CTA = 8 time steps of one outer index; the [1025 x 8] spectrogram tile is staged in shared
// memory (whole 32-byte sectors along whichever axis is contiguous), then 128 mels x 8 steps from the sparse filterbank.
constexpr int MEL_TT = 8;
__global__ void __launch_bounds__(256) mel_kernel(MelParams p) {
  __shared__ float tile[1025][MEL_TT + 1];
  const long o = blockIdx.y;
  const long t0 = (long)blockIdx.x * MEL_TT;
  const int nt = (int)min((long)MEL_TT, p.T - t0);
  const float* base = p.in + o * p.so + t0 * p.st;
  if (p.st == 1) {           // [..., freq, time] contiguous: time fastest
    for (int idx = threadIdx.x; idx < 1025 * MEL_TT; idx += 256) {
      const int f = idx / MEL_TT, tt = idx % MEL_TT;
      tile[f][tt] = tt < nt ? __ldg(base + (long)f * p.sf + tt) : 0.f;
    }
  } else {                   // e.g. the permuted view of a [.., time, freq] tensor: frequency fastest
    for (int idx = threadIdx.x; idx < 1025 * MEL_TT; idx += 256) {
      const int tt = idx / 1025, f = idx % 1025;
      tile[f][tt] = tt < nt ? __ldg(base + (long)f * p.sf + (long)tt * p.st) : 0.f;
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 128 * MEL_TT; idx += 256) {
    const int tt = idx >> 7, m = idx & 127;
    if (tt >= nt) continue;
    const int f0 = __ldg(p.fb_f0 + m), len = __ldg(p.fb_len + m);
    const float* w = p.fb_val + __ldg(p.fb_ofs + m);
    float acc = 0.f;
    for (int j = 0; j < len; ++j) acc = fmaf(tile[f0 + j][tt], __ldg(w + j), acc);
    p.out[(o * p.T + t0 + tt) * 128 + m] = acc;
  }
}
cudaError_t launch_mel(const MelParams& p, cudaStream_t stream) {
  dim3 grid((unsigned)((p.T + MEL_TT - 1) / MEL_TT), (unsigned)p.n_outer);
  mel_kernel<<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) peak_kernel(const float* __restrict__ wav, long L, unsigned int* peak_bits) {
  const int b = blockIdx.y;
  float m = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += (long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(__ldg(wav + (size_t)b * L + i)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(peak_bits + b, __float_as_uint(m));
}
cudaError_t launch_peak(const float* wav, int batch, long L, unsigned int* peak_bits, cudaStream_t stream) {
  dim3 grid((unsigned)std::min<long>((L + 255) / 256, 64), batch);
  peak_kernel<<<grid, 256, 0, stream>>>(wav, L, peak_bits);
  return cudaGetLastError();
}

}  // namespace vf
