// HBM-bound helper kernels around the GEMMs: first UNet layer (Cin = 1), 2x2 average pooling, log/exp
// maps, vocoder conditioning, reflection padding, the Cout = 1 tail conv + tanh + peak, peak-normalise + trim.
// All of them are one-pass, vectorised (16-byte accesses on the channel-innermost planes) and write the
// fp16 hi/lo planes the next tcgen05 GEMM consumes, so no tensor is re-read for an elementwise step.
#include "gemm.cuh"
#include "kernels.cuh"

namespace vf {

__device__ __forceinline__ float lrelu(float a, float slope) { return a > 0.f ? a : a * slope; }

// ---------------------------------------------------------------------------------------------
// Per-clip table of a varlen call (kernels.cuh VarlenImage): one thread per clip, the lengths by value.
__global__ void varlen_setup_kernel(const __grid_constant__ VarlenSetupParams p) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.batch) return;
  VarlenImage r;
  r.n = (int)p.n[b];
  r.T = 1 + r.n / p.hop;
  r.Tp = (r.T + 63) / 64 * 64;
  for (int l = 0; l < 7; ++l) r.unet_rows[l] = (r.Tp >> l) * ((p.W0 >> l) + 1);
  r.voc_len[0] = r.T + r.T % 2 + p.tail_base;
  for (int s = 0; s < 8; ++s) r.voc_len[s + 1] = s < p.num_stages ? r.voc_len[s] * p.scales[s] : 0;
  r.L = r.voc_len[p.num_stages];
  r.skip = (r.L - r.n) / 2;
  r.pad_[0] = r.pad_[1] = r.pad_[2] = 0;
  p.out[b] = r;
}
cudaError_t launch_varlen_setup(const VarlenSetupParams& p, cudaStream_t stream) {
  varlen_setup_kernel<<<(p.batch + 127) / 128, 128, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) unet_first_kernel(UnetFirstParams p) {
  const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int Wp = p.W + 1;
  const size_t total = (size_t)p.batch * p.Tp * Wp;
  if (pix >= total) return;
  const size_t row = pix / Wp;
  const int f = (int)(pix - row * Wp);
  const int t = (int)(row % p.Tp);
  const int b = (int)(row / p.Tp);
  int T = p.T, Tp = p.Tp;          // frames / padded frames of this clip (T is also the row stride of logmel)
  if (p.vl) { T = p.vl[b].T; Tp = p.vl[b].Tp; }
  float out_a[32], out_r[32];
  if (f == p.W || t >= Tp) {       // pad column, or past this clip's padded frames: zeros
#pragma unroll
    for (int c = 0; c < 32; ++c) { out_a[c] = 0.f; out_r[c] = 0.f; }
  } else {
    float a[9];
    float xc = 0.f;
#pragma unroll
    for (int dh = 0; dh < 3; ++dh)
#pragma unroll
      for (int dw = 0; dw < 3; ++dw) {
        const int tt = t + dh - 1, ff = f + dw - 1;
        float v = 0.f;
        if (tt >= 0 && tt < Tp && ff >= 0 && ff < p.W) {
          const float x = tt < T ? __ldg(p.logmel + ((size_t)b * p.T + tt) * p.in_ld + ff) : 0.f;
          if (dh == 1 && dw == 1) xc = x;
          v = lrelu(fmaf(x, p.bn1_scale, p.bn1_shift), p.slope);
        }
        a[dh * 3 + dw] = v;
      }
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      float y = 0.f;
#pragma unroll
      for (int j = 0; j < 9; ++j) y = fmaf(a[j], __ldg(p.w1 + c * 9 + j), y);
      out_a[c] = lrelu(fmaf(y, __ldg(p.bn2_scale + c), __ldg(p.bn2_shift + c)), p.slope);
      out_r[c] = fmaf(xc, __ldg(p.w_sc + c), __ldg(p.b_sc + c));
    }
    bool ovf = false;
#pragma unroll
    for (int c = 0; c < 32; ++c) ovf |= !(fabsf(out_a[c]) <= 65504.f);
    if (ovf && p.err) atomicCAS(p.err, 0, ERR_FP16_OVERFLOW);
  }
  float4* rp = reinterpret_cast<float4*>(p.sc_raw + pix * 32);
#pragma unroll
  for (int i = 0; i < 8; ++i) rp[i] = make_float4(out_r[4 * i], out_r[4 * i + 1], out_r[4 * i + 2], out_r[4 * i + 3]);
#pragma unroll
  for (int i = 0; i < 4; ++i) split_store8(p.a2.hi, p.a2.lo, pix * 32 + 8 * i, out_a + 8 * i);
}
cudaError_t launch_unet_first(const UnetFirstParams& p, cudaStream_t stream) {
  const size_t total = (size_t)p.batch * p.Tp * (p.W + 1);
  unet_first_kernel<<<(unsigned)((total + 127) / 128), 128, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pool_kernel(PoolParams p) {
  const int cg = p.C / 8;
  const int Ho = p.H / 2, Wpo = p.Wpo;
  const size_t total = (size_t)p.batch * Ho * Wpo * cg;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int g = idx % cg;
  const size_t opix = idx / cg;
  const int w = opix % Wpo;
  const int h = (opix / Wpo) % Ho;
  const int b = opix / ((size_t)Wpo * Ho);
  float v[8], a[8];
  if (w == Wpo - 1 || (p.vl && (int)(opix - (size_t)b * Wpo * Ho) >= p.vl[b].unet_rows[p.vl_level])) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i] = 0.f; a[i] = 0.f; }
  } else {
    const float* base = p.in + (((size_t)b * p.H + 2 * h) * p.Wp + 2 * w) * p.C + g * 8;
    float s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float* src = base + ((size_t)(q >> 1) * p.Wp + (q & 1)) * p.C;
      const float4 x0 = __ldg(reinterpret_cast<const float4*>(src));
      const float4 x1 = __ldg(reinterpret_cast<const float4*>(src) + 1);
      s[0] += x0.x; s[1] += x0.y; s[2] += x0.z; s[3] += x0.w;
      s[4] += x1.x; s[5] += x1.y; s[6] += x1.z; s[7] += x1.w;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[i] = s[i] * 0.25f;
      a[i] = v[i];
      if (p.a_scale) a[i] = fmaf(a[i], __ldg(p.a_scale + g * 8 + i), __ldg(p.a_shift + g * 8 + i));
      a[i] = lrelu(a[i], p.slope);
      if (!(fabsf(a[i]) <= 65504.f) && p.err) atomicCAS(p.err, 0, ERR_FP16_OVERFLOW);
    }
  }
  const size_t o = opix * p.C + g * 8;
  if (p.out_raw) {
    reinterpret_cast<float4*>(p.out_raw + o)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p.out_raw + o)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
  if (p.out_r.hi) split_store8(p.out_r.hi, p.out_r.lo, o, v);
  if (p.out_a.hi) split_store8(p.out_a.hi, p.out_a.lo, o, a);
}
cudaError_t launch_pool(const PoolParams& p, cudaStream_t stream) {
  const size_t total = (size_t)p.batch * (p.H / 2) * p.Wpo * (p.C / 8);
  pool_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void to_log_kernel(const float* in, float* out, size_t n, int* neg_count) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = in[i];
  if (x < 0.f && neg_count) atomicAdd(neg_count, 1);
  out[i] = log10f(fmaxf(x, 1e-8f));
}
__global__ void from_log_kernel(const float* in, float* out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = exp10f(fminf(in[i], 5.f));
}
cudaError_t launch_to_log(const float* in, float* out, size_t n, int* neg_count, cudaStream_t stream) {
  to_log_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(in, out, n, neg_count);
  return cudaGetLastError();
}
cudaError_t launch_from_log(const float* in, float* out, size_t n, cudaStream_t stream) {
  from_log_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(in, out, n);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) voc_condition_kernel(VocCondParams p) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // (b, tv, group of 8 mel bins)
  const size_t total = (size_t)p.batch * p.Tv * 16;
  if (idx >= total) return;
  const int g = idx & 15;
  const int tv = (idx >> 4) % p.Tv;
  const int b = (idx >> 4) / p.Tv;
  float c[8];
  int T = p.T;                       // this clip's frames (p.T is also the row stride of mel)
  if (p.vl) {
    T = p.vl[b].T;
    if (tv >= p.vl[b].voc_len[0]) T = -1;
  }
  if (T < 0) {                       // past this clip's conditioning rows: zeros
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = 0.f;
  } else if (tv >= T) {
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = p.tail_value;
  } else {
    const float* src = p.mel + ((size_t)b * p.T + tv) * 128 + g * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float m = __ldg(src + i);
      if (p.is_log) m = exp10f(fminf(m, 5.f));                            // from_log, pytorch_util.py:161-163
      if (p.band_sums) m *= __ldg(p.band_sums + 2 * b) / __ldg(p.band_sums + 2 * b + 1);
      const float v = fabsf(m) / __ldg(p.weight + g * 8 + i);
      const float s = 20.f * log10f(fmaxf(v, p.amp_floor)) - p.ref_db;
      c[i] = fminf(fmaxf((s - p.min_db) / (-p.min_db), 0.f), 1.f);
    }
  }
  split_store8(p.out.hi, p.out.lo, ((size_t)b * p.Tv + tv) * 128 + g * 8, c);
}
// One CTA per clip, fixed reduction order: the scale amp_to_original_f applies (and with it every output sample) is
// reproducible run to run (a multi-CTA atomicAdd version differed in the last bits between identical calls).
__global__ void __launch_bounds__(256) band_energy_kernel(const float* tgt, const float* logest, int T, float* sums,
                                                          const VarlenImage* vl) {
  __shared__ float sh[2][8];
  const int b = blockIdx.x;
  const int Tb = vl ? vl[b].T : T;   // frames of this clip; T stays the row stride
  float st = 0.f, se = 0.f;
  for (int i = threadIdx.x; i < Tb * 20; i += 256) {
    const size_t idx = ((size_t)b * T + i / 20) * 128 + 5 + i % 20;
    st += __ldg(tgt + idx);
    se += exp10f(fminf(__ldg(logest + idx), 5.f));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    st += __shfl_xor_sync(0xffffffffu, st, o);
    se += __shfl_xor_sync(0xffffffffu, se, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = st; sh[1][threadIdx.x >> 5] = se; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f;
    for (int i = 0; i < 8; ++i) { a += sh[0][i]; c += sh[1][i]; }
    sums[2 * b] = a;
    sums[2 * b + 1] = c;
  }
}
cudaError_t launch_band_energy(const float* mel_target_lin, const float* logmel_est, int batch, int T, float* sums,
                               cudaStream_t stream, const VarlenImage* vl) {
  band_energy_kernel<<<batch, 256, 0, stream>>>(mel_target_lin, logmel_est, T, sums, vl);
  return cudaGetLastError();
}

// amp_to_original_f (tools/utils.py:50-55) as a stand-alone op on linear mels [B, T, 128]: est * (mean_low(target) / mean_low(est)),
// low band = mel bins [5, int(128 * 0.2)); one CTA per clip, fixed reduction order.
__global__ void __launch_bounds__(256) amp_to_original_kernel(const float* __restrict__ est, const float* __restrict__ tgt, int T, float* __restrict__ out) {
  __shared__ float sh[2][8];
  __shared__ float ratio;
  const int b = blockIdx.x;
  const size_t base = (size_t)b * T * 128;
  float st = 0.f, se = 0.f;
  for (int i = threadIdx.x; i < T * 20; i += 256) {
    const size_t idx = base + (size_t)(i / 20) * 128 + 5 + i % 20;
    st += __ldg(tgt + idx);
    se += __ldg(est + idx);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    st += __shfl_xor_sync(0xffffffffu, st, o);
    se += __shfl_xor_sync(0xffffffffu, se, o);
  }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = st; sh[1][threadIdx.x >> 5] = se; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f;
    for (int i = 0; i < 8; ++i) { a += sh[0][i]; c += sh[1][i]; }
    ratio = a / c;              // the 1 / (T * 20) of both means cancels
  }
  __syncthreads();
  const float r = ratio;
  for (size_t i = threadIdx.x; i < (size_t)T * 128; i += 256) out[base + i] = __ldg(est + base + i) * r;
}
cudaError_t launch_amp_to_original(const float* est, const float* tgt, int batch, int T, float* out, cudaStream_t stream) {
  amp_to_original_kernel<<<batch, 256, 0, stream>>>(est, tgt, T, out);
  return cudaGetLastError();
}

cudaError_t launch_voc_condition(const VocCondParams& p, cudaStream_t stream) {
  const size_t total = (size_t)p.batch * p.Tv * 16;
  voc_condition_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void reflect_fill_kernel(PlanePtr pl, int batch, int Lmax, int C, int pad, const VarlenImage* vl, int vl_stage) {
  const int cg = C / 8;
  const size_t total = (size_t)batch * 2 * pad * cg;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int g = idx % cg;
  const int j = (idx / cg) % (2 * pad);
  const int b = idx / ((size_t)cg * 2 * pad);
  const int L = vl ? vl[b].voc_len[vl_stage] : Lmax;     // this clip's length; Lmax sets the row pitch
  int dst, src;
  if (j < pad) { dst = j; src = 2 * pad - j; }
  else { const int i = j - pad; dst = L + pad + i; src = L - 2 - i + pad; }
  const size_t rows = (size_t)Lmax + 2 * pad;
  const size_t d = ((size_t)b * rows + dst) * C + g * 8, s = ((size_t)b * rows + src) * C + g * 8;
  *reinterpret_cast<uint4*>(pl.hi + d) = *reinterpret_cast<const uint4*>(pl.hi + s);
  *reinterpret_cast<uint4*>(pl.lo + d) = *reinterpret_cast<const uint4*>(pl.lo + s);
}
cudaError_t launch_reflect_fill(PlanePtr planes, int batch, int L, int C, int pad, cudaStream_t stream, const VarlenImage* vl,
                                int vl_stage) {
  const size_t total = (size_t)batch * 2 * pad * (C / 8);
  reflect_fill_kernel<<<(unsigned)((total + 127) / 128), 128, 0, stream>>>(planes, batch, L, C, pad, vl, vl_stage);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Tile = 320 output samples of one clip, 5 consecutive samples per thread.  The (320 + 6) x C input rows are
// copied global -> shared as fp16 with cp.async (no register staging, deep memory-level parallelism).  For each
// group of 8 channels a thread converts its 11 rows once and reuses them for all 5 outputs x 7 taps, and each
// weight vector for all 5 outputs: ~5x fewer shared-memory reads per FMA than one-output-per-thread.
// Row pitch C + 8 halfs = odd multiple of 16 bytes and an odd row stride per thread (5): conflict-free LDS.128.
constexpr int TAIL_RT = 5, TAIL_THREADS = 64, TAIL_TILE = TAIL_RT * TAIL_THREADS;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}

template <bool THREE>
__global__ void __launch_bounds__(TAIL_THREADS) voc_tail_kernel(VocTailParams p) {
  extern __shared__ __align__(16) uint8_t tail_smem[];
  const int C = p.C, pitch = C + 8;
  float* w_s = reinterpret_cast<float*>(tail_smem);                       // [7][C]
  __half* x_h = reinterpret_cast<__half*>(tail_smem + 7 * C * 4);         // [TAIL_TILE + 6][pitch]
  __half* x_l = x_h + (size_t)(TAIL_TILE + 6) * pitch;                    // THREE only
  const int b = blockIdx.y;
  const long t0 = (long)blockIdx.x * TAIL_TILE;
  const size_t rows = (size_t)p.L + 6;
  const int nrows = (int)min((long)TAIL_TILE + 6, (long)rows - t0);
  const int cg = C / 8;
  for (int idx = threadIdx.x; idx < (TAIL_TILE + 6) * cg; idx += TAIL_THREADS) {
    const int rr = idx / cg, g = idx - rr * cg;
    if (rr < nrows) {
      const size_t off = ((size_t)b * rows + t0 + rr) * C + g * 8;
      cp_async16(x_h + rr * pitch + g * 8, p.in.hi + off);
      if (THREE) cp_async16(x_l + rr * pitch + g * 8, p.in.lo + off);
    } else {                                                              // rows past the clip: never read as valid
      *reinterpret_cast<uint4*>(x_h + rr * pitch + g * 8) = make_uint4(0, 0, 0, 0);
      if (THREE) *reinterpret_cast<uint4*>(x_l + rr * pitch + g * 8) = make_uint4(0, 0, 0, 0);
    }
  }
  for (int i = threadIdx.x; i < 7 * C; i += TAIL_THREADS) w_s[i] = __ldg(p.w + i);
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();

  float acc[TAIL_RT];
#pragma unroll
  for (int o = 0; o < TAIL_RT; ++o) acc[o] = 0.f;
  const int r0 = threadIdx.x * TAIL_RT;
  for (int c8 = 0; c8 < cg; ++c8) {
    float a[TAIL_RT + 6][8];
#pragma unroll
    for (int rr = 0; rr < TAIL_RT + 6; ++rr) {
      const uint4 hq = *reinterpret_cast<const uint4*>(x_h + (r0 + rr) * pitch + c8 * 8);
      const __half2* h2 = reinterpret_cast<const __half2*>(&hq);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h2[j]);
        a[rr][2 * j] = f.x; a[rr][2 * j + 1] = f.y;
      }
      if (THREE) {
        const uint4 lq = *reinterpret_cast<const uint4*>(x_l + (r0 + rr) * pitch + c8 * 8);
        const __half2* l2 = reinterpret_cast<const __half2*>(&lq);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = __half22float2(l2[j]);
          a[rr][2 * j] += f.x; a[rr][2 * j + 1] += f.y;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      const float4 w0 = *reinterpret_cast<const float4*>(w_s + k * C + c8 * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(w_s + k * C + c8 * 8 + 4);
#pragma unroll
      for (int o = 0; o < TAIL_RT; ++o) {
        float s = acc[o];
        s = fmaf(a[o + k][0], w0.x, s); s = fmaf(a[o + k][1], w0.y, s); s = fmaf(a[o + k][2], w0.z, s); s = fmaf(a[o + k][3], w0.w, s);
        s = fmaf(a[o + k][4], w1.x, s); s = fmaf(a[o + k][5], w1.y, s); s = fmaf(a[o + k][6], w1.z, s); s = fmaf(a[o + k][7], w1.w, s);
        acc[o] = s;
      }
    }
  }
  float mag = 0.f;
  const long Lb = p.vl ? p.vl[b].L : p.L;     // this clip's samples (p.L is the row pitch)
#pragma unroll
  for (int o = 0; o < TAIL_RT; ++o) {
    const long t = t0 + r0 + o;
    if (t < Lb) {
      const float y = p.tanh_out ? tanhf(acc[o] + p.bias) : acc[o] + p.bias;
      p.wav[(size_t)b * p.L + t] = y;
      mag = fmaxf(mag, fabsf(y));
    } else if (t < p.L) {
      p.wav[(size_t)b * p.L + t] = 0.f;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mag = fmaxf(mag, __shfl_xor_sync(0xffffffffu, mag, o));
  __shared__ float wmax[TAIL_THREADS / 32];
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = mag;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int i = 0; i < TAIL_THREADS / 32; ++i) m = fmaxf(m, wmax[i]);
    atomicMax(p.peak_bits + b, __float_as_uint(m));
  }
}
cudaError_t launch_voc_tail(const VocTailParams& p, cudaStream_t stream) {
  dim3 grid((unsigned)((p.L + TAIL_TILE - 1) / TAIL_TILE), p.batch);
  const bool three = p.terms == 3;
  const size_t smem = (size_t)7 * p.C * 4 + (size_t)(three ? 2 : 1) * (TAIL_TILE + 6) * (p.C + 8) * 2;
  static bool attr_set[2] = {false, false};     // once per variant (not while a graph is being captured)
  if (!attr_set[three]) {
    cudaError_t e = three ? cudaFuncSetAttribute(voc_tail_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)
                          : cudaFuncSetAttribute(voc_tail_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    attr_set[three] = true;
  }
  if (three) voc_tail_kernel<true><<<grid, TAIL_THREADS, smem, stream>>>(p);
  else voc_tail_kernel<false><<<grid, TAIL_THREADS, smem, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
__global__ void finalize_kernel(FinalizeParams p) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (i >= p.n) return;
  long skip = p.skip;
  if (p.vl) {                        // clip of its own length: its own trim offset, zeros past its samples
    if (i >= p.vl[b].n) { p.out[(size_t)b * p.out_ld + p.out_off + i] = 0.f; return; }
    skip = p.vl[b].skip;
  }
  const float peak = __uint_as_float(p.peak_bits[b]);
  float v = p.wav[(size_t)b * p.L + skip + i];
  if (peak > 1.0f) v = v / peak;
  p.out[(size_t)b * p.out_ld + p.out_off + i] = v;
}
cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t stream) {
  dim3 grid((unsigned)((p.n + 255) / 256), p.batch);
  finalize_kernel<<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// tools/file/wav.py:22-24 (save_wave): frames *= 2^15; frames.astype(np.short).  The numpy cast on the reference's
// x86 hosts truncates toward zero through a 32-bit integer and keeps the low 16 bits, so +1.0 (a peak-normalised
// maximum) becomes -32768; reproduced bit for bit.
__global__ void pcm16_kernel(const float* __restrict__ in, int16_t* __restrict__ out, size_t n, int saturate) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = in[i] * 32768.0f;
    if (saturate) v = fminf(fmaxf(v, -32768.f), 32767.f);       // production option: no wrap of a +1.0 peak
    out[i] = static_cast<int16_t>(static_cast<uint16_t>(static_cast<uint32_t>(__float2int_rz(v)) & 0xffffu));
  }
}
cudaError_t launch_pcm16(const float* in, int16_t* out, size_t n, int saturate, cudaStream_t stream) {
  const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, 148 * 16);
  pcm16_kernel<<<blocks, 256, 0, stream>>>(in, out, n, saturate);
  return cudaGetLastError();
}

}  // namespace vf
