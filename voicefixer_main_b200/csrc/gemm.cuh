// Flat-shift multi-tap GEMM: the one contraction every conv on the VoiceFixer hot path maps to.
//
//   D[m, n] = sum_taps sum_c  A_src(tap)[img, m + a_off(tap), c_off(tap) + c] * W[n, k_off(tap) + c]
//
// Activations live in HBM as "rows x channels" fp16 planes (channels innermost): rows are flattened
// (h, w) pixels with one shared zero pad column per image row for the 2-D UNet (row pitch Wp = W + 1),
// or time steps for the 1-D vocoder.  A conv tap is then a constant row offset; zero padding above /
// below an image is the TMA out-of-bounds fill.  Each fp32 value a is stored as the pair
// hi = fp16(a), lo = fp16(a - hi); the product uses the three terms hi*hi + hi*lo + lo*hi with fp32
// accumulation (error ~2^-22, measured 5e-6 max on the full UNet - see DESIGN.md), or hi*hi only
// (terms = 1) where the stage tolerance allows.
//
// Reference ops covered (file:line in /root/reference):
//   Conv2d 3x3 pad 1 no bias          models/components/modules.py:235-243   9 taps
//   1x1 shortcut Conv2d + bias        models/components/modules.py:245-247   +1 tap, fused in the same accumulator
//   ConvTranspose2d k3 s2             models/components/modules.py:192-194   4 taps, N = 4 phases x Cout
//   Conv1d / ConvTranspose1d          vocoder restatement (oracle/vf_oracle.py:vocoder_generator)
// The epilogue fuses everything the reference does between two convs: bias, residual add
// (modules.py:268-271), eval-mode BatchNorm as a per-channel affine + LeakyReLU/ReLU/ELU of the
// *consumer* (modules.py:263-266, 213), prune/concat placement (modules.py:205-215), the 1x1 head
// with the log-mel residual (unet.py:96-100, gsr_voicefixer.py:90) and the fp16 hi/lo split.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace vf {

constexpr int GEMM_BM = 128;
constexpr int GEMM_MAX_TAPS = 12;

enum { ACT_NONE = 0, ACT_LRELU = 1, ACT_ELU = 2 };
enum { MAP_PLAIN = 0, MAP_CONVT2D = 1, MAP_CONVT1D = 2 };
enum { ERR_FP16_OVERFLOW = 100, ERR_PIPE_PRODUCER = 201, ERR_PIPE_MMA = 202, ERR_PIPE_EPILOGUE = 203 };

struct GemmTap {   // one tap, or a GROUP of up to 3 taps that read row-adjacent windows of the same source
  int a_off;   // row offset of the (group's) window start relative to the output row
  int src;     // which A source (0/1)
  int c_off;   // first channel inside the source
  int k_off;   // first column of the (first) tap's segment in the packed weight matrix
  int nch;     // channels contracted by each tap (multiple of the kernel's BK)
  int both;    // 1: contract hi AND lo planes of A even in 1-term mode (identity tap carrying the fp32-grade
               //    residual stream through the accumulator)
  int g;       // taps in the group (1..3).  Halo load: the A window (128 + 2 rows) is fetched once and tap i is
               // an MMA on the view shifted by shift[i] rows - a descriptor whose start address is advanced by
               // shift * row_bytes; the hardware swizzles on absolute address bits (tools/probe_desc_shift.cu)
  int shift[3];
  int kstride; // columns between consecutive taps' weight segments
};

struct OutPlane {
  __half* hi;
  __half* lo;
  int ld;      // row stride in elements
  int c_off;   // channel offset (concat placement)
};

struct GemmEpilogue {
  int map;             // MAP_*
  int rows_in;         // valid GEMM rows per image
  int Wp;              // 2-D row pitch (pad column = Wp-1); 0 for 1-D data
  int cout;            // channels per phase (N = phases * cout)
  int out_img_rows;    // rows per image in the output allocations
  int out_row0;        // row offset of output row 0 (slack for reflection padding)
  int out_rows_valid;  // MAP_CONVT1D: rows [0, out_rows_valid) exist
  int ct_stride, ct_pad;
  int ct_out_wp;       // MAP_CONVT2D: row pitch of the output level (2*Wp for the mel UNet, modules.py:209 prunes time only;
                       // 2*Wp - 1 for unet_v2's both=True pruning, modules.py:207-208: the column past the pitch is dropped)
  const float* bias;   // [N] or null
  const float* resid;  // fp32 [n_img * rows_in, resid_ld] or null (MAP_PLAIN only)
  int resid_ld;
  const __half* resid_hi;  // residual given as hi/lo planes [n_img * rows_in, resid_ld] (vocoder stacks whose
  const __half* resid_lo;  // GEMM is MMA-bound: cheaper to add in the epilogue than as an identity tap)
  float* out_raw;      // fp32 or null
  int raw_ld;
  OutPlane out_r;      // raw value split hi/lo (consumed by 1x1 shortcut taps)
  OutPlane out_a;      // act(scale * v + shift) split hi/lo (consumed by the next conv)
  const float* a_scale;  // [cout] or null (identity)
  const float* a_shift;
  int act;
  float slope;
  const float* head_w;   // fused 1x1 head over the 32 channels of the row, or null
  float head_b;
  const float* head_in;  // residual input [n_img, head_T, Wp] added to the head (log-mel, gsr_voicefixer.py:90), or null
  float* head_out;       // [n_img, head_T, Wp]: bins 0..Wp-2 = head + bias (+ head_in), bin Wp-1 = 0 (+ head_in): F.pad, unet.py:99
  int head_T;
  // (a, r) residual stream of the hi-only vocoder stacks: x is kept as a = fp16(lrelu_s(x)) - the plane the next conv reads
  // anyway - and r = fp16(x - U(a)), U(a) = min(a, a * inv) the inverse of the LeakyReLU (inv = fp16(1 / s), 0 < s <= 1, in
  // both halves of these words; 0 = off).  Same ~22 significant bits as a hi/lo split of x itself, but a stack moves 4
  // instead of 6 bytes per element out of every residual layer (no separate hi plane of x).
  uint32_t resid_ar;     // the residual planes (resid_hi, resid_lo) hold (a, r): add U(a) + r
  uint32_t out_ar;       // out_a is written as (hi plane = a, lo plane = r); 1-term kernels, ACT_LRELU, no affine
  int tma_out;           // bit 3: MAP_CONVT1D out_a through a 5-D map (see gemm_tc.cu).  MAP_PLAIN layers: bit 0 out_raw, bit 1 out_r, bit 2 out_a leave the staging tiles by TMA store
                         // (GemmTcParams::o_raw / o_r / o_a) instead of LDS + STG: half the LSU wavefronts of the store path
  int* err;
  // Clips of different lengths in one batch (vf_restore_varlen): the per-image table of the call (kernels.cuh VarlenImage).
  // vl_rows[img * vl_stride] = valid OUTPUT rows of image img (before out_row0); every output row at or past it is written
  // as zeros (the value, not the old contents), so the next conv reads the same zero padding a clip of that length alone
  // reads out of bounds.  vl_head_T[img * vl_stride] = frames the fused head writes.  Null: every row is valid.
  const int* vl_rows;
  const int* vl_head_T;
  int vl_stride;
};

struct GemmProblem {
  int n_img;
  int m_tiles;   // ceil(rows_in / 128)
  int N;
  int ntaps;
  int terms;     // 1 or 3
  GemmTap taps[GEMM_MAX_TAPS];
  GemmEpilogue epi;
};

struct GemmTcParams {
  CUtensorMap a_hi[2], a_lo[2];   // [C, rows, n_img] fp16
  CUtensorMap b_hi, b_lo;         // [Ktot, N] fp16 (K-major)
  CUtensorMap i_res;              // epilogue residual by TMA load (resid_tma): fp32 [resid_ld, rows_in, n_img] box 32 x 32 x 1
                                  // SWIZZLE_128B (3-term), or fp16 planes [resid_ld, rows_in, n_img, 2] box 32 x 32 x 1 x 2 SWIZZLE_64B
  int resid_tma;                  // 1: each epilogue warp owns a second 4 KB tile + an mbarrier for it
  CUtensorMap o_raw;              // fp32 [raw_ld, rows, n_img], box 32 x 32 x 1, SWIZZLE_128B (epilogue TMA stores, see tma_out)
  CUtensorMap o_r, o_a;           // fp16 [ld, rows, n_img, planes], box 32 x 32 x 1 x planes, SWIZZLE_64B
  int stages;
  int tile_chunks; // BK-wide K chunks per output tile
  int seg_chunks;  // 3-term mode: chunks per accumulation segment (promotion to registers in between)
  int tmem_cols;   // power of two >= (1 << nbuf_log) accumulator buffers of BN (1-term) or 2 * BN (3-term: [main | correction]) columns
  int nbuf_log;    // log2 of the number of accumulator buffers rotating in TMEM (1 or 2)
  int planes_a;    // smem slots per stage for A: 2 when any tap contracts the lo plane
  int a_box_rows;  // rows per A TMA box: 128, or 130 when taps are grouped (halo)
  int gmax;        // largest tap group: B slots per stage
  int grid;        // persistent CTAs
  uint32_t magic_n, magic_m;   // gemm_tc_magic() of N / BN and m_tiles: division-free tile decoding
  int ctas_per_sm; // co-resident CTAs the launch is sized for (selects the register budget of the kernel variant)
  GemmProblem prob;
};

// Fused residual pair of the C = 64 vocoder stacks (pair_tc.cu): x_new = x + conv_b(lrelu(conv_a(xa) + bias_a)) + bias_b
struct PairParams {
  CUtensorMap a_map;             // activated input plane lrelu(x), hi: [C, L, clips], box 64 x 128 x 1, SWIZZLE_128B
  CUtensorMap wa_map, wb_map;    // packed K-major hi weights [K >= 3C, C], box 64 x C
  CUtensorMap xin_map[2];        // residual x.  in_f32: [0] = the stack's fp32 stream [C, L, clips] (box 32 x 126 x 1, used for
                                 // both channel halves); else [0] / [1] = its hi / lo fp16 planes (box 64 x 126 x 1), written
                                 // by the up-sampling GEMM in front of the stack
  CUtensorMap xo_map;            // x_new, fp32 stream (box 32 x 126 x 1); unused when out_f32 == 0 (last pair of a stage)
  CUtensorMap ao_map;            // lrelu(x_new, slope_out), hi plane [C, out_row0 + L, clips] (box 64 x 126 x 1)
  const float* bias_a;
  const float* bias_b;
  int in_f32, out_f32;
  uint32_t ar_in, ar_out;        // (a, r) stream (see GemmEpilogue): xin_map = the activated and the correction plane of the source,
                                 // xo_map = the correction plane of the destination (fp16, box 64 x 126 x 1); ar_out = 0 on the last pair
  int L, n_img, C, dil, out_img_rows, out_row0, tiles_per_img, stages, grid;
  uint32_t magic_t;              // gemm_tc_magic(tiles_per_img, ...)
  float slope_h, slope_out;
  int* err;
  const int* vl_len;             // per-image clip length L_b = vl_len[img * vl_stride] (varlen batches, see GemmEpilogue), or
  int vl_stride;                 // null: L.  Rows at or past L_b are zero in h and in both outputs
};

__host__ __device__ inline uint32_t fast_div_pair(uint32_t n, uint32_t d, uint32_t magic) {
#ifdef __CUDA_ARCH__
  if (magic == 0u) return n;
  if (magic == 0xffffffffu) return n / d;
  return __umulhi(n, magic);
#else
  (void)magic;
  return n / d;
#endif
}

struct GemmSimtParams {            // validation kernel: same contract, plain pointers
  const __half* a_hi[2];
  const __half* a_lo[2];
  int a_ld[2], a_rows[2], a_img_rows[2];
  const __half* b_hi;
  const __half* b_lo;
  int ktot;
  GemmProblem prob;
};

__device__ __forceinline__ void split_store8(__half* hi, __half* lo, size_t idx, const float* a) {
  __align__(16) __half h[8];
  __align__(16) __half l[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    h[i] = __float2half_rn(a[i]);
    l[i] = __float2half_rn(a[i] - __half2float(h[i]));
  }
  *reinterpret_cast<uint4*>(hi + idx) = *reinterpret_cast<const uint4*>(h);
  *reinterpret_cast<uint4*>(lo + idx) = *reinterpret_cast<const uint4*>(l);
}

// One thread owns GEMM row `r` of image `img`; v holds columns [n_base, n_base + 32).
__device__ __forceinline__ void epilogue_chunk(const GemmEpilogue& e, int img, int r, int n_base, float (&v)[32],
                                               float& head_acc) {
  if (r >= e.rows_in) return;
  int co0 = n_base, phase = 0;
  if (e.map != MAP_PLAIN) {
    phase = n_base / e.cout;
    co0 = n_base - phase * e.cout;
  }
  size_t orow;
  long lrow;               // output row inside the image
  bool pad = false;
  if (e.map == MAP_PLAIN) {
    lrow = r;
    orow = (size_t)img * e.out_img_rows + e.out_row0 + r;
    if (e.Wp > 0) pad = (r % e.Wp) == e.Wp - 1;
  } else if (e.map == MAP_CONVT2D) {
    const int h = r / e.Wp, w = r - h * e.Wp;
    const int ph = phase >> 1, pw = phase & 1;
    const int col = 2 * w + pw;
    if (col >= e.ct_out_wp) return;          // both=True prune: column past the output pitch
    lrow = (long)(2 * h + ph) * e.ct_out_wp + col;
    orow = (size_t)img * e.out_img_rows + lrow;
    pad = col == e.ct_out_wp - 1;
  } else {
    const long t = (long)r * e.ct_stride + phase - e.ct_pad;
    if (t < 0 || t >= e.out_rows_valid) return;
    lrow = t;
    orow = (size_t)img * e.out_img_rows + e.out_row0 + t;
  }
  if (e.vl_rows && lrow >= __ldg(e.vl_rows + (size_t)img * e.vl_stride)) pad = true;   // past this clip: zeros
  if (e.bias) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += __ldg(e.bias + n_base + i);
  }
  if (e.resid) {
    const float4* rp = reinterpret_cast<const float4*>(e.resid + ((size_t)img * e.rows_in + r) * e.resid_ld + co0);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 q = __ldg(rp + i);
      v[4 * i] += q.x; v[4 * i + 1] += q.y; v[4 * i + 2] += q.z; v[4 * i + 3] += q.w;
    }
  }
  if (e.resid_hi) {
    const size_t ro = ((size_t)img * e.rows_in + r) * e.resid_ld + co0;
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] += __half2float(e.resid_hi[ro + i]) + __half2float(e.resid_lo[ro + i]);
  }
  if (pad) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.f;
  }
  if (e.out_raw) {
    float4* op = reinterpret_cast<float4*>(e.out_raw + orow * e.raw_ld + co0);
#pragma unroll
    for (int i = 0; i < 8; ++i) op[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  }
  if (e.out_r.hi) {
    const size_t base = orow * e.out_r.ld + e.out_r.c_off + co0;
#pragma unroll
    for (int i = 0; i < 4; ++i) split_store8(e.out_r.hi, e.out_r.lo, base + 8 * i, v + 8 * i);
  }
  if (e.head_w) {
#pragma unroll
    for (int i = 0; i < 32; ++i) head_acc = fmaf(v[i], __ldg(e.head_w + co0 + i), head_acc);
  }
  if (e.out_a.hi) {
    bool ovf = false;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      float a = v[i];
      if (e.a_scale) a = fmaf(a, __ldg(e.a_scale + co0 + i), __ldg(e.a_shift + co0 + i));
      if (e.act == ACT_LRELU) a = a > 0.f ? a : a * e.slope;
      else if (e.act == ACT_ELU) a = a > 0.f ? a : expm1f(a);
      if (pad) a = 0.f;
      ovf |= !(fabsf(a) <= 65504.f);
      v[i] = a;
    }
    if (ovf && e.err) atomicCAS(e.err, 0, ERR_FP16_OVERFLOW);
    const size_t base = orow * e.out_a.ld + e.out_a.c_off + co0;
#pragma unroll
    for (int i = 0; i < 4; ++i) split_store8(e.out_a.hi, e.out_a.lo, base + 8 * i, v + 8 * i);
  }
}

// unet.py:96-100 + gsr_voicefixer.py:90: out = head(x) padded with a zero bin, plus the input log-mel;
// unet_v2.py:125-132: the same head without the residual (the output is the magnitude itself).
__device__ __forceinline__ void epilogue_head(const GemmEpilogue& e, int img, int r, float head_acc) {
  if (!e.head_w || r >= e.rows_in) return;
  const int t = r / e.Wp, f = r - t * e.Wp;
  if (t >= e.head_T) return;
  if (e.vl_head_T && t >= __ldg(e.vl_head_T + (size_t)img * e.vl_stride)) return;
  const size_t idx = ((size_t)img * e.head_T + t) * e.Wp + f;
  const float y = (f < e.Wp - 1) ? head_acc + e.head_b : 0.f;
  e.head_out[idx] = e.head_in ? y + __ldg(e.head_in + idx) : y;
}

}  // namespace vf
