// Fused residual pair of the vocoder's C = 64 stacks (the last up-sampling stage: 443 k time steps per clip) as ONE kernel:
//     x_new = x + conv_b(lrelu(conv_a(lrelu(x)) + bias_a)) + bias_b          (oracle: vocoder_generator, the `res.s.i` pair)
// conv_a: k = 3, dilation d, zero padding;  conv_b: k = 3, dilation 1, zero padding.  hi-only fp16 operands, fp32
// accumulation (the vocoder's 1-term mode).  What two separate GEMM launches move through HBM in between - the activated
// intermediate h, written by "a" and read back by "b" (4 of 16 bytes per element) - stays in shared memory.  The residual
// stream of a fused stack is the (a, r) pair of gemm.cuh by default (MODE 2: 8 bytes per element), or fp32 (MODE 0 / 1:
// 12 bytes per element, VF_TUNE_AR_STREAM=0).
//
//   tile = 126 output rows t0 .. t0+125 of one clip, m0 = t0 - 1.
//   P1 (conv_a)   A = lrelu(x) rows m0 + (tap-1) d + [0,128) by TMA (out-of-range rows zero filled), accumulator 1 = h rows
//                 m0 .. m0+127 before bias / activation
//   E1            + bias_a, LeakyReLU, rows outside the clip forced to zero (conv_b's zero padding), fp16, written to the
//                 shared-memory tile H in the K-major SWIZZLE_128B layout a TMA load would have produced (h row k sits at
//                 buffer row k + 1: the three taps of conv_b are row-shifted views, start rows 0/1/2 - legal with
//                 base_offset = 0, tools/probe_desc_shift.cu)
//   P2 (conv_b)   A = H views, accumulator 2 = output rows m0 .. m0+127, of which 1..126 are valid
//   E2            + bias_b + x, x_new (fp32) and the activated fp16 plane of the next pair
//
// History of this kernel, all measured on the B200 (B = 32 x 10 s, ms per pair; the two launches it replaces take 2.49):
//   r1   one warp group for E1 and E2, one tile at a time                                            3.23   (serial latency chain)
//   r2a  one warp group per step, double-buffered H / accumulators, resident weights                 2.60
//   r2b  + fp32 stream of the stack instead of hi/lo planes (E2: 640 -> 450 instructions per tile)   2.33
//   r2c  16 E2 warps of 16 columns                                                                    2.72   (more, smaller LSU requests)
//   ncu on r2b/r2c: l1tex__data_pipe_lsu_wavefronts 84 % of peak - the LSU data pipe, fed by the LDG/STG of E2 and the
//   STS/LDS of its row-per-thread <-> row-major staging transposes, is the limiter (DRAM at 58-65 %).  Hence this version:
//   r2d  the residual tile arrives by TMA (SWIZZLE_128B, read conflict-free by the row's own thread), x_new is written
//        back IN PLACE and leaves by TMA store, as does the activated tile: no LDG / STG, no staging transposes.
//
//   r2e  three residual stages re-armed by the store warp, readiness-driven MMA issue order                 1.87   (10.9 GB = 12 B/element
//        at 5.8-6.0 TB/s: HBM-bound, only fewer bytes help)
//   r2f  MODE 2, the (a, r) stream of gemm.cuh: the residual is rebuilt from the activated plane (its TMA re-read is an L2 hit -
//        the centre tap has just fetched those rows) plus an fp16 correction plane, and x_new leaves as the same pair:
//        8 B/element, 1.51-1.58 ms per pair; the output warps' instruction stream is the limit now (FHADD adds, ptx.cuh)
//
// Warp roles (every wait is bounded, ptx.cuh):
//   warp 0       TMA producer: ring of three A tap slots (16 KB each); both weight matrices (2 x 3 x 8 KB) are loaded once and
//                stay resident
//   warp 1       MMA issuer, readiness driven: P2(j) as soon as H(j) is written, P1 taps as they land
//   warps 2-5    E1: accumulator 1 -> H
//   warps 6-13   E2: accumulator 2 + residual tile -> x_new in place + activated tile
//   warp 14      TMA stores of x_new / the activated tile and TMA loads of the residual tiles (three stages of 2 x 16 KB)
#include "gemm.cuh"
#include "ptx.cuh"

namespace vf {

namespace {
constexpr int PAIR_C = 64;
constexpr int PAIR_ROWS = 126;                 // valid output rows per tile
constexpr int PAIR_A_TAP = 128 * 128;          // one A box: 128 rows x 64 channels fp16
constexpr int PAIR_W_TAP = PAIR_C * 128;       // one weight tile: 64 output channels x 64 input channels fp16
constexpr int PAIR_H_BUF = 136 * 128;          // 130 rows used, rounded up to whole 1024-byte swizzle atoms
constexpr int PAIR_X_TILE = 128 * 128;         // residual / output half tile: 126 rows x 128 B (32 fp32 or 64 fp16 channels)
constexpr int PAIR_X_STAGE = 2 * PAIR_X_TILE;
constexpr int PAIR_E1_WARPS = 4, PAIR_E2_WARPS = 8;
constexpr int PAIR_E1_THREADS = 32 * PAIR_E1_WARPS, PAIR_E2_THREADS = 32 * PAIR_E2_WARPS;
constexpr int PAIR_THREADS = 64 + PAIR_E1_THREADS + PAIR_E2_THREADS + 32;
constexpr int PAIR_A_SLOTS = 3, PAIR_X_STAGES = 3;
constexpr int PAIR_SMEM = PAIR_A_SLOTS * PAIR_A_TAP + 6 * PAIR_W_TAP + PAIR_H_BUF + PAIR_X_STAGES * PAIR_X_STAGE + PAIR_X_TILE + 512 + 2 * PAIR_C * 4;

__device__ __forceinline__ void e2_bar_sync() { asm volatile("bar.sync 2, %0;" ::"r"(PAIR_E2_THREADS) : "memory"); }
}  // namespace

// MODE 0: residual in as hi/lo planes of x, out as fp32 (first pair of an fp32-stream stack); 1: fp32 in and out;
// 2: the (a, r) stream of gemm.cuh - residual rebuilt from the activated plane + the correction plane, both out as fp16
template <int MODE>
__global__ void __launch_bounds__(PAIR_THREADS, 1) pair_tc_kernel(const __grid_constant__ PairParams P) {
  constexpr bool F32_IN = MODE == 1, AR = MODE == 2;
  constexpr int C = PAIR_C;
  constexpr uint32_t IDESC = make_idesc_f16(GEMM_BM, C);
  constexpr uint32_t DHI = make_smem_desc_hi(128);

  // 226.8 of the 227 KB a CTA may have: the swizzled tiles need a 1024-byte aligned base, which the declaration requests
  // (no slack to align by hand); a misaligned base is reported instead of silently corrupting the swizzle
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* a_base = smem;                                   // [3] tap slots of 128 x 128 B
  uint8_t* w_base = a_base + PAIR_A_SLOTS * PAIR_A_TAP;     // [Wa tap 0..2][Wb tap 0..2], 8 KB each
  uint8_t* h_base = w_base + 6 * PAIR_W_TAP;                // 136 x 128 B
  uint8_t* x_base = h_base + PAIR_H_BUF;                    // [3 stages][2 half tiles] (fp32: channel halves; planes: hi, lo)
  uint8_t* act_base = x_base + PAIR_X_STAGES * PAIR_X_STAGE;   // activated output tile, 126 x 128 B
  uint64_t* bars = reinterpret_cast<uint64_t*>(act_base + PAIR_X_TILE);
  uint64_t* w_full = bars;            // [1]
  uint64_t* a_full = bars + 1;        // [3]
  uint64_t* a_empty = bars + 4;       // [3]
  uint64_t* acc1_full = bars + 7;     // [2]
  uint64_t* acc1_empty = bars + 9;    // [2]
  uint64_t* h_ready = bars + 11;      // [1]
  uint64_t* h_free = bars + 12;       // [1]
  uint64_t* acc2_full = bars + 13;    // [2]
  uint64_t* acc2_empty = bars + 15;   // [2]
  uint64_t* x_full = bars + 17;       // [3] residual stage loaded
  uint64_t* out_ready = bars + 20;    // [3] E2 has finished the stage and the activated tile
  uint64_t* act_free = bars + 23;     // [1] the activated tile has been read by its TMA store
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 26);
  float* s_bias_a = reinterpret_cast<float*>(bars + 32);   // [C] (16-byte aligned)
  float* s_bias_b = s_bias_a + C;                          // [C]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = P.n_img * P.tiles_per_img;
  const int n_local = total_tiles > (int)blockIdx.x ? (total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  constexpr int TMEM_COLS = 4 * C;               // accumulator 1 x 2 at columns 0 / C, accumulator 2 x 2 at 2C / 3C
  const bool want_f = P.out_f32 != 0;

  if (warp == 0 && lane == 0) {
    if (smem_u32(smem) & 1023u) atomicCAS(P.err, 0, ERR_PIPE_PRODUCER);     // see the declaration of smem
    mbar_init(w_full, 1);
    for (int i = 0; i < PAIR_A_SLOTS; ++i) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(acc1_full + i, 1); mbar_init(acc1_empty + i, PAIR_E1_THREADS);
      mbar_init(acc2_full + i, 1); mbar_init(acc2_empty + i, PAIR_E2_THREADS);
    }
    for (int i = 0; i < PAIR_X_STAGES; ++i) { mbar_init(x_full + i, 1); mbar_init(out_ready + i, PAIR_E2_THREADS); }
    mbar_init(h_ready, PAIR_E1_THREADS); mbar_init(h_free, 1);
    mbar_init(act_free, 1);
    fence_mbar_init();
    tma_prefetch_desc(&P.a_map);
    tma_prefetch_desc(&P.wa_map);
    tma_prefetch_desc(&P.wb_map);
    tma_prefetch_desc(&P.xin_map[0]);
    tma_prefetch_desc(&P.ao_map);
  }
  if (warp == 1) tmem_alloc_dyn(tmem_holder, TMEM_COLS);
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    s_bias_a[i] = __ldg(P.bias_a + i);
    s_bias_b[i] = __ldg(P.bias_b + i);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      mbar_expect_tx(w_full, 6 * PAIR_W_TAP);
      for (int t = 0; t < 3; ++t) {
        tma_load_2d(w_base + t * PAIR_W_TAP, &P.wa_map, w_full, t * C, 0);
        tma_load_2d(w_base + (3 + t) * PAIR_W_TAP, &P.wb_map, w_full, t * C, 0);
      }
      bool ok = true;
      uint32_t sl = 0, ph = 0;        // A tap slot and its phase bit
      for (int j = 0; j < n_local && ok; ++j) {
        const int tile = blockIdx.x + j * gridDim.x;
        const int img = (int)fast_div_pair((uint32_t)tile, (uint32_t)P.tiles_per_img, P.magic_t);
        const int m0 = (tile - img * P.tiles_per_img) * PAIR_ROWS - 1;
        for (int t = 0; t < 3; ++t) {
          if (!mbar_wait(a_empty + sl, ph ^ 1u, P.err, ERR_PIPE_PRODUCER)) { ok = false; break; }
          mbar_expect_tx(a_full + sl, PAIR_A_TAP);
          tma_load_3d(a_base + sl * PAIR_A_TAP, &P.a_map, a_full + sl, 0, m0 + (t - 1) * P.dil, img);
          if (++sl == PAIR_A_SLOTS) { sl = 0; ph ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      const uint32_t da0 = make_smem_desc_lo(smem_u32(a_base));
      const uint32_t dw0 = make_smem_desc_lo(smem_u32(w_base));
      const uint32_t dh = make_smem_desc_lo(smem_u32(h_base));
      bool ok = mbar_wait(w_full, 0, P.err, ERR_PIPE_MMA);
      // Readiness-driven issue order: P2(j) goes as soon as H(j) is written, P1 taps go as they land - so a late tap of
      // tile j+1 never holds back the accumulator the output warps are waiting for (ncu: 20 % of all samples there when
      // P1(j+1) was issued unconditionally before P2(j)).
      int j1 = 0, t1 = 0, j2 = 0;     // next P1 tile / tap, next P2 tile
      uint32_t sl = 0, ph = 0, spins = 0;
      while (j2 < n_local && ok) {
        bool progressed = false;
        if (j2 < j1) {                // ---- P2(j2): conv_b on H into accumulator 2[b]
          const int b = j2 & 1;
          if (mbar_try_wait(h_ready, j2 & 1) && mbar_try_wait(acc2_empty + b, ((j2 >> 1) & 1) ^ 1)) {
            tc_fence_after();
            const uint32_t d = tmem_base + 2 * C + b * C;
#pragma unroll
            for (int t = 0; t < 3; ++t)
#pragma unroll
              for (int k = 0; k < 4; ++k)      // view of tap t starts at buffer row t
                umma_f16_lo(d, dh + t * (128 >> 4) + 2 * k, dw0 + (3 + t) * (PAIR_W_TAP >> 4) + 2 * k, DHI, IDESC, (t | k) ? 1u : 0u);
            umma_commit(acc2_full + b);
            umma_commit(h_free);
            ++j2;
            progressed = true;
          }
        }
        if (!progressed && j1 < n_local && j1 < j2 + 2) {      // ---- one tap of P1(j1): conv_a into accumulator 1[b]
          const int b = j1 & 1;
          if ((t1 > 0 || mbar_try_wait(acc1_empty + b, ((j1 >> 1) & 1) ^ 1)) && mbar_try_wait(a_full + sl, ph)) {
            tc_fence_after();
            const uint32_t d = tmem_base + b * C;
            const uint32_t da = da0 + sl * (PAIR_A_TAP >> 4);
            const uint32_t dw = dw0 + t1 * (PAIR_W_TAP >> 4);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_lo(d, da + 2 * k, dw + 2 * k, DHI, IDESC, (t1 | k) ? 1u : 0u);
            umma_commit(a_empty + sl);
            if (++sl == PAIR_A_SLOTS) { sl = 0; ph ^= 1u; }
            if (++t1 == 3) { umma_commit(acc1_full + b); t1 = 0; ++j1; }
            progressed = true;
          }
        }
        if (progressed) spins = 0;
        else if (++spins > (1u << 24)) { if (P.err) atomicCAS(P.err, 0, ERR_PIPE_MMA); ok = false; }
      }
    }
    __syncwarp();
  } else if (warp < 2 + PAIR_E1_WARPS) {
    // ------------------------------------------------------------------ E1: accumulator 1 -> H
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const uint32_t lane_bits = static_cast<uint32_t>(q * 32) << 16;
    const int jrow = q * 32 + lane;            // this thread's accumulator row = h row
    const int brow = jrow + 1;                 // its row in the H buffer
    const float slope_h = P.slope_h;
    float amax = 0.f;
    bool ok = true;
    // buffer rows 0 and 129 are read by the first / last tap of accumulator rows 0 and 127 (never stored, but they must
    // stay finite for the overflow guard): zero them once, E1 only ever writes rows 1..128
    if (warp == 2 && lane < 8) {
      *reinterpret_cast<uint4*>(h_base + lane * 16) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(h_base + 129 * 128 + lane * 16) = make_uint4(0, 0, 0, 0);
    }
    uint8_t* rowp = h_base + (size_t)brow * 128;
    for (int j = 0; j < n_local && ok; ++j) {
      const int tile = blockIdx.x + j * gridDim.x;
      const int img = (int)fast_div_pair((uint32_t)tile, (uint32_t)P.tiles_per_img, P.magic_t);
      const int m0 = (tile - img * P.tiles_per_img) * PAIR_ROWS - 1;
      const int b = j & 1;
      const int t = m0 + jrow;
      const int len = P.vl_len ? __ldg(P.vl_len + (size_t)img * P.vl_stride) : P.L;     // varlen batch: this clip's length
      const bool in_clip = t >= 0 && t < len;
      if (!mbar_wait(acc1_full + b, (j >> 1) & 1, P.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }
      tc_fence_after();
      if (!mbar_wait(h_free, (j & 1) ^ 1, P.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }      // P2(j-1) has read H
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {              // two passes of 32 columns
        float v[32];
        tmem_ld_32x32(tmem_base + lane_bits + b * C + c * 32, v);
        if (c == 1) {
          tc_fence_before();
          mbar_arrive(acc1_empty + b);           // accumulator 1[b] is in registers: P1(j+2) may start
        }
        const float4* bp = reinterpret_cast<const float4*>(s_bias_a + c * 32);
        uint32_t hw[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 b4 = bp[i];
          float a0 = v[4 * i] + b4.x, a1 = v[4 * i + 1] + b4.y, a2 = v[4 * i + 2] + b4.z, a3 = v[4 * i + 3] + b4.w;
          a0 = fmaxf(a0, a0 * slope_h); a1 = fmaxf(a1, a1 * slope_h); a2 = fmaxf(a2, a2 * slope_h); a3 = fmaxf(a3, a3 * slope_h);
          if (!in_clip) { a0 = a1 = a2 = a3 = 0.f; }     // conv_b pads h with zeros outside the clip
          amax = fmaxf(amax, fmaxf(fmaxf(fabsf(a0), fabsf(a1)), fmaxf(fabsf(a2), fabsf(a3))));
          const __half2 p0 = __floats2half2_rn(a0, a1), p1 = __floats2half2_rn(a2, a3);
          hw[2 * i] = *reinterpret_cast<const uint32_t*>(&p0);
          hw[2 * i + 1] = *reinterpret_cast<const uint32_t*>(&p1);
        }
        // K-major SWIZZLE_128B image: 16-byte chunk index XOR (buffer row & 7)
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<uint4*>(rowp + (((c * 4 + i) ^ (brow & 7)) << 4)) = make_uint4(hw[4 * i], hw[4 * i + 1], hw[4 * i + 2], hw[4 * i + 3]);
      }
      fence_proxy_async();                       // generic-proxy writes -> visible to the tensor core's async proxy
      mbar_arrive(h_ready);
    }
    if (!(amax <= 65504.f) && P.err) atomicCAS(P.err, 0, ERR_FP16_OVERFLOW);
  } else if (warp < 2 + PAIR_E1_WARPS + PAIR_E2_WARPS) {
    // ------------------------------------------------------------------ E2: accumulator 2 + bias_b + x -> x_new (in place), activated tile
    const int ew = warp - (2 + PAIR_E1_WARPS);
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int half = ew >> 2;                  // which 32-column chunk this warp takes (two warps share a lane quarter)
    const uint32_t lane_bits = static_cast<uint32_t>(q * 32) << 16;
    const int jrow = q * 32 + lane;            // this thread's accumulator row
    const bool row_valid = jrow >= 1 && jrow <= PAIR_ROWS;      // accumulator rows 0 and 127 are halo rows
    const int xrow = row_valid ? jrow - 1 : 0; // its row in the residual / output tiles
    const uint32_t sw = (uint32_t)(xrow & 7);  // SWIZZLE_128B: 16-byte chunk index XOR (row & 7)
    const float slope_out = P.slope_out;
    const uint32_t ar_in = P.ar_in, ar_out = P.ar_out;
    float amax = 0.f;
    bool ok = true;
    uint8_t* act_row = act_base + (size_t)xrow * 128;
    int s = 0;                                 // residual stage j % 3 and its phase bit
    uint32_t sph = 0;
    for (int j = 0; j < n_local && ok; ++j) {
      const int b = j & 1;
      const uint32_t pj = (j >> 1) & 1;
      uint8_t* xs = x_base + s * PAIR_X_STAGE;
      if (!mbar_wait(x_full + s, sph, P.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }
      if (!mbar_wait(acc2_full + b, pj, P.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }
      tc_fence_after();
      float v[32];
      tmem_ld_32x32(tmem_base + lane_bits + 2 * C + b * C + half * 32, v);
      tc_fence_before();
      mbar_arrive(acc2_empty + b);
      const float4* bp = reinterpret_cast<const float4*>(s_bias_b + half * 32);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b4 = bp[i];
        v[4 * i] += b4.x; v[4 * i + 1] += b4.y; v[4 * i + 2] += b4.z; v[4 * i + 3] += b4.w;
      }
      if (F32_IN) {
        if (row_valid) {                       // this thread's 32 fp32 channels: the whole 128-byte row of half tile `half`
          const uint8_t* rp = xs + half * PAIR_X_TILE + (size_t)xrow * 128;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 x = *reinterpret_cast<const float4*>(rp + (((uint32_t)i ^ sw) << 4));
            v[4 * i] += x.x; v[4 * i + 1] += x.y; v[4 * i + 2] += x.z; v[4 * i + 3] += x.w;
          }
        }
      } else {
        if (row_valid) {                       // 32 of the 64 fp16 channels of the hi and of the lo tile
          const uint8_t* rh = xs + (size_t)xrow * 128;
          const uint8_t* rl = rh + PAIR_X_TILE;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 yh = *reinterpret_cast<const uint4*>(rh + (((uint32_t)(half * 4 + i) ^ sw) << 4));
            const uint4 yl = *reinterpret_cast<const uint4*>(rl + (((uint32_t)(half * 4 + i) ^ sw) << 4));
            const __half2* ph2 = reinterpret_cast<const __half2*>(&yh);
            const __half2* pl2 = reinterpret_cast<const __half2*>(&yl);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              add_planes(v[8 * i + 2 * k], v[8 * i + 2 * k + 1], reinterpret_cast<const uint32_t*>(ph2)[k], reinterpret_cast<const uint32_t*>(pl2)[k], AR ? ar_in : 0u);
          }
        }
        if (!AR) e2_bar_sync();                // the fp32 result overwrites the plane tiles other warps still read
      }
      if (P.vl_len) {                          // varlen batch: rows past this clip leave as zeros (x_new and the activated tile)
        const int tile = blockIdx.x + j * gridDim.x;
        const int img = (int)fast_div_pair((uint32_t)tile, (uint32_t)P.tiles_per_img, P.magic_t);
        const int t = (tile - img * P.tiles_per_img) * PAIR_ROWS + xrow;
        if (t >= __ldg(P.vl_len + (size_t)img * P.vl_stride)) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
      }
      if (want_f && row_valid) {               // x_new in place: fp32 half tile `half`
        uint8_t* rp = xs + half * PAIR_X_TILE + (size_t)xrow * 128;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<float4*>(rp + (((uint32_t)i ^ sw) << 4)) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      uint32_t hi[16];
      if (AR && ar_out) {                      // x_new leaves as (a, r): the correction plane replaces the r tile in place - each
        uint32_t lo[16];                       // thread rewrites exactly the 16-byte chunks it has just read
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float v0 = v[2 * i], v1 = v[2 * i + 1];
          amax = fmaxf(amax, fmaxf(fabsf(v0), fabsf(v1)));   // |x| bounds |a| and keeps U(a) in range
          ar_split(v0, v1, fmaxf(v0, v0 * slope_out), fmaxf(v1, v1 * slope_out), ar_out, hi[i], lo[i]);
        }
        if (row_valid) {
          uint8_t* rl = xs + PAIR_X_TILE + (size_t)xrow * 128;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            *reinterpret_cast<uint4*>(rl + (((uint32_t)(half * 4 + i) ^ sw) << 4)) = make_uint4(lo[4 * i], lo[4 * i + 1], lo[4 * i + 2], lo[4 * i + 3]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float a0 = fmaxf(v[2 * i], v[2 * i] * slope_out), a1 = fmaxf(v[2 * i + 1], v[2 * i + 1] * slope_out);
          amax = fmaxf(amax, fmaxf(fabsf(a0), fabsf(a1)));     // every row is finite (H border rows are zeroed)
          const __half2 hh = __floats2half2_rn(a0, a1);
          hi[i] = *reinterpret_cast<const uint32_t*>(&hh);
        }
      }
      if (!mbar_wait(act_free, (j & 1) ^ 1, P.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }    // store (j-1) has read the tile
      if (row_valid) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<uint4*>(act_row + (((uint32_t)(half * 4 + i) ^ sw) << 4)) = make_uint4(hi[4 * i], hi[4 * i + 1], hi[4 * i + 2], hi[4 * i + 3]);
      }
      fence_proxy_async();                     // generic-proxy writes -> visible to the TMA store
      mbar_arrive(out_ready + s);
      if (++s == PAIR_X_STAGES) { s = 0; sph ^= 1u; }
    }
    if (!(amax <= 65504.f) && P.err) atomicCAS(P.err, 0, ERR_FP16_OVERFLOW);
  } else {
    // ------------------------------------------------------------------ residual / output warp: the residual tiles arrive and
    // x_new / the activated tile leave by TMA.  The thread that sees a stage's store complete re-arms the stage itself (no
    // hand-off to the producer); three stages cover the HBM round trip at ~1.5 us per tile.
    if (elect_one()) {
      auto load_x = [&](int jj, int st) {       // residual tile of rows t0 .. t0+125 (rows past the clip are zero filled;
        const int tile = blockIdx.x + jj * gridDim.x;      // they are clipped again on the way out)
        const int img = (int)fast_div_pair((uint32_t)tile, (uint32_t)P.tiles_per_img, P.magic_t);
        const int t0 = (tile - img * P.tiles_per_img) * PAIR_ROWS;
        uint8_t* xs = x_base + st * PAIR_X_STAGE;
        mbar_expect_tx(x_full + st, 2 * PAIR_ROWS * 128);
        if (F32_IN) {
          tma_load_3d(xs, &P.xin_map[0], x_full + st, 0, t0, img);                    // channels 0..31
          tma_load_3d(xs + PAIR_X_TILE, &P.xin_map[0], x_full + st, 32, t0, img);     // channels 32..63
        } else {
          tma_load_3d(xs, &P.xin_map[0], x_full + st, 0, t0, img);                    // hi plane
          tma_load_3d(xs + PAIR_X_TILE, &P.xin_map[1], x_full + st, 0, t0, img);      // lo plane
        }
      };
      for (int j = 0; j < PAIR_X_STAGES && j < n_local; ++j) load_x(j, j);
      bool ok = true;
      int s = 0;
      uint32_t sph = 0;
      for (int j = 0; j < n_local && ok; ++j) {
        const int tile = blockIdx.x + j * gridDim.x;
        const int img = (int)fast_div_pair((uint32_t)tile, (uint32_t)P.tiles_per_img, P.magic_t);
        const int t0 = (tile - img * P.tiles_per_img) * PAIR_ROWS;
        if (!mbar_wait(out_ready + s, sph, P.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }
        const uint8_t* xs = x_base + s * PAIR_X_STAGE;
        if (AR) {
          if (P.ar_out) tma_store_3d(&P.xo_map, xs + PAIR_X_TILE, 0, t0, img);      // correction plane, 64 fp16 channels
        } else if (want_f) {                   // rows past the clip are clipped by the tensor map
          tma_store_3d(&P.xo_map, xs, 0, t0, img);
          tma_store_3d(&P.xo_map, xs + PAIR_X_TILE, 32, t0, img);
        }
        tma_store_3d(&P.ao_map, act_base, 0, P.out_row0 + t0, img);
        tma_store_commit();
        tma_store_wait_read();                 // shared memory has been read: the buffers may be reused
        mbar_arrive(act_free);
        if (j + PAIR_X_STAGES < n_local) load_x(j + PAIR_X_STAGES, s);
        if (++s == PAIR_X_STAGES) { s = 0; sph ^= 1u; }
      }
      tma_store_wait_all();                    // global writes complete before the kernel ends
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_dyn(tmem_base, TMEM_COLS);
  }
}

size_t pair_tc_smem_bytes(int C, int /*stages*/) { return C == PAIR_C ? (size_t)PAIR_SMEM : 0; }

template <int MODE>
static cudaError_t launch_pair_t(const PairParams& p, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(pair_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  pair_tc_kernel<MODE><<<p.grid, PAIR_THREADS, PAIR_SMEM, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_pair_tc(const PairParams& p, cudaStream_t stream) {
  if (p.C != PAIR_C) return cudaErrorInvalidValue;
  if (p.ar_in) return launch_pair_t<2>(p, stream);
  return p.in_f32 ? launch_pair_t<1>(p, stream) : launch_pair_t<0>(p, stream);
}

}  // namespace vf
