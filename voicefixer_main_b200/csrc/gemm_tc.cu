// tcgen05 implementation of the flat-shift multi-tap GEMM (see gemm.cuh).
//
// Persistent, warp-specialised: each CTA loops over 128 x BN output tiles (tile = blockIdx.x + i * gridDim.x,
// N tiles of one M tile adjacent so co-running CTAs share the A rows in L2).
//   warp 0     : TMA producer - streams A (activation rows, shifted per tap; one 130..144-row "halo" box serves up to
//                three row-adjacent taps) and B (packed weights) tiles into a `stages`-deep shared-memory ring that
//                runs ahead across tile boundaries (SWIZZLE_128B rows for BK = 64, SWIZZLE_64B for BK = 32); in
//                3-term mode the hi and lo planes of an operand arrive in one 4-D / 3-D box
//   warp 1     : TMEM owner + single-thread tcgen05.mma issuer; 2 or 4 accumulator buffers rotate in TMEM
//   warps 2..  : epilogue (4 or 8 warps; one TMEM lane = output row per thread, two warps share a lane quarter
//                and split the column chunks)
// Both issue loops are run by ONE elected thread each and read the flattened per-chunk table the CTA builds in
// shared memory at start-up (ChunkDesc); their per-chunk instruction count bounds every small-tile layer, which
// is what the table, the 32-bit descriptor arithmetic and the specialised issue bodies (issue_mmas) are for.
//
// Accumulation precision.  The tensor core adds into its fp32 accumulator with truncation, so one long chain
// of K/16 MMAs drifts by ~0.5 ulp per instruction (measured 2e-4 on the UNet log-mel with one accumulator per
// tile).  In 3-term mode the K loop is therefore cut into segments of 24 K steps that rotate through the TMEM
// accumulator buffers; the epilogue warps add each finished segment into registers in fp32 round-to-nearest
// ("promotion") while the tensor core already works on the next one.  Each buffer is [main | correction]: the
// two small correction products (hi*lo, lo*hi) never mix into the main chain.  The same ping-pong is the tile double buffering
// of the 1-term mode (one segment per tile): tile i+1 accumulates while tile i drains.
//
// Epilogue I/O.  A thread owns a row, but global stores are issued row-major by the whole warp: values are
// transposed through a swizzled shared-memory staging tile so every LDG/STG instruction touches whole
// 64/128-byte row segments.  Per-tile constants (bias, BN scale/shift, head weights) live in shared memory.
#include "gemm.cuh"
#include "ptx.cuh"

namespace vf {

namespace {

constexpr int kRowValid = 1, kRowPad = 2;

// A clip's valid output rows (varlen batches, GemmEpilogue::vl_rows), read where it is used: as a volatile load it is not
// hoisted or kept across the epilogue's tile loop (the two-CTA variants have no register to spare).
__device__ __forceinline__ int ld_row_limit(const int* p) {
  int v;
  asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

struct RowInfo {        // published per epilogue thread for its own row, read by the lanes that store that row
  uint32_t orow;        // output row index (already includes image base / row0 / phase mapping)
  uint32_t flags;
};

// Staging tiles: 32 rows x 128 B (fp32 x 32 columns), 16-byte column index XOR (row & 7); and 32 rows x 64 B
// (fp16 x 32 columns), 16-byte column index XOR ((row >> 1) & 3).  See the SO_* / SR_* macros in the epilogue.

__device__ __forceinline__ void epi_bar_sync(int nthreads) {
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// One K chunk (= one ring slot) of a tile, as the two issue threads need it: the tap structure is flattened once per
// CTA into this table, so the per-chunk work of the producer / MMA loops is one 16-byte shared-memory load instead
// of a walk over the tap list in constant memory.
struct ChunkDesc {
  int a_c;          // channel coordinate of the A box
  int a_off;        // row offset of the A box relative to the tile's first row
  uint32_t kk;      // K coordinate of the first weight tile | kstride << 16 (stride between the weight tiles of a group)
  uint32_t flags;   // bit 0 src, bit 1 lo plane of A is needed, bits 2-3 g, bit 4 both, bits 5-6 / 7-8 / 9-10 row shifts
};

// Tile coordinates without loop-carried state: tile = (img * m_tiles + mi) * n_tiles + nt, decoded per tile with the
// host's multiply-high magic numbers (gemm_tc_magic): a handful of instructions instead of two integer divisions,
// and no registers held across the tile loop (the hi-only epilogue runs at a 96-register budget).
__device__ __forceinline__ uint32_t fast_div(uint32_t n, uint32_t d, uint32_t magic) {
  if (magic == 0u) return n;                    // d == 1
  if (magic == 0xffffffffu) return n / d;       // range too large for the 32-bit magic (host decides)
  return __umulhi(n, magic);
}
struct TileCoord {
  int nt, mi, img;
  __device__ __forceinline__ TileCoord(uint32_t tile, const GemmTcParams& P, int n_tiles, int m_tiles) {
    const uint32_t mt = fast_div(tile, (uint32_t)n_tiles, P.magic_n);
    nt = (int)(tile - mt * (uint32_t)n_tiles);
    const uint32_t im = fast_div(mt, (uint32_t)m_tiles, P.magic_m);
    img = (int)im;
    mi = (int)(mt - im * (uint32_t)m_tiles);
  }
};

}  // namespace

// Epilogue helpers: 32 fp32 values of one row -> packed half2 hi (and lo) words.
__device__ __forceinline__ void pack_hi(const float (&v)[32], uint32_t (&hi)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    hi[i] = *reinterpret_cast<const uint32_t*>(&h);
  }
}
__device__ __forceinline__ void pack_hi_lo(const float (&v)[32], uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    hi[i] = *reinterpret_cast<const uint32_t*>(&h);
    lo[i] = residual_h2(v[2 * i], v[2 * i + 1], hi[i]);      // one FHADD per element instead of a conversion and an FSUB
  }
}

// Eight columns (v[8 i .. 8 i + 7]) -> one 16-byte word of the hi plane (and of the lo plane): packing straight into the
// staging tiles keeps 8 instead of 32 packed words live - the two- and three-CTA variants have no registers to spare.
template <bool TWO>
__device__ __forceinline__ void pack8(const float (&v)[32], const int i, uint4& h, uint4& l) {
  uint32_t hw[4], lw[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const __half2 h2 = __floats2half2_rn(v[8 * i + 2 * k], v[8 * i + 2 * k + 1]);
    hw[k] = *reinterpret_cast<const uint32_t*>(&h2);
    if (TWO) lw[k] = residual_h2(v[8 * i + 2 * k], v[8 * i + 2 * k + 1], hw[k]);
  }
  h = make_uint4(hw[0], hw[1], hw[2], hw[3]);
  if (TWO) l = make_uint4(lw[0], lw[1], lw[2], lw[3]);
}

// The MMAs of one K chunk: G taps (row shifts packed 2 bits each in `shifts`) x BK/16 K steps; 3-term mode adds
// lo(A) x hi(B) into the correction half, BOTH (hi-only identity tap) contracts the lo plane into the same accumulator.
template <int BN, int BK, bool THREE, int G, bool BOTH>
__device__ __forceinline__ void issue_mmas(uint32_t d_main, uint32_t da_hi0, uint32_t da_lo0, uint32_t db00, uint32_t shifts,
                                           uint32_t started) {
  constexpr uint32_t idesc = make_idesc_f16(GEMM_BM, BN);
  constexpr uint32_t idesc2 = make_idesc_f16(GEMM_BM, THREE ? 2 * BN : BN);   // hi x [hi | lo]
  constexpr uint32_t dhi = make_smem_desc_hi(BK * 2);
  constexpr uint32_t ROW_UNITS = BK * 2 / 16;
  constexpr uint32_t B_SLOT_UNITS = (THREE ? 2 : 1) * BN * BK * 2 / 16;
  // the tap loop is unrolled where the kernel's register budget has room (narrow tiles): every rolled iteration costs
  // the single issue thread ~25 instructions of loop and shift bookkeeping per 2-4 MMAs
  constexpr int UNROLL_G = BN <= 64 ? G : 1;
#pragma unroll UNROLL_G
  for (int gi = 0; gi < G; ++gi) {
    const uint32_t sh = G == 1 ? 0u : ((shifts >> (2 * gi)) & 3u) * ROW_UNITS;
    const uint32_t db0 = db00 + gi * B_SLOT_UNITS;
#pragma unroll
    for (int k = 0; k < BK / 16; ++k) {
      umma_f16_lo(d_main, da_hi0 + sh + 2 * k, db0 + 2 * k, dhi, idesc2, (gi == 0 && k == 0) ? started : 1u);
      if (THREE) umma_f16_lo(d_main + BN, da_lo0 + sh + 2 * k, db0 + 2 * k, dhi, idesc, 1u);
      else if (BOTH) umma_f16_lo(d_main, da_lo0 + sh + 2 * k, db0 + 2 * k, dhi, idesc, 1u);
    }
  }
}

// MINB = co-resident CTAs per SM the register allocation is budgeted for (the engine picks the variant that
// matches the occupancy shared memory allows: fewer CTAs -> more registers -> no spills in the 3-term epilogue).
template <int BN, int BK, int EPI_WARPS, bool THREE, int MINB>
__global__ void __launch_bounds__(64 + 32 * EPI_WARPS, MINB)
    gemm_tc_kernel(const __grid_constant__ GemmTcParams P) {
  constexpr int B_BYTES = BN * BK * 2;
  constexpr int ROW_BYTES = BK * 2;
  constexpr int EPI_THREADS = 32 * EPI_WARPS;
  constexpr int CHUNK_STEP = EPI_WARPS / 4;             // column chunks are dealt to the warps of a lane quarter
  constexpr int NJ = (BN / 32 + CHUNK_STEP - 1) / CHUNK_STEP;   // chunks per epilogue warp
  constexpr bool PREFETCH = !THREE && MINB == 1;        // residual planes one chunk ahead (needs 32 registers)

  extern __shared__ __align__(16) uint8_t smem_raw[];
  // 1024-byte alignment by offset arithmetic (keeps the pointer in the shared address space: LDS/STS, not generic)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int stages = P.stages;
  const int planes_a = P.planes_a;                      // 2 when any tap contracts the lo plane of A
  constexpr int B_SLOT = (THREE ? 2 : 1) * B_BYTES;      // [B_hi][B_lo] of one tap, contiguous
  const int a_box_bytes = P.a_box_rows * ROW_BYTES;     // bytes one A TMA box delivers
  const int a_slot = (a_box_bytes + 1023) & ~1023;      // halo rows spill into one more swizzle atom
  const int off_b = planes_a * a_slot;
  const int stage_bytes = off_b + P.gmax * B_SLOT;
  uint8_t* stg_base = smem + (size_t)stages * stage_bytes;          // EPI_WARPS x 4 KB staging
  uint8_t* rstg_base = stg_base + EPI_WARPS * 4096;                  // resid_tma: EPI_WARPS x 4 KB residual tiles (TMA destination)
  uint8_t* tail = rstg_base + (size_t)P.resid_tma * EPI_WARPS * 4096;  // P.resid_tma = tiles in flight per warp (0, 1 or 2)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* seg_full_bar = empty_bar + stages;           // [nbuf <= 4] accumulator buffer holds a finished segment
  uint64_t* seg_empty_bar = seg_full_bar + 4;            // [nbuf <= 4] ... has been drained by every epilogue thread
  uint64_t* resid_bar = seg_empty_bar + 4;               // [8][2] per epilogue warp and ring slot: the residual tile has landed
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(resid_bar + 16);   // keep the float arrays 16-byte aligned
  float* s_bias = reinterpret_cast<float*>(tmem_holder + 4);   // [BN]  (16-byte aligned: float4 reads)
  float* s_scale = s_bias + BN;                                // [BN]
  float* s_shift = s_scale + BN;                                // [BN]
  float* s_head = s_shift + BN;                                // [32]
  RowInfo* s_rows = reinterpret_cast<RowInfo*>(s_head + 32);   // [EPI_WARPS * 32]
  ChunkDesc* s_tab = reinterpret_cast<ChunkDesc*>(s_rows + EPI_WARPS * 32);   // [tile_chunks], 16-byte aligned

  const GemmProblem& pr = P.prob;
  const GemmEpilogue& e = pr.epi;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles = pr.N / BN;
  const int total_tiles = pr.n_img * pr.m_tiles * n_tiles;
  const int tile_chunks = P.tile_chunks;                 // K chunks per tile
  const int seg_chunks = THREE ? P.seg_chunks : tile_chunks;   // K chunks per accumulation segment
  const int nbuf_log = P.nbuf_log, nbuf_mask = (1 << nbuf_log) - 1;   // 2 or 4 accumulator buffers rotate in TMEM
  // TMEM columns: 2 or 4 accumulator buffers rotate (as many as 512 columns / co-resident CTAs allow: the MMA
  // thread can run that many segments ahead of the epilogue warps).  1-term: M0 [0,BN) M1 [BN,2BN) ...  3-term: [M0|C0] [M1|C1] ..., each
  // 2*BN wide: hi*hi and hi*lo come from ONE MMA of width 2*BN against the stacked [B_hi; B_lo] tile (A_hi is read
  // from shared memory once instead of twice), lo*hi is a second MMA of width BN into the C half.

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    for (int i = 0; i <= nbuf_mask; ++i) {
      mbar_init(seg_full_bar + i, 1);
      mbar_init(seg_empty_bar + i, EPI_THREADS);
    }
    for (int i = 0; i < 16; ++i) mbar_init(resid_bar + i, 1);
    fence_mbar_init();
    tma_prefetch_desc(&P.a_hi[0]);
    tma_prefetch_desc(&P.b_hi);
    if (!THREE) tma_prefetch_desc(&P.a_lo[0]);
  }
  if (warp == 1) tmem_alloc_dyn(tmem_holder, P.tmem_cols);
  for (int ci = threadIdx.x; ci < tile_chunks; ci += blockDim.x) {   // flatten taps x K chunks (see ChunkDesc)
    int t = 0, first = 0;
    for (; t < pr.ntaps - 1; ++t) {
      const int n = pr.taps[t].nch / BK;
      if (ci < first + n) break;
      first += n;
    }
    const GemmTap& tap = pr.taps[t];
    const int c = (ci - first) * BK;
    ChunkDesc cd;
    cd.a_c = tap.c_off + c;
    cd.a_off = tap.a_off;
    cd.kk = (uint32_t)(tap.k_off + c) | ((uint32_t)tap.kstride << 16);
    cd.flags = (uint32_t)(tap.src & 1) | ((THREE || tap.both) ? 2u : 0u) | ((uint32_t)tap.g << 2) | (tap.both ? 16u : 0u) |
               ((uint32_t)tap.shift[0] << 5) | ((uint32_t)tap.shift[1] << 7) | ((uint32_t)tap.shift[2] << 9);
    s_tab[ci] = cd;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // Each issue warp elects ONE thread (elect.sync) that runs the whole loop.  Running it under `if (lane == 0)`
  // instead makes the compiler wrap every UTMALDG / UTCHMMA / UTCBAR in an ELECT + BRA.U.ANY loop (it cannot prove a
  // single active thread), which measured ~1300 cycles per K chunk on the issue path (ncu, voc.res3.1.a) - the
  // bottleneck of small-chunk layers.  Measured alternatives: all 32 lanes polling (small-chunk layers -17 %, but
  // MMA-bound layers +8 %), lane-0 polling with a shuffle broadcast (+12 % overall).
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {      // ONE elected thread runs the whole loop (see above)
    int s = 0;              // ring slot and its phase bit advance by increment: no division on the issue path
    uint32_t ph = 0;
    bool ok = true;
    for (int tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
      const TileCoord it((uint32_t)tile, P, n_tiles, pr.m_tiles);
      const int img = it.img;
      const int m0 = it.mi * GEMM_BM;
      const int n0 = it.nt * BN;
      ChunkDesc cd = s_tab[0];
      for (int ci = 0; ci < tile_chunks; ++ci) {
        const ChunkDesc cur = cd;
        cd = s_tab[ci + 1 < tile_chunks ? ci + 1 : 0];     // next entry: its load latency hides behind the wait
        if (!mbar_wait(empty_bar + s, ph ^ 1, e.err, ERR_PIPE_PRODUCER)) { ok = false; break; }
        const bool a_lo = (cur.flags & 2u) != 0;
        const int src = cur.flags & 1u;
        const int tg = (cur.flags >> 2) & 3u;
        uint8_t* st = smem + (size_t)s * stage_bytes;
        mbar_expect_tx(full_bar + s, (a_lo ? 2u : 1u) * a_box_bytes + tg * B_SLOT);
        const int k0 = cur.kk & 0xffffu, ks = cur.kk >> 16;
        if (THREE) {      // hi and lo planes of A in one 4-D box, [B_hi][B_lo] of a tap in one 3-D box (a_slot == box bytes)
          tma_load_4d(st, &P.a_hi[src], full_bar + s, cur.a_c, m0 + cur.a_off, img, 0);
          for (int gi = 0; gi < tg; ++gi) tma_load_3d(st + off_b + gi * B_SLOT, &P.b_hi, full_bar + s, k0 + gi * ks, n0, 0);
        } else {
          tma_load_3d(st, &P.a_hi[src], full_bar + s, cur.a_c, m0 + cur.a_off, img);
          if (a_lo) tma_load_3d(st + a_slot, &P.a_lo[src], full_bar + s, cur.a_c, m0 + cur.a_off, img);
          for (int gi = 0; gi < tg; ++gi) tma_load_2d(st + off_b + gi * B_SLOT, &P.b_hi, full_bar + s, k0 + gi * ks, n0);
        }
        if (++s == stages) { s = 0; ph ^= 1; }
      }
    }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
    constexpr int ACC_W = THREE ? 2 * BN : BN;
    int s = 0, g = 0;               // smem ring slot, accumulation-segment counter
    uint32_t ph = 0;                // phase bit of the ring slot
    bool ok = true;
    for (int tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
      uint32_t d_main = 0, started = 0;
      int left_in_seg = 0, buf = 0;                      // countdown: no division on the issue path
      if (!THREE) {                                      // hi-only: one segment per tile, opened here, closed after the loop
        buf = g & nbuf_mask;
        if (!mbar_wait(seg_empty_bar + buf, ((g >> nbuf_log) & 1) ^ 1, e.err, ERR_PIPE_MMA)) { ok = false; break; }
        d_main = tmem_base + buf * ACC_W;
      }
      uint32_t fl = s_tab[0].flags;
      for (int ci = 0; ci < tile_chunks; ++ci) {
        const uint32_t cur = fl;
        fl = s_tab[ci + 1 < tile_chunks ? ci + 1 : 0].flags;
        if (THREE && left_in_seg == 0) {       // open a segment: its accumulator buffer must have been drained
          left_in_seg = min(seg_chunks, tile_chunks - ci);
          buf = g & nbuf_mask;
          if (!mbar_wait(seg_empty_bar + buf, ((g >> nbuf_log) & 1) ^ 1, e.err, ERR_PIPE_MMA)) { ok = false; break; }
          d_main = tmem_base + buf * ACC_W;
          started = 0;
        }
        if (!mbar_wait(full_bar + s, ph, e.err, ERR_PIPE_MMA)) { ok = false; break; }
        tc_fence_after();
        const bool close_seg = THREE ? (--left_in_seg == 0) : (ci + 1 == tile_chunks);
        // descriptors differ only in the 14-bit start-address field of their low word (units of 16 B): +2 per
        // 32-byte K step, +ROW_BYTES/16 per row of halo shift, +B_SLOT/16 per weight tile of a tap group
        const uint32_t da_hi0 = make_smem_desc_lo(smem_u32(smem + (size_t)s * stage_bytes));
        const uint32_t da_lo0 = da_hi0 + (uint32_t)(a_slot >> 4);
        const uint32_t db00 = da_hi0 + (uint32_t)(off_b >> 4);                 // spans [B_hi; B_lo]
        // one straight-line body per chunk kind (the generic loop with its per-MMA predication costs the single
        // issue thread ~2x the instructions of the common single-tap case)
        const uint32_t kind = (cur >> 2) & 7u;                                 // g | both << 2
        if (kind == 1u) {
          issue_mmas<BN, BK, THREE, 1, false>(d_main, da_hi0, da_lo0, db00, 0u, started);
        } else if (kind == 3u) {
          issue_mmas<BN, BK, THREE, 3, false>(d_main, da_hi0, da_lo0, db00, cur >> 5, started);
        } else if (kind == 2u) {
          issue_mmas<BN, BK, THREE, 2, false>(d_main, da_hi0, da_lo0, db00, cur >> 5, started);
        } else {
          issue_mmas<BN, BK, THREE, 1, true>(d_main, da_hi0, da_lo0, db00, 0u, started);
        }
        started = 1;
        umma_commit(empty_bar + s);              // frees the smem slot once these MMAs have read it
        if (close_seg) { umma_commit(seg_full_bar + buf); ++g; }
        if (++s == stages) { s = 0; ph ^= 1; }
      }
    }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue
    const int ew = warp - 2;
    const int q = warp & 3;             // TMEM lane quarter this warp may access
    const int half = ew >> 2;           // with 8 epilogue warps: which column chunks this warp takes
    float4* stg_f = reinterpret_cast<float4*>(stg_base) + (size_t)ew * 256;            // 4 KB per warp
    uint4* stg_h = reinterpret_cast<uint4*>(stg_f);                                    // halves alias the same 4 KB
    uint4* stg_l = stg_h + 128;
    RowInfo* rows = s_rows + ew * 32;
    const int et = threadIdx.x - 64;
    const uint32_t lane_bits = static_cast<uint32_t>(q * 32) << 16;
    // loop-invariant epilogue configuration in registers
    const int map = e.map, Wp = e.Wp, cout = e.cout, rows_in = e.rows_in;
    // hi-only (1-term) kernels serve the vocoder: no BN affine, no fused head, no fp32 streams - compiled out, the
    // 96-register budget of the two-CTA variants has no room for their state
    const bool has_affine = THREE && e.a_scale != nullptr, has_bias = e.bias != nullptr;
    const bool want_a = e.out_a.hi != nullptr, want_r = e.out_r.hi != nullptr, want_raw = THREE && e.out_raw != nullptr;
    const bool has_resid = THREE && e.resid != nullptr, has_resid_planes = e.resid_hi != nullptr, has_head = THREE && e.head_w != nullptr;
    const int act = e.act;
    const float slope = e.slope;
    const uint32_t resid_ar = THREE ? 0u : e.resid_ar, out_ar = THREE ? 0u : e.out_ar;      // (a, r) residual stream, gemm.cuh
    // lane roles for the row-major global accesses
    const int f_row = lane >> 3, f_c16 = lane & 7;       // fp32: 4 rows x 128 B per instruction
    const int h_row = lane >> 2, h_c16 = lane & 3;       // fp16: 8 rows x 64 B per instruction
    const int nseg = (tile_chunks + seg_chunks - 1) / seg_chunks;
    // staging slots: own row (so_*) and row-major role (sr_*); the swizzle terms are lane constants
    const int so_h0 = lane * 4, so_hx = (lane >> 1) & 3;            // sw64(lane, i)      = so_h0 + (i ^ so_hx)
    const int sr_h0 = h_row * 4, sr_hx = h_c16;                     // sw64(8i+h_row, c)  = 32 i + sr_h0 + (c ^ ((h_row >> 1) & 3)) (8i keeps bits 1-2)
    const int so_f0 = lane * 8, so_fx = lane & 7;                   // sw128(lane, i)     = so_f0 + (i ^ so_fx)
    const int sr_f0 = f_row * 8;                                    // sw128(4i+f_row, c) = 32 i + sr_f0 + (c ^ ((4i + f_row) & 7))
#define SO_H(i) (so_h0 + ((i) ^ so_hx))
#define SR_H(i) (32 * (i) + sr_h0 + (sr_hx ^ ((h_row >> 1) & 3)))
#define SO_F(i) (so_f0 + ((i) ^ so_fx))
#define SR_F(i) (32 * (i) + sr_f0 + (f_c16 ^ ((4 * (i) + f_row) & 7)))
    // TMA-store output path (MAP_PLAIN layers, e.tma_out): the staging tiles are written in the layouts SWIZZLE_128B (fp32,
    // 128-byte rows) / SWIZZLE_64B (fp16, 64-byte rows) expect - chunk ^ (row & 7) and chunk ^ ((row >> 1) & 3) are exactly the
    // SO_F / SO_H slots - so lane 0 hands a finished tile to the copy engine instead of the warp reading it back row-major and
    // storing it with 12 STG per lane: half the LSU wavefronts of the store path, which bounds the narrow layers (ncu l1tex 60-86 %)
    // (bit 3: the activated planes of a MAP_CONVT1D layer through a 5-D map [C, phase, q, image, plane] - output row
    // stride * q + phase - the 32 rows of a warp are one box per column chunk)
    const int tma_out = (map == MAP_PLAIN) ? (e.tma_out & 7) : (map == MAP_CONVT1D ? (e.tma_out & 8) : 0);
    bool st_pending = false;             // a TMA store of this warp may still be reading its staging tile (warp-uniform)
    auto stg_release = [&]() {
      if (st_pending) {
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
        st_pending = false;
      }
    };
    // Residual by TMA (P.resid_tma): lane 0 asks the copy engine for the warp's next [32 rows x 32 columns] residual tiles (fp32,
    // or the hi and lo planes) while earlier chunks are processed; the threads read their own rows from the swizzled tile.
    // No LDG, no STS for the residual - the other half of the epilogue's LSU traffic (see tma_out above).  The requests run
    // P.resid_tma (1 or 2) chunks ahead ACROSS tiles: a warp's chunk sequence is known up front (persistent tile loop), and a
    // request issued only at the start of its own tile exposes one HBM round trip per tile (ncu on voc.res2.*.b: 4.8 us per
    // 2-chunk tile, every unit below 62 %).
    const int resid_ring = (map == MAP_PLAIN) ? P.resid_tma : 0;
    const bool resid_tma = resid_ring != 0;
    uint8_t* rstg = rstg_base + (size_t)ew * resid_ring * 4096;
    uint64_t* rbar = resid_bar + ew * 2;
    uint32_t r_cons = 0, r_issued = 0;       // chunks consumed / requested by this warp
    int pf_tile = blockIdx.x, pf_j = half;   // next chunk to request
    auto issue_resid = [&]() {               // warp-uniform control flow, one lane issues
      if (pf_tile >= total_tiles) return;
      if (lane == 0) {
        const TileCoord pt((uint32_t)pf_tile, P, n_tiles, pr.m_tiles);
        const uint32_t slot = r_issued & (uint32_t)(resid_ring - 1);
        uint8_t* dst = rstg + slot * 4096;
        mbar_expect_tx(rbar + slot, 4096);
        if (THREE && e.resid != nullptr) tma_load_3d(dst, &P.i_res, rbar + slot, pt.nt * BN + pf_j * 32, pt.mi * GEMM_BM + q * 32, pt.img);   // fp32 stream
        else tma_load_4d(dst, &P.i_res, rbar + slot, pt.nt * BN + pf_j * 32, pt.mi * GEMM_BM + q * 32, pt.img, 0);                        // hi / lo planes
      }
      ++r_issued;
      pf_j += CHUNK_STEP;
      if (pf_j >= BN / 32) { pf_j = half; pf_tile += gridDim.x; }
    };
    if (resid_tma && half < BN / 32)
      for (int i = 0; i < resid_ring; ++i) issue_resid();
    int prev_n0 = -1, g = 0;
    float amax = 0.f;
    bool ok = true;
    for (int tile = blockIdx.x; tile < total_tiles && ok; tile += gridDim.x) {
      const TileCoord it((uint32_t)tile, P, n_tiles, pr.m_tiles);
      const int img = it.img;
      const int m0 = it.mi * GEMM_BM;
      const int n0 = it.nt * BN;
      if (n0 != prev_n0) {   // per-N-tile constants (uniform branch)
        epi_bar_sync(EPI_THREADS);
        for (int i = et; i < BN; i += EPI_THREADS) {
          s_bias[i] = has_bias ? __ldg(e.bias + n0 + i) : 0.f;
          int co = n0 + i;
          if (map != MAP_PLAIN) co -= (co / cout) * cout;
          s_scale[i] = has_affine ? __ldg(e.a_scale + co) : 1.f;
          s_shift[i] = has_affine ? __ldg(e.a_shift + co) : 0.f;
        }
        if (et < 32) s_head[et] = has_head ? __ldg(e.head_w + et) : 0.f;
        epi_bar_sync(EPI_THREADS);
        prev_n0 = n0;
      }
      const int wrow0 = m0 + q * 32;      // first GEMM row (inside the image) of this warp's 32
      const int r = wrow0 + lane;         // this thread's row
      const bool row_ok = r < rows_in;
      float head_acc = 0.f;
      int cth = 0, ctw = 0;
      uint32_t orow = 0, flags = 0;
      // MAP_PLAIN (everything but the transposed convs): output rows follow the GEMM rows, so the lanes that store
      // row rr of this warp need no exchange: row = obase + rr, valid iff rr < lim.
      const int lim = rows_in - wrow0;
      const uint32_t obase = (uint32_t)((size_t)img * e.out_img_rows + e.out_row0 + wrow0);
      if (map == MAP_PLAIN) {
        if (row_ok) {
          orow = obase + lane;
          flags = kRowValid | ((Wp > 0 && (r % Wp) == Wp - 1) ? kRowPad : 0);
          if (e.vl_rows && r >= __ldg(e.vl_rows + (size_t)img * e.vl_stride)) flags |= kRowPad;   // past this clip: zeros
        }
      } else {
        if (map == MAP_CONVT2D) {
          cth = r / Wp;
          ctw = r - cth * Wp;
        }
        // varlen, 3-term kernels: bit 8 + p of flags = the output row of phase p lies past this clip, decided once per tile
        // (the 1-term kernels test each chunk instead: whichever form costs the variant no spill)
        if (THREE && e.vl_rows && row_ok) {
          const int vlim = ld_row_limit(e.vl_rows + img * e.vl_stride);
          const int nph = map == MAP_CONVT2D ? 4 : e.ct_stride;
          for (int p = 0; p < nph; ++p) {
            const long t = map == MAP_CONVT2D ? (long)(2 * cth + (p >> 1)) * e.ct_out_wp     // vlim: whole rows of pitch ct_out_wp
                                              : (long)r * e.ct_stride + p - e.ct_pad;
            if (t >= vlim) flags |= 1u << (8 + p);
          }
        }
      }
      // store this warp's staged 32 rows x 32 columns of fp16 (hi [+ lo]) row-major: 8 rows x 64 B per instruction
      auto store_rows_h = [&](const OutPlane& op, const int co0, const bool two, const CUtensorMap* tm) {
        if (tm) {                         // staged tile(s) -> TMA store; rows past rows_in are clipped by the tensor map
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(tm, stg_h, op.c_off + co0, e.out_row0 + wrow0, img, 0);
            tma_store_commit();
          }
          st_pending = true;
        } else if (map == MAP_PLAIN) {
          const size_t o0 = (size_t)(obase + h_row) * op.ld + op.c_off + co0;   // one wide multiply per chunk
          uint4* ph = reinterpret_cast<uint4*>(op.hi + o0) + h_c16;
          uint4* pl = reinterpret_cast<uint4*>(op.lo + o0) + h_c16;
          const int step = op.ld;       // 8 rows further, in 16-byte units
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (8 * i + h_row < lim) {
              ph[i * step] = stg_h[SR_H(i)];
              if (two) pl[i * step] = stg_l[SR_H(i)];
            }
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const RowInfo ri = rows[8 * i + h_row];
            if (ri.flags & kRowValid) {
              const size_t o = (size_t)ri.orow * op.ld + op.c_off + co0;
              reinterpret_cast<uint4*>(op.hi + o)[h_c16] = stg_h[SR_H(i)];
              if (two) reinterpret_cast<uint4*>(op.lo + o)[h_c16] = stg_l[SR_H(i)];
            }
          }
        }
      };

      // Residual planes of the NEXT column chunk are fetched into registers while the current one is processed
      // (1-term kernels with a register budget for it): an epilogue warp otherwise has one exposed global-load
      // round trip per chunk, which bounded voc.res*.b (ncu: 31 % of all samples on the first STS after the loads).
      uint4 pre_h[4], pre_l[4];
      auto load_resid = [&](const int j) {     // MAP_PLAIN only (the residual stream follows the GEMM rows)
        const size_t rbase = ((size_t)img * rows_in + wrow0 + h_row) * e.resid_ld + n0 + j * 32;
        const uint4* gh = reinterpret_cast<const uint4*>(e.resid_hi + rbase) + h_c16;
        const uint4* gl = reinterpret_cast<const uint4*>(e.resid_lo + rbase) + h_c16;
        const int step = e.resid_ld;     // 8 rows further, in 16-byte units
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          pre_h[i] = make_uint4(0, 0, 0, 0);
          pre_l[i] = make_uint4(0, 0, 0, 0);
          if (8 * i + h_row < lim) {
            pre_h[i] = __ldg(gh + i * step);
            pre_l[i] = __ldg(gl + i * step);
          }
        }
      };
      if (!resid_tma && PREFETCH && has_resid_planes) load_resid(half);

      // One 32-column chunk of this thread's row: bias, residual, outputs (see gemm.cuh for the semantics).
      auto process_chunk = [&](const int j, float (&v)[32]) {
        const int nb = n0 + j * 32;
        int co0 = nb;
        if (map != MAP_PLAIN) {           // transposed convs: the output row depends on the phase of this chunk
          const int phase = nb / cout;
          co0 = nb - phase * cout;
          const uint32_t keep = THREE ? flags & ~0xffu : 0u;
          const uint32_t past = THREE && ((flags >> (8 + phase)) & 1u) ? (uint32_t)kRowPad : 0u;
          orow = 0; flags = keep;
          if (row_ok) {
            if (map == MAP_CONVT2D) {
              const int ph = phase >> 1, pw = phase & 1;
              const int col = 2 * ctw + pw;
              if (col < e.ct_out_wp) {         // both=True pruning drops the column past the output pitch
                const int lrow = (2 * cth + ph) * e.ct_out_wp + col;
                orow = (uint32_t)((size_t)img * e.out_img_rows + lrow);
                flags = keep | past | kRowValid | (col == e.ct_out_wp - 1 ? kRowPad : 0);
                if (!THREE && e.vl_rows && lrow >= ld_row_limit(e.vl_rows + img * e.vl_stride)) flags |= kRowPad;
              }
            } else {
              const long t = (long)r * e.ct_stride + phase - e.ct_pad;
              if (t >= 0 && t < e.out_rows_valid) {
                orow = (uint32_t)((size_t)img * e.out_img_rows + e.out_row0 + t);
                flags = keep | past | kRowValid;
                if (!THREE && e.vl_rows && t >= ld_row_limit(e.vl_rows + img * e.vl_stride)) flags |= kRowPad;
              }
            }
          }
          __syncwarp();
          rows[lane] = RowInfo{orow, flags};
        }
        if (has_bias) {
          const float4* bp = reinterpret_cast<const float4*>(s_bias + j * 32);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 b4 = bp[i];
            v[4 * i] += b4.x; v[4 * i + 1] += b4.y; v[4 * i + 2] += b4.z; v[4 * i + 3] += b4.w;
          }
        }
        if (THREE && has_resid && resid_tma) {      // the tile was requested one chunk ago (or at the start of the tile)
          const uint32_t slot = r_cons & (uint32_t)(resid_ring - 1);
          if (!mbar_wait(rbar + slot, (r_cons >> (resid_ring >> 1)) & 1u, e.err, ERR_PIPE_EPILOGUE)) ok = false;
          ++r_cons;
          const float4* rt = reinterpret_cast<const float4*>(rstg + slot * 4096);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 x = rt[SO_F(i)];
            v[4 * i] += x.x; v[4 * i + 1] += x.y; v[4 * i + 2] += x.z; v[4 * i + 3] += x.w;
          }
          __syncwarp();                   // every lane has read the tile: it may be refilled
          issue_resid();                  // the slot just read is free again: request the chunk `resid_ring` ahead
        } else if (THREE && has_resid) {         // coalesced global -> staging -> own row (MAP_PLAIN only; fp32 streams exist in 3-term mode only)
          const size_t rbase = ((size_t)img * rows_in + m0 + q * 32) * e.resid_ld + co0;
          stg_release();
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rr = 4 * i + f_row;
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (m0 + q * 32 + rr < rows_in)
              x = __ldg(reinterpret_cast<const float4*>(e.resid + rbase + (size_t)rr * e.resid_ld) + f_c16);
            stg_f[SR_F(i)] = x;
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 x = stg_f[SO_F(i)];
            v[4 * i] += x.x; v[4 * i + 1] += x.y; v[4 * i + 2] += x.z; v[4 * i + 3] += x.w;
          }
        }
        if (has_resid_planes && resid_tma) {
          const uint32_t slot = r_cons & (uint32_t)(resid_ring - 1);
          if (!mbar_wait(rbar + slot, (r_cons >> (resid_ring >> 1)) & 1u, e.err, ERR_PIPE_EPILOGUE)) ok = false;
          ++r_cons;
          const uint4* rth = reinterpret_cast<const uint4*>(rstg + slot * 4096);
          const uint4* rtl = rth + 128;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 xh = rth[SO_H(i)], xl = rtl[SO_H(i)];
            const __half2* ph = reinterpret_cast<const __half2*>(&xh);
            const __half2* pl = reinterpret_cast<const __half2*>(&xl);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              add_planes(v[8 * i + 2 * k], v[8 * i + 2 * k + 1], reinterpret_cast<const uint32_t*>(ph)[k], reinterpret_cast<const uint32_t*>(pl)[k], resid_ar);
          }
          __syncwarp();
          issue_resid();                  // the slot just read is free again: request the chunk `resid_ring` ahead
        } else if (has_resid_planes) {           // residual stream kept as hi/lo planes: coalesced load, sum in fp32
          stg_release();
          __syncwarp();
          if (PREFETCH) {                 // loaded one chunk ahead (see load_resid below): no exposed load latency
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              stg_h[SR_H(i)] = pre_h[i];
              stg_l[SR_H(i)] = pre_l[i];
            }
            if (j + CHUNK_STEP < BN / 32) load_resid(j + CHUNK_STEP);
          } else {
            const size_t rbase = ((size_t)img * rows_in + wrow0) * e.resid_ld + co0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = 8 * i + h_row;
              uint4 xh = make_uint4(0, 0, 0, 0), xl = make_uint4(0, 0, 0, 0);
              if (rr < lim) {
                xh = __ldg(reinterpret_cast<const uint4*>(e.resid_hi + rbase + (size_t)rr * e.resid_ld) + h_c16);
                xl = __ldg(reinterpret_cast<const uint4*>(e.resid_lo + rbase + (size_t)rr * e.resid_ld) + h_c16);
              }
              stg_h[SR_H(i)] = xh;
              stg_l[SR_H(i)] = xl;
            }
          }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 xh = stg_h[SO_H(i)], xl = stg_l[SO_H(i)];
            const __half2* ph = reinterpret_cast<const __half2*>(&xh);
            const __half2* pl = reinterpret_cast<const __half2*>(&xl);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              add_planes(v[8 * i + 2 * k], v[8 * i + 2 * k + 1], reinterpret_cast<const uint32_t*>(ph)[k], reinterpret_cast<const uint32_t*>(pl)[k], resid_ar);
          }
        }
        const bool pad = (flags & kRowPad) != 0;      // pad column, or a row past its clip (varlen): zeros before any range check
        if (pad) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
        if (THREE && want_raw) {          // fp32 output
          stg_release();
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) stg_f[SO_F(i)] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
          if (tma_out & 1) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_3d(&P.o_raw, stg_f, co0, e.out_row0 + wrow0, img);
              tma_store_commit();
            }
            st_pending = true;
          } else {
          __syncwarp();
          if (map == MAP_PLAIN) {
            float4* pr4 = reinterpret_cast<float4*>(e.out_raw + (size_t)(obase + f_row) * e.raw_ld + co0) + f_c16;
            const int step = e.raw_ld;    // 4 rows further, in 16-byte units
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (4 * i + f_row < lim) pr4[i * step] = stg_f[SR_F(i)];
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const RowInfo ri = rows[4 * i + f_row];
              if (ri.flags & kRowValid)
                reinterpret_cast<float4*>(e.out_raw + (size_t)ri.orow * e.raw_ld + co0)[f_c16] = stg_f[SR_F(i)];
            }
          }
          }
        }
        if (want_r) {                     // raw hi/lo planes
          stg_release();
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint4 h, l;
            pack8<true>(v, i, h, l);
            stg_h[SO_H(i)] = h;
            stg_l[SO_H(i)] = l;
          }
          __syncwarp();
          store_rows_h(e.out_r, co0, true, (tma_out & 2) ? &P.o_r : nullptr);
        }
        if (has_head) {                   // fused 1x1 head (N == 32)
#pragma unroll
          for (int i = 0; i < 32; ++i) head_acc = fmaf(v[i], s_head[i], head_acc);
        }
        if (want_a) {                     // activated planes (consumer's BN affine + activation)
          if (has_affine) {
            const float4* sc = reinterpret_cast<const float4*>(s_scale + j * 32);
            const float4* sh = reinterpret_cast<const float4*>(s_shift + j * 32);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 a4 = sc[i], b4 = sh[i];
              v[4 * i] = fmaf(v[4 * i], a4.x, b4.x); v[4 * i + 1] = fmaf(v[4 * i + 1], a4.y, b4.y);
              v[4 * i + 2] = fmaf(v[4 * i + 2], a4.z, b4.z); v[4 * i + 3] = fmaf(v[4 * i + 3], a4.w, b4.w);
            }
          }
          if (out_ar) {                     // (a, r) stream: hi plane = fp16(lrelu(v)), lo plane = fp16(v - U(a)); |v| itself is range-checked
            if (row_ok) {
#pragma unroll
              for (int i = 0; i < 32; ++i) amax = fmaxf(amax, fabsf(v[i]));
            }
            stg_release();
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {   // eight columns at a time straight into the staging tiles: no 32 packed words live at once
              uint32_t h4[4], l4[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float v0 = pad ? 0.f : v[8 * i + 2 * k], v1 = pad ? 0.f : v[8 * i + 2 * k + 1];
                ar_split(v0, v1, fmaxf(v0, v0 * slope), fmaxf(v1, v1 * slope), out_ar, h4[k], l4[k]);
              }
              stg_h[SO_H(i)] = make_uint4(h4[0], h4[1], h4[2], h4[3]);
              stg_l[SO_H(i)] = make_uint4(l4[0], l4[1], l4[2], l4[3]);
            }
          } else {
            if (act == ACT_LRELU) {           // slope in [0, 1]: max(a, slope * a)
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], v[i] * slope);
            } else if (act == ACT_ELU) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = v[i] > 0.f ? v[i] : expm1f(v[i]);
            }
            if (pad) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = 0.f;
            }
            if (row_ok) {
#pragma unroll
              for (int i = 0; i < 32; ++i) amax = fmaxf(amax, fabsf(v[i]));
            }
            stg_release();
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint4 h, l;
              pack8<THREE>(v, i, h, l);
              stg_h[SO_H(i)] = h;
              if (THREE) stg_l[SO_H(i)] = l;
            }
          }
          __syncwarp();
          // A TMA store whose box STARTS at a negative coordinate faults (illegal instruction; tools/probe_tma5d.cu - boxes that
          // run past the upper bound are clipped as documented): the one warp per image and early phase whose first output row
          // would be q = -1 keeps the LDS + STG path.
          if ((tma_out & 8) && !(wrow0 == 0 && nb / cout < e.ct_pad)) {      // t = stride * r + phase - pad = stride * (r - up) + (phase - pad + up * stride)
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              const int d = nb / cout - e.ct_pad;
              const int up = d < 0 ? 1 : 0;
              tma_store_5d(&P.o_a, stg_h, e.out_a.c_off + co0, d + up * e.ct_stride, wrow0 - up, img, 0);
              tma_store_commit();
            }
            st_pending = true;
          } else {
            store_rows_h(e.out_a, co0, THREE || out_ar, (tma_out & 4) ? &P.o_a : nullptr);
          }
        }
      };

      if (THREE) {
        // Promotion: every finished K segment is added into registers in fp32 round-to-nearest, so no chain of
        // truncating tensor-core adds is longer than one segment; the small hi*lo + lo*hi sums join at the end.
        float acc[NJ][32];
        for (int sg = 0; sg < nseg && ok; ++sg, ++g) {
          const int buf = g & nbuf_mask;
          if (!mbar_wait(seg_full_bar + buf, (g >> nbuf_log) & 1, e.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }
          tc_fence_after();
#pragma unroll
          for (int jj = 0; jj < NJ; ++jj) {
            const int j = half + jj * CHUNK_STEP;
            if (j < BN / 32) {
              if constexpr (MINB >= 2) {      // register-capped variants: 16 columns of both accumulators at a time
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                  float w[16], c[16];
                  const uint32_t ta = tmem_base + lane_bits + buf * 2 * BN + j * 32 + hh * 16;
                  tmem_ld2_32x16(ta, ta + BN, w, c);
                  if (sg == 0) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[jj][hh * 16 + i] = w[i] + c[i];
                  } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[jj][hh * 16 + i] += w[i] + c[i];
                  }
                }
              } else {
                float w[32], c[32];
                tmem_ld_32x32(tmem_base + lane_bits + buf * 2 * BN + j * 32, w);
                tmem_ld_32x32(tmem_base + lane_bits + buf * 2 * BN + BN + j * 32, c);
                if (sg == 0) {
#pragma unroll
                  for (int i = 0; i < 32; ++i) acc[jj][i] = w[i] + c[i];
                } else {
#pragma unroll
                  for (int i = 0; i < 32; ++i) acc[jj][i] += w[i] + c[i];
                }
              }
            }
          }
          tc_fence_before();
          mbar_arrive(seg_empty_bar + buf);
        }
        if (ok) {
#pragma unroll
          for (int jj = 0; jj < NJ; ++jj) {
            const int j = half + jj * CHUNK_STEP;
            if (j < BN / 32) process_chunk(j, acc[jj]);
          }
        }
      } else {
        const int buf = g & nbuf_mask;
        if (!mbar_wait(seg_full_bar + buf, (g >> nbuf_log) & 1, e.err, ERR_PIPE_EPILOGUE)) { ok = false; break; }
        tc_fence_after();
#pragma unroll 1
        for (int j = half; j < BN / 32; j += CHUNK_STEP) {
          float v[32];
          tmem_ld_32x32(tmem_base + lane_bits + buf * BN + j * 32, v);
          if (j + CHUNK_STEP >= BN / 32) {   // last chunk is in registers: hand the accumulator back before the math / stores
            tc_fence_before();
            mbar_arrive(seg_empty_bar + buf);
          }
          process_chunk(j, v);
        }
        ++g;
      }
      if (THREE && half == 0) epilogue_head(e, img, r, head_acc);
    }
    if (tma_out && lane == 0) tma_store_wait_all();      // this thread's bulk stores have completed before the CTA exits
    // NaN compares false against everything, inf exceeds the bound
    if (!(amax <= 65504.f) && e.err) atomicCAS(e.err, 0, ERR_FP16_OVERFLOW);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_dyn(tmem_base, P.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------- host side
static int epi_warps_for(int bn, int /*terms*/) { return bn == 32 ? 4 : 8; }

size_t gemm_tc_smem_bytes(int bn, int bk, int stages, int planes_a, int terms, int a_box_rows, int gmax, int tile_chunks, int resid_tma) {
  const size_t a_slot = ((size_t)a_box_rows * bk * 2 + 1023) & ~(size_t)1023;
  const size_t stage = planes_a * a_slot + (size_t)gmax * (terms == 3 ? 2 : 1) * bn * bk * 2;
  const int ew = epi_warps_for(bn, terms);
  return stages * stage + ew * 4096 * (1 + resid_tma) + (2 * stages + 24) * 8 + 32 + (3 * bn + 32) * 4 + ew * 32 * 8 + (size_t)tile_chunks * 16 + 1024;
}

template <int BN, int BK, int EW, bool THREE, int MINB>
static cudaError_t launch_cfg(const GemmTcParams& p, cudaStream_t stream) {
  const size_t smem = gemm_tc_smem_bytes(BN, BK, p.stages, p.planes_a, p.prob.terms, p.a_box_rows, p.gmax, p.tile_chunks, p.resid_tma);
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN, BK, EW, THREE, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  gemm_tc_kernel<BN, BK, EW, THREE, MINB><<<p.grid, 64 + 32 * EW, smem, stream>>>(p);
  return cudaGetLastError();
}
template <int BN, int BK, int EW, int MINB>
static cudaError_t launch_one(const GemmTcParams& p, cudaStream_t stream) {
  return p.prob.terms == 3 ? launch_cfg<BN, BK, EW, true, MINB>(p, stream) : launch_cfg<BN, BK, EW, false, MINB>(p, stream);
}
template <int BK>
static cudaError_t launch_bk(const GemmTcParams& p, int bn, cudaStream_t stream) {
  const int c = p.ctas_per_sm;
  if (bn == 256) return p.prob.terms == 1 ? launch_cfg<256, BK, 8, false, 1>(p, stream) : cudaErrorInvalidValue;
  if (bn == 128) return launch_one<128, BK, 8, 1>(p, stream);
  if (bn == 64) return c >= 2 ? launch_one<64, BK, 8, 2>(p, stream) : launch_one<64, BK, 8, 1>(p, stream);
  if (bn == 32) return c >= 3 ? launch_one<32, BK, 4, 3>(p, stream) : launch_one<32, BK, 4, 2>(p, stream);
  return cudaErrorInvalidValue;
}

// multiply-high magic for n / d with n <= nmax: exact while nmax * d < 2^32 (the error term of ceil(2^32 / d))
uint32_t gemm_tc_magic(uint32_t d, uint64_t nmax) {
  if (d <= 1) return 0u;
  if (nmax * (uint64_t)d >= (1ull << 32)) return 0xffffffffu;
  return (uint32_t)(((1ull << 32) + d - 1) / d);
}

// register-limited CTAs per SM of the variants above (the engine sizes shared memory and the grid against it)
int gemm_tc_max_ctas(int bn) { return bn == 32 ? 3 : (bn == 64 ? 2 : 1); }

cudaError_t launch_gemm_tc(const GemmTcParams& p, int bn, int bk, cudaStream_t stream) {
  if (bk == 64) return launch_bk<64>(p, bn, stream);
  if (bk == 32) return launch_bk<32>(p, bn, stream);
  return cudaErrorInvalidValue;
}

}  // namespace vf
