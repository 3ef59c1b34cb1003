// Host side of libb200vf.so: context, weight packing, per-shape launch plans, and the C ABI (include/b200vf.h).
//
// A plan is the full, pre-resolved launch list for one (batch, frames) shape: every activation buffer is
// allocated once, every TMA tensor map is encoded once, and running a stage is a loop of kernel launches on
// the caller's stream - no allocation, no host synchronisation, no CPU arithmetic on the data path.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

#include "../../include/b200vf.h"
#include "gemm.cuh"
#include "kernels.cuh"

namespace vf {
cudaError_t launch_gemm_tc(const GemmTcParams& p, int bn, int bk, cudaStream_t stream);
size_t gemm_tc_smem_bytes(int bn, int bk, int stages, int planes_a, int terms, int a_box_rows, int gmax, int tile_chunks, int resid_tma = 0);
int gemm_tc_max_ctas(int bn);
uint32_t gemm_tc_magic(uint32_t d, uint64_t nmax);
cudaError_t launch_pair_tc(const PairParams& p, cudaStream_t stream);
size_t pair_tc_smem_bytes(int C, int stages);
cudaError_t launch_gemm_simt(const GemmSimtParams& p, cudaStream_t stream);
}  // namespace vf

using namespace vf;

namespace {

std::string g_create_error;

struct HostT {
  std::vector<float> v;
  std::vector<int64_t> shape;
};

struct GemmW {
  __half* hi = nullptr;
  __half* lo = nullptr;
  float* bias = nullptr;
  int N = 0, K = 0;
  int k_tail = 0;      // trailing identity block (pack_conv1d): a GEMM may contract the K - k_tail columns before it only
};
struct Affine {
  float* scale = nullptr;
  float* shift = nullptr;
};
struct Planes {
  PlanePtr p{nullptr, nullptr};
  int C = 0;
  int img_rows = 0;   // allocated rows per image
  size_t plane_stride = 0;   // elements from the hi plane to the lo plane (same allocation)
};
struct ASrc {
  Planes pl;
  int rows;           // valid rows per image (TMA bound / SIMT bound)
  int row0;           // first valid row inside the allocation (reflection slack), usually 0
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

enum OpKind { OP_GEMM, OP_FIRST, OP_POOL, OP_COND, OP_REFLECT, OP_TAIL, OP_FINALIZE, OP_MEMSET32, OP_PAIR };

struct Op {
  OpKind kind;
  int bn = 0, bk = 0;
  double flops = 0, bytes = 0;   // algorithmic work of this launch (reference op counts), for the roofline
  double exec_flops = 0;         // tensor-core flops actually issued (3 MMAs per product in 3-term mode, K / phase padding,
                                 // identity taps): numerator of the "executed" tensor fraction
  char label[48] = {0};
  GemmTcParams tc;
  GemmSimtParams simt;
  PairParams pair;
  UnetFirstParams first;
  PoolParams pool;
  VocCondParams cond;
  struct { PlanePtr pl; int batch, L, C, pad; const VarlenImage* vl; int vl_stage; } refl;
  VocTailParams tail;
  FinalizeParams fin;
  struct { void* p; size_t bytes; } ms;
};

struct ConvBlockW {
  GemmW conv1, conv2;     // conv2 carries the 1x1 shortcut as an extra K segment when present
  Affine bn1, bn2;
  bool has_sc = false;
  int cin = 0, cout = 0;
};

// One analysis ResUNet (models/components/unet.py / unet_small.py / unet_v2.py share the block structure and key names)
struct UnetW {
  bool loaded = false;
  ConvBlockW enc[6][4], bott, dec[6][4], post;
  GemmW dec_up[6];
  Affine dec_bn1[6];
  float first_bn1_scale = 1, first_bn1_shift = 0;
  float* d_first_w1 = nullptr;
  float* d_first_wsc = nullptr;
  float* d_first_bsc = nullptr;
  float* d_head_w = nullptr;
  float head_b = 0;
};

// PLAN_GSR_VARLEN / PLAN_SSR_VARLEN: the GSR / SSR chain over clips of different lengths (vf_restore_varlen /
// vf_ssr_restore_varlen), keyed by the 64-frame bucket of the longest clip; its kernels take the per-clip lengths from the
// plan's VarlenImage table
enum PlanKind { PLAN_GSR = 0, PLAN_SSR = 1, PLAN_GSR_VARLEN = 2, PLAN_SSR_VARLEN = 3 };

struct Plan {
  int kind = PLAN_GSR;
  uint64_t last_use = 0;
  int batch = 0, T = 0;
  long n_samples = 0;
  std::vector<void*> allocs;
  size_t bytes = 0;
  std::vector<Op> frontend, unet, vocoder, tail;
  float* d_wav = nullptr;        // [B, N]   staged input of the host entry points (buffer 0)
  float* d_out = nullptr;        // [B, N]
  float* d_io[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // [buffer][in / out]: double-buffered host staging
  cudaEvent_t io_ev[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};   // h2d done, input consumed, compute done, d2h done
  unsigned io_seq = 0;
  // a plan's buffers are shared by every call of its shape: uses on different streams are ordered through this event
  cudaEvent_t ev_last = nullptr;
  cudaStream_t last_stream = nullptr;
  bool used = false;
  float* d_mel = nullptr;        // [B, T, 128] linear mel
  float* d_logmel_in = nullptr;  // [B, T, 128] log10 mel (UNet input)
  float* d_logmel_out = nullptr; // [B, T, 128]
  float* d_voc_wav = nullptr;    // [B, L]
  float* d_band = nullptr;       // [B][2] low-band energy sums (unify_energy)
  VarlenImage* d_vl = nullptr;   // [B] per-clip lengths of the current call (PLAN_GSR_VARLEN / PLAN_SSR_VARLEN only)
  unsigned int* d_peak = nullptr;
  long L = 0;
  // SSR plans (unet_v2 + ISTFT)
  float* d_sp = nullptr;         // [B, T, 1025] input magnitude
  float* d_mag = nullptr;        // [B, T, 1025] predicted magnitude
  float* d_frames = nullptr;     // [B, T, 2048] windowed inverse-DFT frames
  // CUDA graphs of the fixed-pointer launch chain (GSR: unet [+ band energy] + vocoder, index = unify flag; SSR: unet),
  // captured on the second use of the plan (the first runs eagerly and sets the kernels' function attributes)
  cudaGraphExec_t graph[2] = {nullptr, nullptr};
  int uses = 0;
  // op slots patched per call
  int fe_op = -1, cond_op = -1, fin_op = -1;
};

}  // namespace

struct vf_ctx {
  int device = 0;
  vf_config cfg;
  std::string err;
  std::unordered_map<std::string, HostT> host_w;
  std::vector<void*> allocs;
  size_t weight_bytes = 0;
  bool loaded = false;
  EncodeTiledFn encode = nullptr;
  int sm_count = 148;
  int unet_terms = 3, voc_terms = 1, validate_simt = 0, unify_energy = 0;
  int64_t launches = 0;
  int* d_err = nullptr;      // [0] device error code, [1] negative-input count
  // tables
  float* d_window = nullptr;
  float2* d_tw1024 = nullptr;
  float2* d_tw2048 = nullptr;
  int *d_fb_f0 = nullptr, *d_fb_len = nullptr, *d_fb_ofs = nullptr;
  float* d_fb_val = nullptr;
  float* d_melw = nullptr;
  // UNet weights: the mel-domain analysis module of VoiceFixer (prefix generator.analysis_module.) and the
  // linear-spectrogram unet_v2 of SSR_UNet / GSR_UNet (prefix generator.unet.); either may be absent
  UnetW gsr, ssr;
  bool voc_loaded = false;
  float* d_win_sq_inv = nullptr;   // ISTFT: 1 / clamp(overlap-added squared window, 1e-11), period hop (steady state)
  // vocoder weights
  std::vector<GemmW> voc_cond;
  GemmW voc_stem;
  std::vector<GemmW> voc_up;
  std::vector<std::vector<GemmW>> voc_res_a, voc_res_b;
  float* d_tail_w = nullptr;
  float tail_b = 0;
  int voc_last_c = 64;
  std::map<std::tuple<int, int, long>, std::unique_ptr<Plan>> plans;   // (kind, batch, frames)
  uint64_t use_clock = 0;
  size_t plan_bytes = 0;               // device bytes held by cached plans
  size_t plan_budget = 0;              // cap for plan_bytes (LRU eviction); 0 = decide at first use from free memory
  int64_t plans_evicted = 0;
  bool use_graphs = true;        // option "graphs"
  cudaStream_t cap_stream = nullptr;   // capture happens on an internal stream (the caller's may be the legacy default stream)
  // host entry points: copies and compute on internal streams, so the H2D of call i+1 and the D2H of call i-1 overlap the
  // compute of call i (option "host_pipeline"); the caller's stream only waits for the call's own D2H
  bool host_pipeline = true;
  cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
  bool op_timing = false;
  struct ProfRec { std::string label; double flops, bytes, exec_flops; int bn, bk, terms; };
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> prof_ev;
  bool timing = false;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  bool ev_valid = false;
};

namespace {

int fail(vf_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(ctx, VF_ECUDA, "%s: %s", #call, cudaGetErrorString(e_));   \
  } while (0)

template <typename T>
int dev_alloc(vf_ctx* ctx, std::vector<void*>& pool, size_t& acct, T** out, size_t count) {
  void* p = nullptr;
  const size_t bytes = std::max<size_t>(count * sizeof(T), 256);
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return fail(ctx, VF_ECUDA, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
  pool.push_back(p);
  acct += bytes;
  *out = static_cast<T*>(p);
  return VF_OK;
}
template <typename T>
int upload(vf_ctx* ctx, T** out, const std::vector<T>& h) {
  int rc = dev_alloc(ctx, ctx->allocs, ctx->weight_bytes, out, h.size());
  if (rc) return rc;
  CK(cudaMemcpy(*out, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  return VF_OK;
}

const HostT* find(vf_ctx* ctx, const std::string& k) {
  auto it = ctx->host_w.find(k);
  return it == ctx->host_w.end() ? nullptr : &it->second;
}
#define NEED(var, key)                                                                \
  const HostT* var = find(ctx, key);                                                  \
  if (!var) return fail(ctx, VF_ESTATE, "missing weight tensor '%s'", std::string(key).c_str());

// fp32 matrix [N][K] -> device fp16 hi/lo pair (+ optional fp32 bias [N])
int upload_gemm(vf_ctx* ctx, GemmW* w, const std::vector<float>& m, int N, int K, const std::vector<float>* bias) {
  std::vector<__half> hi(m.size()), lo(m.size());
  for (size_t i = 0; i < m.size(); ++i) {
    hi[i] = __float2half_rn(m[i]);
    lo[i] = __float2half_rn(m[i] - __half2float(hi[i]));
  }
  w->N = N;
  w->K = K;
  hi.insert(hi.end(), lo.begin(), lo.end());     // [hi matrix][lo matrix]: one 3-D TMA box fetches a tile of both
  int rc = upload(ctx, &w->hi, hi);
  if (rc) return rc;
  w->lo = w->hi + m.size();
  if (bias) return upload(ctx, &w->bias, *bias);
  return VF_OK;
}

// eval-mode BatchNorm2d -> a*x + b (modules.py:232-233, eps 1e-5)
int fold_bn(vf_ctx* ctx, const std::string& p, std::vector<float>* scale, std::vector<float>* shift) {
  NEED(w, p + ".weight");
  NEED(b, p + ".bias");
  NEED(m, p + ".running_mean");
  NEED(v, p + ".running_var");
  const size_t n = w->v.size();
  scale->resize(n);
  shift->resize(n);
  for (size_t i = 0; i < n; ++i) {
    const double a = (double)w->v[i] / std::sqrt((double)v->v[i] + 1e-5);
    (*scale)[i] = (float)a;
    (*shift)[i] = (float)((double)b->v[i] - (double)m->v[i] * a);
  }
  return VF_OK;
}
int upload_bn(vf_ctx* ctx, const std::string& p, Affine* a) {
  std::vector<float> s, h;
  int rc = fold_bn(ctx, p, &s, &h);
  if (rc) return rc;
  rc = upload(ctx, &a->scale, s);
  if (rc) return rc;
  return upload(ctx, &a->shift, h);
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Conv2d 3x3 [Cout][Cin][3][3] (+ optional 1x1 shortcut [Cout][Csc]) -> [Cout][9*Cin + pad64(Csc)]
int pack_conv3x3(vf_ctx* ctx, GemmW* out, const HostT& w, const HostT* sc_w, const HostT* sc_b) {
  const int cout = (int)w.shape[0], cin = (int)w.shape[1];
  const int csc = sc_w ? (int)sc_w->shape[1] : 0;
  const int cscp = sc_w ? round_up(csc, cin >= 64 ? 64 : 32) : 0;
  const int K = 9 * cin + cscp;
  std::vector<float> m((size_t)cout * K, 0.f);
  for (int n = 0; n < cout; ++n) {
    for (int c = 0; c < cin; ++c)
      for (int t = 0; t < 9; ++t) m[(size_t)n * K + t * cin + c] = w.v[((size_t)n * cin + c) * 9 + t];
    for (int c = 0; c < csc; ++c) m[(size_t)n * K + 9 * cin + c] = sc_w->v[(size_t)n * csc + c];
  }
  return upload_gemm(ctx, out, m, cout, K, sc_b ? &sc_b->v : nullptr);
}

// ConvTranspose2d k3 s2 [Cin][Cout][3][3] -> [4*Cout][4*Cin]; phase (ph,pw), tap (dh,dw) <-> kernel index
// kh = ph + 2*dh (valid when <= 2, and dh = 0 for ph = 1).
int pack_convT2d(vf_ctx* ctx, GemmW* out, const HostT& w) {
  const int cin = (int)w.shape[0], cout = (int)w.shape[1];
  const int N = 4 * cout, K = 4 * cin;
  std::vector<float> m((size_t)N * K, 0.f);
  for (int ph = 0; ph < 2; ++ph)
    for (int pw = 0; pw < 2; ++pw)
      for (int dh = 0; dh < 2; ++dh)
        for (int dw = 0; dw < 2; ++dw) {
          const int kh = ph + 2 * dh, kw = pw + 2 * dw;
          if (kh > 2 || kw > 2) continue;
          for (int co = 0; co < cout; ++co)
            for (int ci = 0; ci < cin; ++ci)
              m[(size_t)((ph * 2 + pw) * cout + co) * K + (dh * 2 + dw) * cin + ci] =
                  w.v[(((size_t)ci * cout + co) * 3 + kh) * 3 + kw];
        }
  return upload_gemm(ctx, out, m, N, K, nullptr);
}

// Conv1d [Cout][Cin][k] -> [Cout][k*Cin (+ Cout)]; with `identity` an identity block is appended so the
// residual stream x (kept as fp16 hi/lo planes) is added inside the same accumulator: x' = x + conv(...)
int pack_conv1d(vf_ctx* ctx, GemmW* out, const HostT& w, const HostT& b, bool identity = false) {
  const int cout = (int)w.shape[0], cin = (int)w.shape[1], k = (int)w.shape[2];
  const int K = k * cin + (identity ? cout : 0);
  std::vector<float> m((size_t)cout * K, 0.f);
  for (int n = 0; n < cout; ++n) {
    for (int c = 0; c < cin; ++c)
      for (int t = 0; t < k; ++t) m[(size_t)n * K + t * cin + c] = w.v[((size_t)n * cin + c) * k + t];
    if (identity) m[(size_t)n * K + k * cin + n] = 1.f;
  }
  out->k_tail = identity ? cout : 0;
  return upload_gemm(ctx, out, m, cout, K, &b.v);
}

// ConvTranspose1d [Cin][Cout][2s], stride s -> [s*Cout][2*Cin]: output phase r takes taps (q, k=r) and (q-1, k=r+s)
int pack_convT1d(vf_ctx* ctx, GemmW* out, const HostT& w, const HostT& b, int s) {
  const int cin = (int)w.shape[0], cout = (int)w.shape[1];
  const int N = s * cout, K = 2 * cin;
  std::vector<float> m((size_t)N * K), bias(N);
  for (int r = 0; r < s; ++r)
    for (int co = 0; co < cout; ++co) {
      bias[r * cout + co] = b.v[co];
      for (int j = 0; j < 2; ++j)
        for (int ci = 0; ci < cin; ++ci)
          m[(size_t)(r * cout + co) * K + j * cin + ci] = w.v[((size_t)ci * cout + co) * (2 * s) + r + j * s];
    }
  return upload_gemm(ctx, out, m, N, K, &bias);
}

int load_block(vf_ctx* ctx, const std::string& p, ConvBlockW* blk, bool skip_conv1) {
  NEED(w1, p + ".conv1.weight");
  NEED(w2, p + ".conv2.weight");
  blk->cout = (int)w1->shape[0];
  blk->cin = (int)w1->shape[1];
  const HostT* scw = find(ctx, p + ".shortcut.weight");
  const HostT* scb = find(ctx, p + ".shortcut.bias");
  blk->has_sc = scw != nullptr;
  if (blk->has_sc && !scb) return fail(ctx, VF_ESTATE, "missing weight tensor '%s.shortcut.bias'", p.c_str());
  int rc = upload_bn(ctx, p + ".bn1", &blk->bn1);
  if (rc) return rc;
  rc = upload_bn(ctx, p + ".bn2", &blk->bn2);
  if (rc) return rc;
  if (!skip_conv1) {
    rc = pack_conv3x3(ctx, &blk->conv1, *w1, nullptr, nullptr);
    if (rc) return rc;
  }
  if (skip_conv1) return pack_conv3x3(ctx, &blk->conv2, *w2, nullptr, nullptr);   // Cin = 1: shortcut precomputed
  return pack_conv3x3(ctx, &blk->conv2, *w2, scw, scb);
}

const int ENC_C[6] = {32, 64, 128, 256, 384, 384};
const int DEC_CIN[6] = {384, 384, 384, 256, 128, 64};
const int DEC_COUT[6] = {384, 384, 256, 128, 64, 32};

int build_tables(vf_ctx* ctx) {
  const double PI = 3.14159265358979323846;
  std::vector<float> win(2048);
  for (int i = 0; i < 2048; ++i) win[i] = (float)(0.5 - 0.5 * std::cos(2.0 * PI * i / 2048.0));
  std::vector<float2> t1(1024), t2(1025);
  for (int j = 0; j < 1024; ++j) t1[j] = make_float2((float)std::cos(2 * PI * j / 1024.0), (float)-std::sin(2 * PI * j / 1024.0));
  for (int k = 0; k <= 1024; ++k) t2[k] = make_float2((float)std::cos(2 * PI * k / 2048.0), (float)-std::sin(2 * PI * k / 2048.0));
  int rc = upload(ctx, &ctx->d_window, win);
  if (rc) return rc;
  rc = upload(ctx, &ctx->d_tw1024, t1);
  if (rc) return rc;
  rc = upload(ctx, &ctx->d_tw2048, t2);
  if (rc) return rc;
  std::vector<float> mw(128);
  for (int i = 0; i < 128; ++i) mw[i] = (float)(ctx->cfg.voc_mel_weight_a * std::exp(ctx->cfg.voc_mel_weight_b * i));
  return upload(ctx, &ctx->d_melw, mw);
}

bool has_prefix(vf_ctx* ctx, const std::string& prefix) {
  for (auto& kv : ctx->host_w)
    if (kv.first.compare(0, prefix.size(), prefix) == 0) return true;
  return false;
}

// One ResUNet under state-dict prefix U (unet.py:22-53 / unet_v2.py:46-77 registration names)
int load_unet(vf_ctx* ctx, const std::string& U, UnetW* w) {
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 4; ++j) {
      const std::string p = U + "encoder_block" + std::to_string(i + 1) + ".conv_block" + std::to_string(j + 1);
      int rc = load_block(ctx, p, &w->enc[i][j], i == 0 && j == 0);
      if (rc) return rc;
    }
  int rc;
  {
    const std::string p = U + "encoder_block1.conv_block1";
    std::vector<float> sc, sh;
    rc = fold_bn(ctx, p + ".bn1", &sc, &sh); if (rc) return rc;
    w->first_bn1_scale = sc[0]; w->first_bn1_shift = sh[0];
    NEED(w1, p + ".conv1.weight"); NEED(scw, p + ".shortcut.weight"); NEED(scb, p + ".shortcut.bias");
    if (w1->shape.size() != 4 || w1->shape[1] != 1) return fail(ctx, VF_EINVAL, "%s.conv1.weight: channels_in must be 1", p.c_str());
    rc = upload(ctx, &w->d_first_w1, w1->v); if (rc) return rc;
    rc = upload(ctx, &w->d_first_wsc, scw->v); if (rc) return rc;
    rc = upload(ctx, &w->d_first_bsc, scb->v); if (rc) return rc;
  }
  rc = load_block(ctx, U + "conv_block7", &w->bott, false); if (rc) return rc;
  for (int i = 0; i < 6; ++i) {
    const std::string p = U + "decoder_block" + std::to_string(i + 1);
    NEED(up, p + ".conv1.weight");
    rc = pack_convT2d(ctx, &w->dec_up[i], *up); if (rc) return rc;
    rc = upload_bn(ctx, p + ".bn1", &w->dec_bn1[i]); if (rc) return rc;
    for (int j = 0; j < 4; ++j) {
      rc = load_block(ctx, p + ".conv_block" + std::to_string(j + 2), &w->dec[i][j], false);
      if (rc) return rc;
    }
  }
  rc = load_block(ctx, U + "after_conv_block1", &w->post, false); if (rc) return rc;
  {
    NEED(hw, U + "after_conv2.weight"); NEED(hb, U + "after_conv2.bias");
    rc = upload(ctx, &w->d_head_w, hw->v); if (rc) return rc;
    w->head_b = hb->v[0];
  }
  w->loaded = true;
  return VF_OK;
}

// Residual add of a vocoder stack as an identity tap (through the accumulator, no epilogue loads) up to this channel count;
// above it the epilogue adds the hi/lo planes.  VF_TUNE_IDENT_MAXC overrides (read at weight-load AND plan-build time).
int ident_max_c() {
  if (const char* ov = getenv("VF_TUNE_IDENT_MAXC")) return atoi(ov);
  return 128;
}

int load_vocoder(vf_ctx* ctx) {
  int rc;
  const vf_config& c = ctx->cfg;
  ctx->voc_cond.resize(c.voc_cond_layers);
  for (int i = 0; i < c.voc_cond_layers; ++i) {
    NEED(w, "vocoder.condnet." + std::to_string(i) + ".weight"); NEED(b, "vocoder.condnet." + std::to_string(i) + ".bias");
    rc = pack_conv1d(ctx, &ctx->voc_cond[i], *w, *b); if (rc) return rc;
  }
  {
    NEED(w, "vocoder.stem.weight"); NEED(b, "vocoder.stem.bias");
    rc = pack_conv1d(ctx, &ctx->voc_stem, *w, *b); if (rc) return rc;
  }
  ctx->voc_up.resize(c.voc_num_stages);
  ctx->voc_res_a.assign(c.voc_num_stages, {});
  ctx->voc_res_b.assign(c.voc_num_stages, {});
  for (int s = 0; s < c.voc_num_stages; ++s) {
    NEED(w, "vocoder.up." + std::to_string(s) + ".weight"); NEED(b, "vocoder.up." + std::to_string(s) + ".bias");
    rc = pack_convT1d(ctx, &ctx->voc_up[s], *w, *b, c.voc_scales[s]); if (rc) return rc;
    ctx->voc_res_a[s].resize(c.voc_depth[s]);
    ctx->voc_res_b[s].resize(c.voc_depth[s]);
    for (int i = 0; i < c.voc_depth[s]; ++i) {
      const std::string p = "vocoder.res." + std::to_string(s) + "." + std::to_string(i);
      NEED(wa, p + ".a.weight"); NEED(ba, p + ".a.bias"); NEED(wb, p + ".b.weight"); NEED(bb, p + ".b.bias");
      rc = pack_conv1d(ctx, &ctx->voc_res_a[s][i], *wa, *ba); if (rc) return rc;
      rc = pack_conv1d(ctx, &ctx->voc_res_b[s][i], *wb, *bb, (int)wb->shape[0] <= ident_max_c()); if (rc) return rc;
    }
  }
  {
    NEED(w, "vocoder.tail.weight"); NEED(b, "vocoder.tail.bias");
    const int cl = (int)w->shape[1], k = (int)w->shape[2];
    if (k != 7) return fail(ctx, VF_EINVAL, "vocoder tail kernel must be 7");
    std::vector<float> t((size_t)7 * cl);
    for (int cch = 0; cch < cl; ++cch)
      for (int kk = 0; kk < 7; ++kk) t[(size_t)kk * cl + cch] = w->v[(size_t)cch * 7 + kk];
    rc = upload(ctx, &ctx->d_tail_w, t); if (rc) return rc;
    ctx->tail_b = b->v[0];
    ctx->voc_last_c = cl;
  }
  ctx->voc_loaded = true;
  return VF_OK;
}

const char* const GSR_PREFIX = "generator.analysis_module.";   // models/gsr_voicefixer.py:50,139
const char* const SSR_PREFIX = "generator.unet.";              // models/ssr_unet.py:49, models/gsr_unet.py:49

// Loads whichever of the three networks the descriptors hold (a VoiceFixer checkpoint: analysis module + vocoder;
// an SSR_UNet / GSR_UNet checkpoint: generator.unet.*).  A network that is present must be complete.
int load_all(vf_ctx* ctx) {
  // mel filterbank -> sparse rows (each triangular filter is one contiguous run of bins)
  {
    NEED(fb, "mel.fb");
    if (fb->shape.size() != 2 || fb->shape[0] != 1025 || fb->shape[1] != 128)
      return fail(ctx, VF_EINVAL, "mel.fb must be [1025,128]");
    std::vector<int> f0(128), len(128), ofs(128);
    std::vector<float> val;
    for (int m = 0; m < 128; ++m) {
      int lo = -1, hi = -1;
      for (int f = 0; f < 1025; ++f)
        if (fb->v[(size_t)f * 128 + m] != 0.f) { if (lo < 0) lo = f; hi = f; }
      if (lo < 0) { lo = 0; hi = -1; }
      f0[m] = lo; len[m] = hi - lo + 1; ofs[m] = (int)val.size();
      for (int f = lo; f <= hi; ++f) val.push_back(fb->v[(size_t)f * 128 + m]);
    }
    if (val.empty()) val.push_back(0.f);
    int rc = upload(ctx, &ctx->d_fb_f0, f0); if (rc) return rc;
    rc = upload(ctx, &ctx->d_fb_len, len); if (rc) return rc;
    rc = upload(ctx, &ctx->d_fb_ofs, ofs); if (rc) return rc;
    rc = upload(ctx, &ctx->d_fb_val, val); if (rc) return rc;
  }
  int rc = VF_OK, n_nets = 0;
  if (has_prefix(ctx, GSR_PREFIX)) { rc = load_unet(ctx, GSR_PREFIX, &ctx->gsr); if (rc) return rc; ++n_nets; }
  if (has_prefix(ctx, SSR_PREFIX)) { rc = load_unet(ctx, SSR_PREFIX, &ctx->ssr); if (rc) return rc; ++n_nets; }
  if (has_prefix(ctx, "vocoder.")) { rc = load_vocoder(ctx); if (rc) return rc; ++n_nets; }
  if (n_nets == 0)
    return fail(ctx, VF_ESTATE, "no network in the state: expected keys under '%s', '%s' or 'vocoder.'", GSR_PREFIX, SSR_PREFIX);
  return VF_OK;
}

// ------------------------------------------------------------------------------------------------ plans
struct Builder {
  vf_ctx* ctx;
  Plan* plan;
  int rc = VF_OK;
  std::string label;   // name given to the next op (profiling only)

  template <typename T>
  T* alloc(size_t count) {
    T* p = nullptr;
    if (rc) return nullptr;
    rc = dev_alloc(ctx, plan->allocs, plan->bytes, &p, count);
    return p;
  }
  Planes planes(size_t n_img, int img_rows, int C) {
    Planes pl;
    pl.C = C;
    pl.img_rows = img_rows;
    const size_t cnt = n_img * (size_t)img_rows * C;
    pl.p.hi = alloc<__half>(2 * cnt);        // [hi plane][lo plane]: one 4-D TMA box fetches both (3-term GEMMs)
    pl.p.lo = pl.p.hi ? pl.p.hi + cnt : nullptr;
    pl.plane_stride = cnt;
    return pl;
  }

  int make_map3(CUtensorMap* m, const __half* base, int C, int rows, int img_rows, int n_img, int box_c, bool sw128, int box_rows) {
    cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)rows, (cuuint64_t)n_img};
    cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)img_rows * C * 2};
    cuuint32_t box[3] = {(cuuint32_t)box_c, (cuuint32_t)box_rows, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)base, dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(A: C=%d rows=%d img_rows=%d n=%d box=%d) -> %d", C, rows, img_rows, n_img, box_c, (int)r);
    return VF_OK;
  }
  // generic [C, rows, image] map with SWIZZLE_128B (inner box = 128 bytes): TMA loads / stores of the fused pair kernel
  int make_map3_any(CUtensorMap* m, const void* base, CUtensorMapDataType dt, int esize, int C, int rows, size_t img_rows, int n_img,
                    int box_c, int box_rows) {
    cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)rows, (cuuint64_t)n_img};
    cuuint64_t strides[2] = {(cuuint64_t)C * esize, (cuuint64_t)img_rows * C * esize};
    cuuint32_t box[3] = {(cuuint32_t)box_c, (cuuint32_t)box_rows, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = ctx->encode(m, dt, 3, (void*)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(pair: C=%d rows=%d box=%dx%d esize=%d) -> %d", C, rows, box_c, box_rows, esize, (int)r);
    return VF_OK;
  }
  // epilogue TMA stores: fp16 plane(s) [ld, rows, image, plane], box 32 channels x 32 rows x 1 x planes, SWIZZLE_64B
  int make_map_out4(CUtensorMap* m, const __half* hi, const __half* lo, int planes, int ld, int rows, size_t img_rows, int n_img) {
    const size_t pstride = planes == 2 ? (size_t)(lo - hi) : (size_t)n_img * img_rows * ld;
    cuuint64_t dims[4] = {(cuuint64_t)ld, (cuuint64_t)rows, (cuuint64_t)n_img, (cuuint64_t)planes};
    cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)img_rows * ld * 2, (cuuint64_t)pstride * 2};
    cuuint32_t box[4] = {32, 32, 1, (cuuint32_t)planes};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)hi, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(out planes: ld=%d rows=%d planes=%d) -> %d", ld, rows, planes, (int)r);
    return VF_OK;
  }
  // activated planes of a transposed 1-D conv: output row t = s * q + p as [ld, p, q, image, plane], box 32 x 1 x 32 x 1 x planes
  int make_map_ct5(CUtensorMap* m, const __half* hi, const __half* lo, int planes, int ld, int s, long L, int n_img) {
    const size_t pstride = planes == 2 ? (size_t)(lo - hi) : (size_t)n_img * L * ld;
    cuuint64_t dims[5] = {(cuuint64_t)ld, (cuuint64_t)s, (cuuint64_t)(L / s), (cuuint64_t)n_img, (cuuint64_t)planes};      // strides ascending
    cuuint64_t strides[4] = {(cuuint64_t)ld * 2, (cuuint64_t)ld * 2 * s, (cuuint64_t)L * ld * 2, (cuuint64_t)pstride * 2};
    cuuint32_t box[5] = {32, 1, 32, 1, (cuuint32_t)planes};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)hi, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(convT1d out: ld=%d s=%d L=%ld planes=%d) -> %d", ld, s, L, planes, (int)r);
    return VF_OK;
  }
  // 3-term operands: hi and lo planes in ONE box ([C, rows, image, plane] / [K, N, plane]) - half the TMA issues
  int make_map4(CUtensorMap* m, const __half* base, int C, int rows, int img_rows, int n_img, size_t plane_stride, int box_c, bool sw128, int box_rows) {
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)rows, (cuuint64_t)n_img, 2};
    cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)img_rows * C * 2, (cuuint64_t)plane_stride * 2};
    cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_rows, 1, 2};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)base, dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(A hi+lo: C=%d rows=%d img_rows=%d n=%d box=%dx%d) -> %d", C, rows, img_rows, n_img, box_c, box_rows, (int)r);
    return VF_OK;
  }
  int make_map3w(CUtensorMap* m, const __half* base, int K, int N, int box_k, int box_n, bool sw128) {
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)N, 2};
    cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)N * K * 2};
    cuuint32_t box[3] = {(cuuint32_t)box_k, (cuuint32_t)box_n, 2};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)base, dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(B hi+lo: K=%d N=%d box=%dx%d) -> %d", K, N, box_k, box_n, (int)r);
    return VF_OK;
  }
  int make_map2(CUtensorMap* m, const __half* base, int K, int N, int box_k, int box_n, bool sw128) {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
    cuuint64_t strides[1] = {(cuuint64_t)K * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_k, (cuuint32_t)box_n};
    cuuint32_t es[2] = {1, 1};
    CUresult r = ctx->encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)base, dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, VF_ECUDA, "cuTensorMapEncodeTiled(B: K=%d N=%d box=%dx%d) -> %d", K, N, box_k, box_n, (int)r);
    return VF_OK;
  }

  // taps: nch = real channel count; k segments are laid out back to back, each padded to BK.
  void gemm(std::vector<Op>& ops, const GemmW& W, const ASrc& s0, const ASrc* s1, std::vector<GemmTap> taps,
            GemmEpilogue epi, int n_img, int terms) {
    if (rc) return;
    Op op;
    op.kind = OP_GEMM;
    int bk = 64;
    for (auto& t : taps)
      if (t.nch % 64) bk = 32;
    // a short tail segment (the 32-channel shortcut of a 64-channel conv) may be zero-padded to BK = 64 when
    // the source has exactly that many channels: the TMA box then runs out of bounds and is zero-filled.
    bool promoted = false;
    if (bk == 32) {
      bool main64 = true, padok = true;
      for (auto& t : taps) {
        const ASrc& s = t.src ? *s1 : s0;
        if (t.nch % 64) {
          if (t.nch % 32 || t.c_off + t.nch != s.pl.C) padok = false;
          if (&t != &taps.back()) main64 = false;
        }
      }
      if (main64 && padok && taps.size() > 1) { bk = 64; promoted = true; }
    }
    // K chunk width: every chunk costs the two single-thread issue loops a fixed ~0.5 us round (barrier wait, TMA /
    // MMA operand set-up), so wide chunks win even where narrow ones would allow one more co-resident CTA
    if (bk == 64 && !promoted) {
      int ksum = 0;
      for (auto& t : taps) ksum += t.nch;
      int maxk = 0;   // measured: halving the chunk count beats the extra co-resident CTA (voc.res3.a 1.43 -> 0.96 ms)
      if (const char* ov = getenv("VF_TUNE_BK32_MAXK")) maxk = atoi(ov);
      if (ksum <= maxk) bk = 32;
    }
    const int N = W.N;
    // 1-term (hi-only) GEMMs stream half the operand bytes per MMA, so they are L2-bandwidth bound at 128-wide
    // tiles: use 256-wide N tiles where the accumulator budget allows (one accumulator, double buffered)
    const int bn = (terms == 1 && N % 256 == 0) ? 256 : (N % 128 == 0) ? 128 : (N % 64 == 0) ? 64 : 32;
    if (N % 32) { rc = fail(ctx, VF_EINVAL, "GEMM N=%d not a multiple of 32", N); return; }
    if (terms == 1 && (epi.a_scale || epi.head_w || epi.out_raw || epi.resid)) {
      rc = fail(ctx, VF_EINVAL, "1-term GEMM with an affine / head / fp32 stream epilogue (3-term kernels only)");
      return;
    }
    // epilogue residual by TMA (gemm_tc.cu): one or two more 4 KB tiles per epilogue warp, requested that many chunks ahead;
    // VF_TUNE_TMA_RESID=0 keeps LDG + staging, =1 pins one tile in flight (default: two where the operand ring keeps its depth)
    const char* renv = getenv("VF_TUNE_TMA_RESID");
    const int resid_want = renv ? std::max(0, std::min(2, atoi(renv))) : 2;
    const int resid_tma = (resid_want && !ctx->validate_simt && epi.map == MAP_PLAIN &&
                           ((terms == 3 && epi.resid != nullptr) != (epi.resid_hi != nullptr))) ? 1 : 0;      // exactly one residual source
    int k = 0;
    for (auto& t : taps) {
      t.k_off = k;
      const int padded = round_up(t.nch, bk);
      k += padded;
      t.g = 1; t.shift[0] = t.shift[1] = t.shift[2] = 0; t.kstride = padded;
      if (ctx->validate_simt == 0) t.nch = padded;
    }
    // Halo groups: up to 3 consecutive taps reading row-adjacent windows of the same planes share one A load of
    // 128 + 2 rows; each tap is then an MMA on a row-shifted view (tools/probe_desc_shift.cu).  Worth it where the
    // layer is bound by shared-memory / L2 feed traffic (narrow N); wide-N tiles keep the finer-grained ring.
    int gmax = 1;
    {
      // measured (B = 32 x 10 s, same box): BN = 64 layers gain 8-17 %, BN = 32 layers 15-25 % (9x L2->SM re-reads of
      // the taps become 3x); a grouping whose stage no longer fits twice falls back to single taps
      bool want = ctx->validate_simt == 0;
      if (const char* ov = getenv("VF_TUNE_HALO")) {      // 0: never, 1: only BN = 64 and hi-only BN = 128 tiles
        if (atoi(ov) == 0) want = false;
        if (atoi(ov) == 1) want = want && (bn == 64 || (terms == 1 && bn == 128));
      }
      if (want) {
        std::vector<GemmTap> grouped;
        int gm = 1;
        bool any_both = false;
        for (auto& t : taps) any_both |= t.both != 0;
        for (size_t i = 0; i < taps.size();) {
          GemmTap gt = taps[i];
          size_t n = 1;
          int step = 0;
          while (n < 3 && i + n < taps.size()) {
            const GemmTap& a = taps[i + n - 1];
            const GemmTap& b2 = taps[i + n];
            const int d = b2.a_off - a.a_off;
            if (b2.src != gt.src || b2.c_off != gt.c_off || b2.nch != gt.nch || b2.both || gt.both || (d != 1 && d != -1)) break;
            if (n == 1) step = d; else if (d != step) break;
            ++n;
          }
          const int lo = std::min(taps[i].a_off, taps[i + n - 1].a_off);
          for (size_t j = 0; j < n; ++j) gt.shift[j] = taps[i + j].a_off - lo;
          gt.a_off = lo;
          gt.g = (int)n;
          gm = std::max(gm, gt.g);
          grouped.push_back(gt);
          i += n;
        }
        // a grouped stage holds up to 3 weight tiles: keep the grouping only if a 2-deep ring still fits
        int gchunks = 0;
        for (auto& t : grouped) gchunks += t.nch / bk;
        if (gm > 1 && gemm_tc_smem_bytes(bn, bk, 2, (terms == 3 || any_both) ? 2 : 1, terms, GEMM_BM + 2, gm, gchunks, resid_tma) <= (size_t)226 * 1024) {
          taps.swap(grouped);
          gmax = gm;
        }
      }
    }
    // halo boxes: 128 + 2 rows; 3-term GEMMs fetch the hi and lo planes in one 4-D box, whose planes land back to
    // back in shared memory, so the box is grown to a whole number of 1024-byte swizzle atoms (136 / 144 rows)
    const int a_box_rows = gmax > 1 ? (terms == 3 ? (bk == 64 ? 136 : 144) : GEMM_BM + 2) : GEMM_BM;
    if (k != W.K && k != W.K - W.k_tail) { rc = fail(ctx, VF_EINVAL, "GEMM K mismatch: taps cover %d, packed weight has %d", k, W.K); return; }
    GemmProblem pr;
    memset(&pr, 0, sizeof pr);
    pr.n_img = n_img;
    pr.m_tiles = (epi.rows_in + GEMM_BM - 1) / GEMM_BM;
    pr.N = N;
    pr.ntaps = (int)taps.size();
    pr.terms = terms;
    if (pr.ntaps > GEMM_MAX_TAPS) { rc = fail(ctx, VF_EINVAL, "too many taps"); return; }
    for (int i = 0; i < pr.ntaps; ++i) pr.taps[i] = taps[i];
    epi.err = ctx->d_err;
    pr.epi = epi;
    op.bn = bn;
    op.bk = bk;
    if (ctx->validate_simt) {
      GemmSimtParams& sp = op.simt;
      memset(&sp, 0, sizeof sp);
      const ASrc* srcs[2] = {&s0, s1};
      for (int i = 0; i < 2; ++i) {
        if (!srcs[i]) continue;
        const size_t off = (size_t)srcs[i]->row0 * srcs[i]->pl.C;
        sp.a_hi[i] = srcs[i]->pl.p.hi + off;
        sp.a_lo[i] = srcs[i]->pl.p.lo + off;
        sp.a_ld[i] = srcs[i]->pl.C;
        sp.a_rows[i] = srcs[i]->rows;
        sp.a_img_rows[i] = srcs[i]->pl.img_rows;
      }
      sp.b_hi = W.hi; sp.b_lo = W.lo; sp.ktot = W.K;
      sp.prob = pr;
    } else {
      GemmTcParams& tp = op.tc;
      memset(&tp, 0, sizeof tp);
      const ASrc* srcs[2] = {&s0, s1 ? s1 : &s0};
      for (int i = 0; i < 2 && !rc; ++i) {
        const size_t off = (size_t)srcs[i]->row0 * srcs[i]->pl.C;
        if (terms == 3) {
          if (srcs[i]->pl.plane_stride == 0) rc = fail(ctx, VF_EINVAL, "3-term GEMM source without adjacent hi/lo planes");
          if (!rc) rc = make_map4(&tp.a_hi[i], srcs[i]->pl.p.hi + off, srcs[i]->pl.C, srcs[i]->rows, srcs[i]->pl.img_rows, n_img, srcs[i]->pl.plane_stride, bk, bk == 64, a_box_rows);
        } else {
          rc = make_map3(&tp.a_hi[i], srcs[i]->pl.p.hi + off, srcs[i]->pl.C, srcs[i]->rows, srcs[i]->pl.img_rows, n_img, bk, bk == 64, a_box_rows);
          if (!rc) rc = make_map3(&tp.a_lo[i], srcs[i]->pl.p.lo + off, srcs[i]->pl.C, srcs[i]->rows, srcs[i]->pl.img_rows, n_img, bk, bk == 64, a_box_rows);
        }
      }
      if (terms == 3) {
        if (!rc) rc = make_map3w(&tp.b_hi, W.hi, W.K, N, bk, bn, bk == 64);
      } else {
        if (!rc) rc = make_map2(&tp.b_hi, W.hi, W.K, N, bk, bn, bk == 64);
        if (!rc) rc = make_map2(&tp.b_lo, W.lo, W.K, N, bk, bn, bk == 64);
      }
      // accumulation segments (see gemm_tc.cu): a bounded chain of truncating MMAs, then promotion to registers
      tp.tile_chunks = 0;
      for (auto& t : taps) tp.tile_chunks += t.nch / bk;           // ring slots (group chunks) per tile
      // K steps per truncating accumulation chain.  Longer chains = fewer promotion drains and a longer run-ahead of
      // the MMA thread while the epilogue warps are in their output phase (two TMEM buffers = two segments), but
      // more truncation drift.  Measured on the T = 1001 golden (max log-mel error, UNet ms): 16: 3.1e-5, 33.8;
      // 24: 3.8e-5, 32.0; 32: 4.1e-5, 31.0; 48: 5.5e-5, 30.1 (bar 1e-4).
      int seg_mmas = 24;
      if (const char* ov = getenv("VF_TUNE_SEG_MMAS")) seg_mmas = std::max(4, atoi(ov));
      tp.seg_chunks = std::max(1, seg_mmas / ((bk / 16) * gmax));
      tp.a_box_rows = a_box_rows;
      tp.gmax = gmax;
      bool any_both = false;
      for (auto& t : taps) any_both |= t.both != 0;
      tp.planes_a = (terms == 3 || any_both) ? 2 : 1;
      auto pow2 = [](int x) { int c = 32; while (c < x) c *= 2; return c; };
      // occupancy: small-K tiles are bound by loads/stores -> several persistent CTAs per SM; large-K -> one
      const int reg_limit = gemm_tc_max_ctas(bn);
      int ctas = (k <= 1024) ? reg_limit : 1;
      if (const char* ov = getenv("VF_TUNE_SMALLK_CTAS")) { if (k <= 1024) ctas = std::max(1, std::min(reg_limit, atoi(ov))); }
      {   // per tile shape: VF_TUNE_CTAS_<bn>_<terms>=n
        char key[48];
        snprintf(key, sizeof key, "VF_TUNE_CTAS_%d_%d", bn, terms);
        if (const char* ov = getenv(key)) { if (k <= 1024) ctas = std::max(1, std::min(reg_limit, atoi(ov))); }
      }
      tp.resid_tma = resid_tma;
      int stages = 0;
      for (; ctas >= 1; --ctas) {
        // accumulator buffers: four where TMEM allows (run-ahead of the MMA thread over the epilogue's output phase)
        const int acc_w = (terms == 3 ? 2 : 1) * bn;
        int nb_log = 1;
        if (pow2(4 * acc_w) * ctas <= 512) nb_log = 2;
        if (const char* ov = getenv("VF_TUNE_NBUF")) { if (atoi(ov) == 2) nb_log = 1; }
        tp.nbuf_log = nb_log;
        tp.tmem_cols = pow2((1 << nb_log) * acc_w);
        if (tp.tmem_cols * ctas > 512) continue;
        const size_t per_cta = (size_t)227 * 1024 / ctas - 1024;
        auto fit = [&](int ring) {
          int st = 8;
          for (; st >= 2; --st)
            if (gemm_tc_smem_bytes(bn, bk, st, tp.planes_a, terms, a_box_rows, gmax, tp.tile_chunks, ring) <= per_cta) break;
          return st;
        };
        stages = fit(tp.resid_tma);
        if (tp.resid_tma == 1 && resid_want == 2) {      // a second residual tile in flight if the operand ring stays deep enough
          const int st2 = fit(2);
          if (st2 >= 2 && (st2 == stages || st2 >= 4)) { tp.resid_tma = 2; stages = st2; }
        }
        if (stages >= 2) break;
        tp.resid_tma = resid_tma;
      }
      if (ctas < 1 || stages < 2) { rc = fail(ctx, VF_EINVAL, "no tcgen05 tile configuration fits (bn=%d bk=%d terms=%d)", bn, bk, terms); return; }
      tp.stages = stages;
      tp.ctas_per_sm = ctas;
      // MAP_PLAIN outputs leave the epilogue's staging tiles by TMA store (gemm_tc.cu); VF_TUNE_TMA_STORE=0 keeps LDS + STG
      {
        const char* tenv = getenv("VF_TUNE_TMA_STORE");
        const int want = tenv ? atoi(tenv) : 7;
        GemmEpilogue& pe = pr.epi;
        const int orows = pe.out_row0 + pe.rows_in;
        pe.tma_out = 0;
        if (tp.resid_tma) {
          if (terms == 3 && pe.resid) rc = make_map3_any(&tp.i_res, pe.resid, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, pe.resid_ld, pe.rows_in, (size_t)pe.rows_in, n_img, 32, 32);
          else rc = make_map_out4(&tp.i_res, pe.resid_hi, pe.resid_lo, 2, pe.resid_ld, pe.rows_in, (size_t)pe.rows_in, n_img);
          if (rc) return;
        }
        if (pe.map == MAP_CONVT1D && (want & 4) && !ctx->validate_simt && pe.out_a.hi && !pe.out_r.hi && !pe.out_raw && pe.out_row0 == 0 &&
            pe.out_rows_valid == pe.out_img_rows && pe.out_img_rows % pe.ct_stride == 0 && pe.out_a.ld % 8 == 0) {
          rc = make_map_ct5(&tp.o_a, pe.out_a.hi, pe.out_a.lo, (terms == 3 || pe.out_ar) ? 2 : 1, pe.out_a.ld, pe.ct_stride, pe.out_img_rows, n_img);
          if (rc) return;
          pe.tma_out |= 8;
        }
        if (pe.map == MAP_PLAIN && want) {
          if ((want & 1) && terms == 3 && pe.out_raw && pe.raw_ld % 4 == 0) {
            rc = make_map3_any(&tp.o_raw, pe.out_raw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, pe.raw_ld, orows, (size_t)pe.out_img_rows, n_img, 32, 32);
            if (rc) return;
            pe.tma_out |= 1;
          }
          if ((want & 2) && pe.out_r.hi) {
            rc = make_map_out4(&tp.o_r, pe.out_r.hi, pe.out_r.lo, 2, pe.out_r.ld, orows, (size_t)pe.out_img_rows, n_img);
            if (rc) return;
            pe.tma_out |= 2;
          }
          if ((want & 4) && pe.out_a.hi) {
            rc = make_map_out4(&tp.o_a, pe.out_a.hi, pe.out_a.lo, (terms == 3 || pe.out_ar) ? 2 : 1, pe.out_a.ld, orows, (size_t)pe.out_img_rows, n_img);
            if (rc) return;
            pe.tma_out |= 4;
          }
        }
      }
      const long total_tiles = (long)n_img * pr.m_tiles * (N / bn);
      tp.grid = (int)std::min<long>(total_tiles, (long)ctx->sm_count * ctas);
      tp.magic_n = gemm_tc_magic((uint32_t)(N / bn), (uint64_t)total_tiles);
      tp.magic_m = gemm_tc_magic((uint32_t)pr.m_tiles, (uint64_t)n_img * pr.m_tiles);
      tp.prob = pr;
    }
    {   // algorithmic work: the reference op's own MAC count and the minimum HBM traffic of this launch
      double kreal = 0;
      for (auto& t : taps) if (!t.both) kreal += (double)t.g * std::min(t.nch, (t.src ? s1 : &s0)->pl.C);
      const double wfrac = (epi.Wp > 1) ? double(epi.Wp - 1) / epi.Wp : 1.0;
      double rows = (double)n_img * (epi.map == MAP_CONVT1D ? epi.rows_in - 1 : epi.rows_in) * wfrac;
      op.flops = 2.0 * rows * N * kreal * (epi.map == MAP_CONVT2D ? 9.0 / 16.0 : 1.0);
      // bytes per source element: both fp16 planes in 3-term mode, and for a source that an identity tap contracts
      // with `both` (the hi/lo residual stream of the C <= 128 vocoder stacks); the hi plane alone otherwise
      bool s1_both = false;
      for (auto& t : taps) s1_both |= (t.src == 1 && t.both);
      double a_bytes = (double)n_img * s0.rows * s0.pl.C * (terms == 3 ? 4 : 2);
      if (s1) a_bytes += (double)n_img * s1->rows * s1->pl.C * ((terms == 3 || s1_both) ? 4 : 2);
      double kexec = 0;
      for (auto& t : taps) kexec += (double)t.g * round_up(t.nch, bk) * (terms == 3 ? 3 : (t.both ? 2 : 1));
      op.exec_flops = 2.0 * (double)n_img * pr.m_tiles * GEMM_BM * N * kexec;
      const double out_elems = (double)n_img * (epi.map == MAP_CONVT1D ? (double)epi.out_rows_valid * epi.cout
                                                : (epi.map == MAP_CONVT2D ? 4.0 * epi.rows_in * epi.cout : (double)epi.rows_in * N));
      op.bytes = a_bytes + (double)W.N * W.K * (terms == 3 ? 4 : 2) +
                 out_elems * ((epi.out_raw ? 4 : 0) + (epi.out_r.hi ? 4 : 0) + (epi.out_a.hi ? ((terms == 3 || epi.out_ar) ? 4 : 2) : 0) + ((epi.resid || epi.resid_hi) ? 4 : 0));
      snprintf(op.label, sizeof op.label, "%s", label.c_str());
    }
    ops.push_back(op);
  }
};

// (a, r) residual stream (gemm.cuh): fp16(1 / slope) in both halves of a word, 0 when the LeakyReLU is not invertible that way
uint32_t ar_inv_word(float slope) {
  if (!(slope > 0.f && slope <= 1.f)) return 0;
  const __half h = __float2half(1.f / slope);
  const uint32_t b = *reinterpret_cast<const unsigned short*>(&h);
  return b == 0x7c00u ? 0u : (b | (b << 16));
}

GemmEpilogue epi_plain(int rows_in, int Wp, int cout, int out_img_rows) {
  GemmEpilogue e;
  memset(&e, 0, sizeof e);
  e.map = MAP_PLAIN;
  e.rows_in = rows_in;
  e.Wp = Wp;
  e.cout = cout;
  e.out_img_rows = out_img_rows;
  e.out_rows_valid = out_img_rows;
  return e;
}
void set_out_a(GemmEpilogue& e, const Planes& pl, int c_off, const float* scale, const float* shift, int act, float slope) {
  e.out_a = OutPlane{pl.p.hi, pl.p.lo, pl.C, c_off};
  e.a_scale = scale;
  e.a_shift = shift;
  e.act = act;
  e.slope = slope;
}
// Column `byte_offset` of the per-clip table (null on the equal-length path): output rows at or past it are written as zeros
const int* vl_col(const VarlenImage* vl, size_t byte_offset) {
  return vl ? reinterpret_cast<const int*>(reinterpret_cast<const char*>(vl) + byte_offset) : nullptr;
}
void set_vl_rows(GemmEpilogue& e, const int* col) {
  e.vl_rows = col;
  e.vl_stride = VARLEN_STRIDE;
}
size_t vl_unet(int level) { return offsetof(VarlenImage, unet_rows) + sizeof(int) * level; }
size_t vl_voc(int stage) { return offsetof(VarlenImage, voc_len) + sizeof(int) * stage; }

std::vector<GemmTap> taps3x3(int Wp, int cin) {
  std::vector<GemmTap> t;
  for (int kh = 0; kh < 3; ++kh)
    for (int kw = 0; kw < 3; ++kw) t.push_back(GemmTap{(kh - 1) * Wp + (kw - 1), 0, 0, 0, cin});
  return t;
}

struct Level {
  int lvl, H, W, Wp, C, rows;
  float* raw[2];
  Planes aX, aT, cat_r, cat_a, P_r, P_a;   // P_* : pooled output of this level (input of the next)
  float* P_raw = nullptr;
};

// Geometry of one UNet instance: the mel-domain analysis module (unet.py: W0 = 127 of 128 mel bins, decoders prune the
// time axis only) or unet_v2 on linear magnitudes (unet_v2.py: W0 = 1024 of 1025 bins, both=True pruning).  Row pitch
// of level l is Wp = (W0 >> l) + 1: one shared zero pad column per image row (see gemm.cuh).
struct UnetGeom {
  int W0;                 // valid frequency bins fed to the first block
  const float* in;        // [B, T, W0 + 1] fp32 network input
  const float* head_in;   // [B, T, W0 + 1] residual added to the head output (gsr_voicefixer.py:90) or null (unet_v2.py:132)
  float* head_out;        // [B, T, W0 + 1]
  const char* tag;        // label prefix for profiles
};

int build_unet(vf_ctx* ctx, Builder& b, Plan* plan, const UnetW& U, const UnetGeom& G) {
  const int B = plan->batch, T = plan->T;
  const int Tp = (T + 63) / 64 * 64;
  std::vector<Op>& ops = plan->unet;
  const int terms = ctx->unet_terms;
  const float S = 0.01f;   // LeakyReLU slope, modules.py:265-266
  const VarlenImage* vl = plan->d_vl;
  Level lv[7];
  for (int l = 0; l < 7; ++l) {
    Level& L = lv[l];
    L.lvl = l; L.H = Tp >> l; L.W = G.W0 >> l; L.Wp = L.W + 1; L.C = l < 6 ? ENC_C[l] : 384; L.rows = L.H * L.Wp;
    L.raw[0] = b.alloc<float>((size_t)B * L.rows * L.C);
    L.raw[1] = b.alloc<float>((size_t)B * L.rows * L.C);
    L.aX = b.planes(B, L.rows, L.C);
    L.aT = b.planes(B, L.rows, L.C);
    if (l < 6) {
      L.cat_r = b.planes(B, L.rows, 2 * L.C);
      L.cat_a = b.planes(B, L.rows, 2 * L.C);
      const size_t prow = (size_t)(L.H / 2) * ((L.W >> 1) + 1);      // rows of the pooled level
      L.P_r = b.planes(B, (int)prow, L.C);
      L.P_a = b.planes(B, (int)prow, L.C);
      // the consumer of the pooled tensor needs it in fp32 when its shortcut is the identity (Cin == Cout)
      if (l == 5 || !U.enc[l + 1][0].has_sc) L.P_raw = b.alloc<float>((size_t)B * prow * L.C);
    }
  }
  if (b.rc) return b.rc;

  std::string tag;   // profiling label of the block being emitted
  const std::string pre = G.tag;
  // conv1 of a block: A -> aT with the block's bn2 + LeakyReLU
  auto conv1 = [&](const ConvBlockW& w, Level& L, const Planes& in) {
    b.label = tag + ".conv1";
    GemmEpilogue e = epi_plain(L.rows, L.Wp, w.cout, L.rows);
    set_out_a(e, L.aT, 0, w.bn2.scale, w.bn2.shift, ACT_LRELU, S);
    set_vl_rows(e, vl_col(vl, vl_unet(L.lvl)));
    b.gemm(ops, w.conv1, ASrc{in, L.rows, 0}, nullptr, taps3x3(L.Wp, w.cin), e, B, terms);
  };
  // conv2 of a block: aT (+ 1x1 shortcut of sc_src) (+ residual) -> outputs set by the caller
  auto conv2 = [&](const ConvBlockW& w, Level& L, const Planes* sc_src, const float* resid, GemmEpilogue e) {
    std::vector<GemmTap> taps = taps3x3(L.Wp, w.cout);
    ASrc s1;
    if (sc_src) {
      taps.push_back(GemmTap{0, 1, 0, 0, sc_src->C});
      s1 = ASrc{*sc_src, L.rows, 0};
      e.bias = w.conv2.bias;
    }
    e.resid = resid;
    e.resid_ld = w.cout;
    set_vl_rows(e, vl_col(vl, vl_unet(L.lvl)));
    b.label = tag + (sc_src ? ".conv2+sc" : ".conv2");
    b.gemm(ops, w.conv2, ASrc{L.aT, L.rows, 0}, sc_src ? &s1 : nullptr, taps, e, B, terms);
  };

  // ---------------- encoder
  for (int l = 0; l < 6; ++l) {
    Level& L = lv[l];
    int cur = 0;   // raw[cur] holds the block input
    for (int j = 0; j < 4; ++j) {
      const ConvBlockW& w = U.enc[l][j];
      tag = pre + "enc" + std::to_string(l + 1) + ".b" + std::to_string(j + 1);
      const float* resid = nullptr;
      const Planes* sc = nullptr;
      if (j == 0 && l == 0) {
        Op op; op.kind = OP_FIRST;
        UnetFirstParams& f = op.first;
        memset(&f, 0, sizeof f);
        f.logmel = G.in; f.batch = B; f.T = T; f.Tp = Tp; f.W = G.W0; f.in_ld = G.W0 + 1;
        f.bn1_scale = U.first_bn1_scale; f.bn1_shift = U.first_bn1_shift;
        f.w1 = U.d_first_w1; f.bn2_scale = w.bn2.scale; f.bn2_shift = w.bn2.shift;
        f.w_sc = U.d_first_wsc; f.b_sc = U.d_first_bsc; f.slope = S;
        f.a2 = L.aT.p; f.sc_raw = L.raw[0]; f.err = ctx->d_err; f.vl = vl;
        ops.push_back(op);
        resid = L.raw[0];      // precomputed shortcut(x) acts as the residual
        cur = 0;
      } else if (j == 0) {
        conv1(w, L, lv[l - 1].P_a);
        if (w.has_sc) sc = &lv[l - 1].P_r;
        else resid = lv[l - 1].P_raw;      // encoder_block6: 384 -> 384, identity shortcut
        cur = 1;               // output goes to raw[0]
      } else {
        conv1(w, L, L.aX);
        resid = L.raw[cur];
      }
      GemmEpilogue e = epi_plain(L.rows, L.Wp, w.cout, L.rows);
      const int dst = (j == 0 && l > 0) ? 0 : 1 - cur;
      e.out_raw = L.raw[dst];
      e.raw_ld = L.C;
      if (j < 3) {
        const ConvBlockW& nx = U.enc[l][j + 1];
        set_out_a(e, L.aX, 0, nx.bn1.scale, nx.bn1.shift, ACT_LRELU, S);
      } else {
        // skip connection: raw and activated halves of the decoder's concat buffer (modules.py:215)
        const ConvBlockW& dblk = U.dec[5 - l][0];
        e.out_r = OutPlane{L.cat_r.p.hi, L.cat_r.p.lo, 2 * L.C, L.C};
        set_out_a(e, L.cat_a, L.C, dblk.bn1.scale + L.C, dblk.bn1.shift + L.C, ACT_LRELU, S);
      }
      conv2(w, L, sc, resid, e);
      cur = dst;
    }
    // avg_pool2d(2,2) -> next stage's (or the bottleneck's) bn1 + LeakyReLU
    Op op; op.kind = OP_POOL;
    PoolParams& p = op.pool;
    memset(&p, 0, sizeof p);
    const ConvBlockW& nx = l < 5 ? U.enc[l + 1][0] : U.bott;
    p.in = L.raw[cur]; p.batch = B; p.H = L.H; p.Wp = L.Wp; p.C = L.C; p.Wpo = (L.W >> 1) + 1;
    p.out_r = L.P_r.p; p.out_a = L.P_a.p; p.out_raw = L.P_raw;
    p.a_scale = nx.bn1.scale; p.a_shift = nx.bn1.shift; p.slope = S; p.err = ctx->d_err;
    p.vl = vl; p.vl_level = l + 1;
    ops.push_back(op);
  }
  // ---------------- bottleneck (conv_block7, identity shortcut) -> decoder_block1.bn1 + ReLU
  {
    Level& L = lv[6];
    tag = pre + "bottleneck";
    conv1(U.bott, L, lv[5].P_a);
    GemmEpilogue e = epi_plain(L.rows, L.Wp, 384, L.rows);
    set_out_a(e, L.aX, 0, U.dec_bn1[0].scale, U.dec_bn1[0].shift, ACT_LRELU, 0.f);
    conv2(U.bott, L, nullptr, lv[5].P_raw, e);
  }
  // ---------------- decoder
  for (int k = 0; k < 6; ++k) {
    Level& L = lv[5 - k];
    Level& Lin = lv[6 - k];
    const int cin = DEC_CIN[k], cout = DEC_COUT[k];
    {   // ConvTranspose2d k3 s2 + prune + concat placement (modules.py:213-215)
      GemmEpilogue e;
      memset(&e, 0, sizeof e);
      e.map = MAP_CONVT2D; e.rows_in = Lin.rows; e.Wp = Lin.Wp; e.cout = cout; e.out_img_rows = L.rows;
      e.out_rows_valid = L.rows;
      e.ct_out_wp = L.Wp;      // 2 * Lin.Wp (time-only prune, modules.py:209) or 2 * Lin.Wp - 1 (both=True, modules.py:207-208)
      set_vl_rows(e, vl_col(vl, vl_unet(L.lvl)));
      const ConvBlockW& blk = U.dec[k][0];
      e.out_r = OutPlane{L.cat_r.p.hi, L.cat_r.p.lo, 2 * L.C, 0};
      set_out_a(e, L.cat_a, 0, blk.bn1.scale, blk.bn1.shift, ACT_LRELU, S);
      std::vector<GemmTap> taps;
      for (int dh = 0; dh < 2; ++dh)
        for (int dw = 0; dw < 2; ++dw) taps.push_back(GemmTap{-(dh * Lin.Wp + dw), 0, 0, 0, cin});
      b.label = pre + "dec" + std::to_string(k + 1) + ".convT";
      b.gemm(ops, U.dec_up[k], ASrc{Lin.aX, Lin.rows, 0}, nullptr, taps, e, B, terms);
    }
    int cur = 0;
    for (int j = 0; j < 4; ++j) {
      const ConvBlockW& w = U.dec[k][j];
      tag = pre + "dec" + std::to_string(k + 1) + ".b" + std::to_string(j + 2);
      const float* resid = nullptr;
      const Planes* sc = nullptr;
      if (j == 0) { conv1(w, L, L.cat_a); sc = &L.cat_r; }
      else { conv1(w, L, L.aX); resid = L.raw[cur]; }
      GemmEpilogue e = epi_plain(L.rows, L.Wp, w.cout, L.rows);
      const int dst = j == 0 ? 0 : 1 - cur;
      if (j < 3) {
        const ConvBlockW& nx = U.dec[k][j + 1];
        e.out_raw = L.raw[dst]; e.raw_ld = L.C;
        set_out_a(e, L.aX, 0, nx.bn1.scale, nx.bn1.shift, ACT_LRELU, S);
      } else if (k < 5) {
        set_out_a(e, L.aX, 0, U.dec_bn1[k + 1].scale, U.dec_bn1[k + 1].shift, ACT_LRELU, 0.f);   // ReLU, modules.py:213
      } else {
        e.out_raw = L.raw[dst]; e.raw_ld = L.C;
        set_out_a(e, L.aX, 0, U.post.bn1.scale, U.post.bn1.shift, ACT_LRELU, S);
      }
      conv2(w, L, sc, resid, e);
      cur = dst;
    }
    if (k == 5) {   // after_conv_block1 + after_conv2 head + log-mel residual
      tag = pre + "post";
      conv1(U.post, L, L.aX);
      GemmEpilogue e = epi_plain(L.rows, L.Wp, 32, L.rows);
      e.head_w = U.d_head_w; e.head_b = U.head_b;
      e.head_in = G.head_in; e.head_out = G.head_out; e.head_T = T;
      e.vl_head_T = vl_col(vl, offsetof(VarlenImage, T));      // conv2 sets vl_stride
      conv2(U.post, L, nullptr, L.raw[cur], e);
    }
  }
  return b.rc;
}

int build_vocoder(vf_ctx* ctx, Builder& b, Plan* plan) {
  const vf_config& c = ctx->cfg;
  const int B = plan->batch, T = plan->T;
  const int Tv = T + T % 2 + c.voc_tail_base;
  const int terms = ctx->voc_terms;
  std::vector<Op>& ops = plan->vocoder;
  const int CC = c.voc_cond_channels;
  const VarlenImage* vl = plan->d_vl;

  Planes cond = b.planes(B, Tv, 128);
  Planes c0 = b.planes(B, Tv, CC), c1 = b.planes(B, Tv, CC);
  Planes cpad = b.planes(B, Tv + 6, CC);
  Planes stem = b.planes(B, Tv, c.voc_channels);
  if (b.rc) return b.rc;
  {
    Op op; op.kind = OP_COND;
    VocCondParams& p = op.cond;
    memset(&p, 0, sizeof p);
    p.mel = plan->d_logmel_out; p.is_log = 1; p.batch = B; p.T = T; p.Tv = Tv; p.weight = ctx->d_melw;
    p.amp_floor = c.voc_amp_floor; p.ref_db = c.voc_ref_db; p.min_db = c.voc_min_db; p.tail_value = c.voc_tail_value;
    p.out = cond.p; p.vl = vl;
    plan->cond_op = (int)ops.size();
    ops.push_back(op);
  }
  auto taps1d = [](int k, int dil, int cin, bool centered) {
    std::vector<GemmTap> t;
    for (int i = 0; i < k; ++i) t.push_back(GemmTap{centered ? (i - (k - 1) / 2) * dil : i, 0, 0, 0, cin});
    return t;
  };
  Planes cur = cond;
  for (int i = 0; i < c.voc_cond_layers; ++i) {
    const bool last = i == c.voc_cond_layers - 1;
    Planes dst = last ? cpad : (i % 2 ? c1 : c0);
    GemmEpilogue e = epi_plain(Tv, 0, CC, dst.img_rows);
    e.out_row0 = last ? 3 : 0;
    e.bias = ctx->voc_cond[i].bias;
    set_out_a(e, dst, 0, nullptr, nullptr, ACT_ELU, 0.f);
    set_vl_rows(e, vl_col(vl, vl_voc(0)));
    b.label = "voc.cond" + std::to_string(i);
    b.gemm(ops, ctx->voc_cond[i], ASrc{cur, Tv, 0}, nullptr, taps1d(3, 1, cur.C, true), e, B, terms);
    cur = dst;
  }
  { Op op; op.kind = OP_REFLECT; op.refl.pl = cpad.p; op.refl.batch = B; op.refl.L = Tv; op.refl.C = CC; op.refl.pad = 3;
    op.refl.vl = vl; op.refl.vl_stage = 0; ops.push_back(op); }
  {
    GemmEpilogue e = epi_plain(Tv, 0, c.voc_channels, Tv);
    e.bias = ctx->voc_stem.bias;
    set_out_a(e, stem, 0, nullptr, nullptr, ACT_LRELU, c.voc_stage_slope);
    set_vl_rows(e, vl_col(vl, vl_voc(0)));
    b.label = "voc.stem";
    b.gemm(ops, ctx->voc_stem, ASrc{cpad, Tv + 6, 0}, nullptr, taps1d(7, 1, CC, false), e, B, terms);
  }
  Planes prev = stem;
  long Lprev = Tv;
  int cin = c.voc_channels;
  for (int s = 0; s < c.voc_num_stages; ++s) {
    const int sc = c.voc_scales[s], cout = cin / 2;
    if (vl && sc > 24) return fail(ctx, VF_EINVAL, "varlen vocoder: up-sampling scale %d above 24 (one flag bit per phase)", sc);
    const long L = Lprev * sc;
    const bool last_stage = s == c.voc_num_stages - 1;
    // C = 64 stacks in the hi-only mode: one kernel per residual pair (pair_tc.cu), the intermediate h stays in shared
    // memory and the residual stream of the stack is fp32.  Measured 2.33 vs 2.49 ms per pair against the two GEMM launches
    // (B = 32 x 10 s); VF_TUNE_FUSED_PAIR=0 selects the two-launch path.  Its activated input and output planes must differ
    // (a tile reads rows up to `dil` away from the ones another CTA is writing), so the pairs ping-pong between xa and xa2.
    const char* fenv = getenv("VF_TUNE_FUSED_PAIR");
    const bool fused = !(fenv && atoi(fenv) == 0) && !ctx->validate_simt && terms == 1 && cout == 64;
    // (a, r) residual stream of the hi-only mode (gemm.cuh): x lives in the activated plane the convs read anyway plus one
    // fp16 correction plane (the otherwise unused lo plane of the same allocation), updated in place by every residual layer:
    // 10 instead of 12 bytes per element through a two-launch pair, 8 instead of 12 through a fused pair.  VF_TUNE_AR_STREAM=0
    // keeps separate hi/lo planes of x (and the fp32 stream of the fused stacks).
    const char* aenv = getenv("VF_TUNE_AR_STREAM");
    const uint32_t ar = (!(aenv && atoi(aenv) == 0) && !ctx->validate_simt && terms == 1) ? ar_inv_word(c.voc_res_slope) : 0u;
    // residual stream x as hi/lo planes (ping-pong; a fused stack only reads the first, written by the transposed conv)
    Planes xr[2] = {ar ? Planes() : b.planes(B, (int)L, cout), (fused || ar) ? Planes() : b.planes(B, (int)L, cout)};
    Planes xa = b.planes(B, (int)L, cout), ha = fused ? Planes() : b.planes(B, (int)L, cout);
    Planes tail_in;
    if (last_stage) tail_in = b.planes(B, (int)L + 6, cout);
    if (b.rc) return b.rc;
    {   // ConvTranspose1d: rows q = 0..Lprev produce s phases each
      GemmEpilogue e;
      memset(&e, 0, sizeof e);
      e.map = MAP_CONVT1D; e.rows_in = (int)Lprev + 1; e.cout = cout; e.out_img_rows = (int)L; e.out_rows_valid = (int)L;
      e.ct_stride = sc; e.ct_pad = sc / 2 + sc % 2;
      e.bias = ctx->voc_up[s].bias;
      if (ar) e.out_ar = ar;
      else e.out_r = OutPlane{xr[0].p.hi, xr[0].p.lo, cout, 0};
      set_out_a(e, xa, 0, nullptr, nullptr, ACT_LRELU, c.voc_res_slope);
      set_vl_rows(e, vl_col(vl, vl_voc(s + 1)));
      std::vector<GemmTap> taps = {GemmTap{0, 0, 0, 0, cin}, GemmTap{-1, 0, 0, 0, cin}};
      b.label = "voc.up" + std::to_string(s);
      b.gemm(ops, ctx->voc_up[s], ASrc{prev, (int)Lprev, 0}, nullptr, taps, e, B, terms);
    }
    int curx = 0;
    Planes xa2;
    float* xf[2] = {nullptr, nullptr};       // fp32 residual stream of a fused stack (ping-pong)
    if (fused) {
      xa2 = b.planes(B, (int)L, cout);
      if (!ar) {
        xf[0] = b.alloc<float>((size_t)B * L * cout);
        xf[1] = b.alloc<float>((size_t)B * L * cout);
      }
    }
    if (b.rc) return b.rc;
    int cura = 0;
    for (int i = 0; i < c.voc_depth[s]; ++i) {
      int dil = 1;
      for (int q = 0; q < i % 10; ++q) dil *= 3;
      const bool last = i == c.voc_depth[s] - 1;
      if (fused) {
        Planes src = cura ? xa2 : xa;
        Planes dst = (last && last_stage) ? tail_in : (cura ? xa : xa2);
        Op op;
        op.kind = OP_PAIR;
        PairParams& pp = op.pair;
        memset(&pp, 0, sizeof pp);
        int mrc = b.make_map3(&pp.a_map, src.p.hi, cout, (int)L, src.img_rows, B, 64, true, GEMM_BM);
        if (!mrc) mrc = b.make_map2(&pp.wa_map, ctx->voc_res_a[s][i].hi, ctx->voc_res_a[s][i].K, cout, 64, cout, true);
        if (!mrc) mrc = b.make_map2(&pp.wb_map, ctx->voc_res_b[s][i].hi, ctx->voc_res_b[s][i].K, cout, 64, cout, true);
        if (mrc) return mrc;
        pp.bias_a = ctx->voc_res_a[s][i].bias;
        pp.bias_b = ctx->voc_res_b[s][i].bias;
        const int orow0 = (last && last_stage) ? 3 : 0;
        if (ar) {            // (a, r) stream: the residual is rebuilt from the activated plane (an L2 hit: the centre tap just read
          pp.ar_in = ar;     // these rows) and the correction plane; the new pair leaves as the two planes of `dst`
          mrc = b.make_map3_any(&pp.xin_map[0], src.p.hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, cout, (int)L, (size_t)src.img_rows, B, 64, 126);
          if (!mrc) mrc = b.make_map3_any(&pp.xin_map[1], src.p.lo, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, cout, (int)L, (size_t)src.img_rows, B, 64, 126);
          if (!mrc && !last) {
            pp.ar_out = ar;
            mrc = b.make_map3_any(&pp.xo_map, dst.p.lo, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, cout, (int)L, (size_t)dst.img_rows, B, 64, 126);
          }
        } else if (i == 0) {        // the stack's input: hi / lo planes written by the transposed conv above
          mrc = b.make_map3_any(&pp.xin_map[0], xr[0].p.hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, cout, (int)L, (size_t)L, B, 64, 126);
          if (!mrc) mrc = b.make_map3_any(&pp.xin_map[1], xr[0].p.lo, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, cout, (int)L, (size_t)L, B, 64, 126);
        } else {
          pp.in_f32 = 1;
          mrc = b.make_map3_any(&pp.xin_map[0], xf[curx], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, cout, (int)L, (size_t)L, B, 32, 126);
        }
        if (!mrc && !last && !ar) {
          pp.out_f32 = 1;
          mrc = b.make_map3_any(&pp.xo_map, xf[1 - curx], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, cout, (int)L, (size_t)L, B, 32, 126);
        }
        if (!mrc) mrc = b.make_map3_any(&pp.ao_map, dst.p.hi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, cout, orow0 + (int)L, (size_t)dst.img_rows, B, 64, 126);
        if (mrc) return mrc;
        pp.L = (int)L; pp.n_img = B; pp.C = cout; pp.dil = dil;
        pp.out_img_rows = dst.img_rows;
        pp.out_row0 = (last && last_stage) ? 3 : 0;
        pp.tiles_per_img = (int)((L + 125) / 126);
        const long total_tiles = (long)B * pp.tiles_per_img;
        if (pair_tc_smem_bytes(cout, 0) == 0) return fail(ctx, VF_EINVAL, "fused pair: C=%d not built", cout);
        pp.stages = 2;
        pp.grid = (int)std::min<long>(total_tiles, (long)ctx->sm_count);      // one persistent CTA per SM (211 KB of shared memory)
        pp.magic_t = gemm_tc_magic((uint32_t)pp.tiles_per_img, (uint64_t)total_tiles);
        pp.slope_h = c.voc_res_slope;
        pp.slope_out = last ? c.voc_stage_slope : c.voc_res_slope;
        pp.err = ctx->d_err;
        pp.vl_len = vl_col(vl, vl_voc(s + 1)); pp.vl_stride = VARLEN_STRIDE;
        op.flops = 2.0 * 2.0 * (double)B * L * cout * 3.0 * cout;
        op.exec_flops = 2.0 * 2.0 * (double)B * pp.tiles_per_img * GEMM_BM * cout * 3.0 * cout;
        op.bytes = ar ? (double)B * L * cout * (2 + 2 + (last ? 0 : 2) + 2)    // act in (operand and residual), r in, r out, act out
                      : (double)B * L * cout * (2 + 4 + (last ? 0 : 4) + 2);   // act in, x in, x_new out, act out
        snprintf(op.label, sizeof op.label, "voc.res%d.%d.pair", s, i);
        ops.push_back(op);
        curx = 1 - curx;
        cura = 1 - cura;
        continue;
      }
      {
        GemmEpilogue e = epi_plain((int)L, 0, cout, (int)L);
        e.bias = ctx->voc_res_a[s][i].bias;
        set_out_a(e, ha, 0, nullptr, nullptr, ACT_LRELU, c.voc_res_slope);
        set_vl_rows(e, vl_col(vl, vl_voc(s + 1)));
        b.label = "voc.res" + std::to_string(s) + "." + std::to_string(i) + ".a";
        b.gemm(ops, ctx->voc_res_a[s][i], ASrc{xa, (int)L, 0}, nullptr, taps1d(3, dil, cout, true), e, B, terms);
      }
      {
        Planes dst = (last && last_stage) ? tail_in : xa;
        GemmEpilogue e = epi_plain((int)L, 0, cout, dst.img_rows);
        e.out_row0 = (last && last_stage) ? 3 : 0;
        e.bias = ctx->voc_res_b[s][i].bias;
        if (!last) {
          if (ar) e.out_ar = ar;
          else e.out_r = OutPlane{xr[1 - curx].p.hi, xr[1 - curx].p.lo, cout, 0};
        }
        set_out_a(e, dst, 0, nullptr, nullptr, ACT_LRELU, last ? c.voc_stage_slope : c.voc_res_slope);
        set_vl_rows(e, vl_col(vl, vl_voc(s + 1)));
        b.label = "voc.res" + std::to_string(s) + "." + std::to_string(i) + ".b";
        std::vector<GemmTap> taps = taps1d(3, 1, cout, true);
        ASrc xsrc{xr[curx], (int)L, 0};
        if (ar) {
          // x = U(a) + r from the two planes of xa, rewritten in place: a tile reads exactly the rows it writes, and only
          // the "a" conv of the next pair (a later launch) looks at neighbouring rows
          e.resid_hi = xa.p.hi; e.resid_lo = xa.p.lo; e.resid_ld = cout; e.resid_ar = ar;
          b.gemm(ops, ctx->voc_res_b[s][i], ASrc{ha, (int)L, 0}, nullptr, taps, e, B, terms);
        } else if (cout <= ident_max_c()) {
          // load/store-bound stacks: x rides through the accumulator (identity weights, both planes) and the
          // epilogue issues no global loads
          taps.push_back(GemmTap{0, 1, 0, 0, cout, 1});
          b.gemm(ops, ctx->voc_res_b[s][i], ASrc{ha, (int)L, 0}, &xsrc, taps, e, B, terms);
        } else {
          // MMA-bound stacks: the identity tap would add ~40% tensor work; add the planes in the epilogue instead
          e.resid_hi = xr[curx].p.hi; e.resid_lo = xr[curx].p.lo; e.resid_ld = cout;
          b.gemm(ops, ctx->voc_res_b[s][i], ASrc{ha, (int)L, 0}, nullptr, taps, e, B, terms);
        }
        curx = 1 - curx;
      }
    }
    if (last_stage) {
      { Op op; op.kind = OP_REFLECT; op.refl.pl = tail_in.p; op.refl.batch = B; op.refl.L = (int)L; op.refl.C = cout; op.refl.pad = 3;
        op.refl.vl = vl; op.refl.vl_stage = c.voc_num_stages; ops.push_back(op); }
      plan->L = L;
      plan->d_voc_wav = b.alloc<float>((size_t)B * L);
      plan->d_peak = b.alloc<unsigned int>(B);
      if (b.rc) return b.rc;
      { Op op; op.kind = OP_MEMSET32; op.ms.p = plan->d_peak; op.ms.bytes = (size_t)B * 4; ops.push_back(op); }
      Op op; op.kind = OP_TAIL;
      VocTailParams& p = op.tail;
      memset(&p, 0, sizeof p);
      p.in = tail_in.p; p.batch = B; p.L = (int)L; p.C = cout; p.terms = terms; p.w = ctx->d_tail_w; p.bias = ctx->tail_b;
      p.wav = plan->d_voc_wav; p.peak_bits = plan->d_peak; p.tanh_out = c.voc_tail_tanh; p.vl = vl;
      ops.push_back(op);
    }
    prev = (fused && cura) ? xa2 : xa;
    Lprev = L;
    cin = cout;
  }
  return b.rc;
}

// SSR / GSR-UNet plan (models/ssr_unet.py:145-155 -> unet_v2.py:86-148): STFT magnitude -> unet_v2 on 1024 bins -> the
// predicted magnitude with the input's phase -> ISTFT.  Frames and the magnitude planes are the only extra buffers.
int build_ssr(vf_ctx* ctx, Builder& b, Plan* plan) {
  const size_t sp_n = (size_t)plan->batch * plan->T * 1025;
  plan->d_sp = b.alloc<float>(sp_n);
  plan->d_mag = b.alloc<float>(sp_n);
  plan->d_frames = b.alloc<float>((size_t)plan->batch * plan->T * 2048);
  if (b.rc) return b.rc;
  UnetGeom g{1024, plan->d_sp, nullptr, plan->d_mag, "ssr."};
  return build_unet(ctx, b, plan, ctx->ssr, g);
}

void free_plan(Plan* plan) {
  for (auto& g : plan->graph)
    if (g) { cudaGraphExecDestroy(g); g = nullptr; }
  for (auto& row : plan->io_ev)
    for (auto& e : row)
      if (e) { cudaEventDestroy(e); e = nullptr; }
  if (plan->ev_last) { cudaEventDestroy(plan->ev_last); plan->ev_last = nullptr; }
  for (void* p : plan->allocs) cudaFree(p);
  plan->allocs.clear();
}

void drop_all_plans(vf_ctx* ctx) {
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto& kv : ctx->plans) free_plan(kv.second.get());
  ctx->plans.clear();
  ctx->plan_bytes = 0;
}

// Plans are cached per (kind, batch, frames) - a file-dependent tail segment or a ragged last chunk gets its own
// shape - so the cache is bounded: least-recently-used plans are freed once the cached workspaces exceed the budget
// (option "plan_cache_mb"; default: half of the device memory that was free at the first plan).  The reference
// handler runs in constant memory (eval_gsr_voicefixer.py:49-74); so does a run over any number of distinct lengths.
int evict_plans(vf_ctx* ctx, size_t incoming, const Plan* keep) {
  if (ctx->plan_budget == 0) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return fail(ctx, VF_ECUDA, "cudaMemGetInfo failed");
    ctx->plan_budget = std::max<size_t>((free_b + ctx->plan_bytes) / 2, (size_t)1 << 30);
  }
  bool synced = false;
  while (!ctx->plans.empty() && ctx->plan_bytes + incoming > ctx->plan_budget) {
    auto victim = ctx->plans.end();
    for (auto it = ctx->plans.begin(); it != ctx->plans.end(); ++it)
      if (it->second.get() != keep && (victim == ctx->plans.end() || it->second->last_use < victim->second->last_use)) victim = it;
    if (victim == ctx->plans.end()) break;
    if (!synced) { cudaDeviceSynchronize(); synced = true; }     // the victim may still be executing on some stream
    ctx->plan_bytes -= std::min(ctx->plan_bytes, victim->second->bytes);
    free_plan(victim->second.get());
    ctx->plans.erase(victim);
    ctx->plans_evicted++;
  }
  return VF_OK;
}

int build_ssr(vf_ctx* ctx, Builder& b, Plan* plan);

int get_plan(vf_ctx* ctx, int kind, int batch, int frames, Plan** out) {
  const auto key = std::make_tuple(kind, batch, (long)frames);
  auto it = ctx->plans.find(key);
  if (it != ctx->plans.end()) { it->second->last_use = ++ctx->use_clock; *out = it->second.get(); return VF_OK; }
  if (!ctx->loaded) return fail(ctx, VF_ESTATE, "weights not loaded");
  if ((kind == PLAN_GSR || kind == PLAN_GSR_VARLEN) && !(ctx->gsr.loaded && ctx->voc_loaded))
    return fail(ctx, VF_ESTATE, "this entry point needs the analysis module (generator.analysis_module.*) and the vocoder (vocoder.*) weights");
  if ((kind == PLAN_SSR || kind == PLAN_SSR_VARLEN) && !ctx->ssr.loaded)
    return fail(ctx, VF_ESTATE, "this entry point needs the unet_v2 weights (generator.unet.*)");
  // make room first: a failed cudaMalloc half way through a plan is slower to recover from than an early eviction
  {
    size_t est = 0;
    for (auto& kv : ctx->plans)
      if (std::get<0>(kv.first) == kind) {     // bytes scale with batch * padded frames
        const double r = ((double)batch * ((frames + 63) / 64 * 64)) / ((double)kv.second->batch * ((kv.second->T + 63) / 64 * 64));
        est = (size_t)(r * (double)kv.second->bytes);
        break;
      }
    int rc = evict_plans(ctx, est, nullptr);
    if (rc) return rc;
  }
  std::unique_ptr<Plan> plan(new Plan);
  plan->kind = kind; plan->batch = batch; plan->T = frames;
  Builder b{ctx, plan.get()};
  int rc = VF_OK;
  if (kind == PLAN_GSR || kind == PLAN_GSR_VARLEN) {
    if (kind == PLAN_GSR_VARLEN) plan->d_vl = b.alloc<VarlenImage>(batch);     // before the builders: their ops point into it
    const size_t mel_n = (size_t)batch * frames * 128;
    plan->d_mel = b.alloc<float>(mel_n);
    plan->d_logmel_in = b.alloc<float>(mel_n);
    plan->d_logmel_out = b.alloc<float>(mel_n);
    plan->d_band = b.alloc<float>(2 * (size_t)batch);
    rc = b.rc;
    UnetGeom g{127, plan->d_logmel_in, plan->d_logmel_in, plan->d_logmel_out, ""};
    if (!rc) rc = build_unet(ctx, b, plan.get(), ctx->gsr, g);
    if (!rc) rc = build_vocoder(ctx, b, plan.get());
  } else {
    if (kind == PLAN_SSR_VARLEN) plan->d_vl = b.alloc<VarlenImage>(batch);      // before build_unet: its ops point into it
    rc = b.rc;
    if (!rc) rc = build_ssr(ctx, b, plan.get());
  }
  if (rc == VF_ECUDA && !ctx->plans.empty()) {
    // out of memory with other plans cached: drop them all and retry once
    free_plan(plan.get());
    cudaGetLastError();
    drop_all_plans(ctx);
    return get_plan(ctx, kind, batch, frames, out);
  }
  if (rc) {
    free_plan(plan.get());
    return rc;
  }
  plan->last_use = ++ctx->use_clock;
  ctx->plan_bytes += plan->bytes;
  *out = plan.get();
  Plan* raw = plan.get();
  ctx->plans[key] = std::move(plan);
  return evict_plans(ctx, 0, raw);
}

// staging buffers for the host-pointer entry point, grown on demand
int ensure_io(vf_ctx* ctx, Plan* plan, long n) {
  if (plan->n_samples >= n && plan->d_wav) return VF_OK;
  const size_t before = plan->bytes;
  Builder b{ctx, plan};
  for (int k = 0; k < 2; ++k) {
    plan->d_io[k][0] = b.alloc<float>((size_t)plan->batch * n);
    plan->d_io[k][1] = b.alloc<float>((size_t)plan->batch * n);
  }
  plan->d_wav = plan->d_io[0][0];
  plan->d_out = plan->d_io[0][1];
  plan->n_samples = n;
  ctx->plan_bytes += plan->bytes - before;
  return b.rc;
}

// Orders this use of the plan's buffers after the previous one when that ran on another stream.
int plan_enter(vf_ctx* ctx, Plan* plan, cudaStream_t st) {
  if (plan->used && plan->last_stream != st) CK(cudaStreamWaitEvent(st, plan->ev_last, 0));
  return VF_OK;
}
int plan_exit(vf_ctx* ctx, Plan* plan, cudaStream_t st) {
  if (!plan->ev_last) CK(cudaEventCreateWithFlags(&plan->ev_last, cudaEventDisableTiming));
  CK(cudaEventRecord(plan->ev_last, st));
  plan->last_stream = st;
  plan->used = true;
  return VF_OK;
}

// Host-buffer round trip around `body(d_in, d_out, stream)`.  Pipelined mode: H2D on s_in, compute on s_comp, D2H on
// s_out, two staging buffer pairs; consecutive calls overlap (copy-in of the next, copy-out of the previous) and the
// caller's stream waits only for this call's D2H, so synchronising it still means "out_host is complete".
template <typename F>
int host_roundtrip(vf_ctx* ctx, Plan* plan, const float* in_host, float* out_host, size_t bytes, cudaStream_t st, F body) {
  if (!ctx->host_pipeline) {
    CK(cudaMemcpyAsync(plan->d_wav, in_host, bytes, cudaMemcpyHostToDevice, st));
    int rc = body(plan->d_wav, plan->d_out, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_host, plan->d_out, bytes, cudaMemcpyDeviceToHost, st));
    return VF_OK;
  }
  if (!ctx->s_in) {
    CK(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->s_comp, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
  }
  const int k = (int)(plan->io_seq++ & 1u);
  cudaEvent_t* ev = plan->io_ev[k];
  for (int i = 0; i < 4; ++i)
    if (!ev[i]) CK(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
  float* d_in = plan->d_io[k][0];
  float* d_out = plan->d_io[k][1];
  // (waiting on an event that was never recorded is a no-op)
  CK(cudaStreamWaitEvent(ctx->s_in, ev[1], 0));                 // the compute that read this input buffer two calls ago
  CK(cudaMemcpyAsync(d_in, in_host, bytes, cudaMemcpyHostToDevice, ctx->s_in));
  CK(cudaEventRecord(ev[0], ctx->s_in));
  CK(cudaStreamWaitEvent(ctx->s_comp, ev[0], 0));
  CK(cudaStreamWaitEvent(ctx->s_comp, ev[3], 0));               // the D2H that read this output buffer two calls ago
  int rc = body(d_in, d_out, ctx->s_comp);
  if (rc) return rc;
  CK(cudaEventRecord(ev[1], ctx->s_comp));
  CK(cudaEventRecord(ev[2], ctx->s_comp));
  CK(cudaStreamWaitEvent(ctx->s_out, ev[2], 0));
  CK(cudaMemcpyAsync(out_host, d_out, bytes, cudaMemcpyDeviceToHost, ctx->s_out));
  CK(cudaEventRecord(ev[3], ctx->s_out));
  CK(cudaStreamWaitEvent(st, ev[3], 0));
  return VF_OK;
}

int prof_mark(vf_ctx* ctx, cudaStream_t st) {
  const size_t i = ctx->prof.size();     // event i closes record i-1 and opens record i
  while (ctx->prof_ev.size() <= i) {
    cudaEvent_t ev;
    if (cudaEventCreate(&ev) != cudaSuccess) return fail(ctx, VF_ECUDA, "cudaEventCreate failed");
    ctx->prof_ev.push_back(ev);
  }
  if (cudaEventRecord(ctx->prof_ev[i], st) != cudaSuccess) return fail(ctx, VF_ECUDA, "cudaEventRecord failed");
  return VF_OK;
}

int run_ops(vf_ctx* ctx, std::vector<Op>& ops, cudaStream_t st) {
  for (Op& op : ops) {
    cudaError_t e = cudaSuccess;
    if (ctx->op_timing) {
      int rc = prof_mark(ctx, st);
      if (rc) return rc;
      const char* kinds[] = {"gemm", "unet_first", "pool", "voc_condition", "reflect_fill", "voc_tail", "finalize", "memset", "pair"};
      ctx->prof.push_back({op.label[0] ? std::string(op.label) : std::string(kinds[op.kind]), op.flops, op.bytes, op.exec_flops, op.bn, op.bk, op.kind == OP_GEMM ? op.tc.prob.terms : 0});
    }
    switch (op.kind) {
      case OP_GEMM:
        e = ctx->validate_simt ? launch_gemm_simt(op.simt, st) : launch_gemm_tc(op.tc, op.bn, op.bk, st);
        break;
      case OP_FIRST: e = launch_unet_first(op.first, st); break;
      case OP_POOL: e = launch_pool(op.pool, st); break;
      case OP_COND: e = launch_voc_condition(op.cond, st); break;
      case OP_REFLECT: e = launch_reflect_fill(op.refl.pl, op.refl.batch, op.refl.L, op.refl.C, op.refl.pad, st, op.refl.vl, op.refl.vl_stage); break;
      case OP_TAIL: e = launch_voc_tail(op.tail, st); break;
      case OP_FINALIZE: e = launch_finalize(op.fin, st); break;
      case OP_MEMSET32: e = cudaMemsetAsync(op.ms.p, 0, op.ms.bytes, st); break;
      case OP_PAIR: e = launch_pair_tc(op.pair, st); break;
    }
    if (e != cudaSuccess) return fail(ctx, VF_ECUDA, "kernel launch (op kind %d): %s", (int)op.kind, cudaGetErrorString(e));
    ctx->launches++;
  }
  if (ctx->op_timing) return prof_mark(ctx, st);   // closing event of the last record
  return VF_OK;
}

// The middle of a restore - every launch between the front end and the tail kernel - reads and writes plan-owned
// buffers only, so it is the same work every call: replay it as ONE graph launch instead of ~190 kernel launches
// (SURVEY.md 7 step 6).  `body` enqueues the chain on a stream; it runs eagerly on the first use of the plan, is
// captured on the second, and replayed from then on.  Profiling modes always run eagerly.
template <typename F>
int run_chain(vf_ctx* ctx, Plan* plan, int slot, cudaStream_t st, int64_t n_launches, F body) {
  const bool eager = !ctx->use_graphs || ctx->op_timing || ctx->timing || ctx->validate_simt;
  if (eager || plan->uses++ == 0) return body(st);
  if (!plan->graph[slot]) {
    if (!ctx->cap_stream && cudaStreamCreateWithFlags(&ctx->cap_stream, cudaStreamNonBlocking) != cudaSuccess)
      return fail(ctx, VF_ECUDA, "cudaStreamCreate (graph capture) failed");
    if (cudaStreamBeginCapture(ctx->cap_stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) {
      cudaGetLastError();
      return body(st);
    }
    const int64_t before = ctx->launches;
    const int rc = body(ctx->cap_stream);
    ctx->launches = before;                     // nothing ran yet
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(ctx->cap_stream, &g);
    if (rc || e != cudaSuccess || !g) {
      if (g) cudaGraphDestroy(g);
      cudaGetLastError();
      if (rc) return rc;
      ctx->use_graphs = false;                  // capture is not available here: stay eager
      return body(st);
    }
    const cudaError_t ei = cudaGraphInstantiate(&plan->graph[slot], g, 0);
    cudaGraphDestroy(g);
    if (ei != cudaSuccess) {
      plan->graph[slot] = nullptr;
      cudaGetLastError();
      ctx->use_graphs = false;
      return body(st);
    }
  }
  if (cudaGraphLaunch(plan->graph[slot], st) != cudaSuccess) return fail(ctx, VF_ECUDA, "cudaGraphLaunch: %s", cudaGetErrorString(cudaGetLastError()));
  ctx->launches += n_launches;
  return VF_OK;
}

int frames_of(vf_ctx* ctx, long n) { return 1 + (int)(n / ctx->cfg.hop); }

// vl (varlen plans): n is the row stride of wav, `frames` the plan's frames; each clip's own lengths come from the table
int run_frontend(vf_ctx* ctx, const float* wav, int batch, long n, float* mel, float* logmel, float* sp, float* co,
                 float* si, cudaStream_t st, const VarlenImage* vl = nullptr, int frames = 0) {
  if (n <= 1024) return fail(ctx, VF_EINVAL, "reflect padding needs more than n_fft/2 = 1024 samples (got %ld)", n);
  FrontendParams p;
  memset(&p, 0, sizeof p);
  p.wav = wav; p.n = n; p.batch = batch; p.T = vl ? frames : frames_of(ctx, n); p.vl = vl;
  p.window = ctx->d_window; p.tw1024 = ctx->d_tw1024; p.tw2048 = ctx->d_tw2048;
  p.fb_f0 = ctx->d_fb_f0; p.fb_len = ctx->d_fb_len; p.fb_ofs = ctx->d_fb_ofs; p.fb_val = ctx->d_fb_val;
  p.sp_out = sp; p.cos_out = co; p.sin_out = si; p.mel_out = mel; p.logmel_out = logmel;
  cudaError_t e = launch_frontend(p, st);
  if (e != cudaSuccess) return fail(ctx, VF_ECUDA, "frontend launch: %s", cudaGetErrorString(e));
  ctx->launches++;
  return VF_OK;
}

int check_ready(vf_ctx* ctx) {
  if (!ctx) return VF_EINVAL;
  if (!ctx->loaded) return fail(ctx, VF_ESTATE, "weights not loaded (call vf_load_weights first)");
  cudaError_t e = cudaSetDevice(ctx->device);
  if (e != cudaSuccess) return fail(ctx, VF_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  return VF_OK;
}

}  // namespace

// A batch whose plan would not fit the plan budget is processed in sub-batches through one smaller plan (rows are
// independent, so the result does not change): SSR at 64 x 10 s (143 GB) or a long file's stack of windows then run in two
// or more passes instead of failing with an out-of-memory plan.  Workspace scales with batch x padded frames; the per-frame
// figure is taken from a cached plan of the same path when there is one, else from the measured sizes (DESIGN.md 5).
int choose_sub_batch(vf_ctx* ctx, int kind, int batch, int frames) {
  if (ctx->plan_budget == 0) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) ctx->plan_budget = std::max<size_t>((free_b + ctx->plan_bytes) / 2, (size_t)1 << 30);
  }
  const double tp = (frames + 63) / 64 * 64;
  const bool ssr = kind == PLAN_SSR || kind == PLAN_SSR_VARLEN;
  double per_frame = ssr ? 2.4e6 : 1.7e6;      // bytes per clip and padded frame (measured 2.19e6 / 1.52e6) + margin
  for (auto& kv : ctx->plans)
    if (std::get<0>(kv.first) == kind) {
      per_frame = 1.05 * (double)kv.second->bytes / ((double)kv.second->batch * ((kv.second->T + 63) / 64 * 64));
      break;
    }
  const double fit = (double)ctx->plan_budget / (per_frame * tp);
  if (fit >= batch) return batch;
  int cb = std::max(1, (int)fit);
  for (int d = cb; d >= std::max(1, cb * 3 / 4); --d)         // prefer an even split (one plan shape instead of two)
    if (batch % d == 0) return d;
  return cb;
}

// =============================================================================================== C ABI
extern "C" {

VF_API void vf_default_config(vf_config* c) {
  memset(c, 0, sizeof *c);
  c->sample_rate = 44100; c->n_fft = 2048; c->hop = 441; c->n_mels = 128;
  c->voc_cond_channels = 512; c->voc_cond_layers = 5; c->voc_channels = 1024; c->voc_num_stages = 4;
  const int sc[4] = {7, 7, 3, 3};
  for (int i = 0; i < 4; ++i) { c->voc_scales[i] = sc[i]; c->voc_depth[i] = 8; }
  c->voc_stage_slope = 0.2f; c->voc_res_slope = 0.01f; c->voc_min_db = -115.f; c->voc_ref_db = 20.f;
  c->voc_amp_floor = 1e-5f; c->voc_tail_value = -4.f; c->voc_tail_base = 4;
  c->voc_mel_weight_a = 18.8927416350036; c->voc_mel_weight_b = 0.0269863588184314;
  c->voc_tail_tanh = 1;
}

VF_API const char* vf_last_error(vf_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

VF_API int vf_create(vf_ctx** out, int device, const vf_config* cfg) {
  if (!out) return VF_EINVAL;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, VF_ENODEVICE, "no CUDA device available (%s); libb200vf has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= ndev) return fail(nullptr, VF_EINVAL, "device %d out of range (%d devices)", device, ndev);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(nullptr, VF_ECUDA, "%s", cudaGetErrorString(e));
  if (prop.major != 10) return fail(nullptr, VF_ENODEVICE, "device %d is sm_%d%d; libb200vf is built for sm_100a only", device, prop.major, prop.minor);
  if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(nullptr, VF_ECUDA, "%s", cudaGetErrorString(e));
  std::unique_ptr<vf_ctx> ctx(new vf_ctx);
  ctx->device = device;
  if (cfg) ctx->cfg = *cfg; else vf_default_config(&ctx->cfg);
  const vf_config& c = ctx->cfg;
  if (c.sample_rate != 44100 || c.n_fft != 2048 || c.hop != 441 || c.n_mels != 128)
    return fail(nullptr, VF_EINVAL, "only the reference geometry (44100 Hz, n_fft 2048, hop 441, 128 mels) is built");
  if (c.voc_num_stages < 1 || c.voc_num_stages > 8 || c.voc_cond_layers < 1) return fail(nullptr, VF_EINVAL, "bad vocoder config");
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || !fn) return fail(nullptr, VF_ECUDA, "cuTensorMapEncodeTiled not available from the driver");
  ctx->encode = (EncodeTiledFn)fn;
  cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
  vf_ctx* raw = ctx.get();
  size_t acct = 0;
  int rc = dev_alloc(raw, raw->allocs, acct, &raw->d_err, 4);
  if (rc) { g_create_error = raw->err; return rc; }
  cudaMemset(raw->d_err, 0, 16);
  rc = build_tables(raw);
  if (rc) { g_create_error = raw->err; return rc; }
  *out = ctx.release();
  return VF_OK;
}

VF_API void vf_destroy(vf_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto& kv : ctx->plans) free_plan(kv.second.get());
  for (void* p : ctx->allocs) cudaFree(p);
  for (auto& e : ctx->prof_ev) cudaEventDestroy(e);
  if (ctx->cap_stream) cudaStreamDestroy(ctx->cap_stream);
  for (cudaStream_t st : {ctx->s_in, ctx->s_comp, ctx->s_out})
    if (st) cudaStreamDestroy(st);
  for (auto& e : ctx->ev)
    if (e) cudaEventDestroy(e);
  delete ctx;
}

VF_API int vf_load_weights(vf_ctx* ctx, const vf_tensor_desc* descs, int n) {
  if (!ctx || !descs || n <= 0) return VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  for (int i = 0; i < n; ++i) {
    const vf_tensor_desc& d = descs[i];
    if (!d.name || !d.data || d.ndim < 0 || d.ndim > 4) return fail(ctx, VF_EINVAL, "bad tensor descriptor %d", i);
    HostT t;
    size_t cnt = 1;
    for (int k = 0; k < d.ndim; ++k) { t.shape.push_back(d.shape[k]); cnt *= (size_t)d.shape[k]; }
    t.v.resize(cnt);
    if (d.on_device) CK(cudaMemcpy(t.v.data(), d.data, cnt * 4, cudaMemcpyDeviceToHost));
    else memcpy(t.v.data(), d.data, cnt * 4);
    ctx->host_w[d.name] = std::move(t);
  }
  int rc = load_all(ctx);
  if (rc) return rc;
  ctx->host_w.clear();
  ctx->loaded = true;
  CK(cudaDeviceSynchronize());
  return VF_OK;
}

VF_API int vf_frontend(vf_ctx* ctx, const float* wav, int batch, int64_t n, float* mel_out, float* sp_out, float* cos_out,
                float* sin_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav || batch <= 0) return fail(ctx, VF_EINVAL, "vf_frontend: bad arguments");
  if ((cos_out || sin_out) && !(sp_out && cos_out && sin_out)) return fail(ctx, VF_EINVAL, "cos/sin need sp, cos and sin");
  return run_frontend(ctx, wav, batch, (long)n, mel_out, nullptr, sp_out, cos_out, sin_out, (cudaStream_t)stream);
}

VF_API int vf_unet_mel(vf_ctx* ctx, const float* mel_lin, int batch, int frames, float* logmel_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!mel_lin || !logmel_out || batch <= 0 || frames <= 0) return fail(ctx, VF_EINVAL, "vf_unet_mel: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  Plan* plan;
  rc = get_plan(ctx, PLAN_GSR, batch, frames, &plan);
  if (rc) return rc;
  const size_t n = (size_t)batch * frames * 128;
  rc = plan_enter(ctx, plan, st);
  if (rc) return rc;
  CK(launch_to_log(mel_lin, plan->d_logmel_in, n, ctx->d_err + 1, st));
  ctx->launches++;
  rc = run_ops(ctx, plan->unet, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(logmel_out, plan->d_logmel_out, n * 4, cudaMemcpyDeviceToDevice, st));
  return plan_exit(ctx, plan, st);
}

VF_API int64_t vf_vocoder_out_len(vf_ctx* ctx, int frames) {
  if (!ctx) return -1;
  return (int64_t)(frames + frames % 2 + ctx->cfg.voc_tail_base) * ctx->cfg.hop;
}

VF_API int vf_vocoder(vf_ctx* ctx, const float* mel_lin, int batch, int frames, float* wav_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!mel_lin || !wav_out || batch <= 0 || frames <= 0) return fail(ctx, VF_EINVAL, "vf_vocoder: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  Plan* plan;
  rc = get_plan(ctx, PLAN_GSR, batch, frames, &plan);
  if (rc) return rc;
  rc = plan_enter(ctx, plan, st);
  if (rc) return rc;
  Op& cop = plan->vocoder[plan->cond_op];
  cop.cond.mel = mel_lin;
  cop.cond.is_log = 0;
  cop.cond.band_sums = nullptr;
  rc = run_ops(ctx, plan->vocoder, st);
  cop.cond.mel = plan->d_logmel_out;
  cop.cond.is_log = 1;
  if (rc) return rc;
  CK(cudaMemcpyAsync(wav_out, plan->d_voc_wav, (size_t)batch * plan->L * 4, cudaMemcpyDeviceToDevice, st));
  return plan_exit(ctx, plan, st);
}

// lens == null: every clip has n samples.  Else clip b has lens[b] samples (1024 < lens[b] <= n, checked by the caller), n is the
// row stride of wav and wav_out, and `frames` the 64-frame bucket of the longest clip (the varlen plan's key).
static int restore_impl(vf_ctx* ctx, const float* wav, int batch, int64_t n, float* wav_out, unsigned flags, cudaStream_t st,
                        const int64_t* lens = nullptr, int bucket = 0) {
  const int frames = lens ? bucket : frames_of(ctx, (long)n);
  Plan* plan;
  int rc = get_plan(ctx, lens ? PLAN_GSR_VARLEN : PLAN_GSR, batch, frames, &plan);
  if (rc) return rc;
  if (ctx->op_timing) ctx->prof.clear();
  rc = plan_enter(ctx, plan, st);
  if (rc) return rc;
  const bool tm = ctx->timing;
  if (tm) {
    for (auto& e : ctx->ev)
      if (!e) CK(cudaEventCreate(&e));
    CK(cudaEventRecord(ctx->ev[0], st));
  }
  if (lens) {     // the per-clip table of this call: a plain launch ahead of the frontend and the captured chain
    VarlenSetupParams vp;
    memset(&vp, 0, sizeof vp);
    vp.batch = batch; vp.W0 = 127; vp.hop = ctx->cfg.hop; vp.tail_base = ctx->cfg.voc_tail_base;
    vp.num_stages = ctx->cfg.voc_num_stages;
    for (int s = 0; s < 8; ++s) vp.scales[s] = ctx->cfg.voc_scales[s];
    vp.out = plan->d_vl;
    for (int b = 0; b < batch; ++b) vp.n[b] = (long long)lens[b];
    CK(launch_varlen_setup(vp, st));
    ctx->launches++;
  }
  rc = run_frontend(ctx, wav, batch, (long)n, plan->d_mel, plan->d_logmel_in, nullptr, nullptr, nullptr, st, plan->d_vl, frames);
  if (rc) return rc;
  if (tm) CK(cudaEventRecord(ctx->ev[1], st));
  const bool unify = (flags & VF_RESTORE_UNIFY_ENERGY) != 0;
  auto chain = [&](cudaStream_t s) -> int {
    int r = run_ops(ctx, plan->unet, s);
    if (r) return r;
    if (tm) CK(cudaEventRecord(ctx->ev[2], s));
    // eval_gsr_voicefixer.py:54-55: amp_to_original_f when meta["unify_energy"]
    Op& cop = plan->vocoder[plan->cond_op];
    cop.cond.mel = plan->d_logmel_out;
    cop.cond.is_log = 1;
    cop.cond.band_sums = nullptr;
    if (unify) {
      CK(cudaMemsetAsync(plan->d_band, 0, 2 * (size_t)batch * sizeof(float), s));
      CK(launch_band_energy(plan->d_mel, plan->d_logmel_out, batch, frames, plan->d_band, s, plan->d_vl));
      ctx->launches++;
      cop.cond.band_sums = plan->d_band;
    }
    return run_ops(ctx, plan->vocoder, s);
  };
  rc = run_chain(ctx, plan, unify ? 1 : 0, st, (int64_t)plan->unet.size() + (int64_t)plan->vocoder.size() + (unify ? 1 : 0), chain);
  if (rc) return rc;
  if (tm) CK(cudaEventRecord(ctx->ev[3], st));
  // eval_gsr_voicefixer.py:68-72: peak normalise + trim_center
  FinalizeParams f;
  memset(&f, 0, sizeof f);
  const long d = plan->L - (long)n;
  if (!lens && (d < 0 || d == 1)) return fail(ctx, VF_EINVAL, "vocoder output length %ld incompatible with input %ld (trim_center)", plan->L, (long)n);
  f.wav = plan->d_voc_wav; f.peak_bits = plan->d_peak; f.batch = batch; f.L = plan->L; f.n = (long)n; f.skip = lens ? 0 : d / 2;
  f.out = wav_out; f.out_ld = (long)n; f.out_off = 0; f.vl = plan->d_vl;
  CK(launch_finalize(f, st));
  ctx->launches++;
  if (tm) { CK(cudaEventRecord(ctx->ev[4], st)); ctx->ev_valid = true; }
  return plan_exit(ctx, plan, st);
}

VF_API int vf_restore_ex(vf_ctx* ctx, const float* wav, int batch, int64_t n, float* wav_out, unsigned flags, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav || !wav_out || batch <= 0) return fail(ctx, VF_EINVAL, "vf_restore: bad arguments");
  if (flags & ~(unsigned)VF_RESTORE_UNIFY_ENERGY) return fail(ctx, VF_EINVAL, "vf_restore_ex: unknown flag bits 0x%x", flags);
  const int cb = choose_sub_batch(ctx, PLAN_GSR, batch, frames_of(ctx, (long)n));
  for (int off = 0; off < batch; off += cb) {
    rc = restore_impl(ctx, wav + (size_t)off * n, std::min(cb, batch - off), n, wav_out + (size_t)off * n, flags, (cudaStream_t)stream);
    if (rc) return rc;
  }
  return VF_OK;
}

VF_API int vf_restore_varlen(vf_ctx* ctx, const float* wav, int batch, int64_t n_max, const int64_t* n_samples, float* wav_out,
                             unsigned flags, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav || !wav_out || !n_samples || batch <= 0) return fail(ctx, VF_EINVAL, "vf_restore_varlen: bad arguments");
  if (flags & ~(unsigned)VF_RESTORE_UNIFY_ENERGY) return fail(ctx, VF_EINVAL, "vf_restore_varlen: unknown flag bits 0x%x", flags);
  if (n_max > (int64_t)INT32_MAX / 2) return fail(ctx, VF_EINVAL, "vf_restore_varlen: n_max %ld too large", (long)n_max);
  // every length is checked before anything is launched
  int64_t longest = 0;
  for (int b = 0; b < batch; ++b) {
    if (n_samples[b] <= 1024 || n_samples[b] > n_max)
      return fail(ctx, VF_EINVAL, "vf_restore_varlen: clip %d has %ld samples; need 1024 < n <= n_max = %ld (reflect padding needs "
                  "more than n_fft/2 samples)", b, (long)n_samples[b], (long)n_max);
    longest = std::max(longest, n_samples[b]);
  }
  // one plan per (batch, 64-frame bucket of the longest clip): every call whose longest clip is in the same 0.64 s bucket
  // reuses it and its CUDA graphs
  const int bucket = round_up(frames_of(ctx, (long)longest), 64);
  const int cb = std::min(choose_sub_batch(ctx, PLAN_GSR_VARLEN, batch, bucket), VF_VARLEN_MAX_CLIPS);
  for (int off = 0; off < batch; off += cb) {
    rc = restore_impl(ctx, wav + (size_t)off * n_max, std::min(cb, batch - off), n_max, wav_out + (size_t)off * n_max, flags,
                      (cudaStream_t)stream, n_samples + off, bucket);
    if (rc) return rc;
  }
  return VF_OK;
}

VF_API int vf_restore(vf_ctx* ctx, const float* wav, int batch, int64_t n, float* wav_out, void* stream) {
  return vf_restore_ex(ctx, wav, batch, n, wav_out, ctx && ctx->unify_energy ? VF_RESTORE_UNIFY_ENERGY : 0u, stream);
}

VF_API int vf_restore_host(vf_ctx* ctx, const float* wav_host, int batch, int64_t n, float* out_host, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav_host || !out_host || batch <= 0) return fail(ctx, VF_EINVAL, "vf_restore_host: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned flags = ctx->unify_energy ? VF_RESTORE_UNIFY_ENERGY : 0u;
  const int cb = choose_sub_batch(ctx, PLAN_GSR, batch, frames_of(ctx, (long)n));
  for (int off = 0; off < batch; off += cb) {
    const int b = std::min(cb, batch - off);
    Plan* plan;
    rc = get_plan(ctx, PLAN_GSR, b, frames_of(ctx, (long)n), &plan);
    if (rc) return rc;
    rc = ensure_io(ctx, plan, (long)n);
    if (rc) return rc;
    rc = host_roundtrip(ctx, plan, wav_host + (size_t)off * n, out_host + (size_t)off * n, (size_t)b * n * 4, st,
                        [&](const float* d_in, float* d_out, cudaStream_t s) { return restore_impl(ctx, d_in, b, n, d_out, flags, s); });
    if (rc) return rc;
  }
  return VF_OK;
}

// ---------------------------------------------------------------------------------------------- SSR / GSR-UNet path
// lens == null: every clip has n samples.  Else (a PLAN_SSR_VARLEN plan, sp null) clip b has lens[b] samples
// (1024 < lens[b] <= n, checked by the caller), n is the row stride of wav and wav_out, and plan->T the 64-frame bucket.
static int ssr_impl(vf_ctx* ctx, Plan* plan, const float* sp, const float* wav, int batch, int64_t n, float* wav_out, cudaStream_t st,
                    const int64_t* lens = nullptr) {
  const int frames = plan->T;
  if (ctx->op_timing) ctx->prof.clear();
  int rc = plan_enter(ctx, plan, st);
  if (rc) return rc;
  const bool tm = ctx->timing;
  if (tm) {
    for (auto& e : ctx->ev)
      if (!e) CK(cudaEventCreate(&e));
    CK(cudaEventRecord(ctx->ev[0], st));
  }
  if (lens) {     // the per-clip table of this call (unet_v2 geometry, W0 = 1024): a plain launch ahead of everything else
    VarlenSetupParams vp;
    memset(&vp, 0, sizeof vp);
    vp.batch = batch; vp.W0 = 1024; vp.hop = ctx->cfg.hop;      // the vocoder fields stay 0: no vocoder on this path
    vp.out = plan->d_vl;
    for (int b = 0; b < batch; ++b) vp.n[b] = (long long)lens[b];
    CK(launch_varlen_setup(vp, st));
    ctx->launches++;
  }
  if (!sp) {     // SSR_UNet.pre (ssr_unet.py:140-143): the magnitude of the input itself
    rc = run_frontend(ctx, wav, batch, (long)n, nullptr, nullptr, plan->d_sp, nullptr, nullptr, st, plan->d_vl, frames);
    if (rc) return rc;
  }
  if (tm) CK(cudaEventRecord(ctx->ev[1], st));
  plan->unet[0].first.logmel = sp ? sp : plan->d_sp;       // unet_v2.forward(sp, wav): the caller's sp feeds the net
  if (sp) rc = run_ops(ctx, plan->unet, st);               // caller-owned input pointer: not replayable
  else rc = run_chain(ctx, plan, 0, st, (int64_t)plan->unet.size(), [&](cudaStream_t s) -> int { return run_ops(ctx, plan->unet, s); });
  if (rc) return rc;
  if (tm) CK(cudaEventRecord(ctx->ev[2], st));
  IstftFramesParams fp;
  memset(&fp, 0, sizeof fp);
  fp.mag = plan->d_mag; fp.wav = wav; fp.n = (long)n; fp.batch = batch; fp.T = frames;
  fp.window = ctx->d_window; fp.tw1024 = ctx->d_tw1024; fp.tw2048 = ctx->d_tw2048; fp.frames = plan->d_frames;
  fp.vl = plan->d_vl;
  CK(launch_istft_frames(fp, st));
  IstftOlaParams op;
  memset(&op, 0, sizeof op);
  op.frames = plan->d_frames; op.batch = batch; op.T = frames; op.length = (long)n; op.window = ctx->d_window;
  op.out = wav_out; op.out_ld = (long)n; op.vl = plan->d_vl;
  CK(launch_istft_ola(op, st));
  ctx->launches += 2;
  if (tm) { CK(cudaEventRecord(ctx->ev[3], st)); CK(cudaEventRecord(ctx->ev[4], st)); ctx->ev_valid = true; }
  return plan_exit(ctx, plan, st);
}

VF_API int vf_ssr_forward(vf_ctx* ctx, const float* sp, const float* wav, int batch, int64_t n, float* wav_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav || !wav_out || batch <= 0) return fail(ctx, VF_EINVAL, "vf_ssr_forward: bad arguments");
  if (n <= 1024) return fail(ctx, VF_EINVAL, "reflect padding needs more than n_fft/2 = 1024 samples (got %ld)", (long)n);
  const int frames = frames_of(ctx, (long)n);
  const int cb = choose_sub_batch(ctx, PLAN_SSR, batch, frames);
  for (int off = 0; off < batch; off += cb) {
    const int b = std::min(cb, batch - off);
    Plan* plan;
    rc = get_plan(ctx, PLAN_SSR, b, frames, &plan);
    if (rc) return rc;
    rc = ssr_impl(ctx, plan, sp ? sp + (size_t)off * frames * 1025 : nullptr, wav + (size_t)off * n, b, n, wav_out + (size_t)off * n, (cudaStream_t)stream);
    if (rc) return rc;
  }
  return VF_OK;
}

VF_API int vf_ssr_restore(vf_ctx* ctx, const float* wav, int batch, int64_t n, float* wav_out, void* stream) {
  return vf_ssr_forward(ctx, nullptr, wav, batch, n, wav_out, stream);
}

VF_API int vf_ssr_restore_varlen(vf_ctx* ctx, const float* wav, int batch, int64_t n_max, const int64_t* n_samples,
                                 float* wav_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav || !wav_out || !n_samples || batch <= 0) return fail(ctx, VF_EINVAL, "vf_ssr_restore_varlen: bad arguments");
  if (n_max > (int64_t)INT32_MAX / 2) return fail(ctx, VF_EINVAL, "vf_ssr_restore_varlen: n_max %ld too large", (long)n_max);
  // every length is checked before anything is launched
  int64_t longest = 0;
  for (int b = 0; b < batch; ++b) {
    if (n_samples[b] <= 1024 || n_samples[b] > n_max)
      return fail(ctx, VF_EINVAL, "vf_ssr_restore_varlen: clip %d has %ld samples; need 1024 < n <= n_max = %ld (reflect "
                  "padding needs more than n_fft/2 samples)", b, (long)n_samples[b], (long)n_max);
    longest = std::max(longest, n_samples[b]);
  }
  // one plan per (batch, 64-frame bucket of the longest clip), as for vf_restore_varlen
  const int bucket = round_up(frames_of(ctx, (long)longest), 64);
  const int cb = std::min(choose_sub_batch(ctx, PLAN_SSR_VARLEN, batch, bucket), VF_VARLEN_MAX_CLIPS);
  for (int off = 0; off < batch; off += cb) {
    const int b = std::min(cb, batch - off);
    Plan* plan;
    rc = get_plan(ctx, PLAN_SSR_VARLEN, b, bucket, &plan);
    if (rc) return rc;
    rc = ssr_impl(ctx, plan, nullptr, wav + (size_t)off * n_max, b, n_max, wav_out + (size_t)off * n_max, (cudaStream_t)stream,
                  n_samples + off);
    if (rc) return rc;
  }
  return VF_OK;
}

VF_API int vf_ssr_restore_host(vf_ctx* ctx, const float* wav_host, int batch, int64_t n, float* out_host, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!wav_host || !out_host || batch <= 0) return fail(ctx, VF_EINVAL, "vf_ssr_restore_host: bad arguments");
  if (n <= 1024) return fail(ctx, VF_EINVAL, "reflect padding needs more than n_fft/2 = 1024 samples (got %ld)", (long)n);
  cudaStream_t st = (cudaStream_t)stream;
  const int frames = frames_of(ctx, (long)n);
  const int cb = choose_sub_batch(ctx, PLAN_SSR, batch, frames);
  for (int off = 0; off < batch; off += cb) {
    const int b = std::min(cb, batch - off);
    Plan* plan;
    rc = get_plan(ctx, PLAN_SSR, b, frames, &plan);
    if (rc) return rc;
    rc = ensure_io(ctx, plan, (long)n);
    if (rc) return rc;
    rc = host_roundtrip(ctx, plan, wav_host + (size_t)off * n, out_host + (size_t)off * n, (size_t)b * n * 4, st,
                        [&](const float* d_in, float* d_out, cudaStream_t s) { return ssr_impl(ctx, plan, nullptr, d_in, b, n, d_out, s); });
    if (rc) return rc;
  }
  return VF_OK;
}

VF_API int vf_ssr_unet(vf_ctx* ctx, const float* sp, int batch, int frames, float* mag_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  if (!sp || !mag_out || batch <= 0 || frames <= 0) return fail(ctx, VF_EINVAL, "vf_ssr_unet: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  Plan* plan;
  rc = get_plan(ctx, PLAN_SSR, batch, frames, &plan);
  if (rc) return rc;
  if (ctx->op_timing) ctx->prof.clear();
  rc = plan_enter(ctx, plan, st);
  if (rc) return rc;
  plan->unet[0].first.logmel = sp;
  rc = run_ops(ctx, plan->unet, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(mag_out, plan->d_mag, (size_t)batch * frames * 1025 * 4, cudaMemcpyDeviceToDevice, st));
  return plan_exit(ctx, plan, st);
}

VF_API int vf_ssr_stages(vf_ctx* ctx, int batch, int64_t n, float* sp_out, float* mag_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  Plan* plan;
  const int frames = frames_of(ctx, (long)n);
  rc = get_plan(ctx, PLAN_SSR, batch, frames, &plan);
  if (rc) return rc;
  const size_t bytes = (size_t)batch * frames * 1025 * 4;
  rc = plan_enter(ctx, plan, (cudaStream_t)stream);
  if (rc) return rc;
  if (sp_out) CK(cudaMemcpyAsync(sp_out, plan->d_sp, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (mag_out) CK(cudaMemcpyAsync(mag_out, plan->d_mag, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return plan_exit(ctx, plan, (cudaStream_t)stream);
}

VF_API int vf_istft(vf_ctx* ctx, const float* real, const float* imag, int batch, int frames, int64_t length, float* wav_out, void* stream) {
  if (!ctx || !real || !imag || !wav_out || batch <= 0 || frames <= 0 || length <= 0) return ctx ? fail(ctx, VF_EINVAL, "vf_istft: bad arguments") : VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  if (length + 1024 > (int64_t)(frames - 1) * ctx->cfg.hop + 2048)
    return fail(ctx, VF_EINVAL, "vf_istft: %d frames cover %ld samples, fewer than length %ld + n_fft/2", frames, (long)(frames - 1) * ctx->cfg.hop + 2048, (long)length);
  cudaStream_t st = (cudaStream_t)stream;
  float* frames_buf = nullptr;           // stream-ordered scratch: no plan is tied to a bare ISTFT
  CK(cudaMallocAsync((void**)&frames_buf, (size_t)batch * frames * 2048 * 4, st));
  IstftFramesParams fp;
  memset(&fp, 0, sizeof fp);
  fp.real = real; fp.imag = imag; fp.batch = batch; fp.T = frames;
  fp.window = ctx->d_window; fp.tw1024 = ctx->d_tw1024; fp.tw2048 = ctx->d_tw2048; fp.frames = frames_buf;
  cudaError_t e1 = launch_istft_frames(fp, st);
  IstftOlaParams op;
  memset(&op, 0, sizeof op);
  op.frames = frames_buf; op.batch = batch; op.T = frames; op.length = (long)length; op.window = ctx->d_window;
  op.out = wav_out; op.out_ld = (long)length;
  cudaError_t e2 = e1 == cudaSuccess ? launch_istft_ola(op, st) : e1;
  cudaFreeAsync(frames_buf, st);
  if (e2 != cudaSuccess) return fail(ctx, VF_ECUDA, "istft launch: %s", cudaGetErrorString(e2));
  ctx->launches += 2;
  return VF_OK;
}

// ---------------------------------------------------------------------------------------------- stand-alone boundary ops
VF_API int vf_mel(vf_ctx* ctx, const float* specgram, int64_t n_outer, int64_t frames, int64_t stride_outer, int64_t stride_freq,
                  int64_t stride_time, float* mel_out, void* stream) {
  if (!ctx || !specgram || !mel_out || n_outer <= 0 || frames <= 0 || n_outer > 65535) return ctx ? fail(ctx, VF_EINVAL, "vf_mel: bad arguments") : VF_EINVAL;
  if (!ctx->d_fb_val) return fail(ctx, VF_ESTATE, "mel filterbank not loaded (call vf_load_weights first)");
  CK(cudaSetDevice(ctx->device));
  MelParams p;
  memset(&p, 0, sizeof p);
  p.in = specgram; p.n_outer = (long)n_outer; p.T = (long)frames; p.so = (long)stride_outer; p.sf = (long)stride_freq; p.st = (long)stride_time;
  p.out = mel_out; p.fb_f0 = ctx->d_fb_f0; p.fb_len = ctx->d_fb_len; p.fb_ofs = ctx->d_fb_ofs; p.fb_val = ctx->d_fb_val;
  CK(launch_mel(p, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}

VF_API int vf_resample_poly(vf_ctx* ctx, const float* wav, int batch, int64_t n, int up, int down, const float* taps, int n_taps,
                            float* out, int64_t n_out, void* stream) {
  if (!ctx || !wav || !taps || !out || batch <= 0 || n <= 0 || up <= 0 || down <= 0 || n_taps < 1 || (n_taps & 1) == 0)
    return ctx ? fail(ctx, VF_EINVAL, "vf_resample_poly: bad arguments (n_taps must be odd)") : VF_EINVAL;
  if (n_out != (n * up + down - 1) / down) return fail(ctx, VF_EINVAL, "vf_resample_poly: n_out must be ceil(n * up / down) = %ld", (long)((n * up + down - 1) / down));
  CK(cudaSetDevice(ctx->device));
  CK(launch_resample_poly(wav, batch, (long)n, up, down, taps, n_taps / 2, out, (long)n_out, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}

VF_API int vf_amp_to_original_f(vf_ctx* ctx, const float* mel_est, const float* mel_target, int batch, int frames, float* mel_out, void* stream) {
  if (!ctx || !mel_est || !mel_target || !mel_out || batch <= 0 || frames <= 0) return ctx ? fail(ctx, VF_EINVAL, "vf_amp_to_original_f: bad arguments") : VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(launch_amp_to_original(mel_est, mel_target, batch, frames, mel_out, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}

VF_API int vf_lsd(vf_ctx* ctx, const float* est, const float* target, int images, int frames, int bins, float* out, void* stream) {
  if (!ctx || !est || !target || !out || images <= 0 || frames <= 0 || bins <= 0) return ctx ? fail(ctx, VF_EINVAL, "vf_lsd: bad arguments") : VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(launch_lsd(est, target, images, frames, bins, out, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}

VF_API int vf_sispec(vf_ctx* ctx, const float* est, const float* target, int batch, int64_t n, int est_map, int target_map, float* out, void* stream) {
  if (!ctx || !est || !target || !out || batch <= 0 || n <= 0 || est_map < 0 || est_map > 2 || target_map < 0 || target_map > 2)
    return ctx ? fail(ctx, VF_EINVAL, "vf_sispec: bad arguments") : VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(launch_sispec(est, target, batch, (long)n, est_map, target_map, out, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}

VF_API int vf_finalize(vf_ctx* ctx, const float* wav, int batch, int64_t len, int64_t n, float* wav_out, void* stream) {
  if (!ctx || !wav || !wav_out || batch <= 0 || len <= 0 || n <= 0) return ctx ? fail(ctx, VF_EINVAL, "vf_finalize: bad arguments") : VF_EINVAL;
  const long d = (long)len - (long)n;
  // trim_center (tools/utils.py:57-70) for an estimate at least as long as the reference; d == 1 is the reference's
  // empty-slice case (est[..., 0:-0])
  if (d < 0 || d == 1) return fail(ctx, VF_EINVAL, "vf_finalize: estimate length %ld vs reference %ld is not a trim_center case the path produces", (long)len, (long)n);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned int* peak = nullptr;
  CK(cudaMallocAsync((void**)&peak, (size_t)batch * 4, st));
  CK(cudaMemsetAsync(peak, 0, (size_t)batch * 4, st));
  cudaError_t e1 = launch_peak(wav, batch, (long)len, peak, st);
  FinalizeParams f;
  memset(&f, 0, sizeof f);
  f.wav = wav; f.peak_bits = peak; f.batch = batch; f.L = (long)len; f.n = (long)n; f.skip = d / 2;
  f.out = wav_out; f.out_ld = (long)n; f.out_off = 0;
  cudaError_t e2 = e1 == cudaSuccess ? launch_finalize(f, st) : e1;
  cudaFreeAsync(peak, st);
  if (e2 != cudaSuccess) return fail(ctx, VF_ECUDA, "finalize launch: %s", cudaGetErrorString(e2));
  ctx->launches += 2;
  return VF_OK;
}

VF_API int vf_restore_stages(vf_ctx* ctx, int batch, int64_t n, float* mel_lin_out, float* log_mel_out, void* stream) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  Plan* plan;
  const int frames = frames_of(ctx, (long)n);
  rc = get_plan(ctx, PLAN_GSR, batch, frames, &plan);
  if (rc) return rc;
  const size_t bytes = (size_t)batch * frames * 128 * 4;
  rc = plan_enter(ctx, plan, (cudaStream_t)stream);
  if (rc) return rc;
  if (mel_lin_out) CK(cudaMemcpyAsync(mel_lin_out, plan->d_mel, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (log_mel_out) CK(cudaMemcpyAsync(log_mel_out, plan->d_logmel_out, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return plan_exit(ctx, plan, (cudaStream_t)stream);
}

VF_API int vf_to_log(vf_ctx* ctx, const float* in, float* out, int64_t n, void* stream) {
  if (!ctx || !in || !out || n <= 0) return VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(launch_to_log(in, out, (size_t)n, ctx->d_err + 1, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}
VF_API int vf_from_log(vf_ctx* ctx, const float* in, float* out, int64_t n, void* stream) {
  if (!ctx || !in || !out || n <= 0) return VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(launch_from_log(in, out, (size_t)n, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}

VF_API int vf_to_pcm16_ex(vf_ctx* ctx, const float* in, int16_t* out, int64_t n, int saturate, void* stream) {
  if (!ctx || !in || !out || n <= 0) return VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(launch_pcm16(in, out, (size_t)n, saturate ? 1 : 0, (cudaStream_t)stream));
  ctx->launches++;
  return VF_OK;
}
VF_API int vf_to_pcm16(vf_ctx* ctx, const float* in, int16_t* out, int64_t n, void* stream) {
  return vf_to_pcm16_ex(ctx, in, out, n, 0, stream);
}

VF_API int vf_workspace_bytes(vf_ctx* ctx, int batch, int64_t n, size_t* bytes) {
  int rc = check_ready(ctx);
  if (rc) return rc;
  Plan* plan;
  rc = get_plan(ctx, PLAN_GSR, batch, frames_of(ctx, (long)n), &plan);
  if (rc) return rc;
  if (bytes) *bytes = plan->bytes + ctx->weight_bytes;
  return VF_OK;
}

VF_API int vf_check_errors(vf_ctx* ctx, void* stream) {
  if (!ctx) return VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  int h[2] = {0, 0};
  CK(cudaMemcpy(h, ctx->d_err, 8, cudaMemcpyDeviceToHost));
  if (h[0] || h[1]) CK(cudaMemset(ctx->d_err, 0, 8));
  if (h[0] == ERR_FP16_OVERFLOW) return fail(ctx, VF_EDEVICE, "activation outside the fp16 range (|a| > 65504) in a hi/lo split");
  if (h[0]) return fail(ctx, VF_EDEVICE, "device pipeline error code %d (201 producer / 202 mma / 203 epilogue time-out)", h[0]);
  if (h[1]) return fail(ctx, VF_EASSERT, "input has negative values counts %d", h[1]);
  return VF_OK;
}

VF_API int vf_set_option(vf_ctx* ctx, const char* key, int value) {
  if (!ctx || !key) return VF_EINVAL;
  const std::string k = key;
  int* slot = nullptr;
  if (k == "unet_terms" || k == "vocoder_terms") {
    if (value != 1 && value != 3) return fail(ctx, VF_EINVAL, "%s must be 1 or 3", key);
    // the UNet's fp32 skip streams, BN affines and fused head exist in the 3-term kernels only (the 1e-4 log-mel
    // bar needs fp32-grade products anyway)
    if (k == "unet_terms" && value != 3) return fail(ctx, VF_EINVAL, "unet_terms: only 3 is supported");
    slot = k == "unet_terms" ? &ctx->unet_terms : &ctx->voc_terms;
  } else if (k == "unify_energy") {
    ctx->unify_energy = value ? 1 : 0;     // per-call behaviour, no plan rebuild needed
    return VF_OK;
  } else if (k == "validate_simt") {
    slot = &ctx->validate_simt;
    value = value ? 1 : 0;
  } else if (k == "host_pipeline") {
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    ctx->host_pipeline = value != 0;
    return VF_OK;
  } else if (k == "graphs") {
    ctx->use_graphs = value != 0;
    return VF_OK;
  } else if (k == "plan_cache_mb") {
    if (value < 0) return fail(ctx, VF_EINVAL, "plan_cache_mb must be >= 0 (0: half of the free device memory)");
    ctx->plan_budget = (size_t)value << 20;
    if (value) return evict_plans(ctx, 0, nullptr);
    return VF_OK;
  } else {
    return fail(ctx, VF_EINVAL, "unknown option '%s'", key);
  }
  if (*slot != value) {   // plans bake the option in: drop them
    drop_all_plans(ctx);
    *slot = value;
  }
  return VF_OK;
}

VF_API int64_t vf_launch_count(vf_ctx* ctx) { return ctx ? ctx->launches : -1; }

VF_API int vf_plan_cache_info(vf_ctx* ctx, int* n_plans, size_t* bytes, size_t* budget, int64_t* evicted) {
  if (!ctx) return VF_EINVAL;
  if (n_plans) *n_plans = (int)ctx->plans.size();
  if (bytes) *bytes = ctx->plan_bytes;
  if (budget) *budget = ctx->plan_budget;
  if (evicted) *evicted = ctx->plans_evicted;
  return VF_OK;
}

VF_API int vf_enable_stage_timing(vf_ctx* ctx, int enable) {
  if (!ctx) return VF_EINVAL;
  ctx->timing = enable != 0;
  ctx->ev_valid = false;
  return VF_OK;
}
VF_API int vf_stage_times(vf_ctx* ctx, float ms[4]) {
  if (!ctx || !ms) return VF_EINVAL;
  if (!ctx->ev_valid) return fail(ctx, VF_ESTATE, "no timed vf_restore yet");
  CK(cudaEventSynchronize(ctx->ev[4]));
  for (int i = 0; i < 4; ++i) CK(cudaEventElapsedTime(&ms[i], ctx->ev[i], ctx->ev[i + 1]));
  return VF_OK;
}

VF_API int vf_enable_op_timing(vf_ctx* ctx, int enable) {
  if (!ctx) return VF_EINVAL;
  ctx->op_timing = enable != 0;
  ctx->prof.clear();
  return VF_OK;
}
VF_API int vf_op_count(vf_ctx* ctx) { return ctx ? (int)ctx->prof.size() : -1; }
VF_API int vf_op_info(vf_ctx* ctx, int i, float* ms, double* flops, double* bytes, int* bn, int* bk, int* terms, char* label, int label_cap,
                      double* exec_flops) {
  if (!ctx || i < 0 || i >= (int)ctx->prof.size()) return VF_EINVAL;
  // records of the frontend / finalize launches are not tracked; record i spans events [i, i+1) except that
  // each run_ops() call appends one closing event after its last op, so consecutive event pairs stay aligned
  // only inside one call: look the pair up by walking the event list.
  if ((size_t)i + 1 >= ctx->prof_ev.size()) return fail(ctx, VF_ESTATE, "no events recorded for op %d", i);
  CK(cudaEventSynchronize(ctx->prof_ev[i + 1]));
  float t = 0.f;
  CK(cudaEventElapsedTime(&t, ctx->prof_ev[i], ctx->prof_ev[i + 1]));
  if (ms) *ms = t;
  if (flops) *flops = ctx->prof[i].flops;
  if (bytes) *bytes = ctx->prof[i].bytes;
  if (exec_flops) *exec_flops = ctx->prof[i].exec_flops;
  if (bn) *bn = ctx->prof[i].bn;
  if (bk) *bk = ctx->prof[i].bk;
  if (terms) *terms = ctx->prof[i].terms;
  if (label && label_cap > 0) snprintf(label, label_cap, "%s", ctx->prof[i].label.c_str());
  return VF_OK;
}

VF_API int vf_selftest_gemm(vf_ctx* ctx, int n_img, int rows, int cin, int cout, int ntaps, int dilation, int terms,
                     double* max_abs_diff, double* max_abs_ref) {
  if (!ctx || n_img <= 0 || rows <= 0 || cin % 32 || cout % 32 || ntaps < 1 || ntaps > GEMM_MAX_TAPS || (terms != 1 && terms != 3))
    return ctx ? fail(ctx, VF_EINVAL, "vf_selftest_gemm: bad arguments") : VF_EINVAL;
  CK(cudaSetDevice(ctx->device));
  Plan plan;
  Builder b{ctx, &plan};
  const int K = ntaps * cin;
  // deterministic pseudo-random operands
  uint32_t seed = 12345u + rows * 7 + cin * 3 + cout;
  auto rnd = [&]() { seed = seed * 1664525u + 1013904223u; return ((seed >> 8) & 0xFFFF) / 65536.0f - 0.5f; };
  std::vector<float> wm((size_t)cout * K), bias(cout);
  for (auto& x : wm) x = rnd() * 0.2f;
  for (auto& x : bias) x = rnd();
  GemmW W;
  int rc = upload_gemm(ctx, &W, wm, cout, K, &bias);
  if (rc) return rc;
  const size_t an = (size_t)n_img * rows * cin;
  std::vector<__half> ahi(an), alo(an);
  for (size_t i = 0; i < an; ++i) {
    const float a = rnd() * 4.f;
    ahi[i] = __float2half_rn(a);
    alo[i] = __float2half_rn(a - __half2float(ahi[i]));
  }
  Planes A = b.planes(n_img, rows, cin);
  float* out[2] = {b.alloc<float>((size_t)n_img * rows * cout), b.alloc<float>((size_t)n_img * rows * cout)};
  // hi-only kernels carry no fp32 stream: their result is observed through the raw hi/lo planes (22 bits)
  Planes outp[2] = {b.planes(n_img, rows, cout), b.planes(n_img, rows, cout)};
  if (b.rc) return b.rc;
  CK(cudaMemcpy(A.p.hi, ahi.data(), an * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(A.p.lo, alo.data(), an * 2, cudaMemcpyHostToDevice));
  const int saved = ctx->validate_simt;
  for (int impl = 0; impl < 2; ++impl) {
    ctx->validate_simt = impl;
    std::vector<Op> ops;
    GemmEpilogue e = epi_plain(rows, 0, cout, rows);
    e.bias = W.bias;
    if (terms == 3) {
      e.out_raw = out[impl];
      e.raw_ld = cout;
    } else {
      e.out_r = OutPlane{outp[impl].p.hi, outp[impl].p.lo, cout, 0};
    }
    std::vector<GemmTap> taps;
    for (int t = 0; t < ntaps; ++t) taps.push_back(GemmTap{(t - (ntaps - 1) / 2) * dilation, 0, 0, 0, cin});
    b.gemm(ops, W, ASrc{A, rows, 0}, nullptr, taps, e, n_img, terms);
    if (!b.rc) b.rc = run_ops(ctx, ops, 0);
  }
  ctx->validate_simt = saved;
  cudaError_t se = cudaDeviceSynchronize();
  rc = b.rc;
  double md = 0, mr = 0;
  if (!rc && se == cudaSuccess) {
    const size_t on = (size_t)n_img * rows * cout;
    std::vector<float> h0(on), h1(on);
    if (terms == 3) {
      cudaMemcpy(h0.data(), out[0], on * 4, cudaMemcpyDeviceToHost);
      cudaMemcpy(h1.data(), out[1], on * 4, cudaMemcpyDeviceToHost);
    } else {
      std::vector<__half> ph(on), pl(on);
      for (int impl = 0; impl < 2; ++impl) {
        cudaMemcpy(ph.data(), outp[impl].p.hi, on * 2, cudaMemcpyDeviceToHost);
        cudaMemcpy(pl.data(), outp[impl].p.lo, on * 2, cudaMemcpyDeviceToHost);
        std::vector<float>& h = impl ? h1 : h0;
        for (size_t i = 0; i < on; ++i) h[i] = __half2float(ph[i]) + __half2float(pl[i]);
      }
    }
    for (size_t i = 0; i < on; ++i) {
      const double d = std::fabs((double)h0[i] - (double)h1[i]);
      if (!(d <= md)) md = d;          // NaN-propagating max
      if (std::fabs(h1[i]) > mr) mr = std::fabs(h1[i]);
    }
  }
  for (void* p : plan.allocs) cudaFree(p);
  if (se != cudaSuccess) return fail(ctx, VF_ECUDA, "selftest: %s", cudaGetErrorString(se));
  if (rc) return rc;
  if (max_abs_diff) *max_abs_diff = md;
  if (max_abs_ref) *max_abs_ref = mr;
  return VF_OK;
}

}  // extern "C"
