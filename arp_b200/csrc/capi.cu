// C-ABI implementation of include/arp_b200.h: handle, weight packing, TMA descriptors and the
// stream-ordered pipeline   decode -> patch-embed GEMM -> ln_pre -> 12 x [QKV (ln_1 folded), attention, out-proj (+= x,
// row moments), c_fc (ln_2 folded, QuickGELU), c_proj (+= x, row moments)] (the last block for the class-token row only)
// -> reward head -> per-episode return-to-go scan. The embed entry points stop after the head's image side and return the
// per-frame embedding; arp_label_embeddings runs only the instruction side (head + scan) on such embeddings. The tower
// entry points stop the adapter heads after the frozen CLIP tower; arp_label_tower runs the adapter tail from there.
// Host logic only; every kernel lives in the .cuh next to this file.
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include <cerrno>
#include <unistd.h>

#include "../../include/arp_b200.h"
#include "attention_tc.cuh"
#include "decode.cuh"
#include "fp32_path.cuh"
#include "gemm_tcgen05.cuh"
#include "head.cuh"
#include "inflate.cuh"
#include "layernorm.cuh"
#include "rtgstats.cuh"
#include "scan.cuh"
#include "tower.cuh"

using namespace arp;
static_assert(ARP_MAX_TEXT == HEAD_MAX_TEXT && ARP_MAX_TEXT_GROUPS == HEAD_MAX_GROUPS &&
              ARP_MAX_TEXT_TOTAL == HEAD_MAX_TEXT_TOTAL, "text limits of include/arp_b200.h and head.cuh disagree");
typedef arp::op_t bf16;   // the operand format (common.cuh: bf16 by default, fp16 with -DARP_OP_FP16=1)
#define ARP_OP_DTYPE (ARP_OP_FP16 ? ARP_F16 : ARP_BF16)   // ... as an ArpDType of include/arp_b200.h

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_create_error;

struct ArpHandle;
static int fail(ArpHandle* h, int code, const char* fmt, ...);

#define ARP_CUDA(h, expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return fail(h, ARP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define ARP_TRY(expr)            \
  do {                           \
    int _r = (expr);             \
    if (_r != ARP_OK) return _r; \
  } while (0)

// ------------------------------------------------------------------------------------------------
// driver entry point for TMA descriptors (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(p);
  return fn;
}

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
struct LayerW {
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  bf16 *w_qkv = nullptr, *w_out = nullptr, *w_fc = nullptr, *w_proj = nullptr;
  float *b_qkv = nullptr, *b_out = nullptr, *b_fc = nullptr, *b_proj = nullptr;
  // LayerNorm fold (16-bit residual path): fp32 originals of the two LN-consuming weights, their gamma-folded
  // operands, and the per-output-column vectors of the algebraic LayerNorm (gemm_tcgen05.cuh G2_LNFOLD)
  float *w_qkv_f32 = nullptr, *w_fc_f32 = nullptr;
  bf16 *w_qkv_fold = nullptr, *w_fc_fold = nullptr;
  float *s_qkv = nullptr, *c_qkv = nullptr, *s_fc = nullptr, *c_fc = nullptr;
};

struct WeightSlot {
  void** dst_f32 = nullptr;  // optional extra fp32 copy (weights that get LayerNorm-folded at finalize time)
  void** dst;      // device buffer to fill
  int64_t numel;
  bool as_bf16;    // GEMM operand (bf16) or fp32 parameter
  bool required;
  bool set;
};

struct TmapKey {
  const void* ptr; uint64_t rows, cols, ld; uint32_t box_rows, box_cols, elem;
  bool operator<(const TmapKey& o) const {
    return std::tie(ptr, rows, cols, ld, box_rows, box_cols, elem) <
           std::tie(o.ptr, o.rows, o.cols, o.ld, o.box_rows, o.box_cols, o.elem);
  }
};

struct ArpHandle {
  ArpConfig cfg;
  std::string err;
  int64_t launches = 0;
  // Residual stream format. true (ARP_PREC_BF16, the default 16-bit path): x is kept in the operand format, updated by
  // 16-bit TMA reduce-adds, and IS the A operand of the QKV / c_fc GEMMs, which apply LayerNorm algebraically in their
  // epilogues from per-row moments — no LayerNorm kernels, no normalised copy, no fp32 read-modify-write.
  // false (ARP_PREC_F32RESID): fp32 x, standalone LayerNorm kernels writing a 16-bit copy (round 1's pipeline).
  bool resid16 = true;
  // Snake order: consecutive kernels of a chunk walk the rows in opposite directions, so each starts on what its
  // predecessor wrote last (the tail of a 150-600 MB activation is still in the 126 MB L2). Flipped at every launch.
  int dir = 0;
  bool f32 = false;   // cfg.precision == ARP_PREC_F32: verification path (fp32_path.cuh); GEMM weights are stored as fp32
  int tokens = 0, grid = 0, kp = 0;  // 197, 14, 768
  bool adapter = false, goal = false;
  int n_scales = 0, feat_dim = 0;    // 13, 6656 for adapter heads

  // weights
  bf16* conv1 = nullptr;
  float *class_emb = nullptr, *pos_emb = nullptr, *rowtab = nullptr;
  float *ln_pre_g = nullptr, *ln_pre_b = nullptr, *ln_post_g = nullptr, *ln_post_b = nullptr;
  float* proj = nullptr;
  std::vector<LayerW> layers;
  bf16 *inter_w = nullptr, *fc1_w = nullptr, *fc2_w = nullptr;
  float *fc1_b = nullptr, *fc2_b = nullptr, *res_w = nullptr;
  float res_sigmoid = 0.f;
  bool finalized = false;
  bool adapter_ready = false;   // the image-adapter tensors are set and res_sigmoid is current (arp_label_tower)
  std::map<std::string, WeightSlot> slots;

  // text: n_text rows = n_groups instruction sets concatenated, group g = rows [group_off[g], group_off[g+1])
  float* text = nullptr;             // [HEAD_MAX_TEXT_TOTAL, feat_dim]
  int* group_off = nullptr;          // device int32 [n_groups + 1]
  int group_off_host[HEAD_MAX_GROUPS + 1] = {};
  int n_text = 0, text_dim = 0, n_groups = 1;
  float logit_scale = 0.f;

  // decode tables
  int *h_min = nullptr, *h_cnt = nullptr, *h_k = nullptr, *v_min = nullptr, *v_cnt = nullptr, *v_k = nullptr;
  int h_ksize = 0, v_ksize = 0, max_rows = 0;
  float* lut = nullptr;
  int crop_top = 0, crop_left = 0, src_h = 0, src_w = 0;

  // workspace, sized for cfg.max_batch frames
  struct Work {
    bf16* x16 = nullptr;      // [M, W] 16-bit residual stream (resid16)
    float2* stats = nullptr;  // [M] (rstd, -mean*rstd) of the rows of x16: the LayerNorm the next GEMM folds in
    float* x = nullptr;       // [M, W] fp32 residual stream (!resid16, fp32 path); resid16: fp32 patch-embed output, aliases qkv
    bf16 *xn = nullptr, *qkv = nullptr, *attn = nullptr, *hid = nullptr;
    bf16 *taps = nullptr, *featb = nullptr, *hid2 = nullptr;
    float *featf = nullptr, *mlp = nullptr;
    float* xcls = nullptr;                                       // [B, W] class-token residual rows (last-layer pruning)
    bf16 *xncls = nullptr, *qcls = nullptr, *acls = nullptr, *hcls = nullptr;   // [B,W] x3, [B,4W]
    // fp32 verification path
    float *chw32 = nullptr, *xn32 = nullptr, *qkv32 = nullptr, *attn32 = nullptr, *hid32 = nullptr;
    float *taps32 = nullptr, *hid2_32 = nullptr;
  } ws;

  // scratch that grows with T (goal heads, host path)
  void* scratch[2] = {nullptr, nullptr};  // [0] label temporaries, [1] device outputs of the host path
  size_t scratch_bytes[2] = {0, 0};
  uint8_t* stage_dev[2] = {nullptr, nullptr};
  size_t stage_bytes = 0;
  // compressed-row entry points (arp_*_zfile): two device buffers of one chunk's compressed rows, the inflated rows of one
  // chunk [max_batch, row_bytes], and the call's per-row tables (packed offset, size, inflate status)
  uint8_t* zsrc_dev[2] = {nullptr, nullptr};
  size_t zsrc_bytes = 0;
  uint8_t* zrows_dev = nullptr;
  size_t zrows_bytes = 0;
  void* ztab_dev = nullptr;
  size_t ztab_bytes = 0;
  uint8_t* pin_ring = nullptr;     // pinned staging ring for pageable callers of arp_label_host (STG_SLOTS x STG_SUB frames)
  size_t pin_bytes = 0;
  cudaEvent_t ev_slot[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaStream_t copy_stream = nullptr, own_stream = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};

  std::map<TmapKey, CUtensorMap> tmaps;
  std::vector<void*> allocs;

  // latency mode (arp_online_reward): one CUDA graph per batch size n, rebuilt when weights or text change
  struct OnlineGraph { cudaGraphExec_t exec = nullptr; int64_t launches = 0; uint64_t epoch = 0; };
  std::map<int, OnlineGraph> online_graphs;
  uint64_t online_epoch = 1;
  float* online_out = nullptr;   // device [max_batch * (1 + HEAD_MAX_TEXT + feat_dim)]
  void* stats_dev = nullptr;     // RadixSelectState + min/max keys + 8 result floats (consumer-side statistics)

  // optional per-kernel-class timing (arp_profile_begin/end): CUDA events bracket every launch on its stream
  bool profiling = false;
  struct ProfRec { int cls; double flops; double bytes; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> event_pool;
};

enum ProfClass { PC_GEMM = 0, PC_ATTENTION = 1, PC_LAYERNORM = 2, PC_DECODE = 3, PC_HEAD = 4, PC_SCAN = 5, PC_OTHER = 6, PC_COUNT = 7 };

static cudaEvent_t prof_event(ArpHandle* h) {
  if (!h->event_pool.empty()) { cudaEvent_t e = h->event_pool.back(); h->event_pool.pop_back(); return e; }
  cudaEvent_t e = nullptr;
  cudaEventCreate(&e);
  return e;
}

// RAII bracket: records an event before and after the launches issued inside its scope
struct ProfScope {
  ArpHandle* h; cudaStream_t st; size_t idx; bool on;
  ProfScope(ArpHandle* h_, int cls, double flops, double bytes, cudaStream_t st_) : h(h_), st(st_), idx(0), on(h_->profiling) {
    if (!on) return;
    ArpHandle::ProfRec r{cls, flops, bytes, prof_event(h), prof_event(h)};
    cudaEventRecord(r.e0, st);
    idx = h->prof.size();
    h->prof.push_back(r);
  }
  ~ProfScope() { if (on) cudaEventRecord(h->prof[idx].e1, st); }
};

static int fail(ArpHandle* h, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

template <typename T>
static int dev_alloc(ArpHandle* h, T** p, size_t count) {
  void* q = nullptr;
  ARP_CUDA(h, cudaMalloc(&q, count * sizeof(T) + 256));
  h->allocs.push_back(q);
  // Zeroed once: a partially filled chunk's last frame reads a few rows past its own (the attention kernel's 208-key V
  // box, tile 1's query rows) — rows that must be FINITE (their softmax weight is exactly 0, and 0 x NaN is NaN). Rows
  // ever written by the kernels are finite; never-written rows are these zeros.
  ARP_CUDA(h, cudaMemset(q, 0, count * sizeof(T) + 256));
  *p = reinterpret_cast<T*>(q);
  return ARP_OK;
}

// ------------------------------------------------------------------------------------------------
// Pillow resample tables (SURVEY.md Appendix B; libImaging/Resample.c precompute_coeffs + normalize_coeffs_8bpc)
// ------------------------------------------------------------------------------------------------
static double bicubic_filter(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

static void pil_bicubic_tables(int in_size, int out_size, std::vector<int>& xmin_v, std::vector<int>& cnt_v,
                               std::vector<int>& kk, int& ksize) {
  double scale = static_cast<double>(in_size) / out_size;
  double filterscale = scale < 1.0 ? 1.0 : scale;
  const double support = 2.0 * filterscale;
  ksize = static_cast<int>(std::ceil(support)) * 2 + 1;
  xmin_v.assign(out_size, 0);
  cnt_v.assign(out_size, 0);
  kk.assign(static_cast<size_t>(out_size) * ksize, 0);
  std::vector<double> k(ksize);
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = 0.0 + (xx + 0.5) * scale;
    double ww = 0.0;
    const double ss = 1.0 / filterscale;
    int xmin = static_cast<int>(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = static_cast<int>(center + support + 0.5);
    if (xmax > in_size) xmax = in_size;
    xmax -= xmin;
    for (int x = 0; x < xmax; ++x) {
      const double w = bicubic_filter((x + xmin - center + 0.5) * ss);
      k[x] = w;
      ww += w;
    }
    for (int x = 0; x < xmax; ++x)
      if (ww != 0.0) k[x] /= ww;
    for (int x = 0; x < xmax; ++x) {
      const double v = k[x] * (1 << 22);
      kk[static_cast<size_t>(xx) * ksize + x] = v < 0 ? static_cast<int>(-0.5 + v) : static_cast<int>(0.5 + v);
    }
    xmin_v[xx] = xmin;
    cnt_v[xx] = xmax;
  }
}

static const float kClipMean[3] = {0.48145466f, 0.4578275f, 0.40821073f};
static const float kClipStd[3] = {0.26862954f, 0.26130258f, 0.27577711f};

template <typename T>
static int upload(ArpHandle* h, T** dst, const std::vector<T>& v) {
  ARP_TRY(dev_alloc(h, dst, v.size()));
  ARP_CUDA(h, cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return ARP_OK;
}

static int build_decode_tables(ArpHandle* h) {
  const ArpConfig& c = h->cfg;
  h->src_h = c.in_h;
  h->src_w = c.in_w;
  h->crop_top = h->crop_left = 0;
  if (c.use_crop) {
    if (c.preprocess == ARP_PRE_PIL_BICUBIC) {
      // torchvision CenterCrop(image_size // 2) with image_size = shape[-2] (label_reward.py:96,104):
      // square crop, origin int(round((dim - crop) / 2.0))
      const int cs = c.in_w / 2;  // g[key].shape[-2] is W for [T,F,H,W,3]
      h->src_h = h->src_w = cs;
      h->crop_top = static_cast<int>(std::nearbyint((c.in_h - cs) / 2.0));
      h->crop_left = static_cast<int>(std::nearbyint((c.in_w - cs) / 2.0));
    } else {
      // center_crop(images, (image_size//2, image_size//2)) (label_reward.py:15-36, :203): origin int((dim-crop)/2)
      const int cs = c.in_w / 2;
      h->src_h = h->src_w = cs;
      h->crop_top = (c.in_h - cs) / 2;
      h->crop_left = (c.in_w - cs) / 2;
    }
  }
  if (h->src_h <= 0 || h->src_w <= 0 || h->crop_top < 0 || h->crop_top + h->src_h > c.in_h || h->crop_left < 0 ||
      h->crop_left + h->src_w > c.in_w)
    return fail(h, ARP_ERR_INVALID, "bad crop geometry for %dx%d (a crop larger than the frame would be zero-padded by "
                "torchvision; not supported)", c.in_h, c.in_w);
  if (c.preprocess == ARP_PRE_PIL_BICUBIC) {
    // Resize(224) scales the SHORTER side to 224 and the longer one to int(224 * long / short) (torchvision
    // _compute_resized_output_size), then CenterCrop(224) takes the window at int(round((dim - 224) / 2.0)) — only on the
    // no-crop route (label_reward.py:113-114); the use_crop route resizes its square crop and has no second crop (:96-97).
    // Both passes are separable and a crop is a window, so the tables are the full-size tables restricted to the window.
    int out_w = DEC_OUT, out_h = DEC_OUT;
    if (h->src_w > h->src_h) out_w = static_cast<int>(static_cast<long long>(DEC_OUT) * h->src_w / h->src_h);
    else if (h->src_h > h->src_w) out_h = static_cast<int>(static_cast<long long>(DEC_OUT) * h->src_h / h->src_w);
    const int win_left = static_cast<int>(std::nearbyint((out_w - DEC_OUT) / 2.0));
    const int win_top = static_cast<int>(std::nearbyint((out_h - DEC_OUT) / 2.0));
    std::vector<int> xm, xc, xk, ym, yc, yk;
    {
      std::vector<int> fm, fc, fk;
      pil_bicubic_tables(h->src_w, out_w, fm, fc, fk, h->h_ksize);
      xm.assign(fm.begin() + win_left, fm.begin() + win_left + DEC_OUT);
      xc.assign(fc.begin() + win_left, fc.begin() + win_left + DEC_OUT);
      xk.assign(fk.begin() + (size_t)win_left * h->h_ksize, fk.begin() + (size_t)(win_left + DEC_OUT) * h->h_ksize);
      pil_bicubic_tables(h->src_h, out_h, fm, fc, fk, h->v_ksize);
      ym.assign(fm.begin() + win_top, fm.begin() + win_top + DEC_OUT);
      yc.assign(fc.begin() + win_top, fc.begin() + win_top + DEC_OUT);
      yk.assign(fk.begin() + (size_t)win_top * h->v_ksize, fk.begin() + (size_t)(win_top + DEC_OUT) * h->v_ksize);
    }
    if (h->h_ksize > 64 || h->v_ksize > 64) return fail(h, ARP_ERR_INVALID, "downscale factor too large");
    {
      // Pillow sizes its coefficient rows for the widest possible window (ksize = 2 ceil(support) + 1: 7 for 256 -> 224,
      // 5 when upscaling) but no output pixel uses more than xmax - xmin of them (5 resp. 4 here); the rest are zeros.
      // Re-pack the rows to the largest window that occurs: the kernel applies every tap of a row, and two zero taps of
      // seven were 29 % of its multiply-adds. Exact: only products with a zero coefficient are dropped.
      const int taps = std::max(*std::max_element(xc.begin(), xc.end()), *std::max_element(yc.begin(), yc.end()));
      auto repack = [&](std::vector<int>& k, int old_stride) {
        std::vector<int> r((size_t)DEC_OUT * taps, 0);
        for (int i = 0; i < DEC_OUT; ++i)
          for (int j = 0; j < std::min(old_stride, taps); ++j) r[(size_t)i * taps + j] = k[(size_t)i * old_stride + j];
        k.swap(r);
      };
      repack(xk, h->h_ksize);
      repack(yk, h->v_ksize);
      h->h_ksize = h->v_ksize = taps;
    }
    h->max_rows = 0;
    for (int b = 0; b < DEC_OUT / DEC_BAND; ++b) {
      const int lo = ym[b * DEC_BAND], hi = ym[b * DEC_BAND + DEC_BAND - 1] + yc[b * DEC_BAND + DEC_BAND - 1];
      h->max_rows = std::max(h->max_rows, hi - lo);
    }
    ARP_TRY(upload(h, &h->h_min, xm)); ARP_TRY(upload(h, &h->h_cnt, xc)); ARP_TRY(upload(h, &h->h_k, xk));
    ARP_TRY(upload(h, &h->v_min, ym)); ARP_TRY(upload(h, &h->v_cnt, yc)); ARP_TRY(upload(h, &h->v_k, yk));
    std::vector<float> lut(3 * 256);
    for (int ch = 0; ch < 3; ++ch)
      for (int u = 0; u < 256; ++u) {
        volatile float v = static_cast<float>(u) / 255.0f;  // ToTensor: u8 -> f32, div 255
        volatile float w = v - kClipMean[ch];               // Normalize: sub mean, div std (fp32, separately rounded)
        lut[ch * 256 + u] = w / kClipStd[ch];
      }
    ARP_TRY(upload(h, &h->lut, lut));
  } else {
    const float sc = static_cast<float>(h->src_h) / DEC_OUT;
    h->max_rows = static_cast<int>(sc * DEC_BAND) + 4;
    if (h->max_rows > h->src_h) h->max_rows = h->src_h;
    h->h_ksize = h->v_ksize = 0;
  }
  return ARP_OK;
}

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
static void add_slot(ArpHandle* h, const std::string& name, void** dst, int64_t numel, bool as_bf16, bool required) {
  WeightSlot s;
  s.dst = dst; s.numel = numel; s.as_bf16 = as_bf16; s.required = required; s.set = false;
  h->slots[name] = s;
}

static void register_slots(ArpHandle* h) {
  const ArpConfig& c = h->cfg;
  const int W = c.width, P = c.patch;
  add_slot(h, "visual.conv1.weight", (void**)&h->conv1, (int64_t)W * 3 * P * P, true, true);
  add_slot(h, "visual.class_embedding", (void**)&h->class_emb, W, false, true);
  add_slot(h, "visual.positional_embedding", (void**)&h->pos_emb, (int64_t)h->tokens * W, false, true);
  add_slot(h, "visual.ln_pre.weight", (void**)&h->ln_pre_g, W, false, true);
  add_slot(h, "visual.ln_pre.bias", (void**)&h->ln_pre_b, W, false, true);
  add_slot(h, "visual.ln_post.weight", (void**)&h->ln_post_g, W, false, true);
  add_slot(h, "visual.ln_post.bias", (void**)&h->ln_post_b, W, false, true);
  add_slot(h, "visual.proj", (void**)&h->proj, (int64_t)W * c.embed_dim, false, true);
  h->layers.resize(c.layers);
  for (int l = 0; l < c.layers; ++l) {
    LayerW& L = h->layers[l];
    const std::string p = "visual.transformer.resblocks." + std::to_string(l) + ".";
    add_slot(h, p + "ln_1.weight", (void**)&L.ln1_g, W, false, true);
    add_slot(h, p + "ln_1.bias", (void**)&L.ln1_b, W, false, true);
    add_slot(h, p + "ln_2.weight", (void**)&L.ln2_g, W, false, true);
    add_slot(h, p + "ln_2.bias", (void**)&L.ln2_b, W, false, true);
    add_slot(h, p + "attn.in_proj_weight", (void**)&L.w_qkv, (int64_t)3 * W * W, true, true);
    add_slot(h, p + "attn.in_proj_bias", (void**)&L.b_qkv, 3 * W, false, true);
    add_slot(h, p + "attn.out_proj.weight", (void**)&L.w_out, (int64_t)W * W, true, true);
    add_slot(h, p + "attn.out_proj.bias", (void**)&L.b_out, W, false, true);
    add_slot(h, p + "mlp.c_fc.weight", (void**)&L.w_fc, (int64_t)4 * W * W, true, true);
    add_slot(h, p + "mlp.c_fc.bias", (void**)&L.b_fc, 4 * W, false, true);
    add_slot(h, p + "mlp.c_proj.weight", (void**)&L.w_proj, (int64_t)4 * W * W, true, true);
    add_slot(h, p + "mlp.c_proj.bias", (void**)&L.b_proj, W, false, true);
    h->slots[p + "attn.in_proj_weight"].dst_f32 = (void**)&L.w_qkv_f32;
    h->slots[p + "mlp.c_fc.weight"].dst_f32 = (void**)&L.w_fc_f32;
  }
  if (h->adapter) {
    const int64_t D = h->feat_dim;                       // 13 * 512
    const int64_t Din = (int64_t)c.layers * W;           // 12 * 768
    const int64_t Dmid = (int64_t)c.layers * c.embed_dim;  // 12 * 512 (text_dim * num_clip_layers)
    add_slot(h, "image_intermediate_linear.weight", (void**)&h->inter_w, Dmid * Din, true, true);
    add_slot(h, "image_adapter.layers.0.weight", (void**)&h->fc1_w, 2 * D * D, true, true);
    add_slot(h, "image_adapter.layers.0.bias", (void**)&h->fc1_b, 2 * D, false, true);
    add_slot(h, "image_adapter.layers.3.weight", (void**)&h->fc2_w, 2 * D * D, true, true);
    add_slot(h, "image_adapter.layers.3.bias", (void**)&h->fc2_b, D, false, true);
    add_slot(h, "image_residual_weight", (void**)&h->res_w, 1, false, true);
  }
}

template <typename S, typename D>
__global__ void convert_kernel(const S* __restrict__ src, D* __restrict__ dst, size_t n) {
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    dst[i] = static_cast<D>(static_cast<float>(src[i]));
}

template <typename S, typename D>
static void launch_convert(ArpHandle* h, const void* src, void* dst, size_t n, cudaStream_t st) {
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  convert_kernel<S, D><<<blocks, 256, 0, st>>>(static_cast<const S*>(src), static_cast<D*>(dst), n);
  h->launches++;
}

__global__ void build_rowtab_kernel(const float* __restrict__ pos, const float* __restrict__ cls,
                                    float* __restrict__ tab, int tokens, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= tokens * W) return;
  tab[i] = pos[i] + (i < W ? cls[i] : 0.f);
}

// ------------------------------------------------------------------------------------------------
// C ABI: lifetime
// ------------------------------------------------------------------------------------------------
extern "C" int arp_abi_version(void) { return ARP_B200_ABI_VERSION; }
extern "C" int arp_operand_dtype(void) { return ARP_OP_DTYPE; }

extern "C" const char* arp_last_error(const ArpHandle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" int64_t arp_launch_count(const ArpHandle* h) { return h ? h->launches : 0; }

extern "C" int arp_profile_begin(ArpHandle* h) {
  if (!h) return ARP_ERR_INVALID;
  for (auto& r : h->prof) { h->event_pool.push_back(r.e0); h->event_pool.push_back(r.e1); }
  h->prof.clear();
  h->profiling = true;
  return ARP_OK;
}

extern "C" int arp_profile_end(ArpHandle* h, ArpProfileStats* out, int32_t n_classes) {
  if (!h || !out || n_classes < 1) return fail(h, ARP_ERR_INVALID, "null argument");
  h->profiling = false;
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  ARP_CUDA(h, cudaDeviceSynchronize());
  for (int i = 0; i < n_classes; ++i) out[i] = ArpProfileStats{0, 0.0, 0.0, 0.0};
  for (auto& r : h->prof) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    if (r.cls < n_classes) {
      out[r.cls].launches += 1;
      out[r.cls].total_ms += ms;
      out[r.cls].flops += r.flops;
      out[r.cls].bytes += r.bytes;
    }
    h->event_pool.push_back(r.e0);
    h->event_pool.push_back(r.e1);
  }
  h->prof.clear();
  return ARP_OK;
}

template <typename K>
static int set_smem(ArpHandle* h, K kernel, int bytes) {
  ARP_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return ARP_OK;
}

extern "C" void arp_destroy(ArpHandle* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (void* p : h->allocs) cudaFree(p);
  for (int i = 0; i < 2; ++i) if (h->scratch[i]) cudaFree(h->scratch[i]);
  for (int i = 0; i < 2; ++i) {
    if (h->stage_dev[i]) cudaFree(h->stage_dev[i]);
    if (h->zsrc_dev[i]) cudaFree(h->zsrc_dev[i]);
    if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
    if (h->ev_consumed[i]) cudaEventDestroy(h->ev_consumed[i]);
  }
  if (h->zrows_dev) cudaFree(h->zrows_dev);
  if (h->ztab_dev) cudaFree(h->ztab_dev);
  if (h->pin_ring) cudaFreeHost(h->pin_ring);
  for (cudaEvent_t e : h->ev_slot) if (e) cudaEventDestroy(e);
  for (auto& kv : h->online_graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  for (auto& r : h->prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  for (cudaEvent_t e : h->event_pool) cudaEventDestroy(e);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

extern "C" int arp_create(const ArpConfig* cfg, ArpHandle** out) {
  if (!cfg || !out) return fail(nullptr, ARP_ERR_INVALID, "null argument");
  if (cfg->struct_size != (int32_t)sizeof(ArpConfig))
    return fail(nullptr, ARP_ERR_INVALID, "ArpConfig.struct_size %d != %zu", cfg->struct_size, sizeof(ArpConfig));
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device < 0 || cfg->device >= ndev)
    return fail(nullptr, ARP_ERR_NO_DEVICE, "no CUDA device %d (count %d); this library has no CPU path", cfg->device, ndev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10)
    return fail(nullptr, ARP_ERR_NO_DEVICE, "device %d is sm_%d%d; arp_b200 is built for sm_100a only", cfg->device,
                prop.major, prop.minor);
  if (cfg->width != 768 || cfg->embed_dim != 512 || cfg->heads * 64 != cfg->width)
    return fail(nullptr, ARP_ERR_INVALID, "only ViT-B geometry is built (width 768, 64-wide heads, embed 512)");
  if (cfg->patch != 16 && cfg->patch != 32) return fail(nullptr, ARP_ERR_INVALID, "patch must be 16 or 32");
  if (cfg->layers < 1 || cfg->layers > 48 || cfg->max_batch < 1 || cfg->in_h < 8 || cfg->in_w < 8)
    return fail(nullptr, ARP_ERR_INVALID, "bad layers / max_batch / frame size");
  if (cfg->head < 0 || cfg->head > ARP_HEAD_ADAPTER_GOAL || cfg->preprocess < 0 || cfg->preprocess > 1)
    return fail(nullptr, ARP_ERR_INVALID, "bad head / preprocess enum");
  if (cfg->precision != ARP_PREC_BF16 && cfg->precision != ARP_PREC_F32 && cfg->precision != ARP_PREC_F32RESID)
    return fail(nullptr, ARP_ERR_INVALID, "bad precision enum");
  if (!get_encode_tiled()) return fail(nullptr, ARP_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");

  ArpHandle* h = new ArpHandle();
  h->cfg = *cfg;
  auto bail = [&](int code) { g_create_error = h->err; arp_destroy(h); return code; };
  if (cudaSetDevice(cfg->device) != cudaSuccess) { h->err = "cudaSetDevice failed"; return bail(ARP_ERR_CUDA); }
  h->f32 = cfg->precision == ARP_PREC_F32;
  h->resid16 = cfg->precision == ARP_PREC_BF16;
  h->grid = DEC_OUT / cfg->patch;
  h->tokens = h->grid * h->grid + 1;
  h->kp = 3 * cfg->patch * cfg->patch;
  h->adapter = cfg->head == ARP_HEAD_ADAPTER || cfg->head == ARP_HEAD_ADAPTER_ENSEMBLE || cfg->head == ARP_HEAD_ADAPTER_GOAL;
  h->goal = cfg->head == ARP_HEAD_CLIP_GOAL || cfg->head == ARP_HEAD_ADAPTER_GOAL;
  h->n_scales = cfg->layers + 1;
  h->feat_dim = h->adapter ? h->n_scales * cfg->embed_dim : cfg->embed_dim;
  if (h->adapter && h->n_scales != 13) { h->err = "adapter heads are built for 12-layer CLIP (13 scales)"; return bail(ARP_ERR_INVALID); }

  int r = build_decode_tables(h);
  if (r != ARP_OK) return bail(r);
  register_slots(h);

  const size_t B = cfg->max_batch, M = B * h->tokens, W = cfg->width;
#define CREATE_TRY(e) do { int _r = (e); if (_r != ARP_OK) return bail(_r); } while (0)
  CREATE_TRY(dev_alloc(h, &h->rowtab, (size_t)h->tokens * W));
  {
    ArpHandle::Work& w = h->ws;
    if (h->f32) {
      CREATE_TRY(dev_alloc(h, &w.x, M * W));
      CREATE_TRY(dev_alloc(h, &w.chw32, B * 3 * DEC_OUT * DEC_OUT));
      CREATE_TRY(dev_alloc(h, &w.xn32, M * W));
      CREATE_TRY(dev_alloc(h, &w.qkv32, M * 3 * W));
      CREATE_TRY(dev_alloc(h, &w.attn32, M * W));
      CREATE_TRY(dev_alloc(h, &w.hid32, M * std::max<size_t>(4 * W, h->kp)));
      if (h->adapter) {
        const size_t D = h->feat_dim;
        CREATE_TRY(dev_alloc(h, &w.taps32, B * cfg->layers * W));
        CREATE_TRY(dev_alloc(h, &w.featf, B * D));
        CREATE_TRY(dev_alloc(h, &w.hid2_32, B * 2 * D));
        CREATE_TRY(dev_alloc(h, &w.mlp, B * D));
      }
    } else {
      CREATE_TRY(dev_alloc(h, &w.qkv, M * 3 * W));
      // padded key rows of a frame are the next frame's rows: keep every bit pattern in this buffer finite
      if (cudaMemset(w.qkv, 0, M * 3 * W * sizeof(bf16)) != cudaSuccess) { h->err = "cudaMemset failed"; return bail(ARP_ERR_CUDA); }
      if (h->resid16) {
        CREATE_TRY(dev_alloc(h, &w.x16, M * W));
        CREATE_TRY(dev_alloc(h, &w.stats, M * (2 * W / 256)));   // up to 2*W/256 partials per row (G2_RESID_STATS)
        w.x = reinterpret_cast<float*>(w.qkv);   // fp32 [M, W] patch-embed output: 4MW of the 6MW bytes, dead before QKV
      } else {
        CREATE_TRY(dev_alloc(h, &w.x, M * W));
        CREATE_TRY(dev_alloc(h, &w.xn, M * W));
      }
      CREATE_TRY(dev_alloc(h, &w.attn, M * W));
      CREATE_TRY(dev_alloc(h, &w.hid, M * std::max<size_t>(4 * W, h->kp)));
      CREATE_TRY(dev_alloc(h, &w.xcls, B * W));
      CREATE_TRY(dev_alloc(h, &w.xncls, B * W));
      CREATE_TRY(dev_alloc(h, &w.qcls, B * W));
      CREATE_TRY(dev_alloc(h, &w.acls, B * W));
      CREATE_TRY(dev_alloc(h, &w.hcls, B * 4 * W));
      if (h->adapter) {
        const size_t D = h->feat_dim;
        CREATE_TRY(dev_alloc(h, &w.taps, B * cfg->layers * W));
        CREATE_TRY(dev_alloc(h, &w.featf, B * D));
        CREATE_TRY(dev_alloc(h, &w.featb, B * D));
        CREATE_TRY(dev_alloc(h, &w.hid2, B * 2 * D));
        CREATE_TRY(dev_alloc(h, &w.mlp, B * D));
      }
    }
  }
  // weight buffers
  for (auto& kv : h->slots) {
    WeightSlot& s = kv.second;
    void* p = nullptr;
    if (h->f32) s.as_bf16 = false;   // verification path: every tensor is kept in fp32 (LayerW's bf16* then point at floats)
    if (cudaMalloc(&p, s.numel * (s.as_bf16 ? 2 : 4) + 256) != cudaSuccess) { h->err = "cudaMalloc(weights) failed"; return bail(ARP_ERR_CUDA); }
    h->allocs.push_back(p);
    *s.dst = p;
    if (s.dst_f32 && h->resid16 && !h->f32) {
      float* q = nullptr;
      if (dev_alloc(h, &q, (size_t)s.numel) != ARP_OK) return bail(ARP_ERR_CUDA);
      *s.dst_f32 = q;
    }
  }
  if (h->resid16 && !h->f32) {
    for (auto& L : h->layers) {
      if (dev_alloc(h, &L.w_qkv_fold, (size_t)3 * W * W) != ARP_OK || dev_alloc(h, &L.w_fc_fold, (size_t)4 * W * W) != ARP_OK ||
          dev_alloc(h, &L.s_qkv, (size_t)3 * W) != ARP_OK || dev_alloc(h, &L.c_qkv, (size_t)3 * W) != ARP_OK ||
          dev_alloc(h, &L.s_fc, (size_t)4 * W) != ARP_OK || dev_alloc(h, &L.c_fc, (size_t)4 * W) != ARP_OK)
        return bail(ARP_ERR_CUDA);
    }
  }
  // opt-in shared memory
#define G2_ATTR(T, A, R) CREATE_TRY(set_smem(h, gemm_tcgen05_kernel<T, A, 2, R>, G2Cfg<2>::SMEM_BYTES));
  G2_ATTR(bf16, ACT_NONE, G2_STORE) G2_ATTR(bf16, ACT_QUICKGELU, G2_STORE) G2_ATTR(bf16, ACT_RELU, G2_STORE)
  G2_ATTR(float, ACT_NONE, G2_STORE) G2_ATTR(float, ACT_QUICKGELU, G2_STORE) G2_ATTR(float, ACT_RELU, G2_STORE)
  G2_ATTR(float, ACT_NONE, G2_REDUCE) G2_ATTR(bf16, ACT_NONE, G2_REDUCE)
  G2_ATTR(bf16, ACT_NONE, G2_LNFOLD) G2_ATTR(bf16, ACT_QUICKGELU, G2_LNFOLD) G2_ATTR(bf16, ACT_NONE, G2_RESID_STATS)
#undef G2_ATTR
  CREATE_TRY(set_smem(h, attention_tc_kernel<197>, AtcCfg<197>::SMEM_BYTES));
  CREATE_TRY(set_smem(h, attention_tc_kernel<50>, AtcCfg<50>::SMEM_BYTES));
  CREATE_TRY(set_smem(h, decode_kernel, 160 * 1024));
  CREATE_TRY(set_smem(h, clip_head_kernel<768, 512>, HEAD_SMEM_BYTES));
  CREATE_TRY(set_smem(h, attention_f32_kernel, attn_f32_smem_bytes(197)));
  if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    h->err = "cudaStreamCreate failed";
    return bail(ARP_ERR_CUDA);
  }
  for (int i = 0; i < 2; ++i) {
    cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_consumed[i], cudaEventDisableTiming);
  }
#undef CREATE_TRY
  *out = h;
  return ARP_OK;
}

// ------------------------------------------------------------------------------------------------
// C ABI: weights / text
// ------------------------------------------------------------------------------------------------
static bool is_ignored_key(const std::string& n) {
  static const char* prefixes[] = {"transformer.", "token_embedding.", "positional_embedding", "ln_final.",
                                   "text_projection", "logit_scale", "text_intermediate_linear.", "text_adapter.",
                                   "text_residual_weight", "inverse_layer.", "lambda_id", "input_resolution",
                                   "context_length", "vocab_size", "image_intermediate_linear.", "image_adapter.",
                                   "image_residual_weight"};
  for (const char* p : prefixes)
    if (n.compare(0, strlen(p), p) == 0) return true;
  return false;
}

extern "C" int arp_set_weight(ArpHandle* h, const char* name, const void* data, int32_t dtype, const int64_t* shape,
                              int32_t ndim, void* stream) {
  if (!h || !name || !data || (ndim > 0 && !shape)) return fail(h, ARP_ERR_INVALID, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::string key(name);
  if (key.compare(0, 11, "clip_model.") == 0) key = key.substr(11);  // adapter checkpoints nest CLIP (finetune.py:164)
  auto it = h->slots.find(key);
  if (it == h->slots.end()) {
    if (is_ignored_key(key)) return ARP_OK;
    return fail(h, ARP_ERR_UNKNOWN_KEY, "unknown weight '%s'", name);
  }
  WeightSlot& s = it->second;
  int64_t numel = 1;
  for (int i = 0; i < ndim; ++i) numel *= shape[i];
  if (numel != s.numel) return fail(h, ARP_ERR_INVALID, "weight '%s': %lld elements, expected %lld", name, (long long)numel, (long long)s.numel);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  void* dst = *s.dst;
  const size_t n = static_cast<size_t>(numel);
  if (s.as_bf16) {
    // the CALLER's tensor dtype (ARP_F32 / ARP_F16 / ARP_BF16) -> the library's operand format (bf16 = op_t)
    if (dtype == ARP_F32) launch_convert<float, bf16>(h, data, dst, n, st);
    else if (dtype == ARP_OP_DTYPE) ARP_CUDA(h, cudaMemcpyAsync(dst, data, n * 2, cudaMemcpyDeviceToDevice, st));
    else if (dtype == ARP_F16) launch_convert<__half, bf16>(h, data, dst, n, st);
    else if (dtype == ARP_BF16) launch_convert<__nv_bfloat16, bf16>(h, data, dst, n, st);
    else return fail(h, ARP_ERR_INVALID, "bad dtype %d", dtype);
  } else {
    if (dtype == ARP_F32) ARP_CUDA(h, cudaMemcpyAsync(dst, data, n * 4, cudaMemcpyDeviceToDevice, st));
    else if (dtype == ARP_F16) launch_convert<__half, float>(h, data, dst, n, st);
    else if (dtype == ARP_BF16) launch_convert<__nv_bfloat16, float>(h, data, dst, n, st);
    else return fail(h, ARP_ERR_INVALID, "bad dtype %d", dtype);
  }
  if (s.dst_f32 && *s.dst_f32) {
    void* d32 = *s.dst_f32;
    if (dtype == ARP_F32) ARP_CUDA(h, cudaMemcpyAsync(d32, data, n * 4, cudaMemcpyDeviceToDevice, st));
    else if (dtype == ARP_F16) launch_convert<__half, float>(h, data, d32, n, st);
    else launch_convert<__nv_bfloat16, float>(h, data, d32, n, st);
  }
  ARP_CUDA(h, cudaGetLastError());
  s.set = true;
  h->finalized = false;
  h->adapter_ready = false;
  h->online_epoch++;
  return ARP_OK;
}

extern "C" int arp_missing_weights(const ArpHandle* h, char* names_out, int64_t names_cap) {
  if (!h) return -1;
  int missing = 0;
  std::string names;
  for (const auto& kv : h->slots)
    if (kv.second.required && !kv.second.set) {
      ++missing;
      names += kv.first;
      names += '\n';
    }
  if (names_out && names_cap > 0) {
    const size_t n = std::min<size_t>(names.size(), static_cast<size_t>(names_cap - 1));
    memcpy(names_out, names.data(), n);
    names_out[n] = 0;
  }
  return missing;
}

// the adapter gate sigmoid(image_residual_weight) (clip_multiscale_adapter.py:145-151), read once per weight upload
static int read_res_sigmoid(ArpHandle* h, cudaStream_t st) {
  float w = 0.f;
  ARP_CUDA(h, cudaMemcpyAsync(&w, h->res_w, 4, cudaMemcpyDeviceToHost, st));
  ARP_CUDA(h, cudaStreamSynchronize(st));
  h->res_sigmoid = 1.0f / (1.0f + expf(-w));
  return ARP_OK;
}

static int finalize_weights(ArpHandle* h, cudaStream_t st) {
  if (h->finalized) return ARP_OK;
  char buf[256];
  const int miss = arp_missing_weights(h, buf, sizeof(buf));
  if (miss) return fail(h, ARP_ERR_STATE, "%d weights not set, first: %.200s", miss, buf);
  const int n = h->tokens * h->cfg.width;
  build_rowtab_kernel<<<(n + 255) / 256, 256, 0, st>>>(h->pos_emb, h->class_emb, h->rowtab, h->tokens, h->cfg.width);
  h->launches++;
  if (h->resid16 && !h->f32) {
    const int W = h->cfg.width;
    for (auto& L : h->layers) {
      fold_ln_weights_kernel<<<(3 * W + 7) / 8, 256, 0, st>>>(L.w_qkv_f32, L.ln1_g, L.ln1_b, L.b_qkv, L.w_qkv_fold, L.s_qkv, L.c_qkv, 3 * W, W);
      fold_ln_weights_kernel<<<(4 * W + 7) / 8, 256, 0, st>>>(L.w_fc_f32, L.ln2_g, L.ln2_b, L.b_fc, L.w_fc_fold, L.s_fc, L.c_fc, 4 * W, W);
      h->launches += 2;
    }
  }
  if (h->adapter) ARP_TRY(read_res_sigmoid(h, st));
  ARP_CUDA(h, cudaGetLastError());
  h->finalized = true;
  return ARP_OK;
}

// arp_label_tower's readiness: only the image-adapter tensors are needed (no visual.* slot, no rowtab, no LayerNorm fold),
// and res_sigmoid is computed from image_residual_weight as finalize_weights computes it
static int adapter_weights_ready(ArpHandle* h, cudaStream_t st) {
  if (h->adapter_ready || h->finalized) return ARP_OK;
  static const char* names[] = {"image_intermediate_linear.weight", "image_adapter.layers.0.weight",
                                "image_adapter.layers.0.bias", "image_adapter.layers.3.weight",
                                "image_adapter.layers.3.bias", "image_residual_weight"};
  for (const char* n : names)
    if (!h->slots.at(n).set) return fail(h, ARP_ERR_STATE, "adapter weight '%s' not set", n);
  ARP_TRY(read_res_sigmoid(h, st));
  h->adapter_ready = true;
  return ARP_OK;
}

// arp_set_text is the one-group case of arp_set_text_groups; only the grouped entry point refuses goal heads
static int set_text_rows(ArpHandle* h, const float* text_emb_dev, int32_t n_text_total, int32_t dim,
                         const int32_t* group_offsets_host, int32_t n_groups, float logit_scale_exp, cudaStream_t st) {
  if (!h || !text_emb_dev || !group_offsets_host) return fail(h, ARP_ERR_INVALID, "null argument");
  if (n_groups < 1 || n_groups > HEAD_MAX_GROUPS)
    return fail(h, ARP_ERR_INVALID, "n_groups must be in [1,%d], got %d", HEAD_MAX_GROUPS, n_groups);
  if (n_text_total < 1 || n_text_total > HEAD_MAX_TEXT_TOTAL)
    return fail(h, ARP_ERR_INVALID, "n_text_total must be in [1,%d], got %d", HEAD_MAX_TEXT_TOTAL, n_text_total);
  if (group_offsets_host[0] != 0 || group_offsets_host[n_groups] != n_text_total)
    return fail(h, ARP_ERR_INVALID, "group offsets must run from 0 to n_text_total=%d", n_text_total);
  for (int g = 0; g < n_groups; ++g) {
    const int n = group_offsets_host[g + 1] - group_offsets_host[g];
    if (n < 1 || n > HEAD_MAX_TEXT)
      return fail(h, ARP_ERR_INVALID, "group %d has %d texts, must be in [1,%d]", g, n, HEAD_MAX_TEXT);
  }
  if (dim != h->feat_dim) return fail(h, ARP_ERR_INVALID, "text dim %d, head expects %d", dim, h->feat_dim);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  if (!h->text) ARP_TRY(dev_alloc(h, &h->text, (size_t)HEAD_MAX_TEXT_TOTAL * h->feat_dim));
  if (!h->group_off) ARP_TRY(dev_alloc(h, &h->group_off, (size_t)HEAD_MAX_GROUPS + 1));
  // the handle keeps the host copy: the H2D source stays valid whenever the copy runs
  std::copy(group_offsets_host, group_offsets_host + n_groups + 1, h->group_off_host);
  ARP_CUDA(h, cudaMemcpyAsync(h->text, text_emb_dev, (size_t)n_text_total * dim * 4, cudaMemcpyDeviceToDevice, st));
  ARP_CUDA(h, cudaMemcpyAsync(h->group_off, h->group_off_host, (size_t)(n_groups + 1) * 4, cudaMemcpyHostToDevice, st));
  h->n_text = n_text_total;
  h->n_groups = n_groups;
  h->text_dim = dim;
  h->logit_scale = logit_scale_exp;
  h->online_epoch++;
  return ARP_OK;
}

extern "C" int arp_set_text_groups(ArpHandle* h, const float* text_emb_dev, int32_t n_text_total, int32_t dim,
                                   const int32_t* group_offsets_host, int32_t n_groups, float logit_scale_exp,
                                   void* stream) {
  if (h && h->goal) return fail(h, ARP_ERR_INVALID, "goal-conditioned heads take no text");
  return set_text_rows(h, text_emb_dev, n_text_total, dim, group_offsets_host, n_groups, logit_scale_exp,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int arp_set_text(ArpHandle* h, const float* text_emb_dev, int32_t n_text, int32_t dim, float logit_scale_exp,
                            void* stream) {
  if (h && (n_text < 1 || n_text > HEAD_MAX_TEXT))
    return fail(h, ARP_ERR_INVALID, "n_text must be in [1,%d]", HEAD_MAX_TEXT);
  const int32_t off[2] = {0, n_text};
  return set_text_rows(h, text_emb_dev, n_text, dim, off, 1, logit_scale_exp, static_cast<cudaStream_t>(stream));
}

extern "C" int arp_text_groups(const ArpHandle* h) { return h ? h->n_groups : 0; }

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------
// 2-D row-major tensor [rows, cols] with row pitch ld (elements of `elem` bytes: 2 = bf16, 4 = fp32),
// box [box_rows, box_cols] with a 128-byte inner extent and the 128B swizzle.
static int get_tmap(ArpHandle* h, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                    const CUtensorMap** out, uint32_t box_cols = GEMM_BK, uint32_t elem = 2) {
  TmapKey key{ptr, rows, cols, ld, box_rows, box_cols, elem};
  auto it = h->tmaps.find(key);
  if (it == h->tmaps.end()) {
    if (h->tmaps.size() > 4096) h->tmaps.clear();
    CUtensorMap m;
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {ld * elem};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (gstr[0] & 15))
      return fail(h, ARP_ERR_INVALID, "GEMM operand must be 16-byte aligned with a 16-byte multiple row pitch");
    CUresult r = get_encode_tiled()(&m, elem == 2 ? (ARP_OP_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) : CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                                    2, const_cast<void*>(ptr), gdim, gstr, box,
                                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, ARP_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu", (int)r, (unsigned long long)rows, (unsigned long long)cols);
    it = h->tmaps.emplace(key, m).first;
  }
  *out = &it->second;
  return ARP_OK;
}

// 3-D view [frames, tokens, width] of the attention output with a (1 frame) x 32 tokens x 64 columns box, 128B swizzle:
// one softmax warp's 32 query rows of one head. Rows past `tokens` are out of bounds in dimension 1 and are NOT written,
// so a partially filled warp (tokens = 197: rows 192..196) never touches the next frame's rows.
static int get_tmap_attn_out(ArpHandle* h, const void* ptr, uint64_t frames, uint64_t tokens, uint64_t width,
                             const CUtensorMap** out, uint32_t box_rows = 32) {
  TmapKey key{ptr, frames, tokens, width, box_rows, 64, 0x30002u};
  auto it = h->tmaps.find(key);
  if (it == h->tmaps.end()) {
    if (h->tmaps.size() > 4096) h->tmaps.clear();
    CUtensorMap m;
    cuuint64_t gdim[3] = {width, tokens, frames};
    cuuint64_t gstr[2] = {width * 2, tokens * width * 2};
    cuuint32_t box[3] = {64, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) || (gstr[0] & 15))
      return fail(h, ARP_ERR_INVALID, "attention output must be 16-byte aligned with a 16-byte multiple row pitch");
    CUresult r = get_encode_tiled()(&m, ARP_OP_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3,
                                    const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, ARP_ERR_CUDA, "cuTensorMapEncodeTiled (attention output) failed (%d)", (int)r);
    it = h->tmaps.emplace(key, m).first;
  }
  *out = &it->second;
  return ARP_OK;
}

template <typename K>
static cudaError_t launch_clustered(K kernel, int grid, int cg, int smem, cudaStream_t st, const CUtensorMap& ta,
                                    const CUtensorMap& tb, const CUtensorMap& to, const GemmArgs& g) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(G2_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cg;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, ta, tb, to, g);
}

// LayerNorm fold of one GEMM launch (gemm_tcgen05.cuh G2_LNFOLD): per-row statistics of A, per-column vectors of W
struct LnFoldArgs { const float2* stats; const float* svec; const float* cvec; int nparts = 1; };   // nparts: GemmArgs::ln_nparts

// out[M, N] (ldo) = epilogue(a[M, K] · w[N, K]^T). `resid` (same dtype as out; must alias out on the hot path): the
// output is ACCUMULATED into it by TMA reduce-add. a_rows_alloc: rows addressable behind `a` (>= M); the descriptor
// covers them so that reading a partly filled workspace never depends on M (rows are independent; rows >= M are
// computed and dropped by the clipped store).
static int launch_gemm(ArpHandle* h, const bf16* a, int64_t a_rows_alloc, const bf16* w, void* out, bool out_f32,
                       int act, int64_t M, int N, int K, int ldo, const float* bias, const void* resid, int ldr,
                       const float* rowtab, int period, cudaStream_t st, const LnFoldArgs* fold = nullptr,
                       float2* stats_out = nullptr) {
  if (M <= 0) return ARP_OK;
  if (N % GEMM_BN || K % GEMM_BK) return fail(h, ARP_ERR_INVALID, "GEMM needs N %% 256 == 0 and K %% 64 == 0 (N=%d K=%d)", N, K);
  if (M > 0x7fffffff / 2) return fail(h, ARP_ERR_INVALID, "GEMM M too large");
  constexpr int cg = 2;
  const size_t osz = out_f32 ? 4 : 2;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = (int)M; g.N = N; g.K = K; g.out = out; g.ldo = ldo; g.bias = bias;
  g.rowtab = rowtab; g.period = period > 0 ? period : 1;
  g.reverse = h->dir ^= 1;
  const bool reduce = resid != nullptr;
  if (fold) {
    if (out_f32 || act == ACT_RELU || reduce || rowtab || !fold->stats || !fold->svec || !fold->cvec)
      return fail(h, ARP_ERR_INVALID, "bad LayerNorm-folded GEMM");
    g.ln_stats = fold->stats; g.ln_nparts = fold->nparts; g.svec = fold->svec; g.cvec = fold->cvec; g.eps = 1e-5f;
    g.bias = nullptr;   // cvec carries the bias
  }
  // stats_out: the 16-bit in-place residual update done in registers, emitting the updated rows' LayerNorm statistics
  const bool resid_stats = stats_out != nullptr;
  if (resid_stats) {
    if (!reduce || resid != out || out_f32 || ldr != ldo || rowtab || !bias) return fail(h, ARP_ERR_INVALID, "bad residual+statistics GEMM");
    g.resid = static_cast<const bf16*>(resid); g.ldr = ldr; g.stats_out = stats_out; g.eps = 1e-5f;
  }
  if (reduce) {
    if (act != ACT_NONE) return fail(h, ARP_ERR_INVALID, "the residual epilogue takes no activation");
    if (resid != out)  // out-of-place residual (test hook only): seed the output, then accumulate into it
      ARP_CUDA(h, cudaMemcpy2DAsync(out, (size_t)ldo * osz, resid, (size_t)ldr * osz, (size_t)N * osz, (size_t)M,
                                    cudaMemcpyDeviceToDevice, st));
  }
  const CUtensorMap *ta, *tb, *to;
  ARP_TRY(get_tmap(h, a, (uint64_t)a_rows_alloc, (uint64_t)K, (uint64_t)K, GEMM_BM, &ta));
  ARP_TRY(get_tmap(h, w, (uint64_t)N, (uint64_t)K, (uint64_t)K, GEMM_BN / cg, &tb));
  ARP_TRY(get_tmap(h, out, (uint64_t)M, (uint64_t)N, (uint64_t)ldo, 32, &to, out_f32 ? 32 : 64, out_f32 ? 4 : 2));
  const int row_blocks = (int)((M + GEMM_BM * cg - 1) / (GEMM_BM * cg));
  const int tiles = row_blocks * (N / GEMM_BN);
  const int grid = std::min(tiles * cg, kNumSMs / cg * cg);
  const int smem = G2Cfg<cg>::SMEM_BYTES;
  ProfScope prof(h, PC_GEMM, 2.0 * (double)M * N * K,
                 (double)M * K * 2 + (double)N * K * 2 + (double)M * N * osz * (reduce ? 2 : 1), st);
  cudaError_t e;
#define G2_LAUNCH(T, A, R) e = launch_clustered(gemm_tcgen05_kernel<T, A, cg, R>, grid, cg, smem, st, *ta, *tb, *to, g)
  if (fold) {
    if (act == ACT_NONE) G2_LAUNCH(bf16, ACT_NONE, G2_LNFOLD);
    else G2_LAUNCH(bf16, ACT_QUICKGELU, G2_LNFOLD);
  } else if (resid_stats) {
    G2_LAUNCH(bf16, ACT_NONE, G2_RESID_STATS);
  } else if (reduce) {
    if (out_f32) G2_LAUNCH(float, ACT_NONE, G2_REDUCE);
    else G2_LAUNCH(bf16, ACT_NONE, G2_REDUCE);
  } else if (out_f32) {
    if (act == ACT_NONE) G2_LAUNCH(float, ACT_NONE, G2_STORE);
    else if (act == ACT_QUICKGELU) G2_LAUNCH(float, ACT_QUICKGELU, G2_STORE);
    else G2_LAUNCH(float, ACT_RELU, G2_STORE);
  } else {
    if (act == ACT_NONE) G2_LAUNCH(bf16, ACT_NONE, G2_STORE);
    else if (act == ACT_QUICKGELU) G2_LAUNCH(bf16, ACT_QUICKGELU, G2_STORE);
    else G2_LAUNCH(bf16, ACT_RELU, G2_STORE);
  }
#undef G2_LAUNCH
  h->launches++;
  if (e != cudaSuccess) return fail(h, ARP_ERR_CUDA, "GEMM launch failed: %s", cudaGetErrorString(e));
  return ARP_OK;
}

static int launch_decode(ArpHandle* h, const uint8_t* ob, int64_t n, int64_t stride, void* out, int out_kind,
                         cudaStream_t st) {
  if (n <= 0) return ARP_OK;
  DecodeArgs a;
  memset(&a, 0, sizeof(a));
  a.ob = ob; a.frame_stride = stride; a.in_w = h->cfg.in_w;
  a.crop_top = h->crop_top; a.crop_left = h->crop_left; a.src_h = h->src_h; a.src_w = h->src_w;
  a.T = (int)n; a.mode = h->cfg.preprocess; a.out_kind = out_kind;
  a.h_min = h->h_min; a.h_cnt = h->h_cnt; a.h_k = h->h_k; a.h_ksize = h->h_ksize;
  a.v_min = h->v_min; a.v_cnt = h->v_cnt; a.v_k = h->v_k; a.v_ksize = h->v_ksize;
  a.lut = h->lut;
  for (int c = 0; c < 3; ++c) { a.mean[c] = kClipMean[c]; a.stdv[c] = kClipStd[c]; }
  a.out = out; a.patch = h->cfg.patch; a.grid = h->grid; a.tokens = h->tokens; a.max_rows = h->max_rows;
  const int smem = dec_smem_bytes(h->src_w, h->max_rows, h->h_ksize, h->v_ksize, out_kind);
  if (smem > 160 * 1024) return fail(h, ARP_ERR_INVALID, "frame too large for the decode kernel (%d B smem)", smem);
  ProfScope prof(h, PC_DECODE, 0.0,
                 (double)n * ((double)h->src_h * h->src_w * 3 +
                              (out_kind == DEC_OUT_PATCH_BF16 ? (double)h->tokens * h->kp * 2 : 3.0 * DEC_OUT * DEC_OUT * 4)), st);
  // grid.y is limited to 65535 frames per launch
  for (int64_t f0 = 0; f0 < n; f0 += 32768) {
    const int cnt = (int)std::min<int64_t>(32768, n - f0);
    DecodeArgs b = a;
    b.ob = ob + f0 * stride;
    b.T = cnt;
    if (out_kind == DEC_OUT_PATCH_BF16) b.out = static_cast<bf16*>(out) + (size_t)f0 * h->tokens * h->kp;
    else b.out = static_cast<float*>(out) + (size_t)f0 * 3 * DEC_OUT * DEC_OUT;
    decode_kernel<<<dim3(DEC_OUT / DEC_BAND, cnt), DEC_THREADS, smem, st>>>(b);
    h->launches++;
  }
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

static int launch_ln_bf16(ArpHandle* h, const float* x, const float* g, const float* b, bf16* y, int64_t M,
                          cudaStream_t st) {
  if (M <= 0) return ARP_OK;
  ProfScope prof(h, PC_LAYERNORM, 0.0, (double)M * 768 * 6, st);
  layernorm_f32_bf16_kernel<768><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(x, g, b, y, (int)M, 1e-5f, h->dir ^= 1);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// (rstd, -mean*rstd) of every row of the 16-bit residual stream: the LayerNorm the next GEMM applies in its epilogue
static int launch_row_moments(ArpHandle* h, const bf16* x, float2* stats, int64_t M, cudaStream_t st) {
  if (M <= 0) return ARP_OK;
  ProfScope prof(h, PC_LAYERNORM, 0.0, (double)M * (768 * 2 + 8), st);
  row_moments_kernel<768><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(x, stats, (int)M, 1e-5f, h->dir ^= 1);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

static int launch_attention(ArpHandle* h, const bf16* qkv, bf16* out, int B, int tokens, cudaStream_t st,
                            int64_t rows_alloc = 0) {
  if (B <= 0) return ARP_OK;
  const float scale_log2e = 0.125f * 1.4426950408889634f;
  ProfScope prof(h, PC_ATTENTION, 4.0 * (double)B * h->cfg.heads * tokens * tokens * 64,
                 (double)B * tokens * h->cfg.width * 2 * 4, st);
  if (tokens != 197 && tokens != 50) return fail(h, ARP_ERR_INVALID, "attention is built for 197 or 50 tokens, got %d", tokens);
  const int W = h->cfg.width;
  const uint64_t rows = rows_alloc > 0 ? (uint64_t)rows_alloc : (uint64_t)B * tokens;
  const int nk = (tokens + 15) / 16 * 16;
  const CUtensorMap *tq, *tkv, *to, *tq16, *to16;
  ARP_TRY(get_tmap(h, qkv, rows, 3 * W, 3 * W, 128, &tq));
  ARP_TRY(get_tmap(h, qkv, rows, 3 * W, 3 * W, nk, &tkv));
  ARP_TRY(get_tmap_attn_out(h, out, (uint64_t)B, (uint64_t)tokens, (uint64_t)W, &to));
  ARP_TRY(get_tmap(h, qkv, rows, 3 * W, 3 * W, 16, &tq16));            // 16-row boxes: query tile 1 spread over the quarters
  ARP_TRY(get_tmap_attn_out(h, out, (uint64_t)B, (uint64_t)tokens, (uint64_t)W, &to16, 16));
  const int grid = std::min(B * h->cfg.heads, kNumSMs);
  const int rev = h->dir ^= 1;
  if (tokens == 197)
    attention_tc_kernel<197><<<grid, ATC_THREADS, AtcCfg<197>::SMEM_BYTES, st>>>(*tq, *tkv, *to, *tq16, *to16, B, h->cfg.heads, W, scale_log2e, rev);
  else
    attention_tc_kernel<50><<<grid, ATC_THREADS, AtcCfg<50>::SMEM_BYTES, st>>>(*tq, *tkv, *to, *tq16, *to16, B, h->cfg.heads, W, scale_log2e, rev);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// ------------------------------------------------------------------------------------------------
// the encoder: n frames (n <= max_batch) -> residual stream x after the last block (+ CLS taps)
// ------------------------------------------------------------------------------------------------
static int encode_chunk_f32(ArpHandle* h, const uint8_t* ob, int64_t n, int64_t stride, cudaStream_t st,
                            const float* chw, float* taps32);

// The last resblock for the class-token row only: every head reads just the class-token row of the last block's output
// (ln_post(x[:,0]), adapter taps = class-token rows), so that block computes K/V for all tokens but Q, attention,
// out_proj and the MLP for the class-token row only — same result, 2.4 of 35.1 GFLOP per frame less. K and V of every
// token are already in ws.qkv (columns [W, 3W)); XT = type of the residual stream `x` the class-token rows are gathered
// from. The heads read the result from ws.xcls.
template <typename XT>
static int last_block_cls(ArpHandle* h, const LayerW& L, const XT* x, int64_t n, cudaStream_t st, float* taps32) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const int W = c.width;
  const int64_t B = c.max_batch;
  gather_cls_rows_f32_kernel<768, XT><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(x, ws.xcls, (int)n, h->tokens, W, 0);
  h->launches++;
  ARP_TRY(launch_ln_bf16(h, ws.xcls, L.ln1_g, L.ln1_b, ws.xncls, n, st));
  ARP_TRY(launch_gemm(h, ws.xncls, B, L.w_qkv, ws.qcls, false, ACT_NONE, n, W, W, W, L.b_qkv, nullptr, 0, nullptr, 0, st));
  {
    ProfScope prof(h, PC_ATTENTION, 4.0 * (double)n * c.heads * h->tokens * 64,
                   (double)n * h->tokens * W * 2 * 2 + (double)n * W * 2 * 2, st);
    const unsigned blocks = (unsigned)((n * c.heads + 7) / 8);
    if (h->tokens == 197)
      cls_attention_kernel<197><<<blocks, 256, 0, st>>>(ws.qcls, ws.qkv, ws.acls, (int)n, c.heads, W, 0.125f);
    else if (h->tokens == 50)
      cls_attention_kernel<50><<<blocks, 256, 0, st>>>(ws.qcls, ws.qkv, ws.acls, (int)n, c.heads, W, 0.125f);
    else
      return fail(h, ARP_ERR_INVALID, "attention is built for 197 or 50 tokens, got %d", h->tokens);
    h->launches++;
  }
  ARP_TRY(launch_gemm(h, ws.acls, B, L.w_out, ws.xcls, true, ACT_NONE, n, W, W, W, L.b_out, ws.xcls, W, nullptr, 0, st));
  ARP_TRY(launch_ln_bf16(h, ws.xcls, L.ln2_g, L.ln2_b, ws.xncls, n, st));
  ARP_TRY(launch_gemm(h, ws.xncls, B, L.w_fc, ws.hcls, false, ACT_QUICKGELU, n, 4 * W, W, 4 * W, L.b_fc, nullptr, 0,
                      nullptr, 0, st));
  ARP_TRY(launch_gemm(h, ws.hcls, B, L.w_proj, ws.xcls, true, ACT_NONE, n, W, 4 * W, W, L.b_proj, ws.xcls, W, nullptr,
                      0, st));
  const int l = c.layers - 1;
  if (h->adapter) {
    gather_cls_bf16_kernel<768, float><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ws.xcls, ws.taps, (int)n, 1, c.layers * W, l * W);
    h->launches++;
  }
  if (taps32) {
    gather_cls_rows_f32_kernel<768, float><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ws.xcls, taps32, (int)n, 1,
                                                                                 c.layers * W, l * W);
    h->launches++;
  }
  return ARP_OK;
}

// class-token taps of block l's output: 16-bit for the adapter head, fp32 into taps32 for arp_encode_taps_chw
template <typename XT>
static void gather_taps(ArpHandle* h, const XT* x, int64_t n, int l, cudaStream_t st, float* taps32) {
  const ArpConfig& c = h->cfg;
  if (h->adapter) {
    gather_cls_bf16_kernel<768, XT><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(x, h->ws.taps, (int)n, h->tokens,
                                                                          c.layers * c.width, l * c.width);
    h->launches++;
  }
  if (taps32) {
    gather_cls_rows_f32_kernel<768, XT><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(x, taps32, (int)n, h->tokens,
                                                                              c.layers * c.width, l * c.width);
    h->launches++;
  }
}

// Default path: 16-bit residual stream, LayerNorm folded into the consumer GEMMs (ArpHandle::resid16). The residual
// GEMMs add in registers and emit the next LayerNorm's row statistics themselves (gemm_tcgen05.cuh G2_RESID_STATS): one
// rounding per update and no LayerNorm-class kernel inside the blocks.
static int encode_blocks_r16(ArpHandle* h, int64_t n, cudaStream_t st, float* taps32) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const int W = c.width;
  const int64_t M = n * h->tokens, Mcap = (int64_t)c.max_batch * h->tokens;
  {
    ProfScope prof(h, PC_LAYERNORM, 0.0, (double)M * (768 * 6 + 8), st);
    layernorm_pre_r16_kernel<768><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(ws.x, h->ln_pre_g, h->ln_pre_b, ws.x16,
                                                                          ws.stats, (int)M, 1e-5f);
    h->launches++;
  }
  // format of ws.stats: 1 = (rstd, -mean*rstd) per row (layernorm_pre_r16_kernel), 2*W/256 = partial (mean, M2) per 128
  // columns (written by the residual GEMM's epilogue)
  int parts = 1;
  for (int l = 0; l < c.layers; ++l) {
    const LayerW& L = h->layers[l];
    if (l == c.layers - 1) {
      // K and V of every token: rows [W, 3W) of in_proj, written at column W of the qkv buffer
      const LnFoldArgs f_kv{ws.stats, L.s_qkv + W, L.c_qkv + W, parts};
      ARP_TRY(launch_gemm(h, ws.x16, Mcap, L.w_qkv_fold + (size_t)W * W, ws.qkv + W, false, ACT_NONE, M, 2 * W, W, 3 * W,
                          nullptr, nullptr, 0, nullptr, 0, st, &f_kv));
      ARP_TRY(last_block_cls(h, L, ws.x16, n, st, taps32));
      break;
    }
    const LnFoldArgs f_qkv{ws.stats, L.s_qkv, L.c_qkv, parts};
    ARP_TRY(launch_gemm(h, ws.x16, Mcap, L.w_qkv_fold, ws.qkv, false, ACT_NONE, M, 3 * W, W, 3 * W, nullptr, nullptr, 0,
                        nullptr, 0, st, &f_qkv));
    parts = 2 * W / 256;
    const LnFoldArgs f_fc{ws.stats, L.s_fc, L.c_fc, parts};
    ARP_TRY(launch_attention(h, ws.qkv, ws.attn, (int)n, h->tokens, st, Mcap));
    // x += out_proj(attn) in place; the epilogue also leaves ln_2's row statistics in ws.stats
    ARP_TRY(launch_gemm(h, ws.attn, Mcap, L.w_out, ws.x16, false, ACT_NONE, M, W, W, W, L.b_out, ws.x16, W, nullptr, 0, st,
                        nullptr, ws.stats));
    ARP_TRY(launch_gemm(h, ws.x16, Mcap, L.w_fc_fold, ws.hid, false, ACT_QUICKGELU, M, 4 * W, W, 4 * W, nullptr, nullptr,
                        0, nullptr, 0, st, &f_fc));
    ARP_TRY(launch_gemm(h, ws.hid, Mcap, L.w_proj, ws.x16, false, ACT_NONE, M, W, 4 * W, W, L.b_proj, ws.x16, W, nullptr,
                        0, st, nullptr, ws.stats));   // ... and the next block's ln_1 statistics
    gather_taps(h, ws.x16, n, l, st, taps32);
  }
  return ARP_OK;
}

// ARP_PREC_F32RESID: fp32 residual stream, standalone LayerNorm kernels writing the 16-bit GEMM operand.
static int encode_blocks_r32(ArpHandle* h, int64_t n, cudaStream_t st, float* taps32) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const int W = c.width;
  const int64_t M = n * h->tokens, Mcap = (int64_t)c.max_batch * h->tokens;
  {
    ProfScope prof(h, PC_LAYERNORM, 0.0, (double)M * 768 * 8, st);
    layernorm_f32_inplace_kernel<768><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(ws.x, h->ln_pre_g, h->ln_pre_b, (int)M, 1e-5f);
    h->launches++;
  }
  for (int l = 0; l < c.layers; ++l) {
    const LayerW& L = h->layers[l];
    ARP_TRY(launch_ln_bf16(h, ws.x, L.ln1_g, L.ln1_b, ws.xn, M, st));
    if (l == c.layers - 1) {
      ARP_TRY(launch_gemm(h, ws.xn, Mcap, L.w_qkv + (size_t)W * W, ws.qkv + W, false, ACT_NONE, M, 2 * W, W, 3 * W,
                          L.b_qkv + W, nullptr, 0, nullptr, 0, st));
      ARP_TRY(last_block_cls(h, L, ws.x, n, st, taps32));
      break;
    }
    ARP_TRY(launch_gemm(h, ws.xn, Mcap, L.w_qkv, ws.qkv, false, ACT_NONE, M, 3 * W, W, 3 * W, L.b_qkv, nullptr, 0,
                        nullptr, 0, st));
    ARP_TRY(launch_attention(h, ws.qkv, ws.attn, (int)n, h->tokens, st, Mcap));
    ARP_TRY(launch_gemm(h, ws.attn, Mcap, L.w_out, ws.x, true, ACT_NONE, M, W, W, W, L.b_out, ws.x, W, nullptr, 0, st));
    ARP_TRY(launch_ln_bf16(h, ws.x, L.ln2_g, L.ln2_b, ws.xn, M, st));
    ARP_TRY(launch_gemm(h, ws.xn, Mcap, L.w_fc, ws.hid, false, ACT_QUICKGELU, M, 4 * W, W, 4 * W, L.b_fc, nullptr, 0,
                        nullptr, 0, st));
    ARP_TRY(launch_gemm(h, ws.hid, Mcap, L.w_proj, ws.x, true, ACT_NONE, M, W, 4 * W, W, L.b_proj, ws.x, W, nullptr, 0, st));
    gather_taps(h, ws.x, n, l, st, taps32);
  }
  return ARP_OK;
}

// Input: n dataset frames at ob (row pitch `stride`), or, when chw is set, a caller-preprocessed fp32 image batch
// [n, 3, 224, 224]. taps32 (optional, arp_encode_taps_chw): fp32 [n, layers*W] receives the class-token row of every
// block's output — the frozen-CLIP side of fine-tuning.
static int encode_chunk(ArpHandle* h, const uint8_t* ob, int64_t n, int64_t stride, cudaStream_t st,
                        const float* chw = nullptr, float* taps32 = nullptr) {
  if (h->f32) return encode_chunk_f32(h, ob, n, stride, st, chw, taps32);
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const int W = c.width;
  const int64_t M = n * h->tokens;
  const int64_t Mcap = (int64_t)c.max_batch * h->tokens;
  bf16* patches = ws.hid;  // aliases the MLP hidden buffer (dead until layer 0's c_fc)
  if (chw) {
    ProfScope prof(h, PC_DECODE, 0.0, (double)n * (3.0 * DEC_OUT * DEC_OUT * 4 + (double)h->tokens * h->kp * 2), st);
    patchify_chw_bf16_kernel<<<kNumSMs * 8, 256, 0, st>>>(chw, patches, (int)n, c.patch, h->grid, h->tokens);
    h->launches++;
  } else {
    ARP_TRY(launch_decode(h, ob, n, stride, patches, DEC_OUT_PATCH_BF16, st));
  }
  // patch embed (+ positional embedding, + class embedding on the all-zero row 0 of each frame), fp32 out
  ARP_TRY(launch_gemm(h, patches, Mcap, h->conv1, ws.x, true, ACT_NONE, M, W, h->kp, W, nullptr, nullptr, 0,
                      h->rowtab, h->tokens, st));
  ARP_TRY(h->resid16 ? encode_blocks_r16(h, n, st, taps32) : encode_blocks_r32(h, n, st, taps32));
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// ------------------------------------------------------------------------------------------------
// fp32 verification path (fp32_path.cuh): same schedule, FP32 FMA kernels
// ------------------------------------------------------------------------------------------------
static int launch_sgemm(ArpHandle* h, const float* a, int lda, const void* w, float* out, int ldo, int act, int64_t M,
                        int N, int K, const float* bias, const float* resid, int ldr, const float* rowtab, int period,
                        cudaStream_t st) {
  if (M <= 0) return ARP_OK;
  if (N % SG_BN || K % SG_BK) return fail(h, ARP_ERR_INVALID, "fp32 GEMM needs N %% 128 == 0 and K %% 16 == 0 (N=%d K=%d)", N, K);
  ProfScope prof(h, PC_GEMM, 2.0 * (double)M * N * K, ((double)M * K + (double)N * K + (double)M * N) * 4, st);
  dim3 grid(N / SG_BN, (unsigned)((M + SG_BM - 1) / SG_BM));
  sgemm_nt_f32_kernel<<<grid, SG_THREADS, 0, st>>>(a, static_cast<const float*>(w), out, (int)M, N, K, lda, ldo, bias,
                                                   resid, ldr, rowtab, period > 0 ? period : 1, act);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// The verification path computes every row of every block: the heads read the class-token rows from ws.x.
static int encode_chunk_f32(ArpHandle* h, const uint8_t* ob, int64_t n, int64_t stride, cudaStream_t st,
                            const float* chw, float* taps32) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const int W = c.width;
  const int64_t M = n * h->tokens;
  if (h->tokens != 197 && h->tokens != 50) return fail(h, ARP_ERR_INVALID, "unsupported token count %d", h->tokens);
  float* patches = ws.hid32;   // dead until layer 0's c_fc
  if (!chw) ARP_TRY(launch_decode(h, ob, n, stride, ws.chw32, DEC_OUT_CHW_F32, st));
  im2col_f32_kernel<<<kNumSMs * 8, 256, 0, st>>>(chw ? chw : ws.chw32, patches, (int)n, c.patch, h->grid, h->tokens);
  h->launches++;
  ARP_TRY(launch_sgemm(h, patches, h->kp, h->conv1, ws.x, W, F32_ACT_NONE, M, W, h->kp, nullptr, nullptr, 0, h->rowtab,
                       h->tokens, st));
  auto ln = [&](const float* x, const float* g, const float* b, float* y) {
    ProfScope prof(h, PC_LAYERNORM, 0.0, (double)M * W * 8, st);
    layernorm_f32_f32_kernel<768><<<(unsigned)((M + 7) / 8), 256, 0, st>>>(x, g, b, y, (int)M, 1e-5f);
    h->launches++;
  };
  ln(ws.x, h->ln_pre_g, h->ln_pre_b, ws.x);
  for (int l = 0; l < c.layers; ++l) {
    const LayerW& L = h->layers[l];
    ln(ws.x, L.ln1_g, L.ln1_b, ws.xn32);
    ARP_TRY(launch_sgemm(h, ws.xn32, W, L.w_qkv, ws.qkv32, 3 * W, F32_ACT_NONE, M, 3 * W, W, L.b_qkv, nullptr, 0, nullptr,
                         0, st));
    {
      ProfScope prof(h, PC_ATTENTION, 4.0 * (double)n * c.heads * h->tokens * h->tokens * 64, (double)M * W * 4 * 4, st);
      for (int64_t b0 = 0; b0 < n; b0 += 32768) {
        const int cnt = (int)std::min<int64_t>(32768, n - b0);
        attention_f32_kernel<<<dim3(c.heads, cnt), A32_THREADS, attn_f32_smem_bytes(h->tokens), st>>>(
            ws.qkv32 + (size_t)b0 * h->tokens * 3 * W, ws.attn32 + (size_t)b0 * h->tokens * W, h->tokens, W);
        h->launches++;
      }
    }
    ARP_TRY(launch_sgemm(h, ws.attn32, W, L.w_out, ws.x, W, F32_ACT_NONE, M, W, W, L.b_out, ws.x, W, nullptr, 0, st));
    ln(ws.x, L.ln2_g, L.ln2_b, ws.xn32);
    ARP_TRY(launch_sgemm(h, ws.xn32, W, L.w_fc, ws.hid32, 4 * W, F32_ACT_QUICKGELU, M, 4 * W, W, L.b_fc, nullptr, 0,
                         nullptr, 0, st));
    ARP_TRY(launch_sgemm(h, ws.hid32, 4 * W, L.w_proj, ws.x, W, F32_ACT_NONE, M, W, 4 * W, L.b_proj, ws.x, W, nullptr, 0,
                         st));
    if (h->adapter) {
      gather_cls_rows_f32_kernel<768, float><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ws.x, ws.taps32, (int)n, h->tokens,
                                                                        c.layers * W, l * W);
      h->launches++;
    }
    if (taps32) {
      gather_cls_rows_f32_kernel<768, float><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ws.x, taps32, (int)n, h->tokens,
                                                                        c.layers * W, l * W);
      h->launches++;
    }
  }
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// The adapter heads' final CLIP feature: clip_head_kernel on the class-token rows -> the last 512 columns of ws.featf
// (un-normalised, clip_multiscale_adapter.py:136,145). The tower record stores these columns.
static void adapter_clip_feature(ArpHandle* h, int64_t n, cudaStream_t st) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const float* xsrc = h->f32 ? ws.x : ws.xcls;     // class-token rows: compact after the tensor-core paths' pruned last block
  const int xtok = h->f32 ? h->tokens : 1;
  clip_head_kernel<768, 512><<<(unsigned)((n + HEAD_FR - 1) / HEAD_FR), 256, HEAD_SMEM_BYTES, st>>>(
      xsrc, xtok, h->ln_post_g, h->ln_post_b, 1e-5f, h->proj, nullptr, 0, nullptr, 0, 0.f, 0, ws.featf, h->feat_dim,
      c.layers * c.embed_dim, nullptr, nullptr, 0, (int)n);
  h->launches++;
}

// The adapter tail, from the class-token taps (ws.taps; ws.taps32 on the fp32 path) and the CLIP feature in
// ws.featf[:, Dmid:] of n rows: the intermediate GEMM, the AdapterMLP, then the gate + head. head_chunk runs it after the
// encoder, arp_label_tower after unpacking a tower record: one code path, so both give the same bits from the same values.
// Arguments as head_chunk's.
static int adapter_tail(ArpHandle* h, int64_t n, float* reward_out, int64_t ld, float* logits_out, float* feat_out,
                        cudaStream_t st) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const bool need_text = reward_out || logits_out;
  const int D = h->feat_dim, Dmid = c.layers * c.embed_dim, Din = c.layers * c.width;
  const int64_t B = c.max_batch;
  if (h->f32) {
    ARP_TRY(launch_sgemm(h, ws.taps32, Din, h->inter_w, ws.featf, D, F32_ACT_NONE, n, Dmid, Din, nullptr, nullptr, 0,
                         nullptr, 0, st));
    ARP_TRY(launch_sgemm(h, ws.featf, D, h->fc1_w, ws.hid2_32, 2 * D, F32_ACT_RELU, n, 2 * D, D, h->fc1_b, nullptr, 0,
                         nullptr, 0, st));
    ARP_TRY(launch_sgemm(h, ws.hid2_32, 2 * D, h->fc2_w, ws.mlp, D, F32_ACT_NONE, n, D, 2 * D, h->fc2_b, nullptr, 0,
                         nullptr, 0, st));
  } else {
    // image_intermediate_linear (no bias) over the 12 CLS taps -> first 6144 columns (:143-144)
    ARP_TRY(launch_gemm(h, ws.taps, B, h->inter_w, ws.featf, true, ACT_NONE, n, Dmid, Din, D, nullptr, nullptr, 0,
                        nullptr, 0, st));
    f32_to_bf16_kernel<<<kNumSMs * 4, 256, 0, st>>>(ws.featf, ws.featb, (size_t)n * D);
    h->launches++;
    // AdapterMLP: Linear -> Identity -> ReLU -> Linear (finetune_module/layers.py:42-49)
    ARP_TRY(launch_gemm(h, ws.featb, B, h->fc1_w, ws.hid2, false, ACT_RELU, n, 2 * D, D, 2 * D, h->fc1_b, nullptr, 0,
                        nullptr, 0, st));
    ARP_TRY(launch_gemm(h, ws.hid2, B, h->fc2_w, ws.mlp, true, ACT_NONE, n, D, 2 * D, D, h->fc2_b, nullptr, 0, nullptr,
                        0, st));
  }
  const bool ens = c.head == ARP_HEAD_ADAPTER_ENSEMBLE;
  adapter_head_kernel<13, 512><<<(unsigned)n, 13 * 32, 0, st>>>(
      ws.featf, ws.mlp, h->res_sigmoid, (need_text && !h->goal) ? h->text : nullptr,
      (need_text && !h->goal) ? h->n_text : 0, h->group_off, (need_text && !h->goal) ? h->n_groups : 0,
      h->logit_scale, ens ? 1 : 0, c.reduce, logits_out, h->goal ? nullptr : reward_out, ld, feat_out);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// heads. reward_out [n_groups, ld] (this chunk's column 0; ld = the call's T) / logits_out [n, n_text] /
// feat_out [n, feat_dim] may each be null.
static int head_chunk(ArpHandle* h, int64_t n, float* reward_out, int64_t ld, float* logits_out, float* feat_out,
                      cudaStream_t st) {
  const ArpConfig& c = h->cfg;
  ArpHandle::Work& ws = h->ws;
  const bool need_text = reward_out || logits_out;
  if (need_text && !h->goal && !h->text) return fail(h, ARP_ERR_STATE, "arp_set_text has not been called");
  if (h->adapter) {
    adapter_clip_feature(h, n, st);
    return adapter_tail(h, n, reward_out, ld, logits_out, feat_out, st);
  }
  const float* xsrc = h->f32 ? ws.x : ws.xcls;     // class-token rows: compact after the tensor-core paths' pruned last block
  const int xtok = h->f32 ? h->tokens : 1;
  {
    ProfScope prof(h, PC_HEAD, 2.0 * (double)n * 768 * 512, (double)n * 768 * 4 + 768.0 * 512 * 4, st);
    clip_head_kernel<768, 512><<<(unsigned)((n + HEAD_FR - 1) / HEAD_FR), 256, HEAD_SMEM_BYTES, st>>>(
        xsrc, xtok, h->ln_post_g, h->ln_post_b, 1e-5f, h->proj, (need_text && !h->goal) ? h->text : nullptr,
        h->n_text, h->group_off, h->n_groups, h->logit_scale, c.reduce, feat_out, c.embed_dim, 0, logits_out,
        h->goal ? nullptr : reward_out, ld, (int)n);
    h->launches++;
  }
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// adapter_head_kernel writes the gated, un-normalised feature when asked; normalise rows for encode_image parity
__global__ void l2_normalize_rows_kernel(float* __restrict__ f, int dim, int64_t n) {
  const int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= n) return;
  const int lane = threadIdx.x & 31;
  float* p = f + r * dim;
  float s = 0.f;
  for (int k = lane; k < dim; k += 32) s = fmaf(p[k], p[k], s);
  s = warp_sum(s);
  const float inv = 1.0f / fmaxf(sqrtf(s), 1e-12f);
  for (int k = lane; k < dim; k += 32) p[k] *= inv;
}

__global__ void episode_goal_kernel(const long long* __restrict__ ep_off, int n_eps, long long T,
                                    long long* __restrict__ frame_goal) {
  const int e = blockIdx.x;
  const long long lo = ep_off[e], hi = min(ep_off[e + 1], T);
  for (long long t = lo + threadIdx.x; t < hi; t += blockDim.x) frame_goal[t] = hi - 1;
}

// a device buffer *p of *have bytes grown to at least need (contents not kept)
static int grow(ArpHandle* h, void** p, size_t* have, size_t need) {
  if (*have >= need) return ARP_OK;
  if (*p) { cudaDeviceSynchronize(); cudaFree(*p); *p = nullptr; *have = 0; }
  ARP_CUDA(h, cudaMalloc(p, need));
  *have = need;
  return ARP_OK;
}

static int ensure_scratch(ArpHandle* h, int slot, size_t bytes) {
  return grow(h, &h->scratch[slot], &h->scratch_bytes[slot], bytes);
}

// temporaries of one label call, carved from scratch slot 0
struct LabelTmp {
  float* r = nullptr;            // [n_groups, T] rewards when the caller did not ask for them
  float* g = nullptr;            // [n_groups, T] return-to-go, likewise
  long long* frame_goal = nullptr;  // [T] goal-conditioned heads: index of the episode's last frame
  float* feats = nullptr;        // [T, feat_dim] goal-conditioned heads
};

// with_feats = false: the caller provides the goal heads' features itself (t->feats stays null)
static int carve_label_tmp(ArpHandle* h, int64_t T, LabelTmp* t, bool with_feats = true) {
  auto al = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
  const size_t b_r = al((size_t)h->n_groups * T * 4), b_goal = h->goal ? al((size_t)T * 8) : 0;
  const size_t b_feat = h->goal && with_feats ? al((size_t)T * h->feat_dim * 4) : 0;
  ARP_TRY(ensure_scratch(h, 0, 2 * b_r + b_goal + b_feat + 256));
  uint8_t* p = reinterpret_cast<uint8_t*>(h->scratch[0]);
  t->r = reinterpret_cast<float*>(p); p += b_r;
  t->g = reinterpret_cast<float*>(p); p += b_r;
  if (h->goal) {
    t->frame_goal = reinterpret_cast<long long*>(p); p += b_goal;
    if (with_feats) t->feats = reinterpret_cast<float*>(p);
  }
  return ARP_OK;
}

static int check_ready(ArpHandle* h, const void* ob, int64_t T, int64_t stride, cudaStream_t st) {
  if (!h) return ARP_ERR_INVALID;
  if (T < 0 || (T > 0 && !ob)) return fail(h, ARP_ERR_INVALID, "bad frame buffer / T");
  if (T > 0 && stride < (int64_t)h->cfg.in_h * h->cfg.in_w * 3) return fail(h, ARP_ERR_INVALID, "row stride %lld smaller than one frame", (long long)stride);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return finalize_weights(h, st);
}

// ------------------------------------------------------------------------------------------------
// C ABI: hot path
// ------------------------------------------------------------------------------------------------
extern "C" int arp_compute_reward(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes,
                                  float* reward_dev, float* logits_dev, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_TRY(check_ready(h, ob_dev, T, row_stride_bytes, st));
  if (h->goal) return fail(h, ARP_ERR_INVALID, "goal-conditioned heads need episode boundaries: use arp_label");
  const int64_t B = h->cfg.max_batch;
  for (int64_t t0 = 0; t0 < T; t0 += B) {
    const int64_t n = std::min(B, T - t0);
    ARP_TRY(encode_chunk(h, ob_dev + t0 * row_stride_bytes, n, row_stride_bytes, st));
    ARP_TRY(head_chunk(h, n, reward_dev ? reward_dev + t0 : nullptr, T,
                       logits_dev ? logits_dev + t0 * h->n_text : nullptr, nullptr, st));
  }
  return ARP_OK;
}

extern "C" int arp_encode_image(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes,
                                float* feat_dev, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_TRY(check_ready(h, ob_dev, T, row_stride_bytes, st));
  if (!feat_dev) return fail(h, ARP_ERR_INVALID, "null output");
  const int64_t B = h->cfg.max_batch;
  for (int64_t t0 = 0; t0 < T; t0 += B) {
    const int64_t n = std::min(B, T - t0);
    ARP_TRY(encode_chunk(h, ob_dev + t0 * row_stride_bytes, n, row_stride_bytes, st));
    ARP_TRY(head_chunk(h, n, nullptr, 0, nullptr, feat_dev + t0 * h->feat_dim, st));
  }
  if (h->adapter && T > 0) {
    l2_normalize_rows_kernel<<<(unsigned)((T + 7) / 8), 256, 0, st>>>(feat_dev, h->feat_dim, T);
    h->launches++;
    ARP_CUDA(h, cudaGetLastError());
  }
  return ARP_OK;
}

extern "C" int arp_encode_taps_chw(ArpHandle* h, const float* chw_dev, int64_t T, float* taps_dev, float* feat_dev,
                                   void* stream) {
  if (!h || !chw_dev || (!taps_dev && !feat_dev) || T < 0) return fail(h, ARP_ERR_INVALID, "null argument");
  if (h->adapter) return fail(h, ARP_ERR_INVALID, "arp_encode_taps_chw serves the frozen CLIP tower: use a clip head");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  ARP_TRY(finalize_weights(h, st));
  const int64_t B = h->cfg.max_batch;
  const size_t img = (size_t)3 * DEC_OUT * DEC_OUT, tw = (size_t)h->cfg.layers * h->cfg.width;
  for (int64_t t0 = 0; t0 < T; t0 += B) {
    const int64_t n = std::min(B, T - t0);
    ARP_TRY(encode_chunk(h, nullptr, n, 0, st, chw_dev + t0 * img, taps_dev ? taps_dev + t0 * tw : nullptr));
    if (feat_dev) ARP_TRY(head_chunk(h, n, nullptr, 0, nullptr, feat_dev + t0 * h->feat_dim, st));
  }
  return ARP_OK;
}

// n_groups reward rows [n_groups, T] over the same episodes -> rtg [n_groups, T], rs / gs [n_groups, T, F]
static int scan_launch(ArpHandle* h, const float* reward, int64_t T, const int64_t* ep_off, int n_eps, int F,
                       float gamma, float* rtg, float* rs, float* gs, cudaStream_t st, int n_groups = 1) {
  if (n_eps <= 0 || T <= 0) return ARP_OK;
  if (F < 1 || F > 64) return fail(h, ARP_ERR_INVALID, "num_frames must be in [1,64]");
  if (gs && !rtg) return fail(h, ARP_ERR_INVALID, "rtg_stacked needs an rtg buffer");
  ProfScope prof(h, PC_SCAN, 0.0, (double)n_groups * T * (4 + 4 + 2.0 * F * 4), st);
  rtg_scan_stack_kernel<<<dim3(n_eps, n_groups), SCAN_THREADS, 0, st>>>(
      reward, reinterpret_cast<const long long*>(ep_off), T, F, gamma, rtg, rs, gs);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

extern "C" int arp_scan_only(ArpHandle* h, const float* reward_dev, int64_t T, const int64_t* ep_offsets_dev,
                             int32_t n_eps, int32_t num_frames, float gamma, float* rtg_dev,
                             float* reward_stacked_dev, float* rtg_stacked_dev, void* stream) {
  if (!h || !reward_dev || !ep_offsets_dev) return fail(h, ARP_ERR_INVALID, "null argument");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return scan_launch(h, reward_dev, T, ep_offsets_dev, n_eps, num_frames, gamma, rtg_dev, reward_stacked_dev,
                     rtg_stacked_dev, static_cast<cudaStream_t>(stream));
}

static int label_device(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t stride, const int64_t* ep_off,
                        int n_eps, int F, float* reward, float* rtg, float* rs, float* gs, cudaStream_t st);

extern "C" int arp_label(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes,
                         const int64_t* ep_offsets_dev, int32_t n_eps, int32_t num_frames, float* reward_dev,
                         float* rtg_dev, float* reward_stacked_dev, float* rtg_stacked_dev, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_TRY(check_ready(h, ob_dev, T, row_stride_bytes, st));
  if (!ep_offsets_dev || n_eps < 0) return fail(h, ARP_ERR_INVALID, "bad episode offsets");
  return label_device(h, ob_dev, T, row_stride_bytes, ep_offsets_dev, n_eps, num_frames, reward_dev, rtg_dev,
                      reward_stacked_dev, rtg_stacked_dev, st);
}

// goal heads: rewards from feature distances to the episode's last frame (label_reward.py:159-162, :192-195)
static int goal_rewards(ArpHandle* h, const LabelTmp& tmp, int64_t T, const int64_t* ep_off, int n_eps, float* r,
                        cudaStream_t st) {
  if (h->adapter) {
    l2_normalize_rows_kernel<<<(unsigned)((T + 7) / 8), 256, 0, st>>>(tmp.feats, h->feat_dim, T);
    h->launches++;
  }
  ARP_CUDA(h, cudaMemsetAsync(tmp.frame_goal, 0, (size_t)T * 8, st));
  if (n_eps > 0) {
    episode_goal_kernel<<<n_eps, 128, 0, st>>>(reinterpret_cast<const long long*>(ep_off), n_eps, T, tmp.frame_goal);
    h->launches++;
  }
  goal_distance_kernel<<<(unsigned)((T + 7) / 8), 256, 0, st>>>(tmp.feats, h->feat_dim, tmp.frame_goal, T,
                                                               h->cfg.head == ARP_HEAD_CLIP_GOAL ? -1.f : 1.f, r);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

static int label_device(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t stride, const int64_t* ep_off,
                        int n_eps, int F, float* reward, float* rtg, float* rs, float* gs, cudaStream_t st) {
  if (T == 0) return ARP_OK;
  LabelTmp tmp;
  ARP_TRY(carve_label_tmp(h, T, &tmp));
  float* r = reward ? reward : tmp.r;
  float* g = rtg ? rtg : tmp.g;
  const int64_t B = h->cfg.max_batch;
  for (int64_t t0 = 0; t0 < T; t0 += B) {
    const int64_t n = std::min(B, T - t0);
    ARP_TRY(encode_chunk(h, ob_dev + t0 * stride, n, stride, st));
    if (!h->goal) ARP_TRY(head_chunk(h, n, r + t0, T, nullptr, nullptr, st));
    else ARP_TRY(head_chunk(h, n, nullptr, 0, nullptr, tmp.feats + t0 * h->feat_dim, st));
  }
  if (h->goal) ARP_TRY(goal_rewards(h, tmp, T, ep_off, n_eps, r, st));
  return scan_launch(h, r, T, ep_off, n_eps, F, 1.0f, g, rs, gs, st, h->n_groups);
}

// two device staging buffers of max_batch frames each (host-buffer entry points)
static int ensure_stage(ArpHandle* h) {
  const size_t need = (size_t)h->cfg.in_h * h->cfg.in_w * 3 * h->cfg.max_batch;
  if (h->stage_bytes >= need) return ARP_OK;
  for (int i = 0; i < 2; ++i) {
    if (h->stage_dev[i]) cudaFree(h->stage_dev[i]);
    h->stage_dev[i] = nullptr;
    ARP_CUDA(h, cudaMalloc((void**)&h->stage_dev[i], need));
  }
  h->stage_bytes = need;
  return ARP_OK;
}

// ---- host staging (arp_label_host on pageable memory) -------------------------------------------------------------
// The drop-in hands the library a pointer into a memory-mapped dataset (label_reward.py:268 `g[img_key][traj, -1]`): the
// rows are pageable, file-backed, and only the last stacked frame of each row is wanted. cudaMemcpy from such memory is
// a synchronous driver-side bounce copy; instead a few worker threads gather sub-chunks of frames (page faults and all)
// into a ring of pinned slots while the main thread turns finished slots into asynchronous H2D copies, so that disk /
// page-cache reads, PCIe and the GPU all run concurrently and one call can cover a whole shard.
constexpr int STG_SLOTS = 8;       // pinned ring depth
constexpr int STG_SUB = 64;        // frames per slot (12.6 MB at 256x256x3)
constexpr int STG_WORKERS = 4;

static bool host_ptr_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;   // pageable memory reports cudaMemoryTypeUnregistered
}

// row_bytes: the ring's row pitch (a frame, or the largest compressed chunk of a zfile call)
static int ensure_pinned_ring(ArpHandle* h, size_t row_bytes) {
  const size_t need = row_bytes * STG_SUB * STG_SLOTS;
  if (h->pin_bytes >= need) return ARP_OK;
  if (h->pin_ring) { cudaFreeHost(h->pin_ring); h->pin_ring = nullptr; h->pin_bytes = 0; }
  ARP_CUDA(h, cudaHostAlloc((void**)&h->pin_ring, need, cudaHostAllocDefault));
  h->pin_bytes = need;
  for (int i = 0; i < STG_SLOTS; ++i)
    if (!h->ev_slot[i]) ARP_CUDA(h, cudaEventCreateWithFlags(&h->ev_slot[i], cudaEventDisableTiming));
  return ARP_OK;
}

struct SubChunk { int64_t t0; int n; };   // rows [t0, t0+n) of the call, never straddling a device chunk

// gathers sub-chunk after sub-chunk into the pinned ring; the main thread consumes them in order
// pread() exactly n bytes at off; 0, errno, or -1 at end of file
static int pread_full(int fd, uint8_t* dst, size_t n, int64_t off) {
  size_t got = 0;
  while (got < n) {
    const ssize_t r = pread(fd, dst + got, n - got, (off_t)(off + (int64_t)got));
    if (r <= 0) return r == 0 ? -1 : errno;
    got += (size_t)r;
  }
  return 0;
}

// compressed rows of a zfile call: row t is the zlib stream of bytes[t] bytes at file offset off[t]; pos[t] is its byte
// offset in its device chunk's packed buffer
struct ZRows { const int64_t* off; const int64_t* bytes; std::vector<int64_t> pos; int64_t row_bytes; int64_t max_chunk; };

struct HostStager {
  const uint8_t* src; int64_t stride; size_t frame_bytes; uint8_t* ring; cudaEvent_t* ev_slot; int device;
  int fd = -1; int64_t fd_base = 0;          // fd >= 0: rows are pread() from a file (no page-table traffic) instead of src
  const ZRows* z = nullptr;                  // compressed rows: a slot holds its rows' chunks packed, pitch frame_bytes
  std::atomic<int> io_error{0};
  const std::vector<SubChunk>* subs;
  std::atomic<int64_t> next{0}, issued{0};   // next task to start | sub-chunks whose H2D has been enqueued
  std::atomic<bool> abort{false};
  std::mutex mu; std::condition_variable cv;
  std::vector<char> done;
  std::vector<std::thread> threads;

  void run() {
    cudaSetDevice(device);
    const int64_t n = (int64_t)subs->size();
    for (;;) {
      const int64_t j = next.fetch_add(1);
      if (j >= n || abort.load()) return;
      const int slot = (int)(j % STG_SLOTS);
      if (j >= STG_SLOTS) {                      // the slot's previous tenant must have left for the device
        while (issued.load(std::memory_order_acquire) < j - STG_SLOTS + 1) {
          if (abort.load()) return;
          std::this_thread::yield();
        }
        cudaEventSynchronize(ev_slot[slot]);
      }
      const SubChunk& sc = (*subs)[j];
      uint8_t* dst = ring + (size_t)slot * STG_SUB * frame_bytes;
      if (z) {
        for (int f = 0; f < sc.n && !io_error.load(); ++f) {
          const int64_t t = sc.t0 + f;
          if (const int e = pread_full(fd, dst + (z->pos[t] - z->pos[sc.t0]), (size_t)z->bytes[t], z->off[t])) io_error.store(e);
        }
      } else if (fd < 0) {
        for (int f = 0; f < sc.n; ++f) memcpy(dst + (size_t)f * frame_bytes, src + (sc.t0 + f) * stride, frame_bytes);
      } else {
        for (int f = 0; f < sc.n && !io_error.load(); ++f)
          if (const int e = pread_full(fd, dst + (size_t)f * frame_bytes, frame_bytes, fd_base + (sc.t0 + f) * stride))
            io_error.store(e);
      }
      { std::lock_guard<std::mutex> lk(mu); done[j] = 1; }
      cv.notify_all();
    }
  }
  void start() {
    done.assign(subs->size(), 0);
    int want = STG_WORKERS;
    if (const char* e = getenv("ARP_STAGER_THREADS")) want = std::max(1, std::min(STG_SLOTS, atoi(e)));
    const int nw = (int)std::min<size_t>(want, subs->size());
    for (int i = 0; i < nw; ++i) threads.emplace_back([this] { run(); });
  }
  double waited_s = 0.0;       // time the consumer spent waiting for the workers (ARP_STAGER_DEBUG prints it)
  void wait(int64_t j) {
    std::unique_lock<std::mutex> lk(mu);
    if (done[j]) return;
    const auto t0 = std::chrono::steady_clock::now();
    cv.wait(lk, [&] { return done[j] != 0; });
    waited_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }
  void stop() { abort.store(true); for (auto& t : threads) t.join(); threads.clear(); }
};

// ---- compressed rows (arp_*_zfile) --------------------------------------------------------------------------------
struct ZDev { int64_t* pos = nullptr; int64_t* bytes = nullptr; int* status = nullptr; };   // [T] each, device

static int launch_inflate(ArpHandle* h, const uint8_t* src, const int64_t* off, const int64_t* bytes, int64_t n,
                          int64_t row_bytes, uint8_t* out, int* status, cudaStream_t st) {
  if (n <= 0) return ARP_OK;
  ProfScope prof(h, PC_DECODE, 0.0, (double)n * row_bytes * 2, st);
  arp_inflate::inflate_rows_kernel<<<(unsigned)((n + arp_inflate::INF_WARPS - 1) / arp_inflate::INF_WARPS),
                                     arp_inflate::INF_WARPS * 32, 0, st>>>(src, off, bytes, (int)n, row_bytes, out, status);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// packs each max_batch chunk's compressed rows back to back (z->pos), sizes the device buffers from the call's largest
// chunk, and uploads the per-row tables
static int prepare_zrows(ArpHandle* h, ZRows* z, int64_t T, int64_t B, ZDev* zd, cudaStream_t st) {
  z->pos.assign((size_t)T, 0);
  size_t zsrc = 1;
  z->max_chunk = 1;
  for (int64_t t0 = 0; t0 < T; t0 += B) {
    int64_t p = 0;
    for (int64_t t = t0; t < std::min(T, t0 + B); ++t) {
      z->pos[t] = p;
      p += z->bytes[t];
      z->max_chunk = std::max(z->max_chunk, z->bytes[t]);
    }
    zsrc = std::max(zsrc, (size_t)p);
  }
  if (h->zsrc_bytes < zsrc) {
    for (int i = 0; i < 2; ++i) {
      size_t have = h->zsrc_bytes;
      ARP_TRY(grow(h, reinterpret_cast<void**>(&h->zsrc_dev[i]), &have, zsrc));
    }
    h->zsrc_bytes = zsrc;
  }
  ARP_TRY(grow(h, reinterpret_cast<void**>(&h->zrows_dev), &h->zrows_bytes, (size_t)std::min(B, T) * z->row_bytes));
  ARP_TRY(grow(h, &h->ztab_dev, &h->ztab_bytes, (size_t)T * 20));
  zd->pos = reinterpret_cast<int64_t*>(h->ztab_dev);
  zd->bytes = zd->pos + T;
  zd->status = reinterpret_cast<int*>(zd->bytes + T);
  ARP_CUDA(h, cudaMemcpyAsync(zd->pos, z->pos.data(), (size_t)T * 8, cudaMemcpyHostToDevice, st));
  ARP_CUDA(h, cudaMemcpyAsync(zd->bytes, z->bytes, (size_t)T * 8, cudaMemcpyHostToDevice, st));
  return ARP_OK;
}

static const char* inflate_status_name(int s) {
  switch (s) {
    case ARP_INFLATE_TRUNCATED: return "truncated stream";
    case ARP_INFLATE_BAD_HEADER: return "bad zlib header";
    case ARP_INFLATE_BAD_BLOCK: return "bad block type or stored length";
    case ARP_INFLATE_BAD_CODE: return "bad Huffman code";
    case ARP_INFLATE_DISTANCE_TOO_FAR: return "distance before the start of the row";
    case ARP_INFLATE_TOO_LONG: return "output longer than row_bytes";
    case ARP_INFLATE_TOO_SHORT: return "output shorter than row_bytes";
    case ARP_INFLATE_BAD_ADLER: return "Adler-32 mismatch";
    default: return "unknown status";
  }
}

// ARP_ERR_INVALID naming the first row that did not inflate
static int check_zrows(ArpHandle* h, const ZRows& z, const ZDev& zd, int64_t T, cudaStream_t st) {
  std::vector<int> status((size_t)T);
  ARP_CUDA(h, cudaMemcpyAsync(status.data(), zd.status, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
  ARP_CUDA(h, cudaStreamSynchronize(st));
  for (int64_t t = 0; t < T; ++t)
    if (status[t] != ARP_INFLATE_OK)
      return fail(h, ARP_ERR_INVALID, "row %lld of the call (chunk at file offset %lld, %lld bytes) does not inflate to "
                  "%lld bytes: %s (ArpInflateStatus %d)", (long long)t, (long long)z.off[t], (long long)z.bytes[t],
                  (long long)z.row_bytes, inflate_status_name(status[t]), status[t]);
  return ARP_OK;
}

// the checks the zfile entry points share; row_bytes must be F whole frames, F in [1, 64]
static int check_row_bytes(ArpHandle* h, int64_t row_bytes) {
  const int64_t frame = (int64_t)h->cfg.in_h * h->cfg.in_w * 3;
  if (row_bytes <= 0 || row_bytes % frame != 0 || row_bytes / frame > 64)
    return fail(h, ARP_ERR_INVALID, "row_bytes %lld is not F * %lld with F in [1, 64]", (long long)row_bytes, (long long)frame);
  return ARP_OK;
}

static int check_zargs(ArpHandle* h, int32_t fd, const int64_t* off, const int64_t* bytes, int64_t T, int64_t row_bytes) {
  if (!h) return ARP_ERR_INVALID;
  if (fd < 0) return fail(h, ARP_ERR_INVALID, "bad file descriptor");
  if (T < 0) return fail(h, ARP_ERR_INVALID, "bad T");
  if (T > 0 && (!off || !bytes)) return fail(h, ARP_ERR_INVALID, "null chunk table");
  ARP_TRY(check_row_bytes(h, row_bytes));
  for (int64_t t = 0; t < T; ++t)
    if (off[t] < 0 || bytes[t] < 0)
      return fail(h, ARP_ERR_INVALID, "row %lld: negative chunk offset or size", (long long)t);
  return ARP_OK;
}

// arp_embed_tower_*: the adapter head stopped after the CLIP feature; the chunk's taps and feature become n tower records
static int tower_chunk(ArpHandle* h, int64_t n, float* rec, cudaStream_t st) {
  ArpHandle::Work& ws = h->ws;
  adapter_clip_feature(h, n, st);
  const int Dmid = h->cfg.layers * h->cfg.embed_dim;
  ProfScope prof(h, PC_OTHER, 0.0, (double)n * (TOWER_TAPS * (h->f32 ? 4 : 2) + TOWER_FEAT * 4 + TOWER_DIM * 4), st);
  if (h->f32)
    tower_pack_kernel<float><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ws.taps32, ws.featf, h->feat_dim, Dmid, rec, (int)n);
  else
    tower_pack_kernel<bf16><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ws.taps, ws.featf, h->feat_dim, Dmid, rec, (int)n);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

// emb_host != nullptr: embed mode (arp_embed_host / arp_embed_file) — the same staging and encoder pass, the head writes
// the per-frame embedding [T, feat_dim] (head_chunk's feat_out) to the device, and it is copied to emb_host once at the
// end; there is no reward, no scan, and the episode / output arguments are ignored. tower (adapter heads,
// arp_embed_tower_*): the head stops after the CLIP feature and the rows are tower records [T, TOWER_DIM] instead.
static int label_host_impl(ArpHandle* h, const uint8_t* ob_host, int fd, int64_t fd_offset, int64_t T,
                           int64_t row_stride_bytes, const int64_t* ep_offsets_host, int32_t n_eps, int32_t num_frames,
                           float* reward_host, float* rtg_host, float* reward_stacked_host, float* rtg_stacked_host,
                           float* emb_host = nullptr, bool tower = false, ZRows* z = nullptr) {
  if (!h) return ARP_ERR_INVALID;
  cudaStream_t st = h->own_stream;
  const bool embed = emb_host != nullptr;
  const int64_t ew = tower ? TOWER_DIM : h->feat_dim;   // embed mode: floats per row
  if (fd >= 0 && fd_offset < 0) return fail(h, ARP_ERR_INVALID, "bad file offset");
  ARP_TRY(check_ready(h, fd >= 0 ? reinterpret_cast<const uint8_t*>(h) : ob_host, T, row_stride_bytes, st));
  if (!embed && (!ep_offsets_host || n_eps < 0)) return fail(h, ARP_ERR_INVALID, "bad episode offsets");
  if (!embed && (num_frames < 1 || num_frames > 64)) return fail(h, ARP_ERR_INVALID, "num_frames must be in [1,64]");
  if (T == 0) return ARP_OK;
  const ArpConfig& c = h->cfg;
  const size_t frame_bytes = (size_t)c.in_h * c.in_w * 3;
  const int64_t B = c.max_batch;
  const int F = embed ? 1 : num_frames;
  ARP_TRY(ensure_stage(h));
  ZDev zd;
  if (z) ARP_TRY(prepare_zrows(h, z, T, B, &zd, st));
  // device outputs (scratch slot 1), G = n_groups:
  // [ep_off (n_eps+1) i64][reward G*T][rtg G*T][reward_stacked G*T*F][rtg_stacked G*T*F]; embed mode: [emb T*ew]
  const size_t G = (size_t)h->n_groups;
  const size_t off_bytes = embed ? 0 : (((size_t)(n_eps + 1) * 8) + 255) & ~(size_t)255;
  const size_t out_bytes = embed ? (size_t)T * ew * 4 : G * T * 4 * (2 + 2 * F);
  ARP_TRY(ensure_scratch(h, 1, off_bytes + out_bytes + 1024));
  LabelTmp tmp;
  if (!embed) ARP_TRY(carve_label_tmp(h, T, &tmp));
  int64_t* d_off = reinterpret_cast<int64_t*>(h->scratch[1]);
  float* d_r = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(h->scratch[1]) + off_bytes);
  float* d_g = d_r + G * T;
  float* d_rs = d_g + G * T;
  float* d_gs = d_rs + G * T * F;
  float* d_emb = d_r;
  if (!embed)
    ARP_CUDA(h, cudaMemcpyAsync(d_off, ep_offsets_host, (size_t)(n_eps + 1) * 8, cudaMemcpyHostToDevice, st));
  const int64_t nchunks = (T + B - 1) / B;
  // pinned (or registered) caller memory goes to the device directly, one strided 2-D copy per chunk; pageable memory is
  // gathered through the pinned ring by worker threads
  const bool staged = fd >= 0 || !host_ptr_is_pinned(ob_host);
  const size_t pitch = z ? (size_t)z->max_chunk : frame_bytes;   // pinned ring: bytes per row of a slot
  std::vector<SubChunk> subs;
  HostStager stager;
  if (staged) {
    ARP_TRY(ensure_pinned_ring(h, pitch));
    for (int64_t ci = 0; ci < nchunks; ++ci) {
      const int64_t t0 = ci * B, n = std::min(B, T - t0);
      for (int64_t s0 = 0; s0 < n; s0 += STG_SUB) subs.push_back(SubChunk{t0 + s0, (int)std::min<int64_t>(STG_SUB, n - s0)});
    }
    stager.src = ob_host; stager.stride = row_stride_bytes; stager.frame_bytes = pitch; stager.ring = h->pin_ring;
    stager.ev_slot = h->ev_slot; stager.device = c.device; stager.subs = &subs;
    stager.fd = fd; stager.fd_base = fd_offset; stager.z = z;
    stager.start();
  }
  // double-buffered: chunk i+1's frames (only the scored image of each row) cross PCIe while chunk i is encoded
  int rc = ARP_OK;
  int64_t sub_j = 0;
  for (int64_t ci = 0; ci < nchunks && rc == ARP_OK; ++ci) {
    const int buf = (int)(ci & 1);
    const int64_t t0 = ci * B, n = std::min(B, T - t0);
    if (ci >= 2) cudaStreamWaitEvent(h->copy_stream, h->ev_consumed[buf], 0);
    cudaError_t e = cudaSuccess;
    if (!staged) {
      e = cudaMemcpy2DAsync(h->stage_dev[buf], frame_bytes, ob_host + t0 * row_stride_bytes, (size_t)row_stride_bytes,
                            frame_bytes, (size_t)n, cudaMemcpyHostToDevice, h->copy_stream);
    } else {
      for (int64_t s0 = 0; s0 < n && e == cudaSuccess; s0 += STG_SUB, ++sub_j) {
        stager.wait(sub_j);
        const int slot = (int)(sub_j % STG_SLOTS);
        const uint8_t* ring_slot = h->pin_ring + (size_t)slot * STG_SUB * pitch;
        if (z) {   // the sub-chunk's compressed rows, packed, to their place in the chunk's packed buffer
          const int64_t a = t0 + s0, b = a + subs[sub_j].n - 1;
          e = cudaMemcpyAsync(h->zsrc_dev[buf] + z->pos[a], ring_slot, (size_t)(z->pos[b] + z->bytes[b] - z->pos[a]),
                              cudaMemcpyHostToDevice, h->copy_stream);
        } else {
          e = cudaMemcpyAsync(h->stage_dev[buf] + (size_t)s0 * frame_bytes, ring_slot, (size_t)subs[sub_j].n * frame_bytes,
                              cudaMemcpyHostToDevice, h->copy_stream);
        }
        if (e == cudaSuccess) e = cudaEventRecord(h->ev_slot[slot], h->copy_stream);
        stager.issued.store(sub_j + 1, std::memory_order_release);
      }
    }
    if (e != cudaSuccess) { rc = fail(h, ARP_ERR_CUDA, "H2D frames failed: %s", cudaGetErrorString(e)); break; }
    cudaEventRecord(h->ev_copied[buf], h->copy_stream);
    cudaStreamWaitEvent(st, h->ev_copied[buf], 0);
    if (z) {   // whole rows inflated into zrows_dev; the encoder reads each row's last frame with stride row_bytes
      if ((rc = launch_inflate(h, h->zsrc_dev[buf], zd.pos + t0, zd.bytes + t0, n, z->row_bytes, h->zrows_dev,
                               zd.status + t0, st)) != ARP_OK)
        break;
      rc = encode_chunk(h, h->zrows_dev + (z->row_bytes - (int64_t)frame_bytes), n, z->row_bytes, st);
    } else {
      rc = encode_chunk(h, h->stage_dev[buf], n, (int64_t)frame_bytes, st);
    }
    if (rc != ARP_OK) break;
    if (tower) rc = tower_chunk(h, n, d_emb + t0 * ew, st);
    else if (embed) rc = head_chunk(h, n, nullptr, 0, nullptr, d_emb + t0 * ew, st);
    else if (!h->goal) rc = head_chunk(h, n, d_r + t0, T, nullptr, nullptr, st);
    else rc = head_chunk(h, n, nullptr, 0, nullptr, tmp.feats + t0 * h->feat_dim, st);
    cudaEventRecord(h->ev_consumed[buf], st);
  }
  if (staged) {
    stager.stop();
    if (rc == ARP_OK && stager.io_error.load())
      rc = fail(h, ARP_ERR_INVALID, "reading frames from the file failed (%s)",
                stager.io_error.load() < 0 ? "unexpected end of file" : strerror(stager.io_error.load()));
    if (getenv("ARP_STAGER_DEBUG"))
      fprintf(stderr, "arp_label_host: %lld frames staged in %zu sub-chunks, consumer waited %.3f s for the gather threads\n",
              (long long)T, subs.size(), stager.waited_s);
  }
  if (rc == ARP_OK && z) rc = check_zrows(h, *z, zd, T, st);
  if (rc == ARP_OK && embed) {
    cudaError_t e = cudaMemcpyAsync(emb_host, d_emb, (size_t)T * ew * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = fail(h, ARP_ERR_CUDA, "embedding D2H failed: %s", cudaGetErrorString(e));
  }
  if (embed) {
    // the [T, ew] device result (1.9 GB for an adapter head at 73 k frames, 2.8 GB of tower records) is not kept by the
    // handle between calls
    cudaStreamSynchronize(h->copy_stream);
    cudaStreamSynchronize(st);
    cudaFree(h->scratch[1]);
    h->scratch[1] = nullptr;
    h->scratch_bytes[1] = 0;
  }
  if (rc == ARP_OK && !embed && h->goal) rc = goal_rewards(h, tmp, T, d_off, n_eps, d_r, st);
  if (rc == ARP_OK && !embed) rc = scan_launch(h, d_r, T, d_off, n_eps, F, 1.0f, d_g, d_rs, d_gs, st, h->n_groups);
  if (rc == ARP_OK && !embed) {
    cudaError_t e = cudaSuccess;
    const size_t b1 = G * T * 4, bF = G * T * F * 4;   // group-major: one contiguous block per output
    if (reward_host && e == cudaSuccess) e = cudaMemcpyAsync(reward_host, d_r, b1, cudaMemcpyDeviceToHost, st);
    if (rtg_host && e == cudaSuccess) e = cudaMemcpyAsync(rtg_host, d_g, b1, cudaMemcpyDeviceToHost, st);
    if (reward_stacked_host && e == cudaSuccess) e = cudaMemcpyAsync(reward_stacked_host, d_rs, bF, cudaMemcpyDeviceToHost, st);
    if (rtg_stacked_host && e == cudaSuccess) e = cudaMemcpyAsync(rtg_stacked_host, d_gs, bF, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = fail(h, ARP_ERR_CUDA, "label_host tail failed: %s", cudaGetErrorString(e));
  }
  if (rc != ARP_OK) cudaDeviceSynchronize();   // error path: drain the device before the caller frees anything
  cudaStreamSynchronize(h->copy_stream);
  cudaStreamSynchronize(st);
  return rc;
}

extern "C" int arp_label_host(ArpHandle* h, const uint8_t* ob_host, int64_t T, int64_t row_stride_bytes,
                              const int64_t* ep_offsets_host, int32_t n_eps, int32_t num_frames, float* reward_host,
                              float* rtg_host, float* reward_stacked_host, float* rtg_stacked_host) {
  return label_host_impl(h, ob_host, -1, 0, T, row_stride_bytes, ep_offsets_host, n_eps, num_frames, reward_host, rtg_host,
                         reward_stacked_host, rtg_stacked_host);
}

extern "C" int arp_label_file(ArpHandle* h, int32_t fd, int64_t file_offset, int64_t T, int64_t row_stride_bytes,
                              const int64_t* ep_offsets_host, int32_t n_eps, int32_t num_frames, float* reward_host,
                              float* rtg_host, float* reward_stacked_host, float* rtg_stacked_host) {
  if (fd < 0) return fail(h, ARP_ERR_INVALID, "bad file descriptor");
  return label_host_impl(h, nullptr, fd, file_offset, T, row_stride_bytes, ep_offsets_host, n_eps, num_frames, reward_host,
                         rtg_host, reward_stacked_host, rtg_stacked_host);
}

// ------------------------------------------------------------------------------------------------
// C ABI: stored embeddings (relabeling without frames)
// ------------------------------------------------------------------------------------------------
extern "C" int arp_embedding_dim(const ArpHandle* h) { return h ? h->feat_dim : 0; }

extern "C" int arp_embed_host(ArpHandle* h, const uint8_t* ob_host, int64_t T, int64_t row_stride_bytes, float* emb_host) {
  if (!h || T < 0 || (T > 0 && !emb_host)) return fail(h, ARP_ERR_INVALID, "null argument / bad T");
  if (T == 0) return check_ready(h, ob_host, T, row_stride_bytes, h->own_stream);
  return label_host_impl(h, ob_host, -1, 0, T, row_stride_bytes, nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr,
                         emb_host);
}

extern "C" int arp_embed_file(ArpHandle* h, int32_t fd, int64_t file_offset, int64_t T, int64_t row_stride_bytes,
                              float* emb_host) {
  if (fd < 0) return fail(h, ARP_ERR_INVALID, "bad file descriptor");
  if (!h || T < 0 || (T > 0 && !emb_host)) return fail(h, ARP_ERR_INVALID, "null argument / bad T");
  if (T == 0) return check_ready(h, reinterpret_cast<const uint8_t*>(h), T, row_stride_bytes, h->own_stream);
  return label_host_impl(h, nullptr, fd, file_offset, T, row_stride_bytes, nullptr, 0, 0, nullptr, nullptr, nullptr,
                         nullptr, emb_host);
}

// The instruction side of arp_label on stored embeddings: no image-side weight is read (finalize_weights is not called,
// so a handle that never received them works). Text heads: one head launch + one scan launch for any T and G.
extern "C" int arp_label_embeddings(ArpHandle* h, const float* emb_dev, int64_t T, const int64_t* ep_offsets_dev,
                                    int32_t n_eps, int32_t num_frames, float* reward_dev, float* rtg_dev,
                                    float* reward_stacked_dev, float* rtg_stacked_dev, void* stream) {
  if (!h) return ARP_ERR_INVALID;
  if (T < 0 || (T > 0 && !emb_dev)) return fail(h, ARP_ERR_INVALID, "bad embedding buffer / T");
  if (!ep_offsets_dev || n_eps < 0) return fail(h, ARP_ERR_INVALID, "bad episode offsets");
  if (num_frames < 1 || num_frames > 64) return fail(h, ARP_ERR_INVALID, "num_frames must be in [1,64]");
  if (!h->goal && !h->text) return fail(h, ARP_ERR_STATE, "arp_set_text has not been called");
  if (T > 0x7fffffffLL) return fail(h, ARP_ERR_INVALID, "T too large");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  if (T == 0) return ARP_OK;
  LabelTmp tmp;
  // clip_goal_conditioned measures distances on the stored features themselves (goal_rewards only reads them), so no
  // feature scratch is carved for it; the adapter variant normalises a copy, as the frames path normalises
  // LabelTmp::feats in place
  ARP_TRY(carve_label_tmp(h, T, &tmp, h->adapter));
  float* r = reward_dev ? reward_dev : tmp.r;
  float* g = rtg_dev ? rtg_dev : tmp.g;
  if (h->goal) {
    if (h->adapter)
      ARP_CUDA(h, cudaMemcpyAsync(tmp.feats, emb_dev, (size_t)T * h->feat_dim * 4, cudaMemcpyDeviceToDevice, st));
    else
      tmp.feats = const_cast<float*>(emb_dev);
    ARP_TRY(goal_rewards(h, tmp, T, ep_offsets_dev, n_eps, r, st));
  } else if (h->adapter) {
    ProfScope prof(h, PC_HEAD, 2.0 * (double)T * h->n_text * h->feat_dim, (double)T * h->feat_dim * 4, st);
    adapter_head_kernel<13, 512><<<(unsigned)T, 13 * 32, 0, st>>>(
        emb_dev, nullptr, 0.f, h->text, h->n_text, h->group_off, h->n_groups, h->logit_scale,
        h->cfg.head == ARP_HEAD_ADAPTER_ENSEMBLE ? 1 : 0, h->cfg.reduce, nullptr, r, T, nullptr);
    h->launches++;
  } else {
    ProfScope prof(h, PC_HEAD, 2.0 * (double)T * h->n_text * h->feat_dim, (double)T * h->feat_dim * 4, st);
    clip_embedding_head_kernel<512><<<(unsigned)((T + HEAD_FR - 1) / HEAD_FR), 256, 0, st>>>(
        emb_dev, h->text, h->n_text, h->group_off, h->n_groups, h->logit_scale, h->cfg.reduce, nullptr, r, T, T);
    h->launches++;
  }
  ARP_CUDA(h, cudaGetLastError());
  return scan_launch(h, r, T, ep_offsets_dev, n_eps, num_frames, 1.0f, g, reward_stacked_dev, rtg_stacked_dev, st,
                     h->n_groups);
}

// ------------------------------------------------------------------------------------------------
// C ABI: CLIP tower records (relabeling with another adapter checkpoint without frames or the ViT)
// ------------------------------------------------------------------------------------------------
extern "C" int arp_tower_dim(const ArpHandle* h) { return h && h->adapter ? TOWER_DIM : 0; }

extern "C" int arp_embed_tower_host(ArpHandle* h, const uint8_t* ob_host, int64_t T, int64_t row_stride_bytes,
                                    float* rec_host) {
  if (!h || T < 0 || (T > 0 && !rec_host)) return fail(h, ARP_ERR_INVALID, "null argument / bad T");
  if (!h->adapter) return fail(h, ARP_ERR_INVALID, "tower records serve the adapter heads only");
  if (T == 0) return check_ready(h, ob_host, T, row_stride_bytes, h->own_stream);
  return label_host_impl(h, ob_host, -1, 0, T, row_stride_bytes, nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr,
                         rec_host, true);
}

extern "C" int arp_embed_tower_file(ArpHandle* h, int32_t fd, int64_t file_offset, int64_t T, int64_t row_stride_bytes,
                                    float* rec_host) {
  if (fd < 0) return fail(h, ARP_ERR_INVALID, "bad file descriptor");
  if (!h || T < 0 || (T > 0 && !rec_host)) return fail(h, ARP_ERR_INVALID, "null argument / bad T");
  if (!h->adapter) return fail(h, ARP_ERR_INVALID, "tower records serve the adapter heads only");
  if (T == 0) return check_ready(h, reinterpret_cast<const uint8_t*>(h), T, row_stride_bytes, h->own_stream);
  return label_host_impl(h, nullptr, fd, file_offset, T, row_stride_bytes, nullptr, 0, 0, nullptr, nullptr, nullptr,
                         nullptr, rec_host, true);
}

extern "C" int arp_label_zfile(ArpHandle* h, int32_t fd, const int64_t* chunk_offset_host, const int64_t* chunk_bytes_host,
                               int64_t T, int64_t row_bytes, const int64_t* ep_offsets_host, int32_t n_eps,
                               int32_t num_frames, float* reward_host, float* rtg_host, float* reward_stacked_host,
                               float* rtg_stacked_host) {
  ARP_TRY(check_zargs(h, fd, chunk_offset_host, chunk_bytes_host, T, row_bytes));
  ZRows z{chunk_offset_host, chunk_bytes_host, {}, row_bytes, 0};
  return label_host_impl(h, nullptr, fd, 0, T, row_bytes, ep_offsets_host, n_eps, num_frames, reward_host, rtg_host,
                         reward_stacked_host, rtg_stacked_host, nullptr, false, &z);
}

extern "C" int arp_embed_zfile(ArpHandle* h, int32_t fd, const int64_t* chunk_offset_host, const int64_t* chunk_bytes_host,
                               int64_t T, int64_t row_bytes, float* emb_host) {
  ARP_TRY(check_zargs(h, fd, chunk_offset_host, chunk_bytes_host, T, row_bytes));
  if (T > 0 && !emb_host) return fail(h, ARP_ERR_INVALID, "null argument");
  if (T == 0) return check_ready(h, reinterpret_cast<const uint8_t*>(h), T, row_bytes, h->own_stream);
  ZRows z{chunk_offset_host, chunk_bytes_host, {}, row_bytes, 0};
  return label_host_impl(h, nullptr, fd, 0, T, row_bytes, nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr, emb_host,
                         false, &z);
}

extern "C" int arp_embed_tower_zfile(ArpHandle* h, int32_t fd, const int64_t* chunk_offset_host,
                                     const int64_t* chunk_bytes_host, int64_t T, int64_t row_bytes, float* rec_host) {
  ARP_TRY(check_zargs(h, fd, chunk_offset_host, chunk_bytes_host, T, row_bytes));
  if (T > 0 && !rec_host) return fail(h, ARP_ERR_INVALID, "null argument");
  if (!h->adapter) return fail(h, ARP_ERR_INVALID, "tower records serve the adapter heads only");
  if (T == 0) return check_ready(h, reinterpret_cast<const uint8_t*>(h), T, row_bytes, h->own_stream);
  ZRows z{chunk_offset_host, chunk_bytes_host, {}, row_bytes, 0};
  return label_host_impl(h, nullptr, fd, 0, T, row_bytes, nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr, rec_host,
                         true, &z);
}

extern "C" int arp_inflate_rows(ArpHandle* h, const uint8_t* src_dev, const int64_t* src_off_dev,
                                const int64_t* src_bytes_dev, int64_t n, int64_t row_bytes, uint8_t* out_dev,
                                int32_t* status_dev, void* stream) {
  if (!h) return ARP_ERR_INVALID;
  if (n < 0 || n > 0x7fffffffLL) return fail(h, ARP_ERR_INVALID, "bad n");
  if (n > 0 && (!src_dev || !src_off_dev || !src_bytes_dev || !out_dev || !status_dev))
    return fail(h, ARP_ERR_INVALID, "null argument");
  ARP_TRY(check_row_bytes(h, row_bytes));
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return launch_inflate(h, src_dev, src_off_dev, src_bytes_dev, n, row_bytes, out_dev, status_dev,
                        static_cast<cudaStream_t>(stream));
}

// arp_label's outputs from tower records: per max_batch chunk one unpack launch, then adapter_tail — the launches of
// head_chunk's adapter branch after its clip_head_kernel — and one scan for the call. Reads only the image-adapter
// tensors (adapter_weights_ready, not finalize_weights), so a handle whose visual.* weights were never set works.
extern "C" int arp_label_tower(ArpHandle* h, const float* rec_dev, int64_t T, const int64_t* ep_offsets_dev,
                               int32_t n_eps, int32_t num_frames, float* reward_dev, float* rtg_dev,
                               float* reward_stacked_dev, float* rtg_stacked_dev, void* stream) {
  if (!h) return ARP_ERR_INVALID;
  if (!h->adapter) return fail(h, ARP_ERR_INVALID, "tower records serve the adapter heads only");
  if (T < 0 || (T > 0 && !rec_dev)) return fail(h, ARP_ERR_INVALID, "bad record buffer / T");
  if (reinterpret_cast<uintptr_t>(rec_dev) & 15) return fail(h, ARP_ERR_INVALID, "record buffer must be 16-byte aligned");
  if (!ep_offsets_dev || n_eps < 0) return fail(h, ARP_ERR_INVALID, "bad episode offsets");
  if (num_frames < 1 || num_frames > 64) return fail(h, ARP_ERR_INVALID, "num_frames must be in [1,64]");
  if (T > 0x7fffffffLL) return fail(h, ARP_ERR_INVALID, "T too large");
  if (!h->goal && !h->text) return fail(h, ARP_ERR_STATE, "arp_set_text has not been called");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  ARP_TRY(adapter_weights_ready(h, st));
  if (T == 0) return ARP_OK;
  LabelTmp tmp;
  ARP_TRY(carve_label_tmp(h, T, &tmp));
  float* r = reward_dev ? reward_dev : tmp.r;
  float* g = rtg_dev ? rtg_dev : tmp.g;
  ArpHandle::Work& ws = h->ws;
  const int Dmid = h->cfg.layers * h->cfg.embed_dim;
  const int64_t B = h->cfg.max_batch;
  for (int64_t t0 = 0; t0 < T; t0 += B) {
    const int64_t n = std::min(B, T - t0);
    const float* rec = rec_dev + t0 * TOWER_DIM;
    {
      ProfScope prof(h, PC_OTHER, 0.0, (double)n * (TOWER_DIM * 4 + TOWER_TAPS * (h->f32 ? 4 : 2) + TOWER_FEAT * 4), st);
      if (h->f32)
        tower_unpack_kernel<float><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(rec, ws.taps32, ws.featf, h->feat_dim, Dmid,
                                                                           (int)n);
      else
        tower_unpack_kernel<bf16><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(rec, ws.taps, ws.featf, h->feat_dim, Dmid,
                                                                          (int)n);
      h->launches++;
    }
    if (!h->goal) ARP_TRY(adapter_tail(h, n, r + t0, T, nullptr, nullptr, st));
    else ARP_TRY(adapter_tail(h, n, nullptr, 0, nullptr, tmp.feats + t0 * h->feat_dim, st));
  }
  if (h->goal) ARP_TRY(goal_rewards(h, tmp, T, ep_offsets_dev, n_eps, r, st));
  return scan_launch(h, r, T, ep_offsets_dev, n_eps, num_frames, 1.0f, g, reward_stacked_dev, rtg_stacked_dev, st,
                     h->n_groups);
}

extern "C" int arp_wants_weight(const ArpHandle* h, const char* name) {
  if (!h || !name) return 0;
  std::string key(name);
  if (key.compare(0, 11, "clip_model.") == 0) key = key.substr(11);
  return h->slots.find(key) != h->slots.end() ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
// C ABI: consumer side (ProcgenDataset.preprocess_rtgs, data_procgen.py:132-174)
// ------------------------------------------------------------------------------------------------
struct StatsDev {
  RadixSelectState sel;
  uint32_t mm[2];
  float res[8];   // [0] min [1] max | [2] rtg min [3] rtg max | [4] q_lo [5] q_hi
};

static int ensure_stats(ArpHandle* h) {
  if (h->stats_dev) return ARP_OK;
  uint8_t* p = nullptr;
  ARP_TRY(dev_alloc(h, &p, sizeof(StatsDev)));
  h->stats_dev = p;
  return ARP_OK;
}

static int launch_minmax(ArpHandle* h, const float* x, int64_t n, float* res2, cudaStream_t st) {
  StatsDev* sd = static_cast<StatsDev*>(h->stats_dev);
  const uint32_t init[2] = {0xffffffffu, 0u};
  ARP_CUDA(h, cudaMemcpyAsync(sd->mm, init, sizeof(init), cudaMemcpyHostToDevice, st));
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, kNumSMs * 8);
  minmax_f32_kernel<<<blocks, 256, 0, st>>>(x, n, sd->mm);
  minmax_finish_kernel<<<1, 1, 0, st>>>(sd->mm, res2);
  h->launches += 2;
  return ARP_OK;
}

static int launch_select(ArpHandle* h, const float* x, int64_t n, uint64_t k0, uint64_t k1, float* res2, cudaStream_t st) {
  StatsDev* sd = static_cast<StatsDev*>(h->stats_dev);
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, kNumSMs * 8);
  radix_select_init_kernel<<<1, 256, 0, st>>>(&sd->sel, k0, k1);
  h->launches++;
  for (int pass = 0; pass < 4; ++pass) {
    radix_select_hist_kernel<<<blocks, 256, 0, st>>>(x, n, &sd->sel, pass);
    radix_select_pick_kernel<<<1, 256, 0, st>>>(&sd->sel, pass, res2);
    h->launches += 2;
  }
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

extern "C" int arp_quantile_f32(ArpHandle* h, const float* x_dev, int64_t n, int64_t k_lo, int64_t k_hi,
                                float* lo_hi_host, void* stream) {
  if (!h || !x_dev || !lo_hi_host) return fail(h, ARP_ERR_INVALID, "null argument");
  if (n < 1 || k_lo < 0 || k_hi < 0 || k_lo >= n || k_hi >= n) return fail(h, ARP_ERR_INVALID, "ranks must be in [0, n)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  ARP_TRY(ensure_stats(h));
  StatsDev* sd = static_cast<StatsDev*>(h->stats_dev);
  ProfScope prof(h, PC_SCAN, 0.0, (double)n * 4 * 4, st);
  ARP_TRY(launch_select(h, x_dev, n, (uint64_t)k_lo, (uint64_t)k_hi, sd->res + 4, st));
  ARP_CUDA(h, cudaMemcpyAsync(lo_hi_host, sd->res + 4, 8, cudaMemcpyDeviceToHost, st));
  ARP_CUDA(h, cudaStreamSynchronize(st));
  return ARP_OK;
}

extern "C" int arp_preprocess_rtgs(ArpHandle* h, const float* reward_dev, int64_t T, const int64_t* ep_offsets_dev,
                                   int32_t n_eps, int32_t num_frames, int32_t use_normalize, float* shifted_dev,
                                   float* rtg_dev, float* rtg_stacked_dev, float* stats_host, void* stream) {
  if (!h || !reward_dev || !ep_offsets_dev || !rtg_dev || !rtg_stacked_dev || !stats_host)
    return fail(h, ARP_ERR_INVALID, "null argument");
  if (T < 1 || n_eps < 1) return fail(h, ARP_ERR_INVALID, "empty dataset");
  if (use_normalize && !shifted_dev) return fail(h, ARP_ERR_INVALID, "use_normalize needs a [T] scratch buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  ARP_TRY(ensure_stats(h));
  StatsDev* sd = static_cast<StatsDev*>(h->stats_dev);
  ARP_TRY(launch_minmax(h, reward_dev, T, sd->res, st));                      // data_procgen.py:147-148: over ALL rows
  const float* r = reward_dev;
  if (use_normalize) {                                                        // :150-151
    sub_scalar_f32_kernel<<<(int)std::min<int64_t>((T + 255) / 256, kNumSMs * 8), 256, 0, st>>>(reward_dev, sd->res,
                                                                                              shifted_dev, T);
    h->launches++;
    r = shifted_dev;
  }
  // :155-168 — discount_cumsum(gamma=1.0) and the deque window, identical to the labeler's scan + stack
  ARP_TRY(scan_launch(h, r, T, ep_offsets_dev, n_eps, num_frames, 1.0f, rtg_dev, nullptr, rtg_stacked_dev, st));
  // the stacked values are a gather of rtg: min / max over the labeled rows of rtg = over the stacked array (:171)
  int64_t off_last = 0;
  ARP_CUDA(h, cudaMemcpyAsync(&off_last, ep_offsets_dev + n_eps, 8, cudaMemcpyDeviceToHost, st));
  ARP_CUDA(h, cudaStreamSynchronize(st));
  const int64_t rows = std::min<int64_t>(off_last, T);
  if (rows < 1) return fail(h, ARP_ERR_INVALID, "no labeled rows");
  ARP_TRY(launch_minmax(h, rtg_dev, rows, sd->res + 2, st));
  ARP_CUDA(h, cudaMemcpyAsync(stats_host, sd->res, 16, cudaMemcpyDeviceToHost, st));
  ARP_CUDA(h, cudaStreamSynchronize(st));
  return ARP_OK;
}

// Latency mode (envs/vl_reward.py: one frame per environment step). The whole kernel sequence for n frames is
// captured once into a CUDA graph (~100 launches become one submission); per call: H2D of the frames, graph
// launch, D2H of the results, one synchronisation.
extern "C" int arp_online_reward(ArpHandle* h, const uint8_t* ob_host, int32_t n, float* reward_host,
                                 float* logits_host, float* feat_host) {
  if (!h) return ARP_ERR_INVALID;
  cudaStream_t st = h->own_stream;
  const ArpConfig& c = h->cfg;
  const size_t frame_bytes = (size_t)c.in_h * c.in_w * 3;
  if (n < 1 || n > c.max_batch) return fail(h, ARP_ERR_INVALID, "n must be in [1, max_batch=%d]", c.max_batch);
  ARP_TRY(check_ready(h, ob_host, n, (int64_t)frame_bytes, st));
  const bool text_head = !h->goal;
  if (text_head && !h->text) return fail(h, ARP_ERR_STATE, "arp_set_text has not been called");
  if (h->n_groups > 1)
    return fail(h, ARP_ERR_INVALID, "the online reward scores one instruction set: call arp_set_text (%d groups are set)",
                h->n_groups);
  if (!text_head && (reward_host || logits_host))
    return fail(h, ARP_ERR_INVALID, "goal-conditioned heads produce features only (reward = -||f - f_goal||, vl_reward.py:26-41)");
  ARP_TRY(ensure_stage(h));
  const size_t per = 1 + HEAD_MAX_TEXT + (size_t)h->feat_dim;
  if (!h->online_out) ARP_TRY(dev_alloc(h, &h->online_out, per * c.max_batch));
  float* d_r = h->online_out;
  float* d_lg = d_r + c.max_batch;
  float* d_f = d_lg + (size_t)c.max_batch * HEAD_MAX_TEXT;
  auto run = [&]() -> int {
    ARP_TRY(encode_chunk(h, h->stage_dev[0], n, (int64_t)frame_bytes, st));
    ARP_TRY(head_chunk(h, n, text_head ? d_r : nullptr, n, text_head ? d_lg : nullptr, d_f, st));
    if (h->adapter) {
      l2_normalize_rows_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(d_f, h->feat_dim, n);
      h->launches++;
    }
    return ARP_OK;
  };
  ARP_CUDA(h, cudaMemcpyAsync(h->stage_dev[0], ob_host, frame_bytes * n, cudaMemcpyHostToDevice, st));
  if (h->profiling) {
    ARP_TRY(run());
  } else {
    ArpHandle::OnlineGraph& g = h->online_graphs[n];
    if (!g.exec || g.epoch != h->online_epoch) {
      if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
      const int64_t l0 = h->launches;
      cudaGraph_t graph = nullptr;
      ARP_CUDA(h, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      const int rc = run();
      const cudaError_t e = cudaStreamEndCapture(st, &graph);
      if (rc != ARP_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (e != cudaSuccess) return fail(h, ARP_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
      const cudaError_t ei = cudaGraphInstantiate(&g.exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ei != cudaSuccess) { g.exec = nullptr; return fail(h, ARP_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ei)); }
      g.launches = h->launches - l0;
      g.epoch = h->online_epoch;
      h->launches = l0;
    }
    ARP_CUDA(h, cudaGraphLaunch(g.exec, st));
    h->launches += g.launches;
  }
  if (reward_host) ARP_CUDA(h, cudaMemcpyAsync(reward_host, d_r, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  if (logits_host) ARP_CUDA(h, cudaMemcpyAsync(logits_host, d_lg, (size_t)n * h->n_text * 4, cudaMemcpyDeviceToHost, st));
  if (feat_host) ARP_CUDA(h, cudaMemcpyAsync(feat_host, d_f, (size_t)n * h->feat_dim * 4, cudaMemcpyDeviceToHost, st));
  ARP_CUDA(h, cudaStreamSynchronize(st));
  return ARP_OK;
}

// ------------------------------------------------------------------------------------------------
// C ABI: seams / unit-test hooks
// ------------------------------------------------------------------------------------------------
extern "C" int arp_decode_only(ArpHandle* h, const uint8_t* ob_dev, int64_t T, int64_t row_stride_bytes,
                               float* chw_dev, void* stream) {
  if (!h || !chw_dev || (T > 0 && !ob_dev)) return fail(h, ARP_ERR_INVALID, "null argument");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return launch_decode(h, ob_dev, T, row_stride_bytes, chw_dev, DEC_OUT_CHW_F32, static_cast<cudaStream_t>(stream));
}

extern "C" int arp_gemm_bf16(ArpHandle* h, const void* a_dev, const void* w_dev, void* out_dev, int32_t out_dtype,
                             int64_t M, int32_t N, int32_t K, const float* bias_dev, const void* resid_dev,
                             int32_t act, void* stream) {
  if (!h || !a_dev || !w_dev || !out_dev) return fail(h, ARP_ERR_INVALID, "null argument");
  if (act < 0 || act > 2 || (out_dtype != ARP_F32 && out_dtype != ARP_OP_DTYPE)) return fail(h, ARP_ERR_INVALID, "bad act / out_dtype");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return launch_gemm(h, static_cast<const bf16*>(a_dev), M, static_cast<const bf16*>(w_dev), out_dev,
                     out_dtype == ARP_F32, act, M, N, K, N, bias_dev, resid_dev, N, nullptr, 0,
                     static_cast<cudaStream_t>(stream));
}

extern "C" int arp_resid_gemm_stats(ArpHandle* h, const void* a_dev, const void* w_dev, const float* bias_dev, void* x_dev,
                                    float* stats_dev, int64_t M, int32_t N, int32_t K, void* stream) {
  if (!h || !a_dev || !w_dev || !bias_dev || !x_dev || !stats_dev) return fail(h, ARP_ERR_INVALID, "null argument");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nparts = 2 * N / 256;
  ARP_TRY(ensure_scratch(h, 0, (size_t)M * nparts * sizeof(float2) + 256));     // grows once; stream-ordered reuse
  float2* parts = reinterpret_cast<float2*>(h->scratch[0]);
  ARP_TRY(launch_gemm(h, static_cast<const bf16*>(a_dev), M, static_cast<const bf16*>(w_dev), x_dev, false, ACT_NONE, M, N, K,
                      N, bias_dev, x_dev, N, nullptr, 0, st, nullptr, parts));
  // the merge the consuming GEMM's epilogue performs, as a kernel (test seam only)
  merge_row_stats_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(parts, nparts, reinterpret_cast<float2*>(stats_dev), (int)M, 1e-5f);
  h->launches++;
  ARP_CUDA(h, cudaGetLastError());
  return ARP_OK;
}

extern "C" int arp_ln_gemm(ArpHandle* h, const void* x_dev, const float* gamma_dev, const float* beta_dev,
                           const float* w_f32_dev, const float* bias_dev, void* out_dev, int64_t M, int32_t N,
                           int32_t act, void* stream) {
  if (!h || !x_dev || !gamma_dev || !beta_dev || !w_f32_dev || !bias_dev || !out_dev) return fail(h, ARP_ERR_INVALID, "null argument");
  if (act != ACT_NONE && act != ACT_QUICKGELU) return fail(h, ARP_ERR_INVALID, "bad act");
  if (M < 1 || N < 256 || N % 256) return fail(h, ARP_ERR_INVALID, "bad M / N");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int K = 768;
  uint8_t* tmp = nullptr;
  const size_t b_w = (size_t)N * K * sizeof(bf16), b_v = (size_t)N * 4, b_s = (size_t)M * sizeof(float2);
  auto al = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
  ARP_CUDA(h, cudaMalloc((void**)&tmp, al(b_w) + 2 * al(b_v) + al(b_s)));
  bf16* wf = reinterpret_cast<bf16*>(tmp);
  float* svec = reinterpret_cast<float*>(tmp + al(b_w));
  float* cvec = reinterpret_cast<float*>(tmp + al(b_w) + al(b_v));
  float2* stats = reinterpret_cast<float2*>(tmp + al(b_w) + 2 * al(b_v));
  fold_ln_weights_kernel<<<(N + 7) / 8, 256, 0, st>>>(w_f32_dev, gamma_dev, beta_dev, bias_dev, wf, svec, cvec, N, K);
  h->launches++;
  int rc = launch_row_moments(h, static_cast<const bf16*>(x_dev), stats, M, st);
  const LnFoldArgs f{stats, svec, cvec};
  if (rc == ARP_OK)
    rc = launch_gemm(h, static_cast<const bf16*>(x_dev), M, wf, out_dev, false, act, M, N, K, N, nullptr, nullptr, 0,
                     nullptr, 0, st, &f);
  cudaStreamSynchronize(st);
  h->tmaps.clear();          // descriptors of the freed temporaries must not be served from the cache
  cudaFree(tmp);
  return rc;
}

extern "C" int arp_layernorm_bf16(ArpHandle* h, const float* x_dev, const float* gamma_dev, const float* beta_dev,
                                  void* y_dev, int64_t M, void* stream) {
  if (!h || !x_dev || !gamma_dev || !beta_dev || !y_dev) return fail(h, ARP_ERR_INVALID, "null argument");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return launch_ln_bf16(h, x_dev, gamma_dev, beta_dev, static_cast<bf16*>(y_dev), M, static_cast<cudaStream_t>(stream));
}

extern "C" int arp_attention(ArpHandle* h, const void* qkv_dev, void* out_dev, int32_t B, int32_t tokens,
                             void* stream) {
  if (!h || !qkv_dev || !out_dev) return fail(h, ARP_ERR_INVALID, "null argument");
  ARP_CUDA(h, cudaSetDevice(h->cfg.device));
  return launch_attention(h, static_cast<const bf16*>(qkv_dev), static_cast<bf16*>(out_dev), B, tokens,
                          static_cast<cudaStream_t>(stream));
}

#ifdef ARP_ATTN_TRACE
// dev-only (never part of the shipped ABI): the attention timeline of block 0 (last launch)
extern "C" __attribute__((visibility("default"))) int arp_debug_attn_trace(long long* out, int cap) {
  const int n = 2 * ATC_TR_ITEMS * ATC_TR_EVENTS;
  cudaDeviceSynchronize();
  if (cap < n) return -1;
  cudaMemcpyFromSymbol(out, g_attn_trace, (size_t)n * sizeof(long long));
  return n;
}
#endif
