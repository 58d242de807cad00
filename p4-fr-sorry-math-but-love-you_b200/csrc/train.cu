// train.cu -- the teacher-forced TRAINING step of EfficientSATRN behind the C ABI (frx_train_*).
//
// Replaces one iteration of train_modules/train_single_opt.py:72-112:
//   model.train(); output = model(input, expected, True, 1.0)          (BatchNorm batch statistics, teacher forcing,
//                                                                        networks/EfficientSATRN.py:488-495, :697-706)
//   loss = CrossEntropyLoss(ignore_index=PAD)(output.transpose(1, 2), expected[:, 1:])     (:82-86, :690-692)
//   loss.backward(); clip_grad_norm_(params, max_grad_norm); AdamW.step()                  (:92-98, utils/utils.py:91-92)
// fp32 throughout, like the reference (no autocast).  Data-parallel training: frx_train_fwd_bwd leaves the
// gradients in ONE flat buffer (frx_train_grad_buffer) that the host all-reduces with NCCL -- per bucket, as soon as
// the backward pass has enqueued the kernels that produce it (frx_train_set_bucket_callback) -- before
// frx_train_apply clips and applies AdamW.
//
// Parameters live in one flat fp32 buffer in the layouts the kernels consume (conv [O][kh][kw][I], depthwise [9][C],
// q|k|v concatenated); gradients, Adam moments are parallel buffers, so the optimiser, the norm and the all-reduce are
// layout-agnostic.  frx_train_export / frx_train_read_grad convert back to the reference's state_dict layout.
//
// Dropout (opt-in, frx_train_set_dropout; off by default, and then the pass is the one without it) at the reference's
// sites: 0 the 2-D PE output; per encoder layer 1 the attention probabilities, 2 the MHA output before the residual add;
// 3 the decoder input; per decoder layer 4 / 5 self-attention probabilities / output, 6 / 7 cross-attention probabilities
// / output (rate p), 8 / 9 after each feed-forward ReLU (rate p_ffn).  The masks come from Philox4x32-10 (common.cuh
// philox4x32_10 / DropP) with counter (element index / 4, site + 16 * layer, step, rank) and the 64-bit seed as key, over
// the reference's logical layout of each site.  They are never stored: the backward kernels regenerate them.  step counts
// the forward passes since frx_train_create; it lives in device memory and the pass advances it itself, so a replay of the
// pass's CUDA graph draws new masks.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/frx.h"
#include "kernels.h"
#include "runtime.h"
#include "train_kernels.h"

using namespace frx;

namespace {

int tfail(frx_handle* h, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return 1;
}
#define TCK(expr)                                                                                      \
  do {                                                                                                 \
    cudaError_t e__ = (expr);                                                                          \
    if (e__ != cudaSuccess) return tfail(h, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define TKL()                                                                                          \
  do {                                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                                              \
    if (e__ != cudaSuccess) return tfail(h, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
    h->launches++;                                                                                     \
  } while (0)

struct DevGuard {
  int prev = -1;
  bool changed = false;
  void enter(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DevGuard() { if (changed) cudaSetDevice(prev); }
};

enum PKind { P_PLAIN = 0, P_CONV = 1, P_DW = 2 };
struct TParam { std::string name; size_t off, n; int kind; int d[4]; int pad_rows; };
struct TBN { size_t g = 0, b = 0, rs = 0; int C = 0; float eps = 1e-5f; std::string name; };
struct TBlock {
  int kind, cin, cout, k, stride, mid, se_r;
  bool residual;
  size_t w_a = 0, w_dw = 0, w_b = 0, se_w1 = 0, se_b1 = 0, se_w2 = 0, se_b2 = 0;
  TBN bn1, bn2, bn3;
};
struct TEncLayer { size_t ln_g, ln_b, w_qkv, b_qkv, w_o, b_o, w_c0, w_dw, b_dw, w_c1; TBN n0, ndw, n1; };
struct TDecLayer {
  size_t w_sqkv, b_sqkv, w_so, b_so, w_cq, b_cq, w_ckv, b_ckv, w_co, b_co, w_f0, b_f0, w_f1, b_f1;
  size_t ln1_g, ln1_b, ln2_g, ln2_b, ln3_g, ln3_b;
};

// forward records -----------------------------------------------------------------------------------------------------
struct CB {   // convolution (dense 1x1 or 3x3 implicit GEMM) + train-mode BatchNorm + activation (+ residual)
  const float* x = nullptr;
  float *z = nullptr, *y = nullptr, *stat = nullptr;
  const float* res = nullptr;
  int B = 0, H = 0, W = 0, Cin = 0, Cout = 0, k = 1, stride = 1, OH = 0, OW = 0, pt = 0, pl = 0, act = 0;
  size_t w = 0;
  TBN bn;
};
struct DWS { const float* x; float *z, *y, *stat; int B, H, W, C, OH, OW, stride, pt, pl, act; size_t w; size_t bias; bool has_bias; TBN bn; };
struct SES { const float* y2; float *s, *p1, *hh, *p2, *g, *y3; int B, S, C, R; };
struct BlockSave { CB c1, c2; DWS dw; SES se; const float* x_in; float* y_out; };
struct LNS { const float* x; float* y; float* stat; int M, C; size_t g, b; };
// o / o1 / o2: out_linear's result before dropout and the residual add (only with dropout on)
struct EncSave { LNS ln1, ln2; float *qkv, *att, *pre2, *scr; CB c0, c1; DWS dw; const float* x_in; float* o; };
struct DecSave { const float* x_in; float *qkv, *att, *pre1, *q2, *kv, *catt, *pre2, *f0, *f1, *pre3; LNS ln1, ln2, ln3; float *o1, *o2; };

// what the backward pass needs from the forward pass of the same call (or of the preceding frx_train_forward call)
struct Tape {
  bool valid = false;
  int B = 0, L = 0, H = 0, W = 0;
  size_t ws_mark = 0;
  float *stem_z = nullptr, *stem_stat = nullptr;
  std::vector<BlockSave> bs;
  CB last;
  // LiteSATRN's ShallowCNN (networks/LiteSATRN.py:21-70): conv0 reads the image directly, conv1-3 are implicit GEMMs
  float *lite_z0 = nullptr, *lite_y0 = nullptr, *lite_stat0 = nullptr;
  CB lite_cb[3];
  float* lite_pool[4] = {nullptr, nullptr, nullptr, nullptr};
  const float* trunk_out = nullptr;   // [B, H, W, enc_hidden]: what the 2-D positional encoding reads
  float *pe_mean = nullptr, *pe_hp = nullptr, *pe_h = nullptr, *pe_gp = nullptr, *pe_g = nullptr, *pe_out = nullptr;
  std::vector<EncSave> es;
  const float* memory = nullptr;
  long long* text = nullptr;
  unsigned char* mask = nullptr;
  std::vector<DecSave> ds;
  const float* xd = nullptr;
  float *logits = nullptr, *dlogits = nullptr;
};
enum Phase { PH_BOTH = 0, PH_FWD = 1, PH_BWD = 2 };

constexpr long long kSplitKFloats = 8ll << 20;   // 32 MB: e.g. 32 splits of a 512 x 512 output

struct TrainState {
  Tape tape;
  float *P = nullptr, *G = nullptr, *M = nullptr, *V = nullptr, *RS = nullptr;
  size_t n = 0, n_rs = 0;
  std::vector<TParam> params;
  std::map<std::string, size_t> rs_off;   // "<bn prefix>" -> offset of running_mean (running_var follows at +C)
  std::map<std::string, int> rs_C;
  std::vector<float> hostP, hostRS;
  char* ws = nullptr;
  size_t ws_bytes = 0, ws_used = 0;
  double *acc = nullptr, *sumsq = nullptr;
  float *scal = nullptr, *ones = nullptr, *zeros = nullptr;
  float* splitk_ws = nullptr;   // partial tiles of the split-K GEMM launches (kSplitKFloats floats, re-used stream-ordered)
  int step = 0, max_B = 0, max_L = 0;
  bool own_G = true;
  long long launches = 0;
  // network description
  size_t stem_w = 0; TBN stem_bn;
  bool lite = false;                 // LiteSATRN: ShallowCNN trunk instead of the EfficientNetV2-S blocks
  size_t lite_w[4] = {0, 0, 0, 0}; TBN lite_bn[4];
  std::vector<TBlock> blocks;
  size_t last_w = 0; TBN last_bn;
  size_t pe_w0 = 0, pe_b0 = 0, pe_w1 = 0, pe_b1 = 0;
  std::vector<TEncLayer> enc;
  std::vector<TDecLayer> dec;
  size_t emb = 0, gen_w = 0, gen_b = 0;
  int VP = 0;   // vocabulary rows padded to a multiple of 4
  // gradient buckets (contiguous ranges of G in the order the backward pass completes them)
  std::vector<std::pair<size_t, size_t>> buckets;   // (offset, count)
  size_t mark_trunk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  void (*bucket_cb)(void*, int64_t, int64_t) = nullptr;
  void* bucket_ctx = nullptr;
  // named views into the activation / gradient tape of the LAST frx_train_fwd_bwd call (frx_train_read_tap)
  std::map<std::string, std::pair<const float*, size_t>> taps;
  // CUDA graphs of the whole forward + backward pass, one per (batch, length): the pass is ~12 600 launches of mostly
  // small kernels (launch-bound at the reference's batch size of 16).  Inputs are staged so the graph reads fixed
  // addresses; the activation tape is a bump allocator, so every buffer address is a function of (batch, length) only.
  struct GraphEntry { cudaGraphExec_t exec = nullptr; long long nodes = 0; int seen = 0; unsigned long long last_use = 0; };
  std::map<std::pair<int, int>, GraphEntry> graphs;
  unsigned long long graph_clock = 0;
  float* img_stage = nullptr;
  long long* exp_stage = nullptr;
  // dropout (frx_train_set_dropout)
  float drop_p = 0.f, drop_pffn = 0.f;
  uint64_t drop_seed = 0;
  int drop_rank = 0;
  uint32_t* drop_ctr = nullptr;   // device: forward passes so far, advanced by the passes that run with dropout
  uint32_t drop_pending = 0;      // forward passes without dropout not yet added to *drop_ctr
  float graph_p = 0.f, graph_pffn = 0.f;   // the setting the cached graphs with dropout were captured with
  uint64_t graph_seed = 0;
  int graph_rank = 0;
  bool drop_on() const { return drop_p > 0.f || drop_pffn > 0.f; }
};

struct Ctx {   // one training call
  frx_handle* h;
  TrainState* T;
  cudaStream_t st;
  int B, L;
};

float* walloc(TrainState* T, size_t floats) {
  size_t bytes = (floats * 4 + 255) / 256 * 256;
  if (T->ws_used + bytes > T->ws_bytes) return nullptr;
  float* p = reinterpret_cast<float*>(T->ws + T->ws_used);
  T->ws_used += bytes;
  return p;
}
#define WALLOC(var, floats)                                                                       \
  do {                                                                                            \
    (var) = walloc(c.T, (size_t)(floats));                                                        \
    if (!(var)) return tfail(c.h, "training workspace exhausted (%zu MB): raise max_batch", c.T->ws_bytes >> 20); \
  } while (0)

void same_pad(int in, int k, int stride, int* out, int* pad_lo) {   // timm 0.4.9 layers/padding.py (as runtime.cu)
  *out = (in + stride - 1) / stride;
  if (stride == 1) { *pad_lo = (k - 1) / 2; return; }
  int pad = (*out - 1) * stride + k - in;
  if (pad < 0) pad = 0;
  *pad_lo = pad / 2;
}

const int kArch[6][7] = {{0, 2, 3, 1, 1, 24, 0},  {1, 4, 3, 2, 4, 48, 0},    {1, 4, 3, 2, 4, 64, 0},
                         {2, 6, 3, 2, 4, 128, 25}, {2, 9, 3, 1, 6, 160, 25}, {2, 15, 3, 2, 6, 256, 25}};

// ---------------------------------------------------------------------------------------------------------------------
// parameter registration (host)
// ---------------------------------------------------------------------------------------------------------------------
struct Builder {
  frx_handle* h;
  TrainState* T;
  bool ok = true;
  const HostTensor* get(const std::string& name) {
    auto it = h->raw.find(name);
    if (it == h->raw.end()) { tfail(h, "training: missing tensor '%s'", name.c_str()); ok = false; return nullptr; }
    return &it->second;
  }
  size_t add(const std::string& name, int kind, int pad_rows = 0) {
    const HostTensor* t = get(name);
    if (!t) return 0;
    TParam p{};
    p.name = name; p.kind = kind; p.pad_rows = pad_rows;
    for (int i = 0; i < 4; ++i) p.d[i] = i < (int)t->shape.size() ? (int)t->shape[i] : 1;
    size_t n = t->f.size();
    size_t off = (T->hostP.size() + 3) / 4 * 4;
    const size_t rowlen = t->shape.size() > 1 ? n / (size_t)t->shape[0] : 1;
    const size_t total = n + (size_t)pad_rows * rowlen;
    T->hostP.resize(off + total, 0.f);
    float* d = T->hostP.data() + off;
    if (kind == P_CONV) {          // [O][I][kh][kw] -> [O][kh*kw][I]
      const int O = p.d[0], I = p.d[1], kk = p.d[2] * p.d[3];
      for (int o = 0; o < O; ++o)
        for (int i = 0; i < I; ++i)
          for (int t2 = 0; t2 < kk; ++t2) d[((size_t)o * kk + t2) * I + i] = t->f[((size_t)o * I + i) * kk + t2];
    } else if (kind == P_DW) {     // [C][1][3][3] -> [9][C]
      const int C = p.d[0];
      for (int cc = 0; cc < C; ++cc)
        for (int t2 = 0; t2 < 9; ++t2) d[(size_t)t2 * C + cc] = t->f[(size_t)cc * 9 + t2];
    } else {
      memcpy(d, t->f.data(), n * 4);
    }
    p.off = off; p.n = total;
    T->params.push_back(p);
    return off;
  }
  TBN bn(const std::string& prefix, int C, float eps) {
    TBN b;
    b.C = C; b.eps = eps; b.name = prefix;
    b.g = add(prefix + ".weight", P_PLAIN);
    b.b = add(prefix + ".bias", P_PLAIN);
    const HostTensor *m = get(prefix + ".running_mean"), *v = get(prefix + ".running_var");
    b.rs = T->hostRS.size();
    if (m && v) {
      T->hostRS.insert(T->hostRS.end(), m->f.begin(), m->f.end());
      T->hostRS.insert(T->hostRS.end(), v->f.begin(), v->f.end());
    }
    T->rs_off[prefix] = b.rs;
    T->rs_C[prefix] = C;
    return b;
  }
};

int build_network(frx_handle* h, TrainState* T) {
  const frx_config& c = h->cfg;
  Builder bd{h, T};
  const std::string e = "encoder.shallow_cnn.";
  T->lite = c.network == FRX_NET_LITE_SATRN;
  if (T->lite) {
    // LiteSATRN.py:24-44: conv0 [C/2][Cin][3][3] (read by the direct kernel as is), conv1-3 as implicit GEMMs
    for (int i = 0; i < 4; ++i) {
      T->lite_w[i] = bd.add(e + "conv" + std::to_string(i) + ".weight", i == 0 ? P_PLAIN : P_CONV);
      T->lite_bn[i] = bd.bn(e + "batch_norm" + std::to_string(i), i == 0 ? c.enc_hidden / 2 : c.enc_hidden, 1e-5f);
    }
    for (int s = 0; s < 6; ++s) T->mark_trunk[s] = T->hostP.size();   // one trunk bucket (the last one in backward order)
  } else {
  T->stem_w = bd.add(e + "conv_stem.weight", P_PLAIN);   // [24][Cin][3][3], read by the direct stem kernel as is
  T->stem_bn = bd.bn(e + "bn1", 24, 1e-3f);
  int cin = 24;
  for (int s = 0; s < 6; ++s) {
    for (int r = 0; r < kArch[s][1]; ++r) {
      TBlock b{};
      b.kind = kArch[s][0]; b.k = kArch[s][2]; b.stride = r == 0 ? kArch[s][3] : 1;
      b.cin = cin; b.cout = kArch[s][5]; b.mid = cin * kArch[s][4]; b.se_r = cin * kArch[s][6] / 100;
      b.residual = b.cin == b.cout && b.stride == 1;
      const std::string p = e + "eff_block." + std::to_string(s) + "." + std::to_string(r);
      if (b.kind == 0) {
        b.w_a = bd.add(p + ".conv.weight", P_CONV);
        b.bn1 = bd.bn(p + ".bn1", b.cout, 1e-3f);
      } else if (b.kind == 1) {
        b.w_a = bd.add(p + ".conv_exp.weight", P_CONV);
        b.bn1 = bd.bn(p + ".bn1", b.mid, 1e-3f);
        b.w_b = bd.add(p + ".conv_pwl.weight", P_CONV);
        b.bn2 = bd.bn(p + ".bn2", b.cout, 1e-3f);
      } else {
        b.w_a = bd.add(p + ".conv_pw.weight", P_CONV);
        b.bn1 = bd.bn(p + ".bn1", b.mid, 1e-3f);
        b.w_dw = bd.add(p + ".conv_dw.weight", P_DW);
        b.bn2 = bd.bn(p + ".bn2", b.mid, 1e-3f);
        b.se_w1 = bd.add(p + ".se.conv_reduce.weight", P_PLAIN);
        b.se_b1 = bd.add(p + ".se.conv_reduce.bias", P_PLAIN);
        b.se_w2 = bd.add(p + ".se.conv_expand.weight", P_PLAIN);
        b.se_b2 = bd.add(p + ".se.conv_expand.bias", P_PLAIN);
        b.w_b = bd.add(p + ".conv_pwl.weight", P_CONV);
        b.bn3 = bd.bn(p + ".bn3", b.cout, 1e-3f);
      }
      T->blocks.push_back(b);
      cin = b.cout;
    }
    T->mark_trunk[s] = T->hostP.size();
  }
  T->last_w = bd.add(e + "conv_last.weight", P_CONV);
  T->last_bn = bd.bn(e + "bn2", c.enc_hidden, 1e-5f);
  }
  const std::string pe = "encoder.positional_encoding.";
  T->pe_w0 = bd.add(pe + "dense0.weight", P_PLAIN); T->pe_b0 = bd.add(pe + "dense0.bias", P_PLAIN);
  T->pe_w1 = bd.add(pe + "dense1.weight", P_PLAIN); T->pe_b1 = bd.add(pe + "dense1.bias", P_PLAIN);
  for (int i = 0; i < c.enc_layers; ++i) {
    TEncLayer L{};
    const std::string p = "encoder.attention_layers." + std::to_string(i) + ".";
    L.ln_g = bd.add(p + "norm.weight", P_PLAIN); L.ln_b = bd.add(p + "norm.bias", P_PLAIN);
    const std::string a = p + "attention_layer.";
    L.w_qkv = bd.add(a + "q_linear.weight", P_PLAIN); bd.add(a + "k_linear.weight", P_PLAIN); bd.add(a + "v_linear.weight", P_PLAIN);
    L.b_qkv = bd.add(a + "q_linear.bias", P_PLAIN); bd.add(a + "k_linear.bias", P_PLAIN); bd.add(a + "v_linear.bias", P_PLAIN);
    L.w_o = bd.add(a + "out_linear.weight", P_PLAIN); L.b_o = bd.add(a + "out_linear.bias", P_PLAIN);
    L.w_c0 = bd.add(p + "conv0.weight", P_CONV); L.n0 = bd.bn(p + "norm0", c.enc_filter, 1e-5f);
    L.w_dw = bd.add(p + "depthwise.weight", P_DW); L.b_dw = bd.add(p + "depthwise.bias", P_PLAIN);
    L.ndw = bd.bn(p + "depthwise_norm", c.enc_filter, 1e-5f);
    L.w_c1 = bd.add(p + "conv1.weight", P_CONV); L.n1 = bd.bn(p + "norm1", c.enc_hidden, 1e-5f);
    T->enc.push_back(L);
  }
  T->mark_trunk[6] = T->hostP.size();   // end of the encoder
  T->emb = bd.add("decoder.embedding.weight", P_PLAIN);
  for (int l = 0; l < c.dec_layers; ++l) {
    TDecLayer D{};
    const std::string p = "decoder.attention_layers." + std::to_string(l) + ".";
    const std::string s = p + "self_attention_layer.", a = p + "attention_layer.", f = p + "feedforward_layer.";
    D.w_sqkv = bd.add(s + "q_linear.weight", P_PLAIN); bd.add(s + "k_linear.weight", P_PLAIN); bd.add(s + "v_linear.weight", P_PLAIN);
    D.b_sqkv = bd.add(s + "q_linear.bias", P_PLAIN); bd.add(s + "k_linear.bias", P_PLAIN); bd.add(s + "v_linear.bias", P_PLAIN);
    D.w_so = bd.add(s + "out_linear.weight", P_PLAIN); D.b_so = bd.add(s + "out_linear.bias", P_PLAIN);
    D.ln1_g = bd.add(p + "self_attention_norm.weight", P_PLAIN); D.ln1_b = bd.add(p + "self_attention_norm.bias", P_PLAIN);
    D.w_cq = bd.add(a + "q_linear.weight", P_PLAIN); D.b_cq = bd.add(a + "q_linear.bias", P_PLAIN);
    D.w_ckv = bd.add(a + "k_linear.weight", P_PLAIN); bd.add(a + "v_linear.weight", P_PLAIN);
    D.b_ckv = bd.add(a + "k_linear.bias", P_PLAIN); bd.add(a + "v_linear.bias", P_PLAIN);
    D.w_co = bd.add(a + "out_linear.weight", P_PLAIN); D.b_co = bd.add(a + "out_linear.bias", P_PLAIN);
    D.ln2_g = bd.add(p + "attention_norm.weight", P_PLAIN); D.ln2_b = bd.add(p + "attention_norm.bias", P_PLAIN);
    D.w_f0 = bd.add(f + "linear0.weight", P_PLAIN); D.b_f0 = bd.add(f + "linear0.bias", P_PLAIN);
    D.w_f1 = bd.add(f + "linear1.weight", P_PLAIN); D.b_f1 = bd.add(f + "linear1.bias", P_PLAIN);
    D.ln3_g = bd.add(p + "feedforward_norm.weight", P_PLAIN); D.ln3_b = bd.add(p + "feedforward_norm.bias", P_PLAIN);
    T->dec.push_back(D);
  }
  T->VP = (c.num_classes + 3) / 4 * 4;
  T->gen_w = bd.add("decoder.generator.weight", P_PLAIN, T->VP - c.num_classes);   // zero rows: the logits row stride is VP
  T->gen_b = bd.add("decoder.generator.bias", P_PLAIN, T->VP - c.num_classes);
  if (!bd.ok) return 1;
  // adjacency the fused projections rely on
  for (size_t i = 0; i + 1 < T->params.size(); ++i) {
    const TParam &a = T->params[i], &b = T->params[i + 1];
    const bool fused = (a.name.find("q_linear") != std::string::npos && b.name.find("k_linear") != std::string::npos) ||
                       (a.name.find("k_linear") != std::string::npos && b.name.find("v_linear") != std::string::npos);
    if (fused && a.name.substr(a.name.rfind('.')) == b.name.substr(b.name.rfind('.')) && a.off + a.n != b.off)
      return tfail(h, "training: '%s' and '%s' are not contiguous", a.name.c_str(), b.name.c_str());
  }
  T->n = (T->hostP.size() + 3) / 4 * 4;
  T->hostP.resize(T->n, 0.f);
  T->n_rs = T->hostRS.size();
  // buckets, in backward completion order: decoder | encoder layers + 2-D PE + conv_last | stages 5, 4, 3 | stages 2..0 + stem
  const size_t enc_begin = T->mark_trunk[5], enc_end = T->mark_trunk[6];
  T->buckets = {{enc_end, T->n - enc_end},
                {enc_begin, enc_end - enc_begin},
                {T->mark_trunk[4], T->mark_trunk[5] - T->mark_trunk[4]},
                {T->mark_trunk[3], T->mark_trunk[4] - T->mark_trunk[3]},
                {T->mark_trunk[2], T->mark_trunk[3] - T->mark_trunk[2]},
                {0, T->mark_trunk[2]}};
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// building blocks
// ---------------------------------------------------------------------------------------------------------------------
GemmP dense(const float* A, long long M, int K, const float* W, int N, float* C, int ldc) {
  GemmP g{};
  g.A = A; g.W = W; g.C = C; g.M = (int)M; g.N = N; g.K = K; g.lda = K; g.ldc = ldc; g.conv = 0; g.rows_per_img = 1;
  return g;
}

// y[M, N] = act(x[M, K] * W^T + b) (+ res)
int lin_fwd(Ctx& c, const float* x, long long M, int K, size_t w, size_t b, bool has_b, int N, float* y, int ldy, int act, const float* res) {
  frx_handle* h = c.h;
  GemmP g = dense(x, M, K, c.T->P + w, N, y, ldy);
  if (has_b) g.shift = c.T->P + b;
  g.act = act;
  if (res) { g.res = res; g.ldr = ldy; }
  g.ws = h->opt_train_splitk ? c.T->splitk_ws : nullptr; g.ws_floats = kSplitKFloats; launch_igemm_f32(g, c.st); TKL();
  return 0;
}
// dW += dy^T x; db += colsum(dy); dx (=|+=) dy * W          (dy [M, ldy >= N], x [M, K])
int lin_bwd(Ctx& c, const float* dy, int ldy, const float* x, long long M, int K, size_t w, size_t b, bool has_b, int N, float* dx, bool accumulate) {
  frx_handle* h = c.h;
  WgradP wp{};
  wp.dZ = dy; wp.A = x; wp.dW = c.T->G + w; wp.M = M; wp.N = N; wp.K = K; wp.ldz = ldy; wp.lda = K;
  launch_wgrad(wp, h->num_sms, c.st); TKL();
  if (has_b) { launch_colsum(dy, c.T->G + b, M, N, ldy, c.st); TKL(); }
  if (dx) {
    float* wt;
    WALLOC(wt, (size_t)K * ldy);
    if (ldy != N) TCK(cudaMemsetAsync(wt, 0, (size_t)K * ldy * 4, c.st));
    // W [N][K] -> Wt [K][ldy] (columns N..ldy-1 stay zero)
    if (ldy == N) { launch_repack_dgrad(c.T->P + w, wt, N, 1, K, c.st); TKL(); }
    else {
      float* tmp;
      WALLOC(tmp, (size_t)K * N);
      launch_repack_dgrad(c.T->P + w, tmp, N, 1, K, c.st); TKL();
      TCK(cudaMemcpy2DAsync(wt, (size_t)ldy * 4, tmp, (size_t)N * 4, (size_t)N * 4, K, cudaMemcpyDeviceToDevice, c.st));
    }
    GemmP g = dense(dy, M, ldy, wt, K, dx, K);
    if (accumulate) { g.res = dx; g.ldr = K; }
    g.ws = h->opt_train_splitk ? c.T->splitk_ws : nullptr; g.ws_floats = kSplitKFloats; launch_igemm_f32(g, c.st); TKL();
  }
  return 0;
}

int bn_fwd(Ctx& c, const float* z, long long M, const TBN& bn, int act, const float* res, float* y, float** stat_out) {
  frx_handle* h = c.h;
  float* stat;
  WALLOC(stat, 4 * bn.C);
  launch_bn_stats(z, c.T->acc, c.T->P + bn.g, c.T->P + bn.b, c.T->RS + bn.rs, c.T->RS + bn.rs + bn.C, stat, (int)M, bn.C, bn.eps, 0.1f, c.st);
  TKL();
  launch_bn_apply(z, stat, res, y, M, bn.C, act, c.st); TKL();
  *stat_out = stat;
  return 0;
}

int cb_fwd(Ctx& c, CB& r) {
  frx_handle* h = c.h;
  int pt = 0, pl = 0;
  if (r.k == 1) { r.OH = r.H; r.OW = r.W; }
  else { same_pad(r.H, r.k, r.stride, &r.OH, &pt); same_pad(r.W, r.k, r.stride, &r.OW, &pl); }
  r.pt = pt; r.pl = pl;
  const long long M = (long long)r.B * r.OH * r.OW;
  WALLOC(r.z, M * r.Cout);
  WALLOC(r.y, M * r.Cout);
  GemmP g{};
  g.A = r.x; g.W = c.T->P + r.w; g.C = r.z; g.M = (int)M; g.N = r.Cout; g.K = r.k * r.k * r.Cin; g.lda = g.K; g.ldc = r.Cout;
  g.rows_per_img = 1;
  if (r.k > 1) {
    g.conv = 1; g.H = r.H; g.Wd = r.W; g.Cin = r.Cin; g.OH = r.OH; g.OW = r.OW; g.KH = r.k; g.KW = r.k; g.stride = r.stride; g.pad_t = pt; g.pad_l = pl;
    g.lda = 0;
  }
  g.ws = h->opt_train_splitk ? c.T->splitk_ws : nullptr; g.ws_floats = kSplitKFloats; launch_igemm_f32(g, c.st); TKL();
  return bn_fwd(c, r.z, M, r.bn, r.act, r.res, r.y, &r.stat);
}

// dy: gradient of the record's output.  Produces dx (when want_dx) in a fresh buffer; the caller adds dy to the skip path.
int cb_bwd(Ctx& c, const CB& r, const float* dy, float** dx_out, bool want_dx) {
  frx_handle* h = c.h;
  const long long M = (long long)r.B * r.OH * r.OW;
  float* dz;
  WALLOC(dz, M * r.Cout);
  launch_bn_bwd(dy, r.z, r.stat, c.T->acc, dz, c.T->G + r.bn.g, c.T->G + r.bn.b, (int)M, r.Cout, r.act, c.st); TKL();
  WgradP wp{};
  wp.dZ = dz; wp.A = r.x; wp.dW = c.T->G + r.w; wp.M = M; wp.N = r.Cout; wp.K = r.k * r.k * r.Cin; wp.ldz = r.Cout; wp.lda = wp.K;
  if (r.k > 1) { wp.conv = 1; wp.H = r.H; wp.Wd = r.W; wp.Cin = r.Cin; wp.OH = r.OH; wp.OW = r.OW; wp.KW = r.k; wp.stride = r.stride; wp.pad_t = r.pt; wp.pad_l = r.pl; }
  launch_wgrad(wp, h->num_sms, c.st); TKL();
  if (!want_dx) return 0;
  const int T2 = r.k * r.k;
  float* wt;
  WALLOC(wt, (size_t)r.Cin * T2 * r.Cout);
  launch_repack_dgrad(c.T->P + r.w, wt, r.Cout, T2, r.Cin, c.st); TKL();   // [Cout][T][Cin] -> [Cin][flipped T][Cout]
  const long long Min = (long long)r.B * r.H * r.W;
  float* dx;
  WALLOC(dx, Min * r.Cin);
  GemmP g{};
  g.W = wt; g.C = dx; g.M = (int)Min; g.N = r.Cin; g.K = T2 * r.Cout; g.ldc = r.Cin; g.rows_per_img = 1;
  if (r.k == 1) {
    g.A = dz; g.lda = r.Cout;
  } else {
    const float* zsrc = dz;
    int ZH = r.OH, ZW = r.OW;
    if (r.stride > 1) {
      ZH = (r.OH - 1) * r.stride + 1; ZW = (r.OW - 1) * r.stride + 1;
      float* zs;
      WALLOC(zs, (size_t)r.B * ZH * ZW * r.Cout);
      launch_zero_stuff(dz, zs, r.B, r.OH, r.OW, r.Cout, r.stride, ZH, ZW, c.st); TKL();
      zsrc = zs;
    }
    g.A = zsrc; g.conv = 1; g.H = ZH; g.Wd = ZW; g.Cin = r.Cout; g.OH = r.H; g.OW = r.W; g.KH = r.k; g.KW = r.k; g.stride = 1;
    g.pad_t = r.k - 1 - r.pt; g.pad_l = r.k - 1 - r.pl;
  }
  g.ws = h->opt_train_splitk ? c.T->splitk_ws : nullptr; g.ws_floats = kSplitKFloats; launch_igemm_f32(g, c.st); TKL();
  *dx_out = dx;
  return 0;
}

int dw_fwd(Ctx& c, DWS& r) {
  frx_handle* h = c.h;
  same_pad(r.H, 3, r.stride, &r.OH, &r.pt);
  same_pad(r.W, 3, r.stride, &r.OW, &r.pl);
  const long long M = (long long)r.B * r.OH * r.OW;
  WALLOC(r.z, M * r.C);
  WALLOC(r.y, M * r.C);
  DwP d{r.x, c.T->P + r.w, c.T->ones, r.has_bias ? c.T->P + r.bias : c.T->zeros, r.z, r.B, r.H, r.W, r.C, r.OH, r.OW, r.stride, r.pt, r.pl, ACT_NONE};
  launch_dwconv_f32(d, c.st); TKL();
  return bn_fwd(c, r.z, M, r.bn, r.act, nullptr, r.y, &r.stat);
}
int dw_bwd(Ctx& c, const DWS& r, const float* dy, float** dx_out) {
  frx_handle* h = c.h;
  const long long M = (long long)r.B * r.OH * r.OW;
  float *dz, *dx;
  WALLOC(dz, M * r.C);
  launch_bn_bwd(dy, r.z, r.stat, c.T->acc, dz, c.T->G + r.bn.g, c.T->G + r.bn.b, (int)M, r.C, r.act, c.st); TKL();
  WALLOC(dx, (size_t)r.B * r.H * r.W * r.C);
  launch_dw_bwd(dz, r.x, c.T->P + r.w, dx, c.T->G + r.w, r.has_bias ? c.T->G + r.bias : nullptr, r.B, r.H, r.W, r.C, r.OH, r.OW, r.stride, r.pt,
                r.pl, c.st);
  TKL();
  *dx_out = dx;
  return 0;
}

int se_fwd(Ctx& c, SES& r, const TBlock& b) {
  frx_handle* h = c.h;
  WALLOC(r.s, (size_t)r.B * r.C); WALLOC(r.p1, (size_t)r.B * r.R); WALLOC(r.hh, (size_t)r.B * r.R);
  WALLOC(r.p2, (size_t)r.B * r.C); WALLOC(r.g, (size_t)r.B * r.C); WALLOC(r.y3, (size_t)r.B * r.S * r.C);
  launch_spatial_dot(r.y2, nullptr, r.s, r.B, r.S, r.C, 1.f / (float)r.S, c.st); TKL();
  if (lin_fwd(c, r.s, r.B, r.C, b.se_w1, b.se_b1, true, r.R, r.p1, r.R, ACT_NONE, nullptr)) return 1;
  launch_act_fwd(r.p1, r.hh, ACT_SILU, (long long)r.B * r.R, c.st); TKL();
  if (lin_fwd(c, r.hh, r.B, r.R, b.se_w2, b.se_b2, true, r.C, r.p2, r.C, ACT_NONE, nullptr)) return 1;
  launch_act_fwd(r.p2, r.g, ACT_SIGMOID, (long long)r.B * r.C, c.st); TKL();
  launch_spatial_scale(r.y2, r.g, nullptr, r.y3, r.B, r.S, r.C, c.st); TKL();
  return 0;
}
int se_bwd(Ctx& c, const SES& r, const TBlock& b, const float* dy3, float** dy2_out) {
  frx_handle* h = c.h;
  float *dg, *dp2, *dh, *dp1, *ds, *dy2;
  WALLOC(dg, (size_t)r.B * r.C); WALLOC(dp2, (size_t)r.B * r.C); WALLOC(dh, (size_t)r.B * r.R); WALLOC(dp1, (size_t)r.B * r.R);
  WALLOC(ds, (size_t)r.B * r.C); WALLOC(dy2, (size_t)r.B * r.S * r.C);
  launch_spatial_dot(dy3, r.y2, dg, r.B, r.S, r.C, 1.f, c.st); TKL();
  launch_act_bwd(dg, r.p2, dp2, ACT_SIGMOID, (long long)r.B * r.C, c.st); TKL();
  if (lin_bwd(c, dp2, r.C, r.hh, r.B, r.R, b.se_w2, b.se_b2, true, r.C, dh, false)) return 1;
  launch_act_bwd(dh, r.p1, dp1, ACT_SILU, (long long)r.B * r.R, c.st); TKL();
  if (lin_bwd(c, dp1, r.R, r.s, r.B, r.C, b.se_w1, b.se_b1, true, r.R, ds, false)) return 1;
  launch_axpy(ds, ds, 1.f / (float)r.S, (long long)r.B * r.C, 0, c.st); TKL();
  launch_spatial_scale(dy3, r.g, ds, dy2, r.B, r.S, r.C, c.st); TKL();
  *dy2_out = dy2;
  return 0;
}

int ln_fwd(Ctx& c, LNS& r) {
  frx_handle* h = c.h;
  WALLOC(r.y, (size_t)r.M * r.C);
  WALLOC(r.stat, (size_t)r.M * 2);
  launch_ln_fwd(r.x, c.T->P + r.g, c.T->P + r.b, r.y, r.stat, r.M, r.C, c.st); TKL();
  return 0;
}
int ln_bwd(Ctx& c, const LNS& r, const float* dy, float** dx_out) {
  frx_handle* h = c.h;
  float* dx;
  WALLOC(dx, (size_t)r.M * r.C);
  launch_ln_bwd(dy, r.x, r.stat, c.T->P + r.g, dx, c.T->G + r.g, c.T->G + r.b, r.M, r.C, c.st); TKL();
  *dx_out = dx;
  return 0;
}

void tap(Ctx& c, const std::string& name, const float* p, size_t n) { c.T->taps[name] = {p, n}; }

// dropout site `site` of layer `layer` (ffn: rate p_ffn, else p); back = 1 in the backward pass, which runs after the forward
// pass has advanced the step counter.  step == nullptr when the site's rate is 0.
DropP drop_site(const TrainState* T, int site, int layer, bool ffn, int back) {
  DropP d{};
  const float p = ffn ? T->drop_pffn : T->drop_p;
  if (p <= 0.f) return d;
  d.step = T->drop_ctr;
  d.back = (uint32_t)back;
  d.site = (uint32_t)(site + 16 * layer);
  d.rank = (uint32_t)T->drop_rank;
  d.key_lo = (uint32_t)T->drop_seed;
  d.key_hi = (uint32_t)(T->drop_seed >> 32);
  d.thresh = (uint32_t)std::min(4294967295.0, std::floor((double)p * 4294967296.0));
  d.scale = 1.0f / (1.0f - p);
  return d;
}

// out_linear of an attention block: y = dropout(x W^T + b) + res, or with the site off the GEMM with the residual in its
// epilogue.  o: tape buffer for the undropped GEMM result.
int attn_out_fwd(Ctx& c, const float* x, long long M, int N, size_t w, size_t b, const float* res, float* y, float** o, const DropP& d) {
  frx_handle* h = c.h;
  if (!d.step) return lin_fwd(c, x, M, N, w, b, true, N, y, N, ACT_NONE, res);
  WALLOC(*o, M * N);
  if (lin_fwd(c, x, M, N, w, b, true, N, *o, N, ACT_NONE, nullptr)) return 1;
  launch_dropout(*o, res, y, M * N, d, 0, 0, c.st); TKL();
  return 0;
}
// gradient of out_linear's output under dropout: dy * M * s into a fresh buffer (dy itself when the site is off)
int drop_bwd(Ctx& c, const float* dy, long long n, const DropP& d, const float** out) {
  frx_handle* h = c.h;
  *out = dy;
  if (!d.step) return 0;
  float* m;
  WALLOC(m, n);
  launch_dropout(dy, nullptr, m, n, d, 0, 0, c.st); TKL();
  *out = m;
  return 0;
}

void bucket_done(Ctx& c, int idx) {
  if (c.T->bucket_cb && idx < (int)c.T->buckets.size() && c.T->buckets[idx].second > 0)
    c.T->bucket_cb(c.T->bucket_ctx, (int64_t)c.T->buckets[idx].first, (int64_t)c.T->buckets[idx].second);
}

// ---------------------------------------------------------------------------------------------------------------------
// forward + backward of the whole model
// ---------------------------------------------------------------------------------------------------------------------
// phase PH_BOTH: one training pass (forward, loss, backward).  PH_FWD: the train-mode forward alone (logits_out [B, L, V],
// loss_out optional) leaving the tape for a later PH_BWD, which starts from dlogits_in [B, L, V] (the gradient a caller's
// own criterion produced: EfficientSATRN.forward under model.train() + loss.backward()).
int fwd_bwd(Ctx& c, const float* images, const long long* expected, float* loss_out, int phase = PH_BOTH, float* logits_out = nullptr,
            const float* dlogits_in = nullptr) {
  frx_handle* h = c.h;
  TrainState* T = c.T;
  Tape& tp = T->tape;
  const frx_config& cf = h->cfg;
  const int B = c.B, L = c.L;
  const int H0 = (cf.height - 3) / 2 + 1, W0 = (cf.width - 3) / 2 + 1;
  const int C = cf.enc_hidden, F = cf.enc_filter;
  const int D = cf.dec_hidden, FF = cf.dec_filter, V = cf.num_classes, VP = T->VP, Md = B * L, heads = cf.dec_heads, HD = D / heads;
  const float temp = sqrtf((float)D);
  const float* peh = h->arena + h->pe_h;   // host-built tables (not parameters), uploaded by frx_finalize_weights
  const float* pew = h->arena + h->pe_w;
  if (phase != PH_BWD) {
  T->ws_used = 0;
  T->taps.clear();
  tp.valid = false;
  // ================= forward =================
  if (T->lite) {
    // ShallowCNN: 4 x (conv3x3 p1 -> train-mode BN -> ReLU -> maxpool 2x2), LiteSATRN.py:50-70
    const int C0 = C / 2;
    int Hc = cf.height, Wc = cf.width;
    WALLOC(tp.lite_z0, (size_t)B * Hc * Wc * C0); WALLOC(tp.lite_y0, (size_t)B * Hc * Wc * C0);
    launch_direct_conv3x3(images, T->P + T->lite_w[0], T->ones, T->zeros, tp.lite_z0, B, cf.in_ch, Hc, Wc, Hc, Wc, C0, 1, 1, ACT_NONE, c.st);
    TKL();
    if (bn_fwd(c, tp.lite_z0, (long long)B * Hc * Wc, T->lite_bn[0], ACT_RELU, nullptr, tp.lite_y0, &tp.lite_stat0)) return 1;
    WALLOC(tp.lite_pool[0], (size_t)B * (Hc / 2) * (Wc / 2) * C0);
    launch_maxpool2_fwd(tp.lite_y0, tp.lite_pool[0], B, Hc, Wc, C0, c.st); TKL();
    Hc /= 2; Wc /= 2;
    for (int i = 1; i < 4; ++i) {
      CB& r = tp.lite_cb[i - 1];
      r = CB{};
      r.x = tp.lite_pool[i - 1]; r.B = B; r.H = Hc; r.W = Wc; r.Cin = i == 1 ? C0 : C; r.Cout = C; r.k = 3; r.stride = 1; r.act = ACT_RELU;
      r.w = T->lite_w[i]; r.bn = T->lite_bn[i];
      if (cb_fwd(c, r)) return 1;
      WALLOC(tp.lite_pool[i], (size_t)B * (Hc / 2) * (Wc / 2) * C);
      launch_maxpool2_fwd(r.y, tp.lite_pool[i], B, Hc, Wc, C, c.st); TKL();
      Hc /= 2; Wc /= 2;
    }
    tp.H = Hc; tp.W = Wc;
    tp.trunk_out = tp.lite_pool[3];
  } else {
  float* stem_y;
  WALLOC(tp.stem_z, (size_t)B * H0 * W0 * 24); WALLOC(stem_y, (size_t)B * H0 * W0 * 24);
  launch_direct_conv3x3(images, T->P + T->stem_w, T->ones, T->zeros, tp.stem_z, B, cf.in_ch, cf.height, cf.width, H0, W0, 24, 2, 0, ACT_NONE, c.st);
  TKL();
  if (bn_fwd(c, tp.stem_z, (long long)B * H0 * W0, T->stem_bn, ACT_SILU, nullptr, stem_y, &tp.stem_stat)) return 1;
  tp.bs.assign(T->blocks.size(), BlockSave{});
  const float* x = stem_y;
  tp.H = H0; tp.W = W0;
  for (size_t i = 0; i < T->blocks.size(); ++i) {
    const TBlock& b = T->blocks[i];
    BlockSave& s = tp.bs[i];
    s.x_in = x;
    if (b.kind == 0) {
      s.c1 = CB{}; s.c1.x = x; s.c1.B = B; s.c1.H = tp.H; s.c1.W = tp.W; s.c1.Cin = b.cin; s.c1.Cout = b.cout; s.c1.k = b.k; s.c1.stride = b.stride;
      s.c1.act = ACT_SILU; s.c1.w = b.w_a; s.c1.bn = b.bn1; s.c1.res = b.residual ? x : nullptr;
      if (cb_fwd(c, s.c1)) return 1;
      x = s.c1.y; tp.H = s.c1.OH; tp.W = s.c1.OW;
    } else if (b.kind == 1) {
      s.c1 = CB{}; s.c1.x = x; s.c1.B = B; s.c1.H = tp.H; s.c1.W = tp.W; s.c1.Cin = b.cin; s.c1.Cout = b.mid; s.c1.k = b.k; s.c1.stride = b.stride;
      s.c1.act = ACT_SILU; s.c1.w = b.w_a; s.c1.bn = b.bn1;
      if (cb_fwd(c, s.c1)) return 1;
      s.c2 = CB{}; s.c2.x = s.c1.y; s.c2.B = B; s.c2.H = s.c1.OH; s.c2.W = s.c1.OW; s.c2.Cin = b.mid; s.c2.Cout = b.cout; s.c2.k = 1;
      s.c2.act = ACT_NONE; s.c2.w = b.w_b; s.c2.bn = b.bn2; s.c2.res = b.residual ? x : nullptr;
      if (cb_fwd(c, s.c2)) return 1;
      x = s.c2.y; tp.H = s.c1.OH; tp.W = s.c1.OW;
    } else {
      s.c1 = CB{}; s.c1.x = x; s.c1.B = B; s.c1.H = tp.H; s.c1.W = tp.W; s.c1.Cin = b.cin; s.c1.Cout = b.mid; s.c1.k = 1;
      s.c1.act = ACT_SILU; s.c1.w = b.w_a; s.c1.bn = b.bn1;
      if (cb_fwd(c, s.c1)) return 1;
      s.dw = DWS{}; s.dw.x = s.c1.y; s.dw.B = B; s.dw.H = tp.H; s.dw.W = tp.W; s.dw.C = b.mid; s.dw.stride = b.stride; s.dw.act = ACT_SILU;
      s.dw.w = b.w_dw; s.dw.has_bias = false; s.dw.bn = b.bn2;
      if (dw_fwd(c, s.dw)) return 1;
      s.se = SES{}; s.se.y2 = s.dw.y; s.se.B = B; s.se.S = s.dw.OH * s.dw.OW; s.se.C = b.mid; s.se.R = b.se_r;
      if (se_fwd(c, s.se, b)) return 1;
      s.c2 = CB{}; s.c2.x = s.se.y3; s.c2.B = B; s.c2.H = s.dw.OH; s.c2.W = s.dw.OW; s.c2.Cin = b.mid; s.c2.Cout = b.cout; s.c2.k = 1;
      s.c2.act = ACT_NONE; s.c2.w = b.w_b; s.c2.bn = b.bn3; s.c2.res = b.residual ? x : nullptr;
      if (cb_fwd(c, s.c2)) return 1;
      x = s.c2.y; tp.H = s.dw.OH; tp.W = s.dw.OW;
    }
  }
  tp.last = CB{};
  tp.last.x = x; tp.last.B = B; tp.last.H = tp.H; tp.last.W = tp.W; tp.last.Cin = 256; tp.last.Cout = cf.enc_hidden; tp.last.k = 1; tp.last.act = ACT_SILU; tp.last.w = T->last_w;
  tp.last.bn = T->last_bn;
  if (cb_fwd(c, tp.last)) return 1;
  tp.trunk_out = tp.last.y;
  }
  if (tp.H != h->feat_h || tp.W != h->feat_w) return tfail(h, "training: trunk output %dx%d != %dx%d", tp.H, tp.W, h->feat_h, h->feat_w);
  const int S = tp.H * tp.W;
  // ---- adaptive 2-D positional encoding (:135-154) ----
  WALLOC(tp.pe_mean, (size_t)B * C); WALLOC(tp.pe_hp, (size_t)B * C / 2); WALLOC(tp.pe_h, (size_t)B * C / 2); WALLOC(tp.pe_gp, (size_t)B * 2 * C);
  WALLOC(tp.pe_g, (size_t)B * 2 * C); WALLOC(tp.pe_out, (size_t)B * S * C);
  launch_spatial_dot(tp.trunk_out, nullptr, tp.pe_mean, B, S, C, 1.f / (float)S, c.st); TKL();
  if (lin_fwd(c, tp.pe_mean, B, C, T->pe_w0, T->pe_b0, true, C / 2, tp.pe_hp, C / 2, ACT_NONE, nullptr)) return 1;
  launch_act_fwd(tp.pe_hp, tp.pe_h, ACT_RELU, (long long)B * C / 2, c.st); TKL();
  if (lin_fwd(c, tp.pe_h, B, C / 2, T->pe_w1, T->pe_b1, true, 2 * C, tp.pe_gp, 2 * C, ACT_NONE, nullptr)) return 1;
  launch_act_fwd(tp.pe_gp, tp.pe_g, ACT_SIGMOID, (long long)B * 2 * C, c.st); TKL();
  launch_pe2d_apply(tp.trunk_out, tp.pe_g, peh, pew, tp.pe_out, B, tp.H, tp.W, C, drop_site(T, 0, 0, false, 0), c.st); TKL();
  // ---- encoder layers (:259-281) ----
  tp.es.assign(T->enc.size(), EncSave{});
  const float* xe = tp.pe_out;
  const int Me = B * S;
  for (size_t i = 0; i < T->enc.size(); ++i) {
    const TEncLayer& Lw = T->enc[i];
    EncSave& s = tp.es[i];
    s.x_in = xe;
    s.ln1 = LNS{xe, nullptr, nullptr, Me, C, Lw.ln_g, Lw.ln_b};
    if (ln_fwd(c, s.ln1)) return 1;
    WALLOC(s.qkv, (size_t)Me * 3 * C); WALLOC(s.att, (size_t)Me * C); WALLOC(s.pre2, (size_t)Me * C); WALLOC(s.scr, (size_t)Me * C);
    if (lin_fwd(c, s.ln1.y, Me, C, Lw.w_qkv, Lw.b_qkv, true, 3 * C, s.qkv, 3 * C, ACT_NONE, nullptr)) return 1;
    const DropP dpa = drop_site(T, 1, (int)i, false, 0);
    if (dpa.step) launch_enc_attn_f32_drop(s.qkv, s.att, B, S, C, cf.enc_heads, dpa, c.st);
    else launch_enc_attn_f32(s.qkv, s.att, B, S, C, cf.enc_heads, c.st);
    TKL();
    if (attn_out_fwd(c, s.att, Me, C, Lw.w_o, Lw.b_o, xe, s.pre2, &s.o, drop_site(T, 2, (int)i, false, 0))) return 1;
    s.ln2 = LNS{s.pre2, nullptr, nullptr, Me, C, Lw.ln_g, Lw.ln_b};
    if (ln_fwd(c, s.ln2)) return 1;
    launch_scramble(s.ln2.y, s.scr, B, S, C, 0, c.st); TKL();
    s.c0 = CB{}; s.c0.x = s.scr; s.c0.B = B; s.c0.H = tp.H; s.c0.W = tp.W; s.c0.Cin = C; s.c0.Cout = F; s.c0.k = 1; s.c0.act = ACT_RELU; s.c0.w = Lw.w_c0;
    s.c0.bn = Lw.n0;
    if (cb_fwd(c, s.c0)) return 1;
    s.dw = DWS{}; s.dw.x = s.c0.y; s.dw.B = B; s.dw.H = tp.H; s.dw.W = tp.W; s.dw.C = F; s.dw.stride = 1; s.dw.act = ACT_RELU; s.dw.w = Lw.w_dw;
    s.dw.bias = Lw.b_dw; s.dw.has_bias = true; s.dw.bn = Lw.ndw;
    if (dw_fwd(c, s.dw)) return 1;
    s.c1 = CB{}; s.c1.x = s.dw.y; s.c1.B = B; s.c1.H = tp.H; s.c1.W = tp.W; s.c1.Cin = F; s.c1.Cout = C; s.c1.k = 1; s.c1.act = ACT_RELU; s.c1.w = Lw.w_c1;
    s.c1.bn = Lw.n1; s.c1.res = xe;
    if (cb_fwd(c, s.c1)) return 1;
    xe = s.c1.y;
  }
  tp.memory = xe;   // [B, S, C]
  // ---- teacher-forced decoder (:488-495) ----
  { float* t; WALLOC(t, (size_t)Md * 2); tp.text = reinterpret_cast<long long*>(t); }
  TCK(cudaMemcpy2DAsync(tp.text, (size_t)L * 8, expected, (size_t)(L + 1) * 8, (size_t)L * 8, B, cudaMemcpyDeviceToDevice, c.st));
  { float* t; WALLOC(t, (size_t)(Md + 3) / 4); tp.mask = reinterpret_cast<unsigned char*>(t); }
  launch_pad_mask(tp.text, tp.mask, B, L, cf.pad_id, c.st); TKL();
  float* x0;
  WALLOC(x0, (size_t)Md * D);
  launch_dec_embed_f32(nullptr, tp.text, 0, T->P + T->emb, h->arena + h->pe1d, 0, nullptr, L, temp, x0, Md, D, c.st); TKL();
  if (const DropP d = drop_site(T, 3, 0, false, 0); d.step) { launch_dropout(x0, nullptr, x0, (long long)Md * D, d, 0, 0, c.st); TKL(); }
  tp.ds.assign(T->dec.size(), DecSave{});
  tp.xd = x0;
  for (size_t l = 0; l < T->dec.size(); ++l) {
    const TDecLayer& Wl = T->dec[l];
    DecSave& s = tp.ds[l];
    s.x_in = tp.xd;
    WALLOC(s.qkv, (size_t)Md * 3 * D); WALLOC(s.att, (size_t)Md * D); WALLOC(s.pre1, (size_t)Md * D); WALLOC(s.q2, (size_t)Md * D);
    WALLOC(s.kv, (size_t)B * S * 2 * D); WALLOC(s.catt, (size_t)Md * D); WALLOC(s.pre2, (size_t)Md * D); WALLOC(s.f0, (size_t)Md * FF);
    WALLOC(s.f1, (size_t)Md * D); WALLOC(s.pre3, (size_t)Md * D);
    if (lin_fwd(c, tp.xd, Md, D, Wl.w_sqkv, Wl.b_sqkv, true, 3 * D, s.qkv, 3 * D, ACT_NONE, nullptr)) return 1;
    {
      AttnP a{};
      a.q = s.qkv; a.ldq = 3 * D; a.kcache = s.qkv + D; a.vcache = s.qkv + 2 * D; a.rows_per_img = L; a.D = 3 * D;
      a.causal_L = L; a.key_mask = tp.mask; a.q_per_img = L; a.temperature = temp; a.out = s.att; a.ldo = D; a.M = Md; a.heads = heads;
      const DropP d = drop_site(T, 4, (int)l, false, 0);
      if (d.step) launch_dec_attn_f32_drop(a, HD, d, c.st);
      else launch_dec_attn_f32(a, HD, c.st);
      TKL();
    }
    if (attn_out_fwd(c, s.att, Md, D, Wl.w_so, Wl.b_so, tp.xd, s.pre1, &s.o1, drop_site(T, 5, (int)l, false, 0))) return 1;
    s.ln1 = LNS{s.pre1, nullptr, nullptr, Md, D, Wl.ln1_g, Wl.ln1_b};
    if (ln_fwd(c, s.ln1)) return 1;
    if (lin_fwd(c, s.ln1.y, Md, D, Wl.w_cq, Wl.b_cq, true, D, s.q2, D, ACT_NONE, nullptr)) return 1;
    if (lin_fwd(c, tp.memory, (long long)B * S, cf.dec_src, Wl.w_ckv, Wl.b_ckv, true, 2 * D, s.kv, 2 * D, ACT_NONE, nullptr)) return 1;
    {
      AttnP a{};
      a.q = s.q2; a.ldq = D; a.kcache = s.kv; a.vcache = s.kv + D; a.rows_per_img = S; a.D = 2 * D; a.n_hist = S; a.q_per_img = L;
      a.temperature = temp; a.out = s.catt; a.ldo = D; a.M = Md; a.heads = heads;
      const DropP d = drop_site(T, 6, (int)l, false, 0);
      if (d.step) launch_dec_attn_f32_drop(a, HD, d, c.st);
      else launch_dec_attn_f32(a, HD, c.st);
      TKL();
    }
    if (attn_out_fwd(c, s.catt, Md, D, Wl.w_co, Wl.b_co, s.ln1.y, s.pre2, &s.o2, drop_site(T, 7, (int)l, false, 0))) return 1;
    s.ln2 = LNS{s.pre2, nullptr, nullptr, Md, D, Wl.ln2_g, Wl.ln2_b};
    if (ln_fwd(c, s.ln2)) return 1;
    // feed-forward dropout after each ReLU, in place: f0 / f1 hold the dropped activations
    if (lin_fwd(c, s.ln2.y, Md, D, Wl.w_f0, Wl.b_f0, true, FF, s.f0, FF, ACT_RELU, nullptr)) return 1;
    if (const DropP d = drop_site(T, 8, (int)l, true, 0); d.step) { launch_dropout(s.f0, nullptr, s.f0, (long long)Md * FF, d, 0, 0, c.st); TKL(); }
    if (lin_fwd(c, s.f0, Md, FF, Wl.w_f1, Wl.b_f1, true, D, s.f1, D, ACT_RELU, nullptr)) return 1;
    if (const DropP d = drop_site(T, 9, (int)l, true, 0); d.step) { launch_dropout(s.f1, nullptr, s.f1, (long long)Md * D, d, 0, 0, c.st); TKL(); }
    launch_axpy(s.pre3, s.f1, 1.f, (long long)Md * D, 0, c.st); TKL();
    launch_axpy(s.pre3, s.ln2.y, 1.f, (long long)Md * D, 1, c.st); TKL();
    s.ln3 = LNS{s.pre3, nullptr, nullptr, Md, D, Wl.ln3_g, Wl.ln3_b};
    if (ln_fwd(c, s.ln3)) return 1;
    tp.xd = s.ln3.y;
  }
  WALLOC(tp.logits, (size_t)Md * VP); WALLOC(tp.dlogits, (size_t)Md * VP);
  if (lin_fwd(c, tp.xd, Md, D, T->gen_w, T->gen_b, true, VP, tp.logits, VP, ACT_NONE, nullptr)) return 1;
  tp.B = B; tp.L = L;
  tp.valid = true;
  if (logits_out) TCK(cudaMemcpy2DAsync(logits_out, (size_t)V * 4, tp.logits, (size_t)VP * 4, (size_t)V * 4, Md, cudaMemcpyDeviceToDevice, c.st));
  // ---- loss (:82-86; ignore_index = PAD) ----
  if (phase == PH_BOTH || loss_out) {
    // the CE kernel walks dense rows of width V: copy the V valid columns of the padded logits into a dense [Md, V]
    // buffer and its gradient back
    TCK(cudaMemsetAsync(tp.dlogits, 0, (size_t)Md * VP * 4, c.st));
    float *ld, *dd;
    WALLOC(ld, (size_t)Md * V); WALLOC(dd, (size_t)Md * V);
    TCK(cudaMemcpy2DAsync(ld, (size_t)V * 4, tp.logits, (size_t)VP * 4, (size_t)V * 4, Md, cudaMemcpyDeviceToDevice, c.st));
    launch_cross_entropy(ld, expected, dd, T->scal, B, L, V, cf.pad_id, c.st); TKL();
    TCK(cudaMemcpy2DAsync(tp.dlogits, (size_t)VP * 4, dd, (size_t)V * 4, (size_t)V * 4, Md, cudaMemcpyDeviceToDevice, c.st));
    if (loss_out) TCK(cudaMemcpyAsync(loss_out, T->scal, 4, cudaMemcpyDefault, c.st));
  }
  if (T->drop_on()) { launch_counter_add(T->drop_ctr, 1, c.st); TKL(); }   // the next forward pass draws new masks
  tp.ws_mark = T->ws_used;
  }  // forward phase
  if (phase == PH_FWD) return 0;
  if (phase == PH_BWD) {
    if (!tp.valid || tp.B != B || tp.L != L) return tfail(h, "train_backward: no forward pass of batch %d / length %d to continue from", B, L);
    T->ws_used = tp.ws_mark;
    TCK(cudaMemsetAsync(tp.dlogits, 0, (size_t)Md * VP * 4, c.st));
    TCK(cudaMemcpy2DAsync(tp.dlogits, (size_t)VP * 4, dlogits_in, (size_t)V * 4, (size_t)V * 4, Md, cudaMemcpyDeviceToDevice, c.st));
    tp.valid = false;   // the backward pass re-uses the tape's scratch space
  }
  const int S = tp.H * tp.W, Me = B * S;
  TCK(cudaMemsetAsync(T->G, 0, T->n * 4, c.st));

  // ================= backward =================
  float* dy;   // gradient flowing into the current op's output
  WALLOC(dy, (size_t)Md * D);
  if (lin_bwd(c, tp.dlogits, VP, tp.xd, Md, D, T->gen_w, T->gen_b, true, VP, dy, false)) return 1;
  float* dmem;
  WALLOC(dmem, (size_t)B * S * cf.dec_src);
  TCK(cudaMemsetAsync(dmem, 0, (size_t)B * S * cf.dec_src * 4, c.st));
  for (int l = (int)T->dec.size() - 1; l >= 0; --l) {
    const TDecLayer& Wl = T->dec[l];
    const DecSave& s = tp.ds[l];
    float *dpre3, *df1, *df0, *dw, *dpre2, *dcatt, *du, *dq2, *dkv, *dpre1, *datt, *dqkv, *dx;
    if (ln_bwd(c, s.ln3, dy, &dpre3)) return 1;
    // pre3 = f1 + w ; f1 = relu(linear1(f0)) ; f0 = relu(linear0(w))
    WALLOC(df1, (size_t)Md * D); WALLOC(df0, (size_t)Md * FF); WALLOC(dw, (size_t)Md * D);
    // relu'(pre) == (out > 0); with feed-forward dropout the stored out is the dropped activation (> 0 iff kept and
    // pre > 0), so dropout's M is in the same test and only its scale remains
    launch_act_bwd(dpre3, s.f1, df1, ACT_RELU, (long long)Md * D, c.st); TKL();
    if (T->drop_pffn > 0.f) { launch_axpy(df1, df1, 1.0f / (1.0f - T->drop_pffn), (long long)Md * D, 0, c.st); TKL(); }
    if (lin_bwd(c, df1, D, s.f0, Md, FF, Wl.w_f1, Wl.b_f1, true, D, df0, false)) return 1;
    launch_act_bwd(df0, s.f0, df0, ACT_RELU, (long long)Md * FF, c.st); TKL();
    if (T->drop_pffn > 0.f) { launch_axpy(df0, df0, 1.0f / (1.0f - T->drop_pffn), (long long)Md * FF, 0, c.st); TKL(); }
    {
      const std::string tp = "dec" + std::to_string(l) + ".";
      tap(c, tp + "d_ffn_out", dpre3, (size_t)Md * D); tap(c, tp + "d_linear1", df1, (size_t)Md * D); tap(c, tp + "d_linear0", df0, (size_t)Md * FF);
      tap(c, tp + "f0", s.f0, (size_t)Md * FF); tap(c, tp + "f1", s.f1, (size_t)Md * D);
    }
    launch_axpy(dw, dpre3, 1.f, (long long)Md * D, 0, c.st); TKL();
    if (lin_bwd(c, df0, FF, s.ln2.y, Md, D, Wl.w_f0, Wl.b_f0, true, FF, dw, true)) return 1;
    if (ln_bwd(c, s.ln2, dw, &dpre2)) return 1;
    // pre2 = out_linear(catt) + u
    WALLOC(dcatt, (size_t)Md * D); WALLOC(du, (size_t)Md * D); WALLOC(dq2, (size_t)Md * D); WALLOC(dkv, (size_t)B * S * 2 * D);
    launch_axpy(du, dpre2, 1.f, (long long)Md * D, 0, c.st); TKL();
    const float* dco;
    if (drop_bwd(c, dpre2, (long long)Md * D, drop_site(T, 7, l, false, 1), &dco)) return 1;
    if (lin_bwd(c, dco, D, s.catt, Md, D, Wl.w_co, Wl.b_co, true, D, dcatt, false)) return 1;
    {
      AttnBwdP a{};
      a.q = s.q2; a.k = s.kv; a.v = s.kv + D; a.dout = dcatt; a.dq = dq2; a.dk = dkv; a.dv = dkv + D;
      a.ldq = D; a.ldk = 2 * D; a.ldv = 2 * D; a.ldo = D; a.lddq = D; a.lddk = 2 * D; a.lddv = 2 * D;
      a.Lq = L; a.Lk = S; a.heads = heads; a.HD = HD; a.causal = 0; a.key_mask = nullptr; a.temperature = temp;
      a.drop = drop_site(T, 6, l, false, 1);
      int rc = launch_attn_bwd(a, B, c.st);
      if (rc) return tfail(h, "attention backward configuration failed (%d)", rc);
      TKL();
    }
    if (lin_bwd(c, dkv, 2 * D, tp.memory, (long long)B * S, cf.dec_src, Wl.w_ckv, Wl.b_ckv, true, 2 * D, dmem, true)) return 1;
    if (lin_bwd(c, dq2, D, s.ln1.y, Md, D, Wl.w_cq, Wl.b_cq, true, D, du, true)) return 1;
    if (ln_bwd(c, s.ln1, du, &dpre1)) return 1;
    // pre1 = out_linear(att) + x
    WALLOC(datt, (size_t)Md * D); WALLOC(dqkv, (size_t)Md * 3 * D); WALLOC(dx, (size_t)Md * D);
    launch_axpy(dx, dpre1, 1.f, (long long)Md * D, 0, c.st); TKL();
    const float* dso;
    if (drop_bwd(c, dpre1, (long long)Md * D, drop_site(T, 5, l, false, 1), &dso)) return 1;
    if (lin_bwd(c, dso, D, s.att, Md, D, Wl.w_so, Wl.b_so, true, D, datt, false)) return 1;
    {
      AttnBwdP a{};
      a.q = s.qkv; a.k = s.qkv + D; a.v = s.qkv + 2 * D; a.dout = datt; a.dq = dqkv; a.dk = dqkv + D; a.dv = dqkv + 2 * D;
      a.ldq = a.ldk = a.ldv = 3 * D; a.ldo = D; a.lddq = a.lddk = a.lddv = 3 * D;
      a.Lq = L; a.Lk = L; a.heads = heads; a.HD = HD; a.causal = 1; a.key_mask = tp.mask; a.temperature = temp;
      a.drop = drop_site(T, 4, l, false, 1);
      int rc = launch_attn_bwd(a, B, c.st);
      if (rc) return tfail(h, "attention backward configuration failed (%d)", rc);
      TKL();
    }
    if (lin_bwd(c, dqkv, 3 * D, s.x_in, Md, D, Wl.w_sqkv, Wl.b_sqkv, true, 3 * D, dx, true)) return 1;
    dy = dx;
  }
  if (const DropP d = drop_site(T, 3, 0, false, 1); d.step) { launch_dropout(dy, nullptr, dy, (long long)Md * D, d, 0, 0, c.st); TKL(); }
  launch_embed_bwd(tp.text, dy, T->G + T->emb, Md, D, temp, c.st); TKL();
  bucket_done(c, 0);
  // ---- encoder layers ----
  float* de = dmem;   // gradient of the layer output [B, S, C]
  for (int i = (int)T->enc.size() - 1; i >= 0; --i) {
    const TEncLayer& Lw = T->enc[i];
    const EncSave& s = tp.es[i];
    float *d_dw, *d_c0, *d_scr, *d_ln2, *d_pre2, *d_att, *d_qkv, *d_ln1, *d_x, *dxin;
    WALLOC(dxin, (size_t)Me * C);
    launch_axpy(dxin, de, 1.f, (long long)Me * C, 0, c.st); TKL();     // residual of conv1
    if (cb_bwd(c, s.c1, de, &d_dw, true)) return 1;
    if (dw_bwd(c, s.dw, d_dw, &d_c0)) return 1;
    if (cb_bwd(c, s.c0, d_c0, &d_scr, true)) return 1;
    WALLOC(d_ln2, (size_t)Me * C);
    launch_scramble(d_scr, d_ln2, B, S, C, 1, c.st); TKL();
    if (ln_bwd(c, s.ln2, d_ln2, &d_pre2)) return 1;
    launch_axpy(dxin, d_pre2, 1.f, (long long)Me * C, 1, c.st); TKL();  // pre2 = dropout(out_linear(att)) + x
    WALLOC(d_att, (size_t)Me * C); WALLOC(d_qkv, (size_t)Me * 3 * C); WALLOC(d_ln1, (size_t)Me * C);
    const float* d_o;
    if (drop_bwd(c, d_pre2, (long long)Me * C, drop_site(T, 2, i, false, 1), &d_o)) return 1;
    if (lin_bwd(c, d_o, C, s.att, Me, C, Lw.w_o, Lw.b_o, true, C, d_att, false)) return 1;
    {
      AttnBwdP a{};
      a.q = s.qkv; a.k = s.qkv + C; a.v = s.qkv + 2 * C; a.dout = d_att; a.dq = d_qkv; a.dk = d_qkv + C; a.dv = d_qkv + 2 * C;
      a.ldq = a.ldk = a.ldv = 3 * C; a.ldo = C; a.lddq = a.lddk = a.lddv = 3 * C;
      a.Lq = S; a.Lk = S; a.heads = cf.enc_heads; a.HD = C / cf.enc_heads; a.causal = 0; a.key_mask = nullptr; a.temperature = sqrtf((float)C);
      a.drop = drop_site(T, 1, i, false, 1);
      int rc = launch_attn_bwd(a, B, c.st);
      if (rc) return tfail(h, "attention backward configuration failed (%d)", rc);
      TKL();
    }
    if (lin_bwd(c, d_qkv, 3 * C, s.ln1.y, Me, C, Lw.w_qkv, Lw.b_qkv, true, 3 * C, d_ln1, false)) return 1;
    if (ln_bwd(c, s.ln1, d_ln1, &d_x)) return 1;
    launch_axpy(dxin, d_x, 1.f, (long long)Me * C, 1, c.st); TKL();
    de = dxin;
  }
  // ---- 2-D positional encoding ----
  float* dtrunk;   // gradient of conv_last's output
  {
    float *dg, *dgp, *dh, *dhp, *dmean;
    WALLOC(dtrunk, (size_t)Me * C); WALLOC(dg, (size_t)B * 2 * C); WALLOC(dgp, (size_t)B * 2 * C); WALLOC(dh, (size_t)B * C / 2);
    WALLOC(dhp, (size_t)B * C / 2); WALLOC(dmean, (size_t)B * C);
    if (const DropP d = drop_site(T, 0, 0, false, 1); d.step) {   // the PE output's dropout, NCHW mask
      float* dm;
      WALLOC(dm, (size_t)Me * C);
      launch_dropout(de, nullptr, dm, (long long)Me * C, d, S, C, c.st); TKL();
      de = dm;
    }
    launch_axpy(dtrunk, de, 1.f, (long long)Me * C, 0, c.st); TKL();
    launch_pe2d_bwd_gate(de, peh, pew, dg, B, tp.H, tp.W, C, c.st); TKL();
    launch_act_bwd(dg, tp.pe_gp, dgp, ACT_SIGMOID, (long long)B * 2 * C, c.st); TKL();
    if (lin_bwd(c, dgp, 2 * C, tp.pe_h, B, C / 2, T->pe_w1, T->pe_b1, true, 2 * C, dh, false)) return 1;
    launch_act_bwd(dh, tp.pe_hp, dhp, ACT_RELU, (long long)B * C / 2, c.st); TKL();
    if (lin_bwd(c, dhp, C / 2, tp.pe_mean, B, C, T->pe_w0, T->pe_b0, true, C / 2, dmean, false)) return 1;
    launch_spatial_add(dtrunk, dmean, B, S, C, 1.f / (float)S, c.st); TKL();
  }
  if (T->lite) {
    bucket_done(c, 1);
    const int C0 = C / 2;
    float* d = dtrunk;   // gradient of pool[3]
    for (int i = 3; i >= 1; --i) {
      const CB& r = tp.lite_cb[i - 1];
      float* dyc;
      WALLOC(dyc, (size_t)B * r.OH * r.OW * C);
      launch_maxpool2_bwd(r.y, d, dyc, B, r.OH, r.OW, C, c.st); TKL();
      if (cb_bwd(c, r, dyc, &d, true)) return 1;
    }
    const long long M0 = (long long)B * cf.height * cf.width;
    float *dy0, *dz0;
    WALLOC(dy0, (size_t)M0 * C0); WALLOC(dz0, (size_t)M0 * C0);
    launch_maxpool2_bwd(tp.lite_y0, d, dy0, B, cf.height, cf.width, C0, c.st); TKL();
    launch_bn_bwd(dy0, tp.lite_z0, tp.lite_stat0, T->acc, dz0, T->G + T->lite_bn[0].g, T->G + T->lite_bn[0].b, (int)M0, C0, ACT_RELU, c.st); TKL();
    if (launch_image_conv_wgrad(dz0, images, T->G + T->lite_w[0], B, cf.in_ch, cf.height, cf.width, cf.height, cf.width, C0, 1, 1, c.st))
      return tfail(h, "training: conv0 weight gradient does not support %d output channels", C0);
    TKL();
    bucket_done(c, 5);
    return 0;
  }
  float* dx;
  if (cb_bwd(c, tp.last, dtrunk, &dx, true)) return 1;
  bucket_done(c, 1);
  // ---- trunk blocks ----
  int stage_of_block = 5, left_in_stage = kArch[5][1];
  for (int i = (int)T->blocks.size() - 1; i >= 0; --i) {
    const TBlock& b = T->blocks[i];
    const BlockSave& s = tp.bs[i];
    float* dmain = nullptr;
    const long long n_in = (long long)B * s.c1.H * s.c1.W * b.cin;
    if (b.kind == 0) {
      if (cb_bwd(c, s.c1, dx, &dmain, true)) return 1;
    } else if (b.kind == 1) {
      float* d1;
      if (cb_bwd(c, s.c2, dx, &d1, true)) return 1;
      if (cb_bwd(c, s.c1, d1, &dmain, true)) return 1;
    } else {
      float *d3, *d2, *d1;
      if (cb_bwd(c, s.c2, dx, &d3, true)) return 1;
      if (se_bwd(c, s.se, b, d3, &d2)) return 1;
      if (dw_bwd(c, s.dw, d2, &d1)) return 1;
      if (cb_bwd(c, s.c1, d1, &dmain, true)) return 1;
    }
    if (b.residual) { launch_axpy(dmain, dx, 1.f, n_in, 1, c.st); TKL(); }
    dx = dmain;
    if (--left_in_stage == 0) {
      if (stage_of_block >= 3) bucket_done(c, 2 + (5 - stage_of_block));
      --stage_of_block;
      if (stage_of_block >= 0) left_in_stage = kArch[stage_of_block][1];
    }
  }
  // ---- stem ----
  {
    float* dz;
    WALLOC(dz, (size_t)B * H0 * W0 * 24);
    launch_bn_bwd(dx, tp.stem_z, tp.stem_stat, T->acc, dz, T->G + T->stem_bn.g, T->G + T->stem_bn.b, B * H0 * W0, 24, ACT_SILU, c.st); TKL();
    launch_stem_wgrad(dz, images, T->G + T->stem_w, B, cf.in_ch, cf.height, cf.width, H0, W0, 24, c.st); TKL();
  }
  bucket_done(c, 5);
  return 0;
}

TrainState* state_of(frx_handle* h) { return reinterpret_cast<TrainState*>(h->train); }

// before a forward pass: the device step counter only moves in passes with dropout, so passes without it are counted on
// the host and added before the next pass with it
int drop_count_pass(frx_handle* h, TrainState* T, cudaStream_t st) {
  if (!T->drop_on()) { ++T->drop_pending; return 0; }
  if (T->drop_pending) { launch_counter_add(T->drop_ctr, T->drop_pending, st); TKL(); T->drop_pending = 0; }
  return 0;
}

}  // namespace

// =====================================================================================================================
// C ABI
// =====================================================================================================================
extern "C" int frx_train_create(frx_handle* h, int32_t max_batch, int32_t max_len, float* grad_buffer) {
  if (!h) return 1;
  if (!h->finalized) return tfail(h, "train_create: weights not finalized");
  if (h->cfg.network != FRX_NET_EFFICIENT_SATRN && h->cfg.network != FRX_NET_LITE_SATRN)
    return tfail(h, "train_create: EfficientSATRN and LiteSATRN have a training step (SwinTRN has not)");
  if (max_batch <= 0 || max_len <= 0 || max_len > 256) return tfail(h, "train_create: max_batch / max_len out of range (max_len <= 256)");
  DevGuard g; g.enter(h->cfg.device);
  if (h->train) frx_train_destroy(h);
  TrainState* T = new TrainState();
  h->train = T;
  T->max_B = max_batch; T->max_L = max_len;
  if (build_network(h, T)) return 1;
  TCK(cudaMalloc(&T->P, T->n * 4)); TCK(cudaMalloc(&T->M, T->n * 4)); TCK(cudaMalloc(&T->V, T->n * 4));
  if (grad_buffer) { T->G = grad_buffer; T->own_G = false; }   // caller-owned (a torch tensor the host all-reduces with NCCL)
  else TCK(cudaMalloc(&T->G, T->n * 4));
  TCK(cudaMalloc(&T->RS, (T->n_rs + 4) * 4));
  TCK(cudaMemcpy(T->P, T->hostP.data(), T->n * 4, cudaMemcpyHostToDevice));
  TCK(cudaMemcpy(T->RS, T->hostRS.data(), T->n_rs * 4, cudaMemcpyHostToDevice));
  TCK(cudaMemset(T->M, 0, T->n * 4)); TCK(cudaMemset(T->V, 0, T->n * 4)); TCK(cudaMemset(T->G, 0, T->n * 4));
  TCK(cudaMalloc(&T->acc, 2 * 4096 * sizeof(double))); TCK(cudaMalloc(&T->sumsq, 2 * sizeof(double)));
  TCK(cudaMalloc(&T->scal, 64)); TCK(cudaMalloc(&T->ones, 4096 * 4)); TCK(cudaMalloc(&T->zeros, 4096 * 4));
  TCK(cudaMemset(T->zeros, 0, 4096 * 4));
  TCK(cudaMalloc(&T->splitk_ws, kSplitKFloats * 4));
  TCK(cudaMalloc(&T->drop_ctr, sizeof(uint32_t))); TCK(cudaMemset(T->drop_ctr, 0, sizeof(uint32_t)));
  launch_fill(T->ones, 1.f, 4096, 0);
  TCK(cudaDeviceSynchronize());
  // activation tape: ~75 MB (forward) + ~150 MB (backward) of fp32 per image at 128 x 256, plus the decoder's
  // M = B * L rows (~60 KB per row) and a fixed part for repacked weights
  const double per_img = 230e6 * ((double)h->cfg.height * h->cfg.width / (128.0 * 256.0)) + (double)max_len * 80e3;
  T->ws_bytes = (size_t)(per_img * max_batch + 256e6);
  TCK(cudaMalloc(&T->ws, T->ws_bytes));
  TCK(cudaMalloc(&T->img_stage, (size_t)max_batch * h->cfg.in_ch * h->cfg.height * h->cfg.width * 4));
  TCK(cudaMalloc(&T->exp_stage, (size_t)max_batch * (max_len + 1) * 8));
  std::vector<float>().swap(T->hostP);
  return 0;
}

extern "C" int64_t frx_train_param_count(frx_handle* h) {
  if (!h || !h->finalized) return -1;
  if (h->train) return (int64_t)state_of(h)->n;
  TrainState tmp;
  if (build_network(h, &tmp)) return -1;
  return (int64_t)tmp.n;
}

extern "C" void frx_train_destroy(frx_handle* h) {
  if (!h || !h->train) return;
  DevGuard g; g.enter(h->cfg.device);
  TrainState* T = state_of(h);
  cudaFree(T->P); if (T->own_G) cudaFree(T->G); cudaFree(T->M); cudaFree(T->V); cudaFree(T->RS); cudaFree(T->acc); cudaFree(T->sumsq);
  cudaFree(T->scal); cudaFree(T->ones); cudaFree(T->zeros); cudaFree(T->splitk_ws); cudaFree(T->ws); cudaFree(T->img_stage); cudaFree(T->exp_stage);
  cudaFree(T->drop_ctr);
  for (auto& kv : T->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  delete T;
  h->train = nullptr;
}

extern "C" int frx_train_fwd_bwd(frx_handle* h, const float* images, const int64_t* expected, int32_t B, int32_t len_plus_1,
                                 float* loss_out, void* stream) {
  if (!h) return 1;
  TrainState* T = state_of(h);
  if (!T) return tfail(h, "train_fwd_bwd: call frx_train_create first");
  const int L = len_plus_1 - 1;
  if (B <= 0 || B > T->max_B || L <= 0 || L > T->max_L) return tfail(h, "train_fwd_bwd: batch %d / length %d outside (%d, %d)", B, L, T->max_B, T->max_L);
  DevGuard g; g.enter(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  if (drop_count_pass(h, T, st)) return 1;
  // Eager when graphs are off, when a bucket callback wants to start all-reduces between the kernels of the pass, and on
  // the first use of a shape (which also performs the one-time per-device kernel attribute set-up).
  // the launch plan and whether dropout runs are part of the key
  TrainState::GraphEntry& ge = T->graphs[{B, 4 * L + (T->drop_on() ? 2 : 0) + (h->opt_train_splitk ? 1 : 0)}];
  if (!h->opt_graphs || T->bucket_cb || ge.seen++ == 0) {
    Ctx c{h, T, st, B, L};
    return fwd_bwd(c, images, (const long long*)expected, loss_out);
  }
  const size_t img_floats = (size_t)B * h->cfg.in_ch * h->cfg.height * h->cfg.width;
  TCK(cudaMemcpyAsync(T->img_stage, images, img_floats * 4, cudaMemcpyDeviceToDevice, st));
  TCK(cudaMemcpyAsync(T->exp_stage, expected, (size_t)B * len_plus_1 * 8, cudaMemcpyDeviceToDevice, st));
  if (!ge.exec) {
    cudaStream_t cs;
    TCK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    const long long before = h->launches;
    TCK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    Ctx c{h, T, cs, B, L};
    const int rc = fwd_bwd(c, T->img_stage, T->exp_stage, nullptr);
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(cs, &graph);
    cudaStreamDestroy(cs);
    if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
    if (e != cudaSuccess) return tfail(h, "training graph capture failed: %s", cudaGetErrorString(e));
    ge.nodes = h->launches - before;
    h->launches = before;
    const cudaError_t e2 = cudaGraphInstantiate(&ge.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e2 != cudaSuccess) { ge.exec = nullptr; return tfail(h, "training graph instantiate failed: %s", cudaGetErrorString(e2)); }
    // keep at most 4 shapes (variable target lengths would otherwise accumulate ~13 000-node graphs)
    while (T->graphs.size() > 4) {
      auto victim = T->graphs.end();
      for (auto it = T->graphs.begin(); it != T->graphs.end(); ++it)
        if (&it->second != &ge && (victim == T->graphs.end() || it->second.last_use < victim->second.last_use)) victim = it;
      if (victim == T->graphs.end()) break;
      TCK(cudaStreamSynchronize(st));
      if (victim->second.exec) cudaGraphExecDestroy(victim->second.exec);
      T->graphs.erase(victim);
    }
  }
  ge.last_use = ++T->graph_clock;
  TCK(cudaGraphLaunch(ge.exec, st));
  h->launches += ge.nodes;
  if (loss_out) TCK(cudaMemcpyAsync(loss_out, T->scal, 4, cudaMemcpyDefault, st));
  return 0;
}

extern "C" int frx_train_forward(frx_handle* h, const float* images, const int64_t* expected, int32_t B, int32_t len_plus_1,
                                 float* logits_out, float* loss_out, void* stream) {
  if (!h) return 1;
  TrainState* T = state_of(h);
  if (!T) return tfail(h, "train_forward: call frx_train_create first");
  const int L = len_plus_1 - 1;
  if (B <= 0 || B > T->max_B || L <= 0 || L > T->max_L) return tfail(h, "train_forward: batch %d / length %d outside (%d, %d)", B, L, T->max_B, T->max_L);
  DevGuard g; g.enter(h->cfg.device);
  if (drop_count_pass(h, T, (cudaStream_t)stream)) return 1;
  Ctx c{h, T, (cudaStream_t)stream, B, L};
  return fwd_bwd(c, images, (const long long*)expected, loss_out, PH_FWD, logits_out, nullptr);
}

extern "C" int frx_train_backward(frx_handle* h, const float* images, const float* dlogits, int32_t B, int32_t len_plus_1, void* stream) {
  if (!h) return 1;
  TrainState* T = state_of(h);
  if (!T) return tfail(h, "train_backward: call frx_train_create first");
  if (!dlogits || !images) return tfail(h, "train_backward: null argument");
  DevGuard g; g.enter(h->cfg.device);
  Ctx c{h, T, (cudaStream_t)stream, B, len_plus_1 - 1};
  return fwd_bwd(c, images, nullptr, nullptr, PH_BWD, nullptr, dlogits);
}

extern "C" int frx_train_set_dropout(frx_handle* h, float p, float p_ffn, uint64_t seed, int32_t rank) {
  if (!h) return 1;
  TrainState* T = state_of(h);
  if (!T) return tfail(h, "train_set_dropout: call frx_train_create first");
  if (!(p >= 0.f && p < 1.f) || !(p_ffn >= 0.f && p_ffn < 1.f))
    return tfail(h, "train_set_dropout: rates must lie in [0, 1) (p = %g, p_ffn = %g)", (double)p, (double)p_ffn);
  if (rank < 0) return tfail(h, "train_set_dropout: rank %d < 0", (int)rank);
  if (p == T->drop_p && p_ffn == T->drop_pffn && seed == T->drop_seed && rank == T->drop_rank) return 0;
  DevGuard g; g.enter(h->cfg.device);
  // graphs captured with dropout carry the rates and the key as kernel arguments: they go when another setting with
  // dropout takes over (switching dropout off and on again keeps them)
  const bool on = p > 0.f || p_ffn > 0.f;
  if (on && (p != T->graph_p || p_ffn != T->graph_pffn || seed != T->graph_seed || rank != T->graph_rank)) {
    TCK(cudaDeviceSynchronize());
    for (auto it = T->graphs.begin(); it != T->graphs.end();) {
      if (it->first.second & 2) {
        if (it->second.exec) cudaGraphExecDestroy(it->second.exec);
        it = T->graphs.erase(it);
      } else {
        ++it;
      }
    }
    T->graph_p = p; T->graph_pffn = p_ffn; T->graph_seed = seed; T->graph_rank = rank;
  }
  T->drop_p = p; T->drop_pffn = p_ffn; T->drop_seed = seed; T->drop_rank = rank;
  T->tape.valid = false;   // a frx_train_backward continues a forward pass of the same setting only
  return 0;
}

extern "C" int frx_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  if (!ctr || !key || !out) return 1;
  uint4 io[2] = {make_uint4(ctr[0], ctr[1], ctr[2], ctr[3]), make_uint4(key[0], key[1], 0, 0)};
  uint4* d = nullptr;
  if (cudaMalloc(&d, sizeof io) != cudaSuccess) return 1;
  bool ok = cudaMemcpy(d, io, sizeof io, cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok) { launch_philox_probe(d, 0); ok = cudaGetLastError() == cudaSuccess; }
  ok = ok && cudaMemcpy(io, d, sizeof io, cudaMemcpyDeviceToHost) == cudaSuccess;
  cudaFree(d);
  if (!ok) return 1;
  out[0] = io[0].x; out[1] = io[0].y; out[2] = io[0].z; out[3] = io[0].w;
  return 0;
}

extern "C" int frx_train_grad_buffer(frx_handle* h, float** grads, int64_t* count) {
  if (!h || !state_of(h)) return tfail(h, "train_grad_buffer: call frx_train_create first");
  if (grads) *grads = state_of(h)->G;
  if (count) *count = (int64_t)state_of(h)->n;
  return 0;
}

extern "C" int frx_train_set_bucket_callback(frx_handle* h, void (*cb)(void*, int64_t, int64_t), void* ctx) {
  if (!h || !state_of(h)) return tfail(h, "train_set_bucket_callback: call frx_train_create first");
  state_of(h)->bucket_cb = cb;
  state_of(h)->bucket_ctx = ctx;
  return 0;
}

// clip + AdamW over one contiguous range of the flat buffers (the whole model, or the encoder / decoder parameter group
// of the dual-optimizer loop, train_modules/train_dual_opt.py:95-112: separate clip_grad_norm_ and optimizers)
static int apply_range(frx_handle* h, TrainState* T, size_t off, size_t count, float lr, float weight_decay, float max_grad_norm,
                       float grad_scale, float* grad_norm_out, int slot, cudaStream_t st) {
  launch_sumsq(T->G + off, (long long)count, T->sumsq + slot, st); TKL();
  launch_adamw(T->P + off, T->G + off, T->M + off, T->V + off, T->sumsq + slot, T->scal + 4 + slot, (long long)count, lr, weight_decay, T->step,
               max_grad_norm, grad_scale, st);
  TKL();
  if (grad_norm_out) TCK(cudaMemcpyAsync(grad_norm_out, T->scal + 4 + slot, 4, cudaMemcpyDefault, st));
  return 0;
}

extern "C" int frx_train_apply(frx_handle* h, float lr, float weight_decay, float max_grad_norm, float grad_scale, float* grad_norm_out,
                               void* stream) {
  if (!h) return 1;
  TrainState* T = state_of(h);
  if (!T) return tfail(h, "train_apply: call frx_train_create first");
  DevGuard g; g.enter(h->cfg.device);
  T->step += 1;
  return apply_range(h, T, 0, T->n, lr, weight_decay, max_grad_norm, grad_scale, grad_norm_out, 0, (cudaStream_t)stream);
}

extern "C" int frx_train_apply_dual(frx_handle* h, float enc_lr, float dec_lr, float weight_decay, float max_grad_norm, float grad_scale,
                                    float* enc_grad_norm_out, float* dec_grad_norm_out, void* stream) {
  if (!h) return 1;
  TrainState* T = state_of(h);
  if (!T) return tfail(h, "train_apply_dual: call frx_train_create first");
  DevGuard g; g.enter(h->cfg.device);
  T->step += 1;
  const size_t enc_end = T->mark_trunk[6];   // parameters are laid out encoder first (model.encoder.parameters()), decoder after
  if (apply_range(h, T, 0, enc_end, enc_lr, weight_decay, max_grad_norm, grad_scale, enc_grad_norm_out, 0, (cudaStream_t)stream)) return 1;
  return apply_range(h, T, enc_end, T->n - enc_end, dec_lr, weight_decay, max_grad_norm, grad_scale, dec_grad_norm_out, 1, (cudaStream_t)stream);
}

static int unpack_to(frx_handle* h, TrainState* T, const float* flat_dev, const char* name, float* dst) {
  for (const TParam& p : T->params) {
    if (p.name != name) continue;
    std::vector<float> packed(p.n), out;
    TCK(cudaMemcpy(packed.data(), flat_dev + p.off, p.n * 4, cudaMemcpyDeviceToHost));
    size_t n = 1;
    for (int i = 0; i < 4; ++i) n *= (size_t)p.d[i];
    out.resize(n);
    if (p.kind == P_CONV) {
      const int O = p.d[0], I = p.d[1], kk = p.d[2] * p.d[3];
      for (int o = 0; o < O; ++o)
        for (int i = 0; i < I; ++i)
          for (int t = 0; t < kk; ++t) out[((size_t)o * I + i) * kk + t] = packed[((size_t)o * kk + t) * I + i];
    } else if (p.kind == P_DW) {
      const int C = p.d[0];
      for (int cc = 0; cc < C; ++cc)
        for (int t = 0; t < 9; ++t) out[(size_t)cc * 9 + t] = packed[(size_t)t * C + cc];
    } else {
      memcpy(out.data(), packed.data(), n * 4);
    }
    TCK(cudaMemcpy(dst, out.data(), n * 4, cudaMemcpyDefault));
    return 0;
  }
  // BatchNorm running statistics
  std::string nm(name);
  const size_t dot = nm.rfind('.');
  if (dot != std::string::npos) {
    auto it = T->rs_off.find(nm.substr(0, dot));
    if (it != T->rs_off.end() && flat_dev == T->P) {
      const int C = T->rs_C[it->first];
      const std::string leaf = nm.substr(dot + 1);
      if (leaf == "running_mean" || leaf == "running_var") {
        TCK(cudaMemcpy(dst, T->RS + it->second + (leaf == "running_var" ? C : 0), (size_t)C * 4, cudaMemcpyDefault));
        return 0;
      }
    }
  }
  return tfail(h, "training: no parameter named '%s'", name);
}

// inverse of unpack_to for parameters: state_dict layout (host or device pointer) -> the flat parameter buffer
extern "C" int frx_train_import(frx_handle* h, const char* name, const float* src) {
  if (!h || !state_of(h) || !name || !src) return tfail(h, "train_import: bad arguments");
  DevGuard g; g.enter(h->cfg.device);
  TrainState* T = state_of(h);
  for (const TParam& p : T->params) {
    if (p.name != name) continue;
    size_t n = 1;
    for (int i = 0; i < 4; ++i) n *= (size_t)p.d[i];
    std::vector<float> in(n), packed(p.n, 0.f);
    TCK(cudaMemcpy(in.data(), src, n * 4, cudaMemcpyDefault));
    if (p.kind == P_CONV) {
      const int O = p.d[0], I = p.d[1], kk = p.d[2] * p.d[3];
      for (int o = 0; o < O; ++o)
        for (int i = 0; i < I; ++i)
          for (int t = 0; t < kk; ++t) packed[((size_t)o * kk + t) * I + i] = in[((size_t)o * I + i) * kk + t];
    } else if (p.kind == P_DW) {
      const int C = p.d[0];
      for (int cc = 0; cc < C; ++cc)
        for (int t = 0; t < 9; ++t) packed[(size_t)t * C + cc] = in[(size_t)cc * 9 + t];
    } else {
      memcpy(packed.data(), in.data(), n * 4);
    }
    TCK(cudaMemcpy(T->P + p.off, packed.data(), p.n * 4, cudaMemcpyHostToDevice));
    return 0;
  }
  return tfail(h, "training: no parameter named '%s'", name);
}

extern "C" int frx_train_export(frx_handle* h, const char* name, float* dst) {
  if (!h || !state_of(h) || !name || !dst) return tfail(h, "train_export: bad arguments");
  DevGuard g; g.enter(h->cfg.device);
  return unpack_to(h, state_of(h), state_of(h)->P, name, dst);
}

extern "C" int frx_train_read_grad(frx_handle* h, const char* name, float* dst) {
  if (!h || !state_of(h) || !name || !dst) return tfail(h, "train_read_grad: bad arguments");
  DevGuard g; g.enter(h->cfg.device);
  return unpack_to(h, state_of(h), state_of(h)->G, name, dst);
}

extern "C" int64_t frx_train_read_tap(frx_handle* h, const char* name, float* dst, int64_t capacity) {
  if (!h || !state_of(h) || !name) return -1;
  DevGuard g; g.enter(h->cfg.device);
  TrainState* T = state_of(h);
  auto it = T->taps.find(name);
  if (it == T->taps.end()) { tfail(h, "train_read_tap: no tap named '%s'", name); return -1; }
  const int64_t n = (int64_t)it->second.second;
  if (dst) {
    if (capacity < n) { tfail(h, "train_read_tap: '%s' holds %lld floats, capacity %lld", name, (long long)n, (long long)capacity); return -1; }
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpy(dst, it->second.first, (size_t)n * 4, cudaMemcpyDefault) != cudaSuccess) {
      tfail(h, "train_read_tap: copy failed");
      return -1;
    }
  }
  return n;
}

extern "C" int64_t frx_train_step_count(const frx_handle* h) { return h && h->train ? reinterpret_cast<const TrainState*>(h->train)->step : 0; }
